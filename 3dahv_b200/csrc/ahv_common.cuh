// Shared constants and small device helpers for lib3dahv_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ahv_b200.h"

namespace ahv {

constexpr int kC = 16;      // volume channels            modules/modules.py:64
constexpr int kS = 8;       // D = H = W                  modules/modules.py:97-100
constexpr int kVox = 512;   // voxel samples per hypothesis
constexpr int kK = 384;     // tri-plane channels          modules/modules.py:67
constexpr int kO = 32;      // head output channels        modules/model.py:34
constexpr int kP = 64;      // positions of the folded 8x8 plane
constexpr int kMaxK = 32;   // largest supported top-k

// Source volume staged in shared memory with a one-voxel zero halo, channel
// innermost: line L = ((z+1)*10 + (y+1))*10 + (x+1), 16 fp32 (64 B) per line.
// Out-of-range taps of padding_mode='zeros' (utils.py:129) then read zeros and
// need no per-tap bounds test.
constexpr int kHalo = 10;
constexpr int kLines = kHalo * kHalo * kHalo;  // 1000
constexpr int kVolSmemBytes = kLines * kC * 4; // 64000

#define AHV_CUDA_OK(expr)                          \
  do {                                             \
    cudaError_t _e = (expr);                       \
    if (_e != cudaSuccess) return AHV_ECUDA;       \
  } while (0)

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Largest L1 norm of a row of W ([32 rows][kCols], fp32), by `kWarps` warps: warp w sums rows w, w + kWarps, ...  Each
// row's sum has one fixed order (lane partial sums, then the butterfly) whatever kWarps is, so every CTA of the tensor-core
// scoring kernel and of the tcgen05 backward derives the same value.
template <int kCols, int kWarps>
__device__ __forceinline__ float row_l1max(const float* __restrict__ W, int warp, int lane) {
  constexpr int kRowsPerWarp = (kO + kWarps - 1) / kWarps;
  float m = 0.0f;
#pragma unroll
  for (int i = 0; i < kRowsPerWarp; ++i) {
    const int r = warp + i * kWarps;
    if (r < kO) {
      float l1 = 0.0f;
#pragma unroll
      for (int j = 0; j < kCols / 32; ++j) l1 += fabsf(__ldg(W + r * kCols + lane + 32 * j));
      m = fmaxf(m, warp_sum(l1));
    }
  }
  return m;  // this warp's largest row norm (identical in all lanes)
}

// Power-of-two normalisation of a weight matrix: e = floor(log2 of its largest row L1 norm) - `target`, so that W * 2^-e
// has that norm in [2^target, 2^(target+1)) whatever the weights' magnitude.  0 when the weights are all zero or not
// finite.
__device__ __forceinline__ int weight_exponent(float l1max, int target) {
  return (l1max > 0.0f && isfinite(l1max)) ? max(-60, min(60, ilogbf(l1max) - target)) : 0;
}
// W1's normalised row norms land in [4, 8), which keeps the tensor-core scorer's pair-scaled volume in (2^11, 2^13]
// (stage_pair_volume); W2's land in [1, 2) (conv2 accumulates in fp32; only its fp16 operand needs the range).
constexpr int kW1NormTarget = 2, kW2NormTarget = 0;

// Sample position of output voxel (x,y,z base coordinates) under rotation R
// (F.affine_grid, utils.py:126), un-normalised as grid_sample does with
// align_corners=False: i = ((g+1)*8-1)/2.  ((g+1)*8 is exact, so one FFMA
// (g+1)*4-0.5 reproduces ATen's two-step rounding bit for bit.)
struct Tap {
  int line;          // halo line index of the (x0,y0,z0) corner
  float fx, fy, fz;  // fractional parts
};

__device__ __forceinline__ float unnorm(float g) { return fmaf(__fadd_rn(g, 1.0f), 4.0f, -0.5f); }

// Un-normalised, unclamped sample position (ix, iy, iz) of base point (x, y, z): grid = R @ (x, y, z);
// x -> W, y -> H, z -> D
__device__ __forceinline__ float3 sample_coords(const float* R, float x, float y, float z) {
  const float gx = fmaf(R[2], z, fmaf(R[1], y, R[0] * x));
  const float gy = fmaf(R[5], z, fmaf(R[4], y, R[3] * x));
  const float gz = fmaf(R[8], z, fmaf(R[7], y, R[6] * x));
  return make_float3(unnorm(gx), unnorm(gy), unnorm(gz));
}

__device__ __forceinline__ Tap tap_at(float3 u) {
  // clamp to [-1, 8]: anything outside only ever touches the zero halo
  float ix = fminf(fmaxf(u.x, -1.0f), 8.0f);
  float iy = fminf(fmaxf(u.y, -1.0f), 8.0f);
  float iz = fminf(fmaxf(u.z, -1.0f), 8.0f);
  float x0 = fminf(floorf(ix), 7.0f), y0 = fminf(floorf(iy), 7.0f), z0 = fminf(floorf(iz), 7.0f);
  Tap t;
  t.fx = ix - x0;
  t.fy = iy - y0;
  t.fz = iz - z0;
  t.line = (((int)z0 + 1) * kHalo + ((int)y0 + 1)) * kHalo + ((int)x0 + 1);
  return t;
}

__device__ __forceinline__ Tap make_tap(const float* R, float x, float y, float z) {
  return tap_at(sample_coords(R, x, y, z));
}

// (score, index) -> one ordered 64-bit key: larger key = higher score, ties -> lower index
typedef unsigned long long u64;

__device__ __forceinline__ u64 make_key(float score, uint32_t idx) {
  uint32_t u = __float_as_uint(score + 0.0f);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((u64)u << 32) | (u64)(0xFFFFFFFFu - idx);
}
__device__ __forceinline__ float key_score(u64 key) {
  uint32_t u = (uint32_t)(key >> 32);
  u = (u & 0x80000000u) ? (u ^ 0x80000000u) : ~u;
  return __uint_as_float(u);
}
__device__ __forceinline__ uint32_t key_index(u64 key) { return 0xFFFFFFFFu - (uint32_t)key; }

// SM count of the current device, 0 when it cannot be read
inline int sm_count() {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  return sms;
}

namespace peer { struct Args; }  // ahv_peer.cuh

// Launch-side helpers implemented in the .cu files --------------------------
int launch_so3_from_normals(const float* normals, float* R, int64_t n, cudaStream_t s);
int launch_so3_sample(uint64_t seed, int64_t first, float* R, int64_t n, cudaStream_t s);
int launch_so3_grid(int64_t n_total, int64_t first, float* R, int64_t count, cudaStream_t s);
// The nested Hopf x HEALPix grid (ahv_so3.cu): 72 * 8^level cells at level 0..kHopfMaxLevel.
constexpr int kHopfMaxLevel = 16;
__host__ __device__ constexpr int64_t hopf_cells(int level) { return (int64_t)72 << (3 * level); }
int launch_so3_hopf_grid(int level, int64_t first, float* R, int64_t count, cudaStream_t s);
int launch_so3_hopf_children(int level, const int64_t* parent, int64_t n, int64_t* child, float* R, cudaStream_t s);
// Per pair, the k cells out[b,j] = cand[b, pick[b,j]] (cand NULL: pick[b,j] itself; -1 for a pick outside [0,n)), in
// pick's order or, with `sort`, in ascending index order.  k <= 32.
int launch_hopf_pick(const int64_t* cand, int64_t n, const int64_t* pick, int B, int k, bool sort, int64_t* out,
                     cudaStream_t s);
int launch_so3_perturb(const float* centers, int64_t n, int m, float max_angle_deg, uint64_t seed, float* out,
                       cudaStream_t s);
int launch_rotate_volume(const float* vol, int per_rot, const float* R, const float* base,
                         float* out, int64_t n, cudaStream_t s);
int launch_rotate_volume_bwd(const float* grad_out, int per_rot, const float* R, const float* base,
                             float* grad_vol, int64_t n, cudaStream_t s);
int launch_rotate_volume_grad_R(const float* vol, int per_rot, const float* R, const float* base, const float* grad_out,
                                float* grad_R, int64_t n, cudaStream_t s);
// The fused backward kernels (ahv_score_bwd.cu, ahv_score_bwd_tc.cu) on `grid` CTAs, 0: one per SM (at most one per
// item).  det: the deterministic instance, whose outputs are the workspace slots below (launch_score_bwd_det).
int launch_score_bwd(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                     const float* W1, const float* W2, const float* b2, const float* base,
                     const float* grad_scores, float* g_vol, float* g_tgt, float* g_W1, float* g_W2,
                     float* g_b2, int B, int64_t N, cudaStream_t s, const void* h1_saved = nullptr,
                     const float* pair_inv = nullptr, float* g_R = nullptr, unsigned grid = 0, bool det = false);
int launch_score_bwd_tc(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                        const float* W1, const float* W2, const float* b2, const float* base,
                        const float* grad_scores, const void* h1_saved, const float* pair_inv, float* g_vol,
                        float* g_tgt, float* g_W1, float* g_W2, float* g_b2, int B, int64_t N, cudaStream_t s,
                        unsigned grid = 0, bool det = false);
// Deterministic backward (ahv_score_backward_det).  The kernels store what the atomic instances add into global memory
// in per-CTA workspace slots, and score_bwd_det_reduce adds the slots of every output element in increasing slot order.
//   weight slot c (one per CTA, c < grid):   dW1 [32][384] | dW2 [32][32] | db2 [32]              kDetWSlot floats
//   segment slot c + b (CTA c, pair b):     dV_b [16][512] | dT_b [32][64]                         kDetSegSlot floats
// CTA c's items are contiguous, so c + b strictly increases over its segments: grid + B - 1 segment slots.
// grid = min(B*N, SMs, kDetGridCap): the bits depend on the inputs and on min(SMs, kDetGridCap) alone, and the
// workspace size on (B, N) alone.
constexpr int kDetGridCap = 160;
constexpr int kDetWSlot = kO * kK + kO * kO + kO;
constexpr int kDetSegSlot = kC * kVox + kO * kP;
struct DetBwdWs {   // offsets into the workspace in floats (each region 128-byte aligned); total * 4 bytes in all
  int grid_max;
  size_t seg, rot, total;   // rot: grad_R of every item [B*N][9] for a shared R (its sum over pairs)
  DetBwdWs(int B, int64_t N, bool shared_grad_R)
      : grid_max((int)((int64_t)B * N < kDetGridCap ? (int64_t)B * N : kDetGridCap)),
        seg((size_t)grid_max * kDetWSlot),
        rot(seg + (B > 0 && grid_max > 0 ? (size_t)(grid_max + B - 1) * kDetSegSlot : 0)),
        total(rot + (shared_grad_R ? ((size_t)B * (size_t)N * 9 + 63) / 64 * 64 : 0)) {}
};
int launch_score_bwd_det(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                         const float* W1, const float* W2, const float* b2, const float* base, const float* grad_scores,
                         const void* h1_saved, const float* pair_inv, float* g_vol, float* g_tgt, float* g_W1,
                         float* g_W2, float* g_b2, float* g_R, int B, int64_t N, bool tc, float* ws, cudaStream_t s);
int launch_score_tc_train(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair, const float* W1,
                          const float* W2, const float* b2, const float* base, float* scores, void* h1_out,
                          float* pair_inv_out, int B, int64_t N, void* ws, size_t ws_bytes, cudaStream_t s);
int launch_resblock3d(const float* x, const float* Wc1, const float* Wc2, const float* Wd, float* out, int64_t m,
                      cudaStream_t s);
int launch_infonce(const float* scores, const float* R, int r_per_pair, const float* gt, float thr_deg, float temperature,
                   float* loss, float* grad, int B, int64_t N, cudaStream_t s);
int launch_gradient_ascent(const void* vol_src, int vol_dtype, const float* tgt_feat, const float* R_init, const float* W1,
                           const float* W2, const float* b2, const float* base, int steps, float step_deg, float* R_out,
                           float* score_out, int B, int K, cudaStream_t s, const int64_t* skip_idx = nullptr,
                           int64_t item_lo = 0, int64_t item_hi = -1);  // item_hi < 0: every item of B*K
int launch_forward_3d2d(const float* vol, const float* W1, const float* W2, const float* b2,
                        float* feat, int64_t m, cudaStream_t s);
int launch_tgt_feat(const float* vol_tgt, const float* W1, const float* W2, const float* b2,
                    unsigned long long* clear_keys, float* feat, int B, cudaStream_t s);
int launch_score_fp32(const void* vol_src, int vol_dtype, const float* tgt_feat, const float* R,
                      int r_per_pair, const float* W1, const float* W2, const float* b2,
                      const float* base, float* scores, int B, int64_t N, cudaStream_t s);
int launch_score_tc(const void* vol_src, int vol_dtype, const float* tgt_feat, const float* R,
                    int r_per_pair, const float* W1, const float* W2, const float* b2,
                    const float* base, float* scores, int B, int64_t N, void* ws, size_t ws_bytes,
                    cudaStream_t s, bool f16_gather);
size_t score_tc_workspace_bytes(int B, int64_t N);
float* scratch_tgt_feat(void* ws, int B);  // [B,32,64] slot inside the tensor-core scratch
int launch_verify_tc_argmax(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R,
                            int r_per_pair, const float* W1, const float* W2, const float* b2,
                            const float* base, float* scores, float* best_val, int64_t* best_idx,
                            float* R_best, int64_t idx_offset, int B, int64_t N, void* ws, size_t ws_bytes,
                            cudaStream_t s, bool f16_gather, const peer::Args* pa = nullptr);
int launch_verify_tc_screened(const float* vol_src, const float* vol_tgt, const float* R, int r_per_pair, const float* W1,
                              const float* W2, const float* b2, const float* base, float* best_val, int64_t* best_idx,
                              float* R_best, int64_t idx_offset, int B, int64_t N, void* ws, size_t ws_bytes, float* s16,
                              void* lists, cudaStream_t s, const peer::Args* pa = nullptr);
int launch_topk_exchange(const float* val, const int64_t* idx, const float* R, int r_per_pair, int64_t idx_offset,
                         int64_t N, int B, int k, float* out_val, int64_t* out_idx, float* R_best,
                         const peer::Args& pa, cudaStream_t s);
int launch_scores_exchange(const float* part, int B, int64_t N, float* out, const peer::Args& pa, int64_t cap_hyps,
                           cudaStream_t s);
int launch_slot_gather(float* R_all, float* score_all, int64_t item_lo, int64_t item_hi, int B, int k, const peer::Args& pa,
                       cudaStream_t s);
int preload_exchange_kernels();  // see ahv_exchange.cu
int preload_ranged_ascent();
int launch_topk(const float* scores, int B, int64_t N, int k, int64_t idx_offset, float* val,
                int64_t* idx, void* ws, size_t ws_bytes, cudaStream_t s);
size_t topk_workspace_bytes(int B, int64_t N, int k);
int launch_topk_merge(const float* vals, const int64_t* idx, int parts, int B, int k, float* out_val,
                      int64_t* out_idx, cudaStream_t s);
int launch_gather_rotations(const float* R, int r_per_pair, const int64_t* idx, int64_t idx_offset,
                            int B, int64_t N, int k, float* R_out, cudaStream_t s);
int launch_topk_distinct(const float* scores, const float* R, int r_per_pair, int B, int64_t N, int k, float min_sep_deg,
                         float* val, int64_t* idx, float* R_best, cudaStream_t s);
// Screened arg-max of ahv_verify (k = 1, fp32 volumes, AHV_MATH_TC; the passes are described at
// launch_verify_tc_screened in ahv_score_tc.cu).  Per pair a list of kScreenList hypotheses: the contenders (16-bit
// gather score within 2 tau of the pair's screened maximum, at most kScreenCap of them, padded with the first), then
// kScreenProbes fixed strided probes.  tau is in score units (scores are means of cosines): 27x the largest 16-bit vs
// fp32 gather difference on the bench workload (7.3e-5) and at least 8x that of order-one volumes with outliers up to
// 3e7 times the bulk, of the mixed per-pair scales and of the head-weight cases short of one W1 row dominating the
// others by 2^6 (profiles/r11_screen_margin.json); with it the bench workload has at most 22 contenders per pair.
constexpr int kScreenCap = 224;
constexpr int kScreenProbes = 32;
constexpr int kScreenList = kScreenCap + kScreenProbes;
constexpr float kScreenTau = 2e-3f;
struct ScreenLists {  // carved from the verification workspace's top-k partials region (unused when k == 1)
  int* idx;      // [B][kScreenList] hypothesis index
  float* s16;    // [B][kScreenList] its 16-bit gather score
  int* count;    // [B] contenders found (more than kScreenCap: the pair is flagged)
  float* err;    // [B] largest |fp32 score - 16-bit score| over the list
  int* flagged;  // [1 + B]: number of flagged pairs, then the flagged pairs (in no particular order)
  static size_t bytes(int B) { return (size_t)B * kScreenList * 8 + (size_t)B * 8 + (size_t)(B + 1) * 4; }
  ScreenLists(void* p, int B) {
    idx = static_cast<int*>(p);
    s16 = reinterpret_cast<float*>(idx + (size_t)B * kScreenList);
    count = reinterpret_cast<int*>(s16 + (size_t)B * kScreenList);
    err = reinterpret_cast<float*>(count + B);
    flagged = reinterpret_cast<int*>(err + B);
  }
};
int launch_screen_select(const float* s16, const unsigned long long* keys, int B, int64_t N, const float* R, int r_per_pair,
                         const ScreenLists& L, float* R_list, cudaStream_t s);
int launch_screen_guard(const float* s32, const ScreenLists& L, int B, unsigned long long* keys, cudaStream_t s);
size_t posterior_workspace_bytes(int B, int64_t N, int k, bool moments);
// ahv_posterior_mass (moment == nullptr) and ahv_posterior_moments (mean_R, mean_cos and moment set)
int launch_posterior(const float* scores, const float* R, int r_per_pair, const float* centers, int B, int64_t N, int k,
                     float radius_deg, float temperature, float* log_z, float* mass, float* mean_R, float* mean_cos,
                     float* moment, void* ws, cudaStream_t s);

}  // namespace ahv
