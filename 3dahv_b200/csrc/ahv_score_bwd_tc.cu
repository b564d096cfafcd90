// Fused backward of the verification scores with its contractions on tcgen05 (training variant,
// SURVEY.md §8a-8 / §8f-3; the reference: autograd through modules/model.py:43-63).
//
// Same chain as ahv_score_bwd.cu (which stays the exact fp32 form) for a training step that kept conv1's ReLU'd
// output H1 in the forward (ahv_score_train).  One CTA = 256 threads per SM, a contiguous range of (pair, hypothesis)
// items; per item:
//
//   X = rotate(V_b, R_n)                         fp32 gather in shared memory (taps recorded for the adjoint)
//   H2 = H1 W2^T + b2   [64 pos x 32]            tcgen05.mma  M=64 N=16 (x2)  K=32   H1 = the fp16 rows the forward kept
//   F = H2/|H2| ; dH2 ; dT += (g/64) F ; db2     fp32, thread = (position, 8 channels) as the accumulator presents them
//   dH1 = (dH2 W2) * [H1 > 0]                    tcgen05.mma  M=64 N=16 (x2)  K=32   dH2 under one power of two per item
//   dW2 += dH2^T H1                              tcgen05.mma  M=64 N=16 (x2)  K=64   rows = channels (32 + 32 padding)
//   dA   [64 pos x 384]  = dH1 [64 x 32] . W1    tcgen05.mma  M=64 N=192 (x2) K=32
//   dW1^T[384    x 32 ]  = A^T [384 x 64] . dH1  tcgen05.mma  M=128 (x3 views) N=32 K=64
//   dX = fold(dA) (three tri-plane views onto the rotated volume) ; dV_b += rotate^T(dX)   (gather over a work list)
//
// 1.75 of the ~1.8 MFLOP per item are tensor-core work; the fp32 kernel spent 69 % of its time on them.
//
// Operands (fp16, fp32 accumulation in TMEM), all K-major SWIZZLE_NONE core-matrix layouts
// (element (row r, k) at (r/8)*SBO + (k/8)*LBO + (r%8)*16 + (k%8)*2):
//   H1, dH2, dH1 as A [pos][ch] : SBO 512, LBO 128     written by the thread that owns (pos, 8 channels): one 16 B store
//   W2 / W2^T     as B [32][32] : SBO 512, LBO 128     packed once per CTA
//   W1^T as B of dA   [n'][o]   : SBO 512, LBO 128     packed once per CTA; rows PERMUTED n' = g*96 + view*32 + cc*8 + kk
//                                                      (channel c = 4g + cc) so that every fold thread owns 32 columns
//                                                      of every view
//   A^T  as A of dW1  [m][pos]  : SBO 1024, LBO 128    (view z: 1152 / 144) m = view*128 + c*8 + kk; view y is the rotated
//                                                      volume as it lies ([c][d][h][w]), view x its (h,w) transpose, view z
//                                                      its (d,h) one
//   dH1, dH2^T, H1^T  [ch][pos] : SBO 1040, LBO 128    B of dW1, A and B of dW2 (pitch 1040: the eight 2-byte stores of a
//                                                      thread's channel block hit distinct banks across the warp)
// Scales (powers of two, undone in fp32 when the accumulators are read): W1 and W2 are packed as W * 2^-e (largest row
// L1 norm in [4, 8) / [1, 2)), as the forward packs them (same sums, same e); H1 carries the forward's pair scale s and
// W1's normaliser (pair_inv_scale = 2^e1 / s), A^T the pair scale s alone; dH2 a per-item scale from the bound
// 2 |g/64| / min_p |H2_p|; dH1 a per-item scale from max |dH1| (2^13 <= max < 2^14); dX (fp16) a launch-wide one, kappa,
// from the normalised W1's largest column L1 norm (inv_kappa also undoes 2^-e1).
// The M=64 accumulators come in pairs side by side in the lanes (lanes 0-15 / 16-31 of every 32-lane quadrant hold two
// column blocks of the same 16 rows), so all 32 lanes of a warp read; dW1^T and dW2 are read every item into per-thread
// fp32 accumulators (48 + 8), which keeps the accumulation across items in fp32 and lets the scales differ per item.
// dX lies voxel-major, channels innermost, in fp16, over the dead A^T operand; the adjoint walks, per input voxel, a row of up
// to 16 (offset, weight) contributions built in one pass of shared-memory atomics (exact fallback for matrices that are
// not rotations and crowd more contributions onto a voxel).
//
// Gradients are those of the function the tensor-core forward evaluated (its ReLU mask), with fp16 operand rounding:
// checked to 1e-3 of each gradient's maximum against fp64 autograd of that function (tests/test_gpu_training.py).
//
// kDet (ahv_score_backward_det): no float atomics - dV, dT and the weight gradients go to the workspace slots of
// DetBwdWs (ahv_common.cuh: g_vol / g_tgt point at the segment slots, g_W1 / g_W2 / g_b2 at the weight slots) - and
// every input voxel's contributions are summed in increasing output-voxel order: a sorting network over the row in
// registers, an insertion sort of the exact path's lists.  The exact path's work list, the sorts and the flushes of the
// gradients are shared with the fp32 backward (ahv_adjoint.cuh).
#include <cstddef>

#include "ahv_adjoint.cuh"
#include "ahv_head_fp32.cuh"
#include "ahv_tc_ptx.cuh"

// -DAHV_BWD_PHASES: thread 0 of CTA 0 accumulates clock64() per phase and prints the shares (diagnostics builds only)
#ifdef AHV_BWD_PHASES
#include <cstdio>
#define AHV_PH(i)                                                           \
  do {                                                                      \
    if (threadIdx.x == 0) { const long long c_ = clock64(); ph_[i] += c_ - last_; last_ = c_; } \
  } while (0)
#else
#define AHV_PH(i) do {} while (0)
#endif

namespace ahv {

using namespace tc;

namespace {

constexpr int kAtView = 16384;     // bytes of one view of A^T: 128 rows x 64 positions fp16
constexpr int kAtZLbo = 144, kAtZSbo = 8 * kAtZLbo;   // view z: K-chunk pitch 144 B (its stores run over h: distinct banks)
constexpr int kAtBytes = 2 * kAtView + 16 * kAtZSbo;
constexpr int kDh1bPitch = 1040;   // row-group pitch (SBO) of the [channel][position] operands
constexpr int kTmemCols = 512;     // dA: columns 0..191 (both lane halves); dW1^T: 192..287; conv2, dH1, dW2: 288..335
constexpr int kColW = 192;
// rotated volume [c][d][h][w]: channel pitch 584 = 8 mod 32, so the gather's four lanes of a voxel (channels j, j+4, j+8, j+12)
// and its eight voxels along w store to 32 distinct banks
constexpr int kRc = kS * kRotD + 8;
constexpr int kColH2 = 288, kColDh1 = 304, kColW2 = 320;   // conv2, dH1, dW2 accumulators: 16 columns each, both lane halves
// dX (gradient w.r.t. the rotated volume) lives over the A^T operand once its MMAs are done, voxel-major with the 16
// channels innermost, in fp16: the adjoint's random reads of it are what bounds the kernel, and a record of 32 bytes
// costs half the shared-memory wavefronts of an fp32 one.  Element (d, h, w, c) at word d*kDxD + h*kDxH + w*kDxW + c/2
// (pitches in 4-byte words, multiples of 4 so that a record is two aligned LDS.128).  The values are the raw
// accumulators (dH1's per-item scale S, W1's normaliser 2^-e1) times kappa, a power of two fixed per launch from the
// packed W1 so that the sum of the three views cannot overflow fp16: |acc| < 2^14 * max_k sum_o |fp16(W1[o][k] 2^-e1)|,
// kappa <= 2 / (3 * that maximum).
constexpr int kDxW = 12, kDxH = 100, kDxD = 804;
static_assert(8 * kDxD * 4 <= kAtBytes, "dX fits over the A^T operand");

struct __align__(128) BwdTcSmem {
  float vol[kLines * kC];          // halo'd source volume, channel innermost (as the fp32 scorer)
  float rotA[kC * kRc];            // rotated volume X [c][d][h][w] (padded); dead after the operands -> work-list entries
  float dh2[kP * kH1Row];          // scratch behind rotA: tail of the work list, its counters; db2 reduction at the end
  float4 taps[kVox];
  unsigned char at[kAtBytes];      // A^T operand
  unsigned char w1t[kK * kO * 2];  // W1^T operand (permuted rows)
  unsigned char dh1a[kP * kO * 2];
  unsigned char h1a[kP * kO * 2];  // H1 as the forward kept it: A of conv2
  unsigned char dh2a[kP * kO * 2]; // dH2 [pos][o]: A of dH1
  unsigned char w2b[kO * kO * 2];  // W2 as B of conv2 [o][i]
  unsigned char w2tb[kO * kO * 2]; // W2^T as B of dH1 [i][o]
  float2 part[kP * 4];             // per (position, channel block): partial |H2|^2 and <H2, T>
  unsigned char dh1b[4 * kDh1bPitch];
  unsigned char h1t[4 * kDh1bPitch];   // H1^T  [i][pos]: B of dW2
  unsigned char dh2t[8 * kDh1bPitch];  // dH2^T [o][pos]: A of dW2 (M=64: the upper 32 rows are never written, their products never read)
  float base[8];
  float red[8];
  float Rcur[12];
  unsigned long long bar[3];       // dA + dW1 | conv2 | dH1 + dW2
  uint32_t tmem_slot;
  int overflow;                    // some input voxel has more than kListCap contributions (degenerate R): exact path
};
static_assert(sizeof(BwdTcSmem) <= 232448, "shared memory budget");
// adjoint work list: per input voxel a row of kListCap 4-byte entries (dX offset / 4 | weight as unorm16 << 16), row pitch
// 20 words so that eight consecutive rows start in distinct 16-byte bank groups.  It covers the rotated-volume buffer and
// the first 4 KB of the dH2 buffer behind it; the counters follow.
constexpr int kListCap = 16, kListPitch = 20, kListTail = (kVox * kListPitch * 4 - kC * kRc * 4) / 4;   // floats of dh2 it takes
static_assert(kListTail >= 0 && (kListTail + 2 * kVox) <= kP * kH1Row && kVox * 8 * 8 <= kC * kRc * 4, "work list fits the dead buffers");
static_assert(offsetof(BwdTcSmem, dh2) == offsetof(BwdTcSmem, rotA) + kC * kRc * 4, "dh2 follows rotA");

__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// vol_g [16][512] NCDHW -> halo'd lines, the 16 channels of a line in the order 0 4 8 12 | 1 5 9 13 | 2 6 10 14 | 3 7 11 15
__device__ __forceinline__ void stage_volume_interleaved(float* __restrict__ vol, const float* __restrict__ vol_g) {
  for (int i = threadIdx.x; i < kLines * kC; i += kThreads) vol[i] = 0.0f;
  __syncthreads();
  for (int i = threadIdx.x; i < kC * kVox; i += kThreads) {
    const int c = i >> 9, v = i & 511;
    const int z = v >> 6, y = (v >> 3) & 7, x = v & 7;
    const int line = ((z + 1) * kHalo + (y + 1)) * kHalo + (x + 1);
    vol[line * kC + (c & 3) * 4 + (c >> 2)] = __ldg(vol_g + i);
  }
}

// trilinear gather of one hypothesis into rotA, 4 lanes per output voxel (as gather_hypothesis of the fp32 scorer,
// without the transposed copy); lane j==0 of every voxel records the tap for the adjoint
__device__ __forceinline__ void gather_rotated(BwdTcSmem& sm, const float* R) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = lane & 3, q = lane >> 2;
  // warp = h; iteration it = d; the 8 voxels of an iteration run along w (q), 4 lanes (j) per voxel.  The sample
  // position of a voxel is computed ONCE, by lane (d % 4) * 8 + w for the four d of a half, and handed to the voxel's
  // four lanes by shuffles (the four lanes used to recompute it: a third of the gather's instructions).
#pragma unroll 1
  for (int half = 0; half < 2; ++half) {
    const int dl = 4 * half + (lane >> 3), wl = lane & 7;
    const Tap own = make_tap(R, sm.base[wl], sm.base[warp], sm.base[dl]);
    sm.taps[dl * 64 + warp * 8 + wl] = make_float4(__int_as_float(own.line), own.fx, own.fy, own.fz);
#pragma unroll 1
    for (int i = 0; i < 4; ++i) {
      const int d = 4 * half + i, h = warp, w = q, src = i * 8 + q;
      Tap t;
      t.line = __shfl_sync(0xffffffffu, own.line, src);
      t.fx = __shfl_sync(0xffffffffu, own.fx, src);
      t.fy = __shfl_sync(0xffffffffu, own.fy, src);
      t.fz = __shfl_sync(0xffffffffu, own.fz, src);
      const int swap = (t.line ^ q) & 1;  // parity order: the two x-taps of a lane pair never share a bank half
      const float wx_first = swap ? t.fx : 1.0f - t.fx;
      const float wx_second = swap ? 1.0f - t.fx : t.fx;
      const float* p0 = sm.vol + (t.line + swap) * kC + j * 4;
      const float* p1 = sm.vol + (t.line + 1 - swap) * kC + j * 4;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int dz = 0; dz < 2; ++dz)
#pragma unroll
        for (int dy = 0; dy < 2; ++dy) {
          const float wyz = (dy ? t.fy : 1.0f - t.fy) * (dz ? t.fz : 1.0f - t.fz);
          const int off = (dz * kHalo * kHalo + dy * kHalo) * kC;
          const float4 a = *reinterpret_cast<const float4*>(p0 + off);
          const float4 b = *reinterpret_cast<const float4*>(p1 + off);
          const float wa = wyz * wx_first, wb = wyz * wx_second;
          acc.x = fmaf(wa, a.x, acc.x); acc.y = fmaf(wa, a.y, acc.y);
          acc.z = fmaf(wa, a.z, acc.z); acc.w = fmaf(wa, a.w, acc.w);
          acc.x = fmaf(wb, b.x, acc.x); acc.y = fmaf(wb, b.y, acc.y);
          acc.z = fmaf(wb, b.z, acc.z); acc.w = fmaf(wb, b.w, acc.w);
        }
      float* dst = sm.rotA + j * kRc + d * kRotD + h * 8 + w;   // the staged volume interleaves the channels: lane j holds j, j+4, j+8, j+12
      dst[0] = acc.x; dst[4 * kRc] = acc.y; dst[8 * kRc] = acc.z; dst[12 * kRc] = acc.w;
    }
  }
}

// acc[0..15] += w * (the 16 fp16 channels of one dX record)
__device__ __forceinline__ void axpy_record(float* acc, float w, const uint32_t* rec) {
  const uint4 a = *reinterpret_cast<const uint4*>(rec), b = *reinterpret_cast<const uint4*>(rec + 4);
  const uint32_t u[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&u[i]));
    acc[2 * i] = fmaf(w, f.x, acc[2 * i]);
    acc[2 * i + 1] = fmaf(w, f.y, acc[2 * i + 1]);
  }
}
// four channels of a dX record += four accumulator values times kappa
__device__ __forceinline__ void add4_record(uint32_t* p, float kappa, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
  const uint2 x = *reinterpret_cast<const uint2*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&x.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&x.y));
  *reinterpret_cast<uint2*>(p) = make_uint2(pack_h2(fmaf(__uint_as_float(r0), kappa, a.x), fmaf(__uint_as_float(r1), kappa, a.y)),
                                            pack_h2(fmaf(__uint_as_float(r2), kappa, b.x), fmaf(__uint_as_float(r3), kappa, b.y)));
}

// rotated volume (fp32) -> the three views of the A^T operand (fp16, pair scale `sb`)
__device__ __forceinline__ void pack_views(BwdTcSmem& sm, float sb) {
  const int t = threadIdx.x;
#pragma unroll
  for (int i = 0; i < 4; ++i) {  // views y and z: one conversion, two conflict-free 16 B stores; lanes run over (d, h)
    const int task = t + 256 * i, c = task >> 6, d = (task >> 3) & 7, h = task & 7;
    const float* src = sm.rotA + c * kRc + d * kRotD + h * 8;
    const float4 a = *reinterpret_cast<const float4*>(src), b = *reinterpret_cast<const float4*>(src + 4);
    const uint4 pk = make_uint4(pack_h2(a.x * sb, a.y * sb), pack_h2(a.z * sb, a.w * sb), pack_h2(b.x * sb, b.y * sb), pack_h2(b.z * sb, b.w * sb));
    *reinterpret_cast<uint4*>(sm.at + kAtView + c * 1024 + d * 128 + h * 16) = pk;           // [c][d][h][w] as it lies
    *reinterpret_cast<uint4*>(sm.at + 2 * kAtView + c * kAtZSbo + h * kAtZLbo + d * 16) = pk;  // [c][h][d][w], h pitch 144 B
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {  // view x: [c][d][w][h]; lanes run over (d, w), eight h gathered per thread
    const int task = t + 256 * i, c = task >> 6, d = (task >> 3) & 7, w = task & 7;
    const float* src = sm.rotA + c * kRc + d * kRotD + w;
    *reinterpret_cast<uint4*>(sm.at + c * 1024 + d * 128 + w * 16) =
        make_uint4(pack_h2(src[0] * sb, src[8] * sb), pack_h2(src[16] * sb, src[24] * sb), pack_h2(src[32] * sb, src[40] * sb),
                   pack_h2(src[48] * sb, src[56] * sb));
  }
}

template <bool kDet>
__global__ void __launch_bounds__(kThreads, 1)
score_bwd_tc_kernel(const float* __restrict__ vol_src, const float* __restrict__ tgt_feat,
                    const float* __restrict__ R, int r_per_pair, const float* __restrict__ W1,
                    const float* __restrict__ W2, const float* __restrict__ b2, const float* __restrict__ base,
                    const float* __restrict__ grad_scores, const __half* __restrict__ h1_saved,
                    const float* __restrict__ pair_inv, float* __restrict__ g_vol, float* __restrict__ g_tgt,
                    float* __restrict__ g_W1, float* __restrict__ g_W2, float* __restrict__ g_b2, int B, int64_t N) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  BwdTcSmem& sm = *reinterpret_cast<BwdTcSmem*>(smem_raw);
  const int64_t total = (int64_t)B * N;
  const int64_t lo = total * blockIdx.x / gridDim.x, hi = total * (blockIdx.x + 1) / gridDim.x;
  if (lo >= hi) return;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  // shared-window address of the struct, made opaque once: ptxas otherwise re-derives it (S2UR SR_CgaCtaId + 5 uniform
  // ops) in front of every MMA it issues
  uint32_t sbase;
  asm volatile("mov.u32 %0, %1;" : "=r"(sbase) : "r"(smem_u32(smem_raw)));
  const uint32_t bar_s = sbase + (uint32_t)offsetof(BwdTcSmem, bar);

  // ---- set-up: weight normalisers, W2 operands, W1^T operand (fp16, permuted rows), base coordinates, barrier, TMEM ----
  sm.part[warp] = make_float2(row_l1max<kK, kThreads / 32>(W1, warp, lane), row_l1max<kO, kThreads / 32>(W2, warp, lane));
  __syncthreads();
  float n1, w1s, w2s;   // 2^-e1, 2^e1, 2^e2
  {
    float m1 = sm.part[0].x, m2 = sm.part[0].y;
#pragma unroll
    for (int w = 1; w < kThreads / 32; ++w) { m1 = fmaxf(m1, sm.part[w].x); m2 = fmaxf(m2, sm.part[w].y); }
    const int e1 = weight_exponent(m1, kW1NormTarget), e2 = weight_exponent(m2, kW2NormTarget);
    n1 = scalbnf(1.0f, -e1);
    w1s = scalbnf(1.0f, e1);
    w2s = scalbnf(1.0f, e2);
    const float n2 = scalbnf(1.0f, -e2);
    for (int i = t; i < kO * kO; i += kThreads) {
      const int o = i / kO, c = i % kO;
      const __half w = __float2half_rn(__ldg(W2 + i) * n2);
    *reinterpret_cast<__half*>(sm.w2b + (o >> 3) * 512 + (c >> 3) * 128 + (o & 7) * 16 + (c & 7) * 2) = w;   // rows o, K = i
      *reinterpret_cast<__half*>(sm.w2tb + (c >> 3) * 512 + (o >> 3) * 128 + (c & 7) * 16 + (o & 7) * 2) = w;  // rows i, K = o
    }
  }
  for (int i = t; i < kO * kK; i += kThreads) {
    const int o = i / kK, k = i - o * kK;  // coalesced read of W1[o][k]
    const int view = k >> 7, c = (k >> 3) & 15, kk = k & 7;
    const int grp = (c >> 2) * 12 + view * 4 + (c & 3);  // n' / 8
    *reinterpret_cast<__half*>(sm.w1t + grp * 512 + (o >> 3) * 128 + kk * 16 + (o & 7) * 2) = __float2half_rn(__ldg(W1 + i) * n1);
  }
  if (t < 8) sm.base[t] = base ? base[t] : 0.0f;
  {  // largest L1 norm of a packed W1 column (normalised, fp16-rounded, as the MMA sees it): bounds |dA acc| / max|dH1 S|
    float cmax = 0.0f;
    for (int k = t; k < kK; k += kThreads) {
      float c1 = 0.0f;
      for (int o = 0; o < kO; ++o) c1 += fabsf(__half2float(__float2half_rn(__ldg(W1 + o * kK + k) * n1)));
      cmax = fmaxf(cmax, c1);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
    if (lane == 0) sm.red[warp] = cmax;
  }
  if (warp == 0) {
    if (lane == 0) {
      mbar_init(bar_s, 1);
      mbar_init(bar_s + 8, 1);
      mbar_init(bar_s + 16, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    tmem_alloc(smem_u32(&sm.tmem_slot), kTmemCols);
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_slot;
  float kappa = 1.0f, inv_kappa = w1s;   // dX = acc * kappa; dA = dX * inv_kappa / S (inv_kappa undoes W1's normaliser too)
  {
    float c = sm.red[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) c = fmaxf(c, sm.red[w]);
    if (c > 0.0f) {
      const float x = 2.0f / (3.0f * c);
      const int e = min(max(((__float_as_int(x) >> 23) & 0xff) - 127, -60), 60);   // floor(log2 x)
      kappa = __int_as_float((127 + e) << 23);
      inv_kappa = __int_as_float((127 - e) << 23) * w1s;
    }
  }
  const uint32_t at_s = sbase + (uint32_t)offsetof(BwdTcSmem, at), w1t_s = sbase + (uint32_t)offsetof(BwdTcSmem, w1t);
  const uint32_t dh1a_s = sbase + (uint32_t)offsetof(BwdTcSmem, dh1a), dh1b_s = sbase + (uint32_t)offsetof(BwdTcSmem, dh1b);
  const uint32_t h1t_s = sbase + (uint32_t)offsetof(BwdTcSmem, h1t), dh2t_s = sbase + (uint32_t)offsetof(BwdTcSmem, dh2t);
  const uint32_t h1a_s = sbase + (uint32_t)offsetof(BwdTcSmem, h1a), dh2a_s = sbase + (uint32_t)offsetof(BwdTcSmem, dh2a);
  const uint32_t w2b_s = sbase + (uint32_t)offsetof(BwdTcSmem, w2b), w2tb_s = sbase + (uint32_t)offsetof(BwdTcSmem, w2tb);
  constexpr uint32_t idA = instr_desc(64, kColW), idW = instr_desc(128, 32), idC = instr_desc(64, 16);

  // accumulator read-out mapping: TMEM quadrant of this warp, column half
  const int qd = warp & 3, hf = warp >> 2;
  // head mapping: thread = (position, 8 channels cg2*8 ..) as the M=64 accumulators present them: the two lane halves
  // of a quadrant hold two 16-column accumulators of the same 16 rows, warps w and w+4 split each into 8 + 8 columns
  const int pos = 16 * qd + (lane & 15), cg2 = (lane >> 4) * 2 + hf;
  const uint32_t tq = tmem + ((uint32_t)(32 * qd) << 16);
  // fold mapping: lanes 0-15 / 16-31 hold the two M=64 accumulators: position 16 qd + lane%16, channel group g
  const int fpos = 16 * qd + (lane & 15), fp = fpos >> 3, fq = fpos & 7, fg = (lane >> 4) * 2 + hf;

  float b2r[8], tg[8];
#pragma unroll
  for (int oo = 0; oo < 8; ++oo) b2r[oo] = b2[cg2 * 8 + oo];
  float aW1[3][16];  // dW1[o = 16 hf + oo][k = view*128 + 32 qd + lane]
  float aW2[8];      // dW2[o = 16 qd + lane % 16][i = 16 (lane / 16) + 8 hf ..]  (quadrants 0 and 1 only)
  float ab2[8];      // db2[cg2*8 + oo] (this thread's position only)
  float aT[8];       // dT_b[cg2*8 + oo][pos]
  float aV[2][kC];   // dV_b[c][voxel t + 256 j]
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int oo = 0; oo < 16; ++oo) aW1[v][oo] = 0.0f;
#pragma unroll
  for (int i = 0; i < 8; ++i) aW2[i] = 0.0f;
#pragma unroll
  for (int i = 0; i < 8; ++i) ab2[i] = aT[i] = 0.0f;
#pragma unroll
  for (int j = 0; j < 2; ++j)
#pragma unroll
    for (int c = 0; c < kC; ++c) aV[j][c] = 0.0f;

  auto flush = [&](int b) { flush_pair<kDet>(g_tgt, g_vol, b, aT, aV, cg2, pos, true, true); };

  // ---- the adjoint's work list ----
  // Output voxel vo feeds the 8 input voxels of its tap with weight w.  Turned round: every INPUT voxel gets the list
  // of its (vo, w) contributions, so that the adjoint is one flat loop per input voxel.  A rigid rotation puts about 8
  // (at most ~12) contributions on a voxel: the list is a fixed row of kListCap entries per voxel, filled in ONE pass
  // (the counter's atomic returns the place in the row) while the tensor core works.  A matrix that is not a rotation
  // can exceed the row: then the item takes the exact path (counting sort with prefix sums) - valid for any matrix R.
  int* cnt = reinterpret_cast<int*>(sm.dh2 + kListTail);   // [512] contributions per input voxel
  int* start = cnt + kVox;                                 // [512] exclusive prefix sum (exact path)
  uint32_t* ent16 = reinterpret_cast<uint32_t*>(sm.rotA);  // [512][kListPitch]
  uint2* ent = reinterpret_cast<uint2*>(sm.rotA);          // exact path: [<= 4096] (offset of dX[vo], weight)
  // The thread's two output voxels (one per pass) are chosen two apart in x and y and four in z across the lanes of a
  // warp, so that the taps of one warp's voxels rarely meet in the same counter.
  auto list_pass = [&](int j) {
    const int vo = adjoint_out_voxel(t, j);
    const uint32_t off4 = (uint32_t)((vo >> 6) * kDxD + ((vo >> 3) & 7) * kDxH + (vo & 7) * kDxW) >> 2;   // record, in 16-byte units
    const float4 tp = sm.taps[vo];
    const int line = __float_as_int(tp.x);   // ((z0+1)*10 + (y0+1))*10 + (x0+1), corner in [-1, 7]^3
    const int zl = line / (kHalo * kHalo), rl = line - zl * (kHalo * kHalo), yl = rl / kHalo, xl = rl - yl * kHalo;
    const int x0 = xl - 1, y0 = yl - 1, z0 = zl - 1;
    const int tgt0 = z0 * 64 + y0 * 8 + x0;
    bool over = false;
#pragma unroll
    for (int dlt = 0; dlt < 8; ++dlt) {
      const int dx = dlt & 1, dy = (dlt >> 1) & 1, dz = dlt >> 2;
      if ((unsigned)(x0 + dx) < 8u && (unsigned)(y0 + dy) < 8u && (unsigned)(z0 + dz) < 8u) {
        const int v = tgt0 + dz * 64 + dy * 8 + dx;
        const float w = (dx ? tp.y : 1.0f - tp.y) * (dy ? tp.z : 1.0f - tp.z) * (dz ? tp.w : 1.0f - tp.w);
        const int r = atomicAdd(&cnt[v], 1);
        if (r < kListCap) ent16[v * kListPitch + r] = off4 | (__float2uint_rn(w * 65535.0f) << 16);
        else over = true;
      }
    }
    if (over) sm.overflow = 1;
  };

  int cur_b = -1;
  float pinv = 1.0f, pvol = 1.0f;   // H1 = h1 * pinv (2^e1 / s); 1/s, the volume's scale in A^T
  uint32_t phase = 0;
  float r_next = 0.0f;
  if (t < 9) r_next = __ldg(R + (r_per_pair ? (size_t)lo : (size_t)(lo % N)) * 9 + t);
#ifdef AHV_BWD_PHASES
  long long ph_[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, last_ = clock64();
#endif
  for (int64_t it = lo; it < hi; ++it) {
    const int b = (int)(it / N);
    if (b != cur_b) {
      if (cur_b >= 0) flush(cur_b);
      __syncthreads();
      stage_volume_interleaved(sm.vol, vol_src + (size_t)b * kC * kVox);
#pragma unroll
      for (int oo = 0; oo < 8; ++oo) tg[oo] = tgt_feat[((size_t)b * kO + cg2 * 8 + oo) * kP + pos];
      pinv = __ldg(pair_inv + b);
      pvol = pinv * n1;
      cur_b = b;
    }
    cnt[t] = 0;   // the work list's counters (the previous item's adjoint is behind a barrier)
    cnt[t + 256] = 0;
    if (t == 0) sm.overflow = 0;
    if (t < 9) {   // this item's rotation was fetched one item ago; fetch the next one's
      sm.Rcur[t] = r_next;
      if (it + 1 < hi) r_next = __ldg(R + (r_per_pair ? (size_t)(it + 1) : (size_t)((it + 1) % N)) * 9 + t);
    }
    // H1 of this item as the forward kept it (fp16, pair-scaled): in flight during the gather
    const uint4 hq = __ldg(reinterpret_cast<const uint4*>(h1_saved + ((size_t)it * kP + pos) * kO + cg2 * 8));
    const float g64 = grad_scores[it] * (1.0f / 64.0f);  // d mean over the 64 positions
    float inv_s2 = 1.0f;
    __syncthreads();
    float Rr[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) Rr[e] = sm.Rcur[e];
    AHV_PH(0);

    // ---------------- X = rotate(V_b, R); H1 as the operand of conv2 and of dW2 ----------------
    gather_rotated(sm, Rr);
    {
      *reinterpret_cast<uint4*>(sm.h1a + (pos >> 3) * 512 + cg2 * 128 + (pos & 7) * 16) = hq;
      const __half* hp = reinterpret_cast<const __half*>(&hq);   // and transposed, as the B operand of dW2
      unsigned char* bb = sm.h1t + cg2 * kDh1bPitch + (pos >> 3) * 128 + (pos & 7) * 2;
#pragma unroll
      for (int j = 0; j < 8; ++j) *reinterpret_cast<__half*>(bb + j * 16) = hp[j];
    }
    fence_proxy_async();
    __syncthreads();
    AHV_PH(1);

    // ---------------- conv2 on the tensor core (the forward's own arithmetic), A^T operand meanwhile ----------------
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int half = 0; half < 2; ++half)  // output channels 16 half .. +15 -> lanes 16 half .. of every quadrant
#pragma unroll
          for (int j = 0; j < 2; ++j)
            umma_f16_raw(tmem + kColH2 + ((uint32_t)(16 * half) << 16), smem_desc(h1a_s + j * 256, 128, 512),
                         smem_desc(w2b_s + half * 1024 + j * 256, 128, 512), idC, j);
        umma_commit_raw(bar_s + 8);
      }
      __syncwarp();
    }
    pack_views(sm, 1.0f / pvol);
    AHV_PH(2);
    mbar_wait(bar_s + 8, phase);
    tc_fence_after();
    float v[8];
    {
      uint32_t r8[8];
      tmem_ld8(tq + kColH2 + hf * 8, r8);
      tmem_ld_wait();
      const float sc = pinv * w2s;   // undo the pair scale and both weight normalisers
#pragma unroll
      for (int oo = 0; oo < 8; ++oo) v[oo] = fmaf(__uint_as_float(r8[oo]), sc, b2r[oo]);  // + bias
    }
    float ss = 0.0f, ft = 0.0f;
#pragma unroll
    for (int oo = 0; oo < 8; ++oo) { ss = fmaf(v[oo], v[oo], ss); ft = fmaf(v[oo], tg[oo], ft); }
    sm.part[pos * 4 + cg2] = make_float2(ss, ft);
    __syncthreads();
    {
      const float4 p01 = *reinterpret_cast<const float4*>(&sm.part[pos * 4]), p23 = *reinterpret_cast<const float4*>(&sm.part[pos * 4 + 2]);
      ss = (p01.x + p01.z) + (p23.x + p23.z);   // fixed order: the four threads of a position agree bit for bit
      ft = (p01.y + p01.w) + (p23.y + p23.w);
    }
    {
      // F = v / max(|v|, eps) (modules/modules.py:122).  d<F,T>/dv = (T - F <F,T>) / |v| above the clamp, T / eps below
      const float nraw = sqrtf(ss), nr = fmaxf(nraw, 1e-12f), inv = 1.0f / nr;
      const float fdot = ft * inv;
      const bool clamped = nraw < 1e-12f;
#pragma unroll
      for (int oo = 0; oo < 8; ++oo) {
        const float F = v[oo] * inv;
        const float d2 = g64 * inv * (clamped ? tg[oo] : tg[oo] - F * fdot);
        aT[oo] = fmaf(g64, F, aT[oo]);
        ab2[oo] += d2;
        v[oo] = d2;
      }
      // dH2 as fp16 operands - rows = positions for dH1 = dH2 W2, rows = channels for dW2 = dH2^T H1 - under ONE power of
      // two per item (dW2 contracts over the positions): every |dH2| is below 2 |g/64| / min_p |H2_p|, which the scale maps
      // into [2^13, 2^14).  The smallest |H2_p|^2 comes from the partial sums every thread can see (fixed order: all
      // warps derive the same scale).
      float ssmin;
      {
        const float4 a01 = *reinterpret_cast<const float4*>(&sm.part[lane * 4]), a23 = *reinterpret_cast<const float4*>(&sm.part[lane * 4 + 2]);
        const float4 b01 = *reinterpret_cast<const float4*>(&sm.part[(lane + 32) * 4]), b23 = *reinterpret_cast<const float4*>(&sm.part[(lane + 32) * 4 + 2]);
        ssmin = fminf((a01.x + a01.z) + (a23.x + a23.z), (b01.x + b01.z) + (b23.x + b23.z));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ssmin = fminf(ssmin, __shfl_xor_sync(0xffffffffu, ssmin, o));
      }
      const float bnd = 2.0f * fabsf(g64) / fmaxf(sqrtf(ssmin), 1e-12f);
      int e = ((__float_as_int(bnd) >> 23) & 0xff) - 127;
      e = bnd > 0.0f ? min(max(e, -100), 100) : 13;
      const float S2 = __int_as_float((127 + 13 - e) << 23);
      inv_s2 = __int_as_float((127 - 13 + e) << 23);
      __half hv[8];
#pragma unroll
      for (int oo = 0; oo < 8; ++oo) hv[oo] = __float2half_rn(v[oo] * S2);
      *reinterpret_cast<uint4*>(sm.dh2a + (pos >> 3) * 512 + cg2 * 128 + (pos & 7) * 16) = *reinterpret_cast<const uint4*>(hv);
      unsigned char* bb = sm.dh2t + cg2 * kDh1bPitch + (pos >> 3) * 128 + (pos & 7) * 2;
#pragma unroll
      for (int oo = 0; oo < 8; ++oo) *reinterpret_cast<__half*>(bb + oo * 16) = hv[oo];
    }
    fence_proxy_async();
    tc_fence_before();  // conv2's accumulator has been read
    __syncthreads();
    AHV_PH(3);

    // ---------------- dH1 = (dH2 W2) * [H1 > 0] and dW2 += dH2^T H1 on the tensor core; half of the work list meanwhile ----------------
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int half = 0; half < 2; ++half)
#pragma unroll
          for (int j = 0; j < 2; ++j)
            umma_f16_raw(tmem + kColDh1 + ((uint32_t)(16 * half) << 16), smem_desc(dh2a_s + j * 256, 128, 512),
                         smem_desc(w2tb_s + half * 1024 + j * 256, 128, 512), idC, j);
#pragma unroll
        for (int half = 0; half < 2; ++half)  // rows = channels o of dH2 (the upper 32 of the M=64 rows are padding), K = positions
#pragma unroll
          for (int j = 0; j < 4; ++j)
            umma_f16_raw(tmem + kColW2 + ((uint32_t)(16 * half) << 16), smem_desc(dh2t_s + j * 256, 128, kDh1bPitch),
                         smem_desc(h1t_s + half * 2 * kDh1bPitch + j * 256, 128, kDh1bPitch), idC, j);
        umma_commit_raw(bar_s + 16);
      }
      __syncwarp();
    }
    AHV_PH(10);
    list_pass(0);
    AHV_PH(11);
    float dh1[8];
    {
      mbar_wait(bar_s + 16, phase);
      tc_fence_after();
      uint32_t r8[8];
      tmem_ld8(tq + kColDh1 + hf * 8, r8);
      tmem_ld_wait();
      const uint4 hm = *reinterpret_cast<const uint4*>(sm.h1a + (pos >> 3) * 512 + cg2 * 128 + (pos & 7) * 16);
      const __half* hp = reinterpret_cast<const __half*>(&hm);  // ReLU mask (modules/modules.py:68)
      float mx = 0.0f;
      const float dsc = inv_s2 * w2s;   // undo the dH2 scale and W2's normaliser
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        dh1[j] = __half2float(hp[j]) > 0.0f ? __uint_as_float(r8[j]) * dsc : 0.0f;
        mx = fmaxf(mx, fabsf(dh1[j]));
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      if (lane == 0) sm.red[warp] = mx;
      if (qd < 2) {  // dW2 rows o = 16 qd + lane % 16 (quadrants 2, 3 hold the padding rows)
        tmem_ld8(tq + kColW2 + hf * 8, r8);
        tmem_ld_wait();
        const float sc = inv_s2 * pinv;  // undo the dH2 scale and the pair scale of H1
#pragma unroll
        for (int j = 0; j < 8; ++j) aW2[j] = fmaf(__uint_as_float(r8[j]), sc, aW2[j]);
      }
    }
    tc_fence_before();
    __syncthreads();
    AHV_PH(4);

    // ---------------- dH1 -> fp16 operands under the item's power-of-two scale ----------------
    float invS;
    {
      float m = sm.red[0];
#pragma unroll
      for (int w = 1; w < 8; ++w) m = fmaxf(m, sm.red[w]);
      int e = ((__float_as_int(m) >> 23) & 0xff) - 127;  // floor(log2 max|dH1|)
      e = m > 0.0f ? min(max(e, -100), 100) : 13;
      const float S = __int_as_float((127 + 13 - e) << 23);  // 2^13 <= max * S < 2^14
      invS = __int_as_float((127 - 13 + e) << 23);
      *reinterpret_cast<uint4*>(sm.dh1a + (pos >> 3) * 512 + cg2 * 128 + (pos & 7) * 16) =
          make_uint4(pack_h2(dh1[0] * S, dh1[1] * S), pack_h2(dh1[2] * S, dh1[3] * S), pack_h2(dh1[4] * S, dh1[5] * S),
                     pack_h2(dh1[6] * S, dh1[7] * S));
      unsigned char* bb = sm.dh1b + cg2 * kDh1bPitch + (pos >> 3) * 128 + (pos & 7) * 2;
#pragma unroll
      for (int j = 0; j < 8; ++j) *reinterpret_cast<__half*>(bb + j * 16) = __float2half_rn(dh1[j] * S);
    }
    fence_proxy_async();  // A^T, dH1 operands: generic-proxy stores -> async proxy
    __syncthreads();
    AHV_PH(5);

    // ---------------- the two contractions on the tensor core ----------------
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int half = 0; half < 2; ++half)  // dA: rows = positions, columns = 192 of the permuted W1^T rows
#pragma unroll
          for (int j = 0; j < 2; ++j)
            umma_f16_raw(tmem + ((uint32_t)(16 * half) << 16), smem_desc(dh1a_s + j * 256, 128, 512),
                         smem_desc(w1t_s + half * (kColW / 8) * 512 + j * 256, 128, 512), idA, j);
#pragma unroll
        for (int view = 0; view < 3; ++view)  // dW1^T: rows = (c, kk) of the view, K = the 64 positions
#pragma unroll
          for (int j = 0; j < 4; ++j)
            umma_f16_raw(tmem + kColW + view * 32,
                         view < 2 ? smem_desc(at_s + view * kAtView + j * 256, 128, 1024)
                                  : smem_desc(at_s + 2 * kAtView + j * 2 * kAtZLbo, kAtZLbo, kAtZSbo),
                         smem_desc(dh1b_s + j * 256, 128, kDh1bPitch), idW, j);
        umma_commit_raw(bar_s);
      }
      __syncwarp();
    }

    list_pass(1);   // second half of the adjoint's work list, in the shadow of the MMAs

    AHV_PH(6);
    // ---------------- accumulators: dW1^T -> registers, dA -> dX (fold of the three views) ----------------
    mbar_wait(bar_s, phase);
    AHV_PH(7);
    phase ^= 1;
    tc_fence_after();
    {
      const float sc = invS * pvol;  // undo the item's dH1 scale and the pair's volume scale
      uint32_t r[16];
#pragma unroll
      for (int view = 0; view < 3; ++view) {
        tmem_ld16(tq + kColW + view * 32 + hf * 16, r);
        tmem_ld_wait();
#pragma unroll
        for (int oo = 0; oo < 16; ++oo) aW1[view][oo] = fmaf(__uint_as_float(r[oo]), sc, aW1[view][oo]);
      }
    }
    uint32_t* dX = reinterpret_cast<uint32_t*>(sm.at);  // the A^T operand is dead: its MMAs have completed
    {
      uint32_t r[32];
      // view x: dX[d=p, h=q, w=kk, c] = ...   (every element of dX written exactly once: no zeroing needed)
      tmem_ld32(tq + hf * 96, r);
      tmem_ld_wait();
      {
        uint32_t* dst = dX + fp * kDxD + fq * kDxH + 2 * fg;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
          *reinterpret_cast<uint2*>(dst + kk * kDxW) = make_uint2(pack_h2(__uint_as_float(r[kk]) * kappa, __uint_as_float(r[8 + kk]) * kappa),
                                                                  pack_h2(__uint_as_float(r[16 + kk]) * kappa, __uint_as_float(r[24 + kk]) * kappa));
      }
      tmem_ld32(tq + hf * 96 + 32, r);  // view y, in flight across the barrier
      tmem_ld_wait();
      __syncthreads();
      {  // dX[d=p, h=kk, w=q, c] += ...
        uint32_t* dst = dX + fp * kDxD + fq * kDxW + 2 * fg;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) add4_record(dst + kk * kDxH, kappa, r[kk], r[8 + kk], r[16 + kk], r[24 + kk]);
      }
      tmem_ld32(tq + hf * 96 + 64, r);  // view z
      tmem_ld_wait();
      tc_fence_before();                // the next item's MMAs overwrite these accumulators
      __syncthreads();
      {  // dX[d=kk, h=p, w=q, c] += ...
        uint32_t* dst = dX + fp * kDxH + fq * kDxW + 2 * fg;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) add4_record(dst + kk * kDxD, kappa, r[kk], r[8 + kk], r[16 + kk], r[24 + kk]);
      }
    }
    const float unscale = invS * inv_kappa;   // dX holds dA * S * 2^-e1 * kappa
    __syncthreads();
    AHV_PH(8);

    // ---------------- dV_b += rotate^T(dX): adjoint of utils.py:113-131, one flat list per input voxel ----------------
    if (sm.overflow == 0) {
      const float wq = unscale * (1.0f / 65535.0f);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int vi = t + 256 * j;
        const int nn = cnt[vi];
        int nmax = nn;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, o));
        uint32_t en[kListCap];
        {
          const uint4* row = reinterpret_cast<const uint4*>(ent16 + vi * kListPitch);
#pragma unroll
          for (int q = 0; q < kListCap / 4; ++q) {
            const uint4 x = row[q];
            en[4 * q] = x.x; en[4 * q + 1] = x.y; en[4 * q + 2] = x.z; en[4 * q + 3] = x.w;
          }
        }
        if constexpr (kDet) {
          // the row in increasing record offset: halves swapped (offset on top, unique per output voxel), the unused
          // places above every entry; the network's size follows the warp's longest row
#pragma unroll
          for (int i = 0; i < kListCap; ++i) en[i] = i < nn ? __byte_perm(en[i], 0, 0x1032) : 0xffffffffu;
          sort_row(en, nmax);
        }
#pragma unroll
        for (int i = 0; i < kListCap; ++i) {
          if (i >= nmax) break;   // warp-uniform
          if (i < nn) {
            const uint32_t off4 = kDet ? en[i] >> 16 : en[i] & 0xffffu, w16 = kDet ? en[i] & 0xffffu : en[i] >> 16;
            axpy_record(aV[j], (float)w16 * wq, dX + (off4 << 2));
          }
        }
      }
    } else {
      // exact path (some voxel has more than kListCap contributions): counting sort with prefix sums, 8-byte entries
      __syncthreads();
      build_exact_list<kDxD, kDxH, kDxW>(sm.taps, cnt, start, ent, reinterpret_cast<int*>(sm.red));
      __syncthreads();
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int vi = t + 256 * j;
        const int nn = cnt[vi];
        uint2* e = ent + start[vi];
        if constexpr (kDet) sort_list(e, nn);   // the atomics ranked the list in arrival order: sort it by dX offset
        walk_list(e, nn, [&](uint2 en) { axpy_record(aV[j], __uint_as_float(en.y) * unscale, dX + en.x); });
      }
    }
    __syncthreads();  // dX (the operand buffer), taps and the work list are re-used by the next hypothesis
    AHV_PH(9);
  }
#ifdef AHV_BWD_PHASES
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    long long tot = 0;
    for (int i = 0; i < 10; ++i) tot += ph_[i];
    printf("dW2+dH1 detail: MMA issue %lld | list pass 0 %lld | rest = wait + read-outs + barrier\n", ph_[10] / (hi - lo), ph_[11] / (hi - lo));
    ph_[4] += ph_[10] + ph_[11];
    printf("bwd_tc phases, cycles per item (CTA 0, %lld items): loop+R %lld | gather+H1 %lld | pack views %lld | conv2+dH2 %lld | dW2+dH1 %lld | "
           "operands %lld | MMA issue+sort %lld | MMA wait %lld | dW1 read+fold %lld | adjoint %lld | total %lld\n",
           (long long)(hi - lo), ph_[0] / (hi - lo), ph_[1] / (hi - lo), ph_[2] / (hi - lo), ph_[3] / (hi - lo), ph_[4] / (hi - lo),
           ph_[5] / (hi - lo), ph_[6] / (hi - lo), ph_[7] / (hi - lo), ph_[8] / (hi - lo), ph_[9] / (hi - lo), tot / (hi - lo));
  }
#endif
  flush(cur_b);
  // weight gradients: one atomic per accumulator and CTA (kDet: one store into the CTA's weight slot)
#pragma unroll
  for (int view = 0; view < 3; ++view)
#pragma unroll
    for (int oo = 0; oo < 16; ++oo)
      flush_weight<kDet>(g_W1 + (16 * hf + oo) * kK + view * 128 + 32 * qd + lane, aW1[view][oo]);
  if (qd < 2) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      flush_weight<kDet>(g_W2 + (16 * qd + (lane & 15)) * kO + 16 * (lane >> 4) + 8 * hf + i, aW2[i]);
  }
  flush_b2<kDet>(sm.dh2, ab2, cg2, pos, g_b2, true);   // sm.dh2: [4 cg2][8 oo][64 pos]
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, kTmemCols);
  }
}

}  // namespace

int launch_score_bwd_tc(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                        const float* W1, const float* W2, const float* b2, const float* base,
                        const float* grad_scores, const void* h1_saved, const float* pair_inv, float* g_vol,
                        float* g_tgt, float* g_W1, float* g_W2, float* g_b2, int B, int64_t N, cudaStream_t s,
                        unsigned grid, bool det) {
  const int64_t total = (int64_t)B * N;
  if (total == 0) return AHV_OK;
  if (!h1_saved || !pair_inv) return AHV_EINVAL;
  if (grid == 0) {
    const int sms = sm_count();
    if (sms <= 0) return AHV_ECUDA;
    grid = (unsigned)(total < sms ? total : sms);
  }
  const auto kernel = det ? score_bwd_tc_kernel<true> : score_bwd_tc_kernel<false>;
  const size_t smem = sizeof(BwdTcSmem);
  AHV_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<grid, kThreads, smem, s>>>(vol_src, tgt_feat, R, r_per_pair, W1, W2, b2, base, grad_scores,
                                      static_cast<const __half*>(h1_saved), pair_inv, g_vol, g_tgt, g_W1, g_W2, g_b2, B, N);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

}  // namespace ahv
