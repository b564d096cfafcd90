// Fused hypothesis-and-verification kernels on tcgen05 tensor cores (AHV_MATH_TC*).
//
// Replace modules/model.py:186-193 (rotate_volume -> forward_3d2d -> correlate -> mean) for every
// (pair, hypothesis) without materialising anything in HBM: algorithmic HBM traffic is 36 B of
// rotation in and 4 B of score out (nothing at all when only the arg-max is requested).
//
// One persistent CTA per SM, 13 warps, warp-specialised (both kernels):
//   warps 0-7   GATHER   trilinear resampling (utils.py:113-131) of the source volume held in shared
//                        memory (zero halo, channel innermost).  One lane per output voxel, all 16
//                        channels.  The 16-byte chunks of a voxel line are visited in a per-lane
//                        rotated order and the two taps that sit in adjacent lines in bank-parity
//                        order, which makes every LDS.128 phase conflict-free by construction.
//                        Results are rounded to fp16 and become the tri-plane A operand of conv1.
//   warp  12    MMA      converged warp, one elect.sync lane issues tcgen05.mma (kind::f16, fp32
//                        accumulate in TMEM): conv1 = 24 K slices (view,k) of (N=32,K=16) per hypothesis -
//                        slice (view,k) multiplies the 16 channels at a fixed k, so the rearrange/cat of
//                        modules/modules.py:115-118 is pure descriptor arithmetic - two hypotheses
//                        interleaved in the two 16-lane halves of each TMEM sub-partition (M=64 per
//                        hypothesis for views y/z, one M=128 MMA per slice for view x in the TS kernel);
//                        conv2 = 2 x (M=128,N=32,K=16) per pair.
//   warps 8-11  EPILOGUE tcgen05.ld D1 -> ReLU -> fp16 -> conv2 operand; tcgen05.ld D2 -> +bias ->
//                        L2 norm -> dot with the target features (registers) -> mean over 64
//                        positions -> score (+ running arg-max key, one atomicMax per CTA and pair);
//                        the last CTA to finish decodes the winners and, when the hypothesis set is
//                        sharded over GPUs, exchanges them with the peers' kernels over NVLink.
// Pipelines (mbarrier): A-operand stages full/empty (3 deep), TMEM D1 full/empty, A2 full, D2 full.
// Set-up: every CTA packs W1/W2 to fp16 operand layouts itself (MMA/epilogue warps) and derives each
// pair's scale while staging its volume (gather warps), so the kernel depends on the target-feature
// prologue only through its epilogue warps (programmatic dependent launch).
//
//   score_tc_ts_kernel   view x of conv1 and conv2's A operand go register -> TMEM (tcgen05.st) and are
//                        consumed in the TS form of tcgen05.mma; only the YZ operand copy lives in shared
//                        memory; a stage is a hypothesis pair.  (An earlier SS-form kernel - both operand
//                        copies and A2 in shared memory - is gone from the build; see git history.)
// It exists for fp32-staged volumes (fp32 FFMA interpolation) and for 16-bit staged volumes
// (K16: bf16 inputs or AHV_MATH_TC_F16GATHER; x-pair lines, packed HFMA2 interpolation).
//
// Precision: normalisation and correlation are fp32; the two 1x1 convs use fp16 operands (10-bit
// mantissa = TF32-equivalent) with fp32 accumulation.  The source volume is pre-scaled per pair by a
// power of two (exact) so fp16 can neither overflow nor go subnormal; the scale is undone after
// conv2 (ReLU and the bias-free conv1 are positively homogeneous).
//
// Files: ahv_tc_ptx.cuh (PTX wrappers), ahv_peer.cuh (NVLink exchange buffer), ahv_tc_common.cuh (roles, tile
// iterator, weight packing, volume staging, epilogue), ahv_score_tc_ts.cuh (the kernel), this file
// (target-feature prologue, workspace carve-up, launchers).
#include "ahv_score_tc_ts.cuh"

namespace ahv {

namespace tc {

// ---- prologue: target features forward_3d2d(vol_tgt[b]) (modules/model.py:191) in fp32, + arg-max key clear ----
// grid (16, B), 128 threads: CTA (j, b) computes the 4 positions (p = j>>1, q = 4*(j&1) .. +3) of pair b for
// all 32 channels.  The scoring kernel is launched programmatically dependent on this grid and only its
// epilogue warps wait for it.  (In practice the two kernels do not share an SM although 6.7 KB of shared
// memory would fit beside the scoring CTA, so this kernel is built to be SHORT: all of a warp's W1 rows are
// fetched in one L2 round trip - the scoring CTAs of the 16 SMs it occupies start that much later.)
//   A[q][k]   tri-plane operand of the 4 positions (modules/modules.py:115-118):
//             k = c*8+kk       -> V[c, p, q, kk]   (view x)
//             k = 128+c*8+kk   -> V[c, p, kk, q]   (view y)
//             k = 256+c*8+kk   -> V[c, kk, p, q]   (view z)
//   conv1: warp w owns output rows o = w, w+4, ..., w+28; lanes stride k (coalesced W1 row reads);
//          ReLU -> h1[q][o].
//   conv2 + bias + L2 normalise: warp = position, lane = output channel.
constexpr int kTgtThreads = 128, kTgtCtasPerPair = 16;
__global__ void __launch_bounds__(kTgtThreads, 2)
tc_tgt_feat_kernel(const float* __restrict__ vol_tgt, const float* __restrict__ W1, const float* __restrict__ W2,
                   const float* __restrict__ b2, u64* __restrict__ best_keys, unsigned* __restrict__ done_counter,
                   float* __restrict__ tgt_feat, int B) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // let the scoring kernel start its setup now
  __shared__ float A[4][kK];
  __shared__ float h1[4][kO + 1];
  const int p = blockIdx.x >> 1, q0 = (blockIdx.x & 1) * 4, b = blockIdx.y;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  if (best_keys && blockIdx.x == 0 && t == 0) best_keys[b] = 0ull;
  if (done_counter && blockIdx.x == 0 && b == 0 && t == 32) *done_counter = 0u;
  const float* V = vol_tgt + (size_t)b * kC * kVox;
  float wr[8][12];  // this warp's eight W1 rows: all 96 loads in flight at once (one L2 round trip)
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int j = 0; j < 12; ++j) wr[r][j] = __ldg(W1 + (warp + 4 * r) * kK + lane + 32 * j);
  float4 w2r[kO / 4];  // conv2: this thread's W2 row (lane = output channel), fetched in the same round trip
#pragma unroll
  for (int o = 0; o < kO / 4; ++o) w2r[o] = __ldg(reinterpret_cast<const float4*>(W2 + lane * kO) + o);
  const float bias = __ldg(b2 + lane);
#pragma unroll
  for (int i = 0; i < 4 * kK / kTgtThreads; ++i) {
    const int e = t + kTgtThreads * i;
    const int ql = e / kK, k = e - ql * kK, q = q0 + ql;
    const int view = k >> 7, c = (k >> 3) & 15, kk = k & 7;
    const int d = view == 2 ? kk : p, h = view == 0 ? q : (view == 1 ? kk : p), w = view == 0 ? kk : q;
    A[ql][k] = __ldg(V + c * kVox + d * 64 + h * 8 + w);
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int o = warp + 4 * r;
    float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int j = 0; j < 12; ++j)
#pragma unroll
      for (int ql = 0; ql < 4; ++ql) acc[ql] = fmaf(wr[r][j], A[ql][lane + 32 * j], acc[ql]);
#pragma unroll
    for (int ql = 0; ql < 4; ++ql) {
      const float v = warp_sum(acc[ql]);
      if (lane == ql) h1[ql][o] = fmaxf(v, 0.0f);  // ReLU (modules/modules.py:68)
    }
  }
  __syncthreads();
  {
    const int ql = warp, o2 = lane;  // 4 warps = 4 positions, lanes = output channels
    float v = bias;
#pragma unroll
    for (int o = 0; o < kO; o += 4) {
      const float4 w4 = w2r[o / 4];
      v = fmaf(w4.x, h1[ql][o], v); v = fmaf(w4.y, h1[ql][o + 1], v);
      v = fmaf(w4.z, h1[ql][o + 2], v); v = fmaf(w4.w, h1[ql][o + 3], v);
    }
    const float ss = warp_sum(v * v);
    const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);  // F.normalize eps (modules/modules.py:122)
    tgt_feat[((size_t)b * kO + o2) * kP + p * 8 + q0 + ql] = v * inv;
  }
}

struct Scratch {  // carve-up of the tensor-core path's workspace
  __half* w_packed;
  float2* pair_scale;
  u64* best_keys;
  unsigned* counter;
  float* tgt_feat;
};
__host__ inline size_t scratch_bytes(int B) {
  return (size_t)(kW1Bytes + kW2Bytes) + (size_t)B * (sizeof(float2) + sizeof(u64)) + (size_t)B * kO * kP * 4 + 256;
}
__host__ inline Scratch carve(void* ws, int B) {
  unsigned char* p = static_cast<unsigned char*>(ws);
  Scratch sc;
  sc.w_packed = reinterpret_cast<__half*>(p);
  p += kW1Bytes + kW2Bytes;
  sc.tgt_feat = reinterpret_cast<float*>(p);
  p += (size_t)B * kO * kP * 4;
  sc.pair_scale = reinterpret_cast<float2*>(p);
  p += (size_t)B * sizeof(float2);
  sc.best_keys = reinterpret_cast<u64*>(p);
  sc.counter = reinterpret_cast<unsigned*>(sc.best_keys + B);  // inside the 256-byte tail of scratch_bytes
  return sc;
}

// Tensor map of the source volumes for the TMA staging: [B*16 channels][8 d][64 (h,w)] elements, one box = one
// pair's whole volume (contiguous in HBM; the 3-D form keeps every box dimension <= 256).
static int make_volume_map(const void* vol_src, int B, bool bf16, CUtensorMap* map) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  // the driver's encoder, looked up once (an immutable function pointer, not state)
  static void* const fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      f = nullptr;
    return f;
  }();
  if (!fn) return AHV_ECUDA;
  const cuuint64_t esz = bf16 ? 2 : 4;
  const cuuint64_t dims[3] = {64, 8, (cuuint64_t)B * kC};
  const cuuint64_t strides[2] = {64 * esz, 512 * esz};  // bytes between d slices, between channels
  const cuuint32_t box[3] = {64, 8, (cuuint32_t)kC};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = reinterpret_cast<EncodeFn>(fn)(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                                                    const_cast<void*>(vol_src), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? AHV_OK : AHV_ECUDA;
}

template <typename KernelT, typename... Args>
static int launch_pdl(KernelT kernel, unsigned grid, size_t smem, cudaStream_t s, bool pdl, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreadsTC);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  AHV_CUDA_OK(cudaLaunchKernelEx(&cfg, kernel, args...));
  return AHV_OK;
}

// Launches: [target features + key clear] -> scoring.  The scoring kernel packs the weights and derives
// the per-pair scales itself; when the prologue runs, the scoring kernel is launched programmatically
// dependent on it (its setup, weight packing, volume staging and first gathers overlap the prologue; only
// the epilogue warps wait for the target features).
template <typename T, bool K16, bool kSave = false>
int launch_typed(const T* vol_src, const float* vol_tgt, const float* tgt_feat_in, const float* R,
                 int r_per_pair, const float* W1, const float* W2, const float* b2, const float* base,
                 float* scores, bool want_argmax, int B, int64_t N, const Scratch& sc, Finalize fin, cudaStream_t s,
                 const int* pair_list = nullptr) {
  int dev = 0, sms = 0;
  AHV_CUDA_OK(cudaGetDevice(&dev));
  AHV_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const bool prologue = vol_tgt != nullptr;
  if (prologue) {
    const int st = launch_tgt_feat(vol_tgt, W1, W2, b2, want_argmax ? sc.best_keys : nullptr, sc.tgt_feat, B, s);
    if (st != AHV_OK) return st;
  } else if (want_argmax && !pair_list) {  // a listed-pairs pass adds to the keys (and the cleared counter) it finds
    AHV_CUDA_OK(cudaMemsetAsync(sc.best_keys, 0, (size_t)B * sizeof(u64) + sizeof(unsigned), s));
  }
  fin.counter = sc.counter;
  // a tile is two hypotheses: do not spread tiny problems over more CTAs than tiles
  const int64_t tiles = ((int64_t)B * N + 1) / 2;
  const unsigned grid = (unsigned)(tiles < sms ? tiles : sms);
  if (((int64_t)B * N) / grid >= 0xffffffffLL) return AHV_EINVAL;  // per-CTA tile iterator is 32-bit
  const float* tgt = prologue ? sc.tgt_feat : tgt_feat_in;
  u64* keys = want_argmax ? sc.best_keys : nullptr;
  CUtensorMap vol_map;
  const int mst = make_volume_map(vol_src, B, sizeof(T) == 2, &vol_map);
  if (mst != AHV_OK) return mst;
  AHV_CUDA_OK(cudaFuncSetAttribute(score_tc_ts_kernel<T, K16, kSave>, cudaFuncAttributeMaxDynamicSharedMemorySize, MapTS::smem_bytes));
  // CTAs that inherit the prologue's SMs start late; only worth compensating when the prologue is smaller than this
  // grid and every CTA has tiles to spare (see the work split in the kernel)
  int late = 0;
  if (prologue && kTgtCtasPerPair * (int64_t)B <= grid / 2 && (int64_t)B * N / grid >= 8) late = kTgtCtasPerPair * B;
  return launch_pdl(score_tc_ts_kernel<T, K16, kSave>, grid, MapTS::smem_bytes, s, prologue, vol_map, tgt, R, r_per_pair, b2, base, W1,
                    W2, scores, keys, B, N, fin, late, pair_list);
}

}  // namespace tc

// forward_3d2d for B plain volumes (+ optional clear of B arg-max keys): the fused step's prologue, also
// behind ahv_forward_3d2d for per-pair sizes
int launch_tgt_feat(const float* vol_tgt, const float* W1, const float* W2, const float* b2,
                    unsigned long long* clear_keys, float* feat, int B, cudaStream_t s) {
  // same shared-memory carve-out as the scoring kernel: an SM cannot change its L1/shared split while a CTA
  // is resident, so with the default (small) carve-out the dependent scoring CTAs could not join these SMs
  AHV_CUDA_OK(cudaFuncSetAttribute(tc::tc_tgt_feat_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                   (int)cudaSharedmemCarveoutMaxShared));
  for (int b0 = 0; b0 < B; b0 += 65535) {  // gridDim.y limit
    const int nb = B - b0 < 65535 ? B - b0 : 65535;
    tc::tc_tgt_feat_kernel<<<dim3(tc::kTgtCtasPerPair, nb), tc::kTgtThreads, 0, s>>>(
        vol_tgt + (size_t)b0 * kC * kVox, W1, W2, b2, clear_keys ? clear_keys + b0 : nullptr,
        clear_keys && b0 == 0 ? reinterpret_cast<unsigned*>(clear_keys + B) : nullptr,  // Scratch::counter
        feat + (size_t)b0 * kO * kP, nb);
    AHV_CUDA_OK(cudaGetLastError());
  }
  return AHV_OK;
}

size_t score_tc_workspace_bytes(int B, int64_t N) {
  (void)N;
  return tc::scratch_bytes(B);
}

float* scratch_tgt_feat(void* ws, int B) { return tc::carve(ws, B).tgt_feat; }

// dispatch on (volume dtype, gather precision): bf16 volumes always use the 16-bit staged gather
// (exact staging); fp32 volumes use it only when the caller opts in (AHV_MATH_TC_F16GATHER)
static int dispatch(const void* vol_src, int vol_dtype, bool f16_gather, const float* vol_tgt,
                    const float* tgt_feat, const float* R, int r_per_pair, const float* W1, const float* W2,
                    const float* b2, const float* base, float* scores, bool want_argmax, int B, int64_t N,
                    const tc::Scratch& sc, const tc::Finalize& fin, cudaStream_t s) {
  if (vol_dtype == AHV_VOL_BF16)
    return tc::launch_typed<__nv_bfloat16, true>((const __nv_bfloat16*)vol_src, vol_tgt, tgt_feat, R, r_per_pair, W1,
                                                 W2, b2, base, scores, want_argmax, B, N, sc, fin, s);
  if (f16_gather)
    return tc::launch_typed<float, true>((const float*)vol_src, vol_tgt, tgt_feat, R, r_per_pair, W1, W2, b2, base,
                                         scores, want_argmax, B, N, sc, fin, s);
  return tc::launch_typed<float, false>((const float*)vol_src, vol_tgt, tgt_feat, R, r_per_pair, W1, W2, b2, base,
                                        scores, want_argmax, B, N, sc, fin, s);
}

// scores only (target features supplied by the caller)
int launch_score_tc(const void* vol_src, int vol_dtype, const float* tgt_feat, const float* R,
                    int r_per_pair, const float* W1, const float* W2, const float* b2,
                    const float* base, float* scores, int B, int64_t N, void* ws, size_t ws_bytes,
                    cudaStream_t s, bool f16_gather) {
  if ((int64_t)B * N == 0) return AHV_OK;
  if (ws_bytes < tc::scratch_bytes(B)) return AHV_EWORKSPACE;
  return dispatch(vol_src, vol_dtype, f16_gather, nullptr, tgt_feat, R, r_per_pair, W1, W2, b2, base, scores, false,
                  B, N, tc::carve(ws, B), tc::Finalize{}, s);
}

// training forward (modules/model.py:53-56 before autograd): scores + the ReLU'd conv1 output of every item and the
// pair scales, which ahv_score_backward's saved-activation form reads instead of recomputing conv1
int launch_score_tc_train(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair, const float* W1,
                          const float* W2, const float* b2, const float* base, float* scores, void* h1_out,
                          float* pair_inv_out, int B, int64_t N, void* ws, size_t ws_bytes, cudaStream_t s) {
  if ((int64_t)B * N == 0) return AHV_OK;
  if (ws_bytes < tc::scratch_bytes(B)) return AHV_EWORKSPACE;
  tc::Finalize fin;
  fin.h1_out = static_cast<__half*>(h1_out);
  fin.pair_inv_out = pair_inv_out;
  return tc::launch_typed<float, false, true>(vol_src, nullptr, tgt_feat, R, r_per_pair, W1, W2, b2, base, scores, false, B, N,
                                              tc::carve(ws, B), fin, s);
}

// the fused selection of a k = 1 verification: winners decoded by the scoring kernel's last CTA, or exchanged with the
// peers' kernels when the set is sharded
static int make_finalize(float* best_val, int64_t* best_idx, float* R_best, int64_t idx_offset, int B, const peer::Args* pa,
                         tc::Finalize* fin) {
  fin->val = best_val;
  fin->idx = best_idx;
  fin->R_best = R_best;
  fin->idx_offset = idx_offset;
  if (pa && pa->world > 1) {
    if (pa->world > peer::kMaxPeers || pa->rank < 0 || pa->rank >= pa->world || B > pa->cap_pairs || pa->cap_k < 1)
      return AHV_EINVAL;
    for (int r = 0; r < pa->world; ++r)
      if (!pa->bufs[r]) return AHV_EINVAL;
    fin->peers = *pa;
  }
  return AHV_OK;
}

// the whole verification step with arg-max selection in two launches: prologue (target features, key
// clear) -> fused scoring + arg-max, whose last CTA also decodes the winners (no finalize launch)
int launch_verify_tc_argmax(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R,
                            int r_per_pair, const float* W1, const float* W2, const float* b2,
                            const float* base, float* scores, float* best_val, int64_t* best_idx,
                            float* R_best, int64_t idx_offset, int B, int64_t N, void* ws, size_t ws_bytes,
                            cudaStream_t s, bool f16_gather, const peer::Args* pa) {
  const int world = pa ? pa->world : 1;
  if ((int64_t)B * N == 0) return world > 1 ? AHV_EINVAL : AHV_OK;  // a sharded step needs every rank in the exchange
  if (ws_bytes < tc::scratch_bytes(B)) return AHV_EWORKSPACE;
  tc::Finalize fin;
  const int st = make_finalize(best_val, best_idx, R_best, idx_offset, B, pa, &fin);
  if (st != AHV_OK) return st;
  return dispatch(vol_src, vol_dtype, f16_gather, vol_tgt, nullptr, R, r_per_pair, W1, W2, b2, base, scores, true,
                  B, N, tc::carve(ws, B), fin, s);
}

// The same step for fp32 volumes with the fp32 gather's result, screened by the 16-bit gather (1.6x its rate):
//   pass 1  the 16-bit gather scores every hypothesis into `s16` [B,N]; its arg-max keys give each pair's screened
//           maximum m_b (prologue: target features, key clear);
//   select  per pair the contenders {n : s16[b,n] >= m_b - 2 tau} (at most kScreenCap) and kScreenProbes strided
//           probes; their rotations are copied into s16's space as [B][kScreenList][9] per-pair rotation sets;
//   pass 2  the fp32 gather scores the lists;
//   guard   the list's fp32 arg-max key (original index: ties -> lowest) replaces the pair's screened key; the pair is
//           flagged when some |s32 - s16| on its list exceeds tau / 4, or it had no or too many contenders;
//   pass 3  the fp32 gather scores every hypothesis of the flagged pairs (their number is read on the device: zero
//           items when none), publishes into the same keys, and its last CTA decodes them or runs the exchange.
// A hypothesis's score depends on (pair, rotation) alone, not on the tile or CTA it is scored in, so the fp32 winner is
// the single pass's bit for bit whenever it is on its pair's list - which holds when every 16-bit score lies within
// tau of its fp32 score: then s16[w] >= s32[w] - tau >= s32[n*] - tau >= m_b - 2 tau (n* the screened arg-max).
// `s16` must hold B*N floats and at least kScreenList*40 bytes per pair; `lists` ScreenLists::bytes(B).  No host
// synchronisation: graph-capturable.
int launch_verify_tc_screened(const float* vol_src, const float* vol_tgt, const float* R, int r_per_pair, const float* W1,
                              const float* W2, const float* b2, const float* base, float* best_val, int64_t* best_idx,
                              float* R_best, int64_t idx_offset, int B, int64_t N, void* ws, size_t ws_bytes, float* s16,
                              void* lists, cudaStream_t s, const peer::Args* pa) {
  if (ws_bytes < tc::scratch_bytes(B)) return AHV_EWORKSPACE;
  tc::Finalize fin;
  int st = make_finalize(best_val, best_idx, R_best, idx_offset, B, pa, &fin);
  if (st != AHV_OK) return st;
  const tc::Scratch sc = tc::carve(ws, B);
  const ScreenLists L(lists, B);
  float* R_list = s16;                                          // [B][kScreenList][9], after the selection
  float* s32 = s16 + (size_t)B * kScreenList * 9;               // [B][kScreenList]
  st = tc::launch_typed<float, true>(vol_src, vol_tgt, nullptr, R, r_per_pair, W1, W2, b2, base, s16, true, B, N, sc,
                                     tc::Finalize{}, s);
  if (st != AHV_OK) return st;
  st = launch_screen_select(s16, sc.best_keys, B, N, R, r_per_pair, L, R_list, s);
  if (st != AHV_OK) return st;
  st = tc::launch_typed<float, false>(vol_src, nullptr, sc.tgt_feat, R_list, 1, W1, W2, b2, base, s32, false, B, kScreenList,
                                      sc, tc::Finalize{}, s);
  if (st != AHV_OK) return st;
  st = launch_screen_guard(s32, L, B, sc.best_keys, s);
  if (st != AHV_OK) return st;
  return tc::launch_typed<float, false>(vol_src, nullptr, sc.tgt_feat, R, r_per_pair, W1, W2, b2, base, nullptr, true, B, N,
                                        sc, fin, s, L.flagged);
}

}  // namespace ahv

#ifdef AHV_TIMELINE
extern "C" AHV_API int ahv_diag_timeline(unsigned long long* host_out /*[160][16]*/) {
  return cudaMemcpyFromSymbol(host_out, ahv::tc::g_timeline, sizeof(unsigned long long) * 160 * 16) == cudaSuccess ? AHV_OK : AHV_ECUDA;
}
#endif
