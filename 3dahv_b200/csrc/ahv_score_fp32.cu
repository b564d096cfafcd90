// fp32 CUDA-core kernels of the path (AHV_MATH_FP32 and the refcompat ops).
//
//  * score_fp32_kernel   — fused modules/model.py:186-193: per (pair,
//    hypothesis) trilinear resample (utils.py:113-131) -> tri-plane head
//    (modules/modules.py:112-124) -> cosine vs target -> mean.  Nothing is
//    materialised in HBM except the 4-byte score.
//  * rotate_volume_kernel — utils.py:113-131 materialised (refcompat only).
//  * rotate_volume_bwd_kernel / rotate_volume_grad_R_kernel — its gradients w.r.t. the volume and the
//    rotation (training variant, refcompat under autograd).
//
// Data layout in shared memory (one CTA = 256 threads, 1 CTA / SM):
//   vol   [1000 lines][16 ch] fp32, zero halo          64000 B
//   w1t   [384 k][32 o]      fp32 (W1 transposed)      49152 B
//   rotA  [16 c][8 d][72]    rotated volume, (h,w) rows padded 64->72
//   rotT  [16 c][8 d][72]    same with h<->w swapped (view x reads along h)
//   h1s   [64 pos][36]       ReLU(conv1) rows padded 32->36
//   w2s   [32 rows][36]      W2, row r(o) = (o%8)*4 + o/8
#include "ahv_head_fp32.cuh"

namespace ahv {

// ---- fused scoring kernel ---------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads, 1)
score_fp32_kernel(const T* __restrict__ vol_src, const float* __restrict__ tgt_feat,
                  const float* __restrict__ R, int r_per_pair, const float* __restrict__ W1,
                  const float* __restrict__ W2, const float* __restrict__ b2,
                  const float* __restrict__ base, float* __restrict__ scores, int B, int64_t N) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Fp32Smem& sm = *reinterpret_cast<Fp32Smem*>(smem_raw);
  const int64_t total = (int64_t)B * N;
  const int64_t lo = total * blockIdx.x / gridDim.x, hi = total * (blockIdx.x + 1) / gridDim.x;
  if (lo >= hi) return;
  stage_weights(sm, W1, W2, base);
  const int pos = threadIdx.x >> 2, cg2 = threadIdx.x & 3;
  float b2r[8], tg[8];
#pragma unroll
  for (int oo = 0; oo < 8; ++oo) b2r[oo] = b2[cg2 * 8 + oo];
  int cur_b = -1;
  for (int64_t it = lo; it < hi; ++it) {
    const int b = (int)(it / N);
    const int64_t n = it - (int64_t)b * N;
    if (b != cur_b) {
      __syncthreads();
      stage_volume<T>(sm.vol, vol_src + (size_t)b * kC * kVox);
#pragma unroll
      for (int oo = 0; oo < 8; ++oo) tg[oo] = tgt_feat[((size_t)b * kO + cg2 * 8 + oo) * kP + pos];
      cur_b = b;
    }
    if (threadIdx.x < 9)
      sm.Rcur[threadIdx.x] = R[(r_per_pair ? (size_t)it : (size_t)n) * 9 + threadIdx.x];
    __syncthreads();
    float Rr[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) Rr[e] = sm.Rcur[e];
    gather_hypothesis<false>(sm, Rr, nullptr);
    __syncthreads();
    conv1_relu(sm);
    __syncthreads();
    float v[8];
    conv2_bias(sm, b2r, v);
    float ss, dt;
    head_dots(v, tg, ss, dt);
    mean_cosine(ss, dt, sm.red, scores + it);
  }
}

// ---- rotate_volume materialised (refcompat) --------------------------------
__global__ void __launch_bounds__(kThreads, 1)
rotate_volume_kernel(const float* __restrict__ vol, int per_rot, const float* __restrict__ R,
                     const float* __restrict__ base, float* __restrict__ out, int64_t n,
                     int rot_per_cta) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* svol = reinterpret_cast<float*>(smem_raw);
  float* sbase = svol + kLines * kC;
  float* sR = sbase + 8;
  if (threadIdx.x < 8) sbase[threadIdx.x] = base[threadIdx.x];
  const int64_t first = (int64_t)blockIdx.x * rot_per_cta;
  for (int r = 0; r < rot_per_cta; ++r) {
    const int64_t i = first + r;
    if (i >= n) break;
    if (per_rot || r == 0) {
      __syncthreads();
      stage_volume<float>(svol, vol + (per_rot ? (size_t)i * kC * kVox : 0));
    }
    __syncthreads();
    if (threadIdx.x < 9) sR[threadIdx.x] = R[i * 9 + threadIdx.x];
    __syncthreads();
    float Rr[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) Rr[e] = sR[e];
    // task = (channel quad j, voxel v); consecutive lanes -> consecutive voxels
    for (int task = threadIdx.x; task < 4 * kVox; task += kThreads) {
      const int v = task & 511, j = task >> 9;
      const int d = v >> 6, h = (v >> 3) & 7, w = v & 7;
      Tap t = make_tap(Rr, sbase[w], sbase[h], sbase[d]);
      const float* p = svol + t.line * kC + j * 4;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int dz = 0; dz < 2; ++dz)
#pragma unroll
        for (int dy = 0; dy < 2; ++dy)
#pragma unroll
          for (int dx = 0; dx < 2; ++dx) {
            const float wgt = (dx ? t.fx : 1.0f - t.fx) * (dy ? t.fy : 1.0f - t.fy) *
                              (dz ? t.fz : 1.0f - t.fz);
            const float4 a = *reinterpret_cast<const float4*>(
                p + (dz * kHalo * kHalo + dy * kHalo + dx) * kC);
            acc.x = fmaf(wgt, a.x, acc.x); acc.y = fmaf(wgt, a.y, acc.y);
            acc.z = fmaf(wgt, a.z, acc.z); acc.w = fmaf(wgt, a.w, acc.w);
          }
      float* o = out + ((size_t)i * kC + j * 4) * kVox + v;
      o[0] = acc.x; o[kVox] = acc.y; o[2 * kVox] = acc.z; o[3 * kVox] = acc.w;
    }
  }
}

// ---- rotate_volume backward (training variant, SURVEY.md §8f-3) --------------
// grad_vol += scatter of grad_out through the same 8 trilinear taps the forward used
// (the adjoint of utils.py:113-131 with respect to the volume).  One CTA handles
// `rot_per_cta` rotations; with a shared volume their contributions meet in shared
// memory (ATOMS) and are flushed once per CTA with global atomics.
__global__ void __launch_bounds__(kThreads, 1)
rotate_volume_bwd_kernel(const float* __restrict__ grad_out, int per_rot, const float* __restrict__ R,
                         const float* __restrict__ base, float* __restrict__ grad_vol, int64_t n,
                         int rot_per_cta) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* acc = reinterpret_cast<float*>(smem_raw);  // [1000 lines][16 ch] halo'd like the forward volume
  float* sbase = acc + kLines * kC;
  float* sR = sbase + 8;
  if (threadIdx.x < 8) sbase[threadIdx.x] = base[threadIdx.x];
  const int64_t first = (int64_t)blockIdx.x * rot_per_cta;
  for (int r = 0; r < rot_per_cta; ++r) {
    const int64_t i = first + r;
    if (i >= n) break;
    if (per_rot || r == 0) {
      __syncthreads();
      for (int e = threadIdx.x; e < kLines * kC; e += kThreads) acc[e] = 0.0f;
    }
    __syncthreads();
    if (threadIdx.x < 9) sR[threadIdx.x] = R[i * 9 + threadIdx.x];
    __syncthreads();
    float Rr[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) Rr[e] = sR[e];
    for (int task = threadIdx.x; task < 4 * kVox; task += kThreads) {
      const int v = task & 511, j = task >> 9;
      const int d = v >> 6, h = (v >> 3) & 7, w = v & 7;
      Tap t = make_tap(Rr, sbase[w], sbase[h], sbase[d]);
      const float* go = grad_out + ((size_t)i * kC + j * 4) * kVox + v;
      const float g0 = go[0], g1 = go[kVox], g2 = go[2 * kVox], g3 = go[3 * kVox];
      float* p = acc + t.line * kC + j * 4;
#pragma unroll
      for (int dz = 0; dz < 2; ++dz)
#pragma unroll
        for (int dy = 0; dy < 2; ++dy)
#pragma unroll
          for (int dx = 0; dx < 2; ++dx) {
            const float wgt = (dx ? t.fx : 1.0f - t.fx) * (dy ? t.fy : 1.0f - t.fy) * (dz ? t.fz : 1.0f - t.fz);
            float* q = p + (dz * kHalo * kHalo + dy * kHalo + dx) * kC;
            atomicAdd(q + 0, wgt * g0); atomicAdd(q + 1, wgt * g1);
            atomicAdd(q + 2, wgt * g2); atomicAdd(q + 3, wgt * g3);
          }
    }
    const bool flush = per_rot || r == rot_per_cta - 1 || i + 1 >= n;
    if (flush) {
      __syncthreads();
      float* gv = grad_vol + (per_rot ? (size_t)i * kC * kVox : 0);
      for (int e = threadIdx.x; e < kC * kVox; e += kThreads) {
        const int c = e >> 9, v = e & 511;
        const int z = v >> 6, y = (v >> 3) & 7, x = v & 7;
        const float val = acc[(((z + 1) * kHalo + (y + 1)) * kHalo + (x + 1)) * kC + c];  // halo lines are discarded
        if (per_rot) gv[e] = val;
        else if (val != 0.0f) atomicAdd(gv + e, val);
      }
    }
  }
}

int launch_rotate_volume_bwd(const float* grad_out, int per_rot, const float* R, const float* base,
                             float* grad_vol, int64_t n, cudaStream_t s) {
  if (n == 0) return AHV_OK;
  const int rpc = per_rot ? 1 : 8;
  const int64_t grid = (n + rpc - 1) / rpc;
  const size_t smem = (kLines * kC + 8 + 12) * sizeof(float);
  AHV_CUDA_OK(cudaFuncSetAttribute(rotate_volume_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  rotate_volume_bwd_kernel<<<(unsigned)grid, kThreads, smem, s>>>(grad_out, per_rot, R, base, grad_vol, n, rpc);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

// ---- rotate_volume gradient with respect to the rotation ---------------------
// grad_R[i] = dL/dR_i of out = rotate_volume(vol, R) given grad_out = dL/dout (rot_grad_accum, the same
// formula as the fused backward's rotation phase).  The source volume is staged with its zero halo once per
// CTA (shared) or once per rotation; one CTA handles `rot_per_cta` rotations and overwrites their grad_R.
__global__ void __launch_bounds__(kThreads, 1)
rotate_volume_grad_R_kernel(const float* __restrict__ vol, int per_rot, const float* __restrict__ R,
                            const float* __restrict__ base, const float* __restrict__ grad_out,
                            float* __restrict__ grad_R, int64_t n, int rot_per_cta) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* svol = reinterpret_cast<float*>(smem_raw);
  float* sbase = svol + kLines * kC;
  float* sR = sbase + 8;
  float* red = sR + 12;  // [8 warps][9]
  if (threadIdx.x < 8) sbase[threadIdx.x] = base[threadIdx.x];
  const int64_t first = (int64_t)blockIdx.x * rot_per_cta;
  for (int r = 0; r < rot_per_cta; ++r) {
    const int64_t i = first + r;
    if (i >= n) break;
    if (per_rot || r == 0) {
      __syncthreads();
      stage_volume<float>(svol, vol + (per_rot ? (size_t)i * kC * kVox : 0));
    }
    __syncthreads();
    if (threadIdx.x < 9) sR[threadIdx.x] = R[i * 9 + threadIdx.x];
    __syncthreads();
    float Rr[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) Rr[e] = sR[e];
    float G[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) G[e] = 0.0f;
    // task = (channel quad j, voxel v); consecutive lanes -> consecutive voxels (coalesced grad_out)
    for (int task = threadIdx.x; task < 4 * kVox; task += kThreads) {
      const int v = task & 511, j = task >> 9;
      const int d = v >> 6, h = (v >> 3) & 7, w = v & 7;
      const float* go = grad_out + ((size_t)i * kC + j * 4) * kVox + v;
      rot_grad_accum(svol, Rr, sbase[w], sbase[h], sbase[d], j, make_float4(go[0], go[kVox], go[2 * kVox], go[3 * kVox]), G);
    }
    const float s = block_sum9(G, red, 4.0f);
    if (threadIdx.x < 9) grad_R[i * 9 + threadIdx.x] = s;
  }
}

int launch_rotate_volume_grad_R(const float* vol, int per_rot, const float* R, const float* base, const float* grad_out,
                                float* grad_R, int64_t n, cudaStream_t s) {
  if (n == 0) return AHV_OK;
  const int rpc = per_rot ? 1 : 8;
  const int64_t grid = (n + rpc - 1) / rpc;
  const size_t smem = (kLines * kC + 8 + 12 + 72) * sizeof(float);
  AHV_CUDA_OK(cudaFuncSetAttribute(rotate_volume_grad_R_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  rotate_volume_grad_R_kernel<<<(unsigned)grid, kThreads, smem, s>>>(vol, per_rot, R, base, grad_out, grad_R, n, rpc);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

// ---- launchers --------------------------------------------------------------

int launch_score_fp32(const Scored& p, const float* tgt_feat, float* scores, cudaStream_t s) {
  const int64_t total = (int64_t)p.B * p.N;
  if (total == 0) return AHV_OK;
  const int sms = sm_count();
  if (sms <= 0) return AHV_ECUDA;
  const unsigned grid = (unsigned)(total < sms ? total : sms);
  const size_t smem = sizeof(Fp32Smem);
  if (p.vol_dtype == AHV_VOL_F32) {
    AHV_CUDA_OK(cudaFuncSetAttribute(score_fp32_kernel<float>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    score_fp32_kernel<float><<<grid, kThreads, smem, s>>>(p.vol_f32(), tgt_feat, p.R, p.r_per_pair, p.W1, p.W2, p.b2,
                                                          p.base, scores, p.B, p.N);
  } else {
    AHV_CUDA_OK(cudaFuncSetAttribute(score_fp32_kernel<__nv_bfloat16>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    score_fp32_kernel<__nv_bfloat16><<<grid, kThreads, smem, s>>>(
        (const __nv_bfloat16*)p.vol_src, tgt_feat, p.R, p.r_per_pair, p.W1, p.W2, p.b2, p.base, scores, p.B, p.N);
  }
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

int launch_forward_3d2d(const float* vol, const float* W1, const float* W2, const float* b2,
                        float* feat, int64_t m, cudaStream_t s) {
  // every target feature comes from the fused step's prologue kernel, whatever m is, so ahv_score (caller-computed
  // target features), ahv_verify and the refine / search chains agree bit for bit at every batch size
  constexpr int64_t kChunk = 1 << 30;  // launch_tgt_feat counts volumes in an int
  for (int64_t m0 = 0; m0 < m; m0 += kChunk) {
    const int st = launch_tgt_feat(vol + (size_t)m0 * kC * kVox, W1, W2, b2, nullptr, feat + (size_t)m0 * kO * kP,
                                   (int)(m - m0 < kChunk ? m - m0 : kChunk), s);
    if (st != AHV_OK) return st;
  }
  return AHV_OK;
}

int launch_rotate_volume(const float* vol, int per_rot, const float* R, const float* base,
                         float* out, int64_t n, cudaStream_t s) {
  if (n == 0) return AHV_OK;
  const int rpc = per_rot ? 1 : 8;
  const int64_t grid = (n + rpc - 1) / rpc;
  const size_t smem = (kLines * kC + 8 + 12) * sizeof(float);
  AHV_CUDA_OK(cudaFuncSetAttribute(rotate_volume_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)smem));
  rotate_volume_kernel<<<(unsigned)grid, kThreads, smem, s>>>(vol, per_rot, R, base, out, n, rpc);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

}  // namespace ahv
