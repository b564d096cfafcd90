// InfoNCE over hypothesis scores (training variant, modules/model.py:43-63 / model_co3d.py:41-61), fused:
//   positives_b = { n : 180/pi * arccos((clamp(<R[b,n], G[b]>, -1, 3) - 1) / 2) <= ACC_THR }          (:46-49)
//   loss_b = -log( sum_{n in positives_b} exp(s[b,n]/T) / max(sum_n exp(s[b,n]/T), 1e-8) )            (:58-61)
// and, in the same launch, d loss_b / d s[b,n] (what autograd would push into the scores):
//   exp(s/T)/T * ( [sum > 1e-8]/sum_all - [n positive]/sum_pos ).
// The reference builds this from ~15 elementwise / reduction launches plus Python lists of index tensors per
// pair; here it is one CTA per pair, two passes over that pair's N scores and rotations.
//
// Arithmetic.  The positive mass sp and the negative mass sn are summed separately in double, in a fixed order
// (per thread, then warp shuffles, then warps in index order): the result is deterministic.  A confident pair, one
// whose positives hold almost all of the softmax mass, must not form a difference of nearly equal terms: with the
// clamp inactive the loss is log1p(sn/sp) and a positive's coefficient is -sn/(sa*sp) (= 1/sa - 1/sp), both in
// double and cast to fp32 once, so they keep fp32 relative accuracy down to losses far below fp32's epsilon.  When
// the clamp is active (sa <= 1e-8) the loss is -log(sp/1e-8) and no gradient flows through the clamped sum.  No
// positive gives +inf and finite gradients, as the reference does; every hypothesis positive gives exactly 0.
// Domain: exp(s/T) is fp32, so |s|/T must stay below ~88 (the reference overflows there too).
#include "ahv_common.cuh"

namespace ahv {

constexpr int kNceThreads = 256;

__device__ __forceinline__ bool nce_positive(const float* __restrict__ r, const float* g, float thr_deg) {
  float dot = 0.0f;
#pragma unroll
  for (int e = 0; e < 9; ++e) dot = fmaf(__ldg(r + e), g[e], dot);
  const float sim = (fminf(fmaxf(dot, -1.0f), 3.0f) - 1.0f) * 0.5f;
  return 180.0f * (acosf(sim) * 0.318309886183790672f) <= thr_deg;  // 180 * arccos(sim) / pi, as the reference writes it
}

__global__ void __launch_bounds__(kNceThreads)
infonce_kernel(const float* __restrict__ scores, const float* __restrict__ R, int r_per_pair,
               const float* __restrict__ gt, float thr_deg, float inv_T, float* __restrict__ loss,
               float* __restrict__ grad, int64_t N) {
  __shared__ double red[2][kNceThreads / 32];
  __shared__ float coef[2];  // d loss / d e for a positive and for a negative hypothesis
  const int b = blockIdx.x, t = threadIdx.x;
  const float* s = scores + (size_t)b * N;
  const float* Rb = R + (r_per_pair ? (size_t)b * N * 9 : 0);
  float g[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) g[e] = __ldg(gt + b * 9 + e);
  double sp = 0.0, sn = 0.0;
  for (int64_t n = t; n < N; n += kNceThreads) {
    const float e = expf(s[n] * inv_T);
    if (nce_positive(Rb + n * 9, g, thr_deg)) sp += e; else sn += e;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sp += __shfl_xor_sync(0xffffffffu, sp, o);
    sn += __shfl_xor_sync(0xffffffffu, sn, o);
  }
  if ((t & 31) == 0) { red[0][t >> 5] = sp; red[1][t >> 5] = sn; }
  __syncthreads();
  if (t == 0) {
    double p = 0.0, q = 0.0;
    for (int w = 0; w < kNceThreads / 32; ++w) { p += red[0][w]; q += red[1][w]; }  // fixed order: deterministic
    const double a = p + q;
    const bool live = (float)a > 1e-8f;                           // .clamp(min=1e-8) (:61) inactive
    loss[b] = (float)(live ? log1p(q / p) : -log(p / 1e-8));     // p == 0: +inf; q == 0 (live): exactly 0
    coef[0] = (float)(live ? -q / (a * p) : -1.0 / p);            // no positive at all: -inf, never used
    coef[1] = live ? (float)(1.0 / a) : 0.0f;
  }
  if (!grad) return;
  __syncthreads();
  const float c_pos = coef[0], c_neg = coef[1];
  float* gb = grad + (size_t)b * N;
  for (int64_t n = t; n < N; n += kNceThreads) {
    const float e = expf(s[n] * inv_T) * inv_T;
    gb[n] = e * (nce_positive(Rb + n * 9, g, thr_deg) ? c_pos : c_neg);
  }
}

int launch_infonce(const float* scores, const float* R, int r_per_pair, const float* gt, float thr_deg, float temperature,
                   float* loss, float* grad, int B, int64_t N, cudaStream_t s) {
  if (B == 0) return AHV_OK;
  infonce_kernel<<<B, kNceThreads, 0, s>>>(scores, R, r_per_pair, gt, thr_deg, 1.0f / temperature, loss, grad, N);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

}  // namespace ahv
