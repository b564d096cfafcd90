// Gradient ascent of the AHV_MATH_FP32 score on SO(3) (ahv_gradient_ascent; extension, DESIGN.md §4.4).
//
// The algorithm of HypothesisVerifier.refine_gradient (verify.py), which stays as its torch-op restatement, in one
// kernel: backtracking Riemannian gradient ascent from given rotations, a fixed number of steps, each candidate on its
// own.  A candidate's step t+1 depends only on its step t, so one CTA runs every step of an item before it moves on to
// the next - no grid-wide synchronisation, no host step.  Per item:
//
//   evaluation 0   s = S(R), G = dS/dR at R_init (the fused backward's dH2 -> dH1 -> dA fold -> rotation phase)
//   every step     one thread: M = G R^T, w = (M21 - M12, M02 - M20, M10 - M01), u = w / max(|w|, 1e-30),
//                  R~ = (I + sin(th) [u]x + (1 - cos(th)) [u]x^2) R, then R~ <- 1.5 R~ - 0.5 R~ R~^T R~ (one Newton step)
//                  s~ = S(R~) with the fp32 scorer's arithmetic and reduction order (bit-identical scores)
//                  s~ > s: the backward half at R~ for G~; R, s, G <- R~, s~, G~; th *= 1.2
//                  else:   th /= 2, and no backward at all
//
// Only dS/dR is formed: no weight, target or volume gradient, no adjoint of the resampling, no atomics - the result is
// bit-deterministic.  One CTA = 256 threads, 1 CTA / SM, contiguous range of (pair, candidate) items; the pair's
// halo'd volume, target features and the weights are staged once per pair.
#include "ahv_bwd_fp32.cuh"

namespace ahv {

struct AscentSmem {
  Fp32Smem f;               // f.Rcur: the rotation being scored (R_init, then each trial)
  float dh2[kP * kH1Row];   // dL/dH2 [pos][36]; the rotation phase's partial sums once dH1 is formed
  float R[9];               // the item's current rotation
  float G[9];               // dS/dR at R
  float s;                  // the score just computed (thread 0 -> every thread)
};
static_assert(sizeof(AscentSmem) <= 232448, "shared memory budget");

// The trial rotation of one step from R, G = dS/dR and the step angle theta (verify.py, refine_gradient's loop body).
__device__ __forceinline__ void trial_rotation(const float* R, const float* G, float theta, float* out) {
  float M[9];  // G R^T: <G, [e_i]x R> = <G R^T, [e_i]x>
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) M[i * 3 + j] = G[i * 3] * R[j * 3] + G[i * 3 + 1] * R[j * 3 + 1] + G[i * 3 + 2] * R[j * 3 + 2];
  const float w0 = M[7] - M[5], w1 = M[2] - M[6], w2 = M[3] - M[1];
  const float nw = fmaxf(sqrtf(w0 * w0 + w1 * w1 + w2 * w2), 1e-30f);
  const float u0 = w0 / nw, u1 = w1 / nw, u2 = w2 / nw;
  const float K[9] = {0.0f, -u2, u1, u2, 0.0f, -u0, -u1, u0, 0.0f};
  const float sn = sinf(theta), cs = 1.0f - cosf(theta);
  float D[9];  // I + sin(theta) K + (1 - cos(theta)) K^2
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const float kk = K[i * 3] * K[j] + K[i * 3 + 1] * K[3 + j] + K[i * 3 + 2] * K[6 + j];
      D[i * 3 + j] = ((i == j ? 1.0f : 0.0f) + sn * K[i * 3 + j]) + cs * kk;
    }
  float T[9];  // D R
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) T[i * 3 + j] = D[i * 3] * R[j] + D[i * 3 + 1] * R[3 + j] + D[i * 3 + 2] * R[6 + j];
  float P[9];  // T T^T
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) P[i * 3 + j] = T[i * 3] * T[j * 3] + T[i * 3 + 1] * T[j * 3 + 1] + T[i * 3 + 2] * T[j * 3 + 2];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {   // one Newton step towards the nearest rotation: 1.5 T - 0.5 (T T^T) T
      const float q = P[i * 3] * T[j] + P[i * 3 + 1] * T[3 + j] + P[i * 3 + 2] * T[6 + j];
      out[i * 3 + j] = 1.5f * T[i * 3 + j] - 0.5f * q;
    }
}

// kItemRange: the grid covers items [item_lo, item_hi) of the B*K only (one rank's share in
// ahv_refine_gradient_sharded); without it the range is [0, B*K) and the arguments are unused.
template <typename T, bool kItemRange>
__global__ void __launch_bounds__(kThreads, 1)
ascent_fp32_kernel(const T* __restrict__ vol_src, const float* __restrict__ tgt_feat, const float* __restrict__ R_init,
                   const float* __restrict__ W1, const float* __restrict__ W2, const float* __restrict__ b2,
                   const float* __restrict__ base, int steps, float theta0, float* __restrict__ R_out,
                   float* __restrict__ score_out, int B, int K, const int64_t* __restrict__ skip_idx,
                   int64_t item_lo, int64_t item_hi) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  AscentSmem& as = *reinterpret_cast<AscentSmem*>(smem_raw);
  Fp32Smem& sm = as.f;
  const int64_t first = kItemRange ? item_lo : 0;
  const int64_t total = kItemRange ? item_hi - item_lo : (int64_t)B * K;
  const int64_t lo = first + total * blockIdx.x / gridDim.x, hi = first + total * (blockIdx.x + 1) / gridDim.x;
  if (lo >= hi) return;
  const int t = threadIdx.x;
  stage_weights(sm, W1, W2, base);
  const int pos = t >> 2, cg2 = t & 3;
  float b2r[8], tg[8];
#pragma unroll
  for (int oo = 0; oo < 8; ++oo) b2r[oo] = b2[cg2 * 8 + oo];
  int cur_b = -1;
  for (int64_t it = lo; it < hi; ++it) {
    const int b = (int)(it / K);
    __syncthreads();  // the previous item is done with the volume, R and Rcur
    if (skip_idx && skip_idx[it] < 0) {  // an empty selection slot (ahv_refine_gradient_distinct): nothing to ascend
      if (t < 9) R_out[(size_t)it * 9 + t] = nanf("");
      if (t == 0) score_out[it] = -INFINITY;
      continue;
    }
    if (b != cur_b) {
      stage_volume<T>(sm.vol, vol_src + (size_t)b * kC * kVox);
#pragma unroll
      for (int oo = 0; oo < 8; ++oo) tg[oo] = tgt_feat[((size_t)b * kO + cg2 * 8 + oo) * kP + pos];
      cur_b = b;
    }
    if (t < 9) as.R[t] = sm.Rcur[t] = R_init[(size_t)it * 9 + t];
    float s = 0.0f, theta = theta0;  // the same in every thread: the branches below are block-uniform
#pragma unroll 1
    for (int step = 0; step <= steps; ++step) {  // evaluation 0 at R_init, then one per trial
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
      mean_cosine(ss, dt, sm.red, &as.s);
      __syncthreads();
      const float st = as.s;
      const bool accept = step == 0 || st > s;
      if (step > 0) theta = accept ? theta * 1.2f : theta * 0.5f;
      if (!accept) {  // every thread read Rcur before the gather's __syncthreads
        if (step < steps && t == 0) trial_rotation(as.R, as.G, theta, sm.Rcur);
        continue;
      }
      s = st;
      if (step < steps) {  // G at the accepted rotation, for the next trial: the backward half for g = 1
        head_dh2(v, tg, ss, dt, 1.0f / 64.0f, as.dh2, [](int, float, float) {});
        __syncthreads();
        head_dh1(sm, as.dh2, pos, cg2);
        fold_dA(sm, t);
        const float g = rotation_grad(sm, as.dh2, t);
        if (t < 9) {
          as.G[t] = g;
          as.R[t] = sm.Rcur[t];
        }
        __syncthreads();
        if (t == 0) trial_rotation(as.R, as.G, theta, sm.Rcur);
      } else if (t < 9) {
        as.R[t] = sm.Rcur[t];
      }
    }
    if (t < 9) R_out[(size_t)it * 9 + t] = as.R[t];
    if (t == 0) score_out[it] = s;
  }
}

template <bool kItemRange>
void launch_ascent(const Scored& p, const float* tgt_feat, int steps, float theta0, float* R_out, float* score_out,
                   const int64_t* skip_idx, int64_t item_lo, int64_t item_hi, unsigned grid, size_t smem, cudaStream_t s,
                   cudaError_t* err) {
  const int K = (int)p.N;
  if (p.vol_dtype == AHV_VOL_F32) {
    *err = cudaFuncSetAttribute(ascent_fp32_kernel<float, kItemRange>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (*err != cudaSuccess) return;
    ascent_fp32_kernel<float, kItemRange><<<grid, kThreads, smem, s>>>(p.vol_f32(), tgt_feat, p.R, p.W1, p.W2, p.b2, p.base,
                                                                       steps, theta0, R_out, score_out, p.B, K, skip_idx,
                                                                       item_lo, item_hi);
  } else {
    *err = cudaFuncSetAttribute(ascent_fp32_kernel<__nv_bfloat16, kItemRange>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)smem);
    if (*err != cudaSuccess) return;
    ascent_fp32_kernel<__nv_bfloat16, kItemRange><<<grid, kThreads, smem, s>>>((const __nv_bfloat16*)p.vol_src, tgt_feat, p.R,
                                                                               p.W1, p.W2, p.b2, p.base, steps, theta0, R_out,
                                                                               score_out, p.B, K, skip_idx, item_lo, item_hi);
  }
  *err = cudaGetLastError();
}

int launch_gradient_ascent(const Scored& p, const float* tgt_feat, int steps, float step_deg, float* R_out,
                           float* score_out, cudaStream_t s, const int64_t* skip_idx, int64_t item_lo, int64_t item_hi) {
  const bool ranged = item_hi >= 0;
  const int64_t total = ranged ? item_hi - item_lo : (int64_t)p.B * p.N;
  if (total <= 0) return AHV_OK;
  int dev = 0, sms = 0;
  AHV_CUDA_OK(cudaGetDevice(&dev));
  AHV_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const unsigned grid = (unsigned)(total < sms ? total : sms);
  const size_t smem = sizeof(AscentSmem);
  const float theta0 = (float)((double)step_deg * (3.14159265358979323846 / 180.0));  // math.radians, rounded once
  cudaError_t err = cudaSuccess;
  if (ranged)
    launch_ascent<true>(p, tgt_feat, steps, theta0, R_out, score_out, skip_idx, item_lo, item_hi, grid, smem, s, &err);
  else
    launch_ascent<false>(p, tgt_feat, steps, theta0, R_out, score_out, skip_idx, 0, 0, grid, smem, s, &err);
  AHV_CUDA_OK(err);
  return AHV_OK;
}

int preload_ranged_ascent() {
  cudaFuncAttributes a;
  AHV_CUDA_OK(cudaFuncGetAttributes(&a, ascent_fp32_kernel<float, true>));
  AHV_CUDA_OK(cudaFuncGetAttributes(&a, ascent_fp32_kernel<__nv_bfloat16, true>));
  return AHV_OK;
}

}  // namespace ahv
