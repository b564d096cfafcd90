// fp32 CUDA-core building blocks of the verification head (modules/modules.py:112-124),
// shared by the AHV_MATH_FP32 scorer, ahv_forward_3d2d and the tensor-core path's prologue
// (target features).  Shared-memory layout: see ahv_score_fp32.cu.
#pragma once
#include "ahv_common.cuh"

namespace ahv {

constexpr int kThreads = 256;
constexpr int kRotD = 72;          // padded (h,w) plane
constexpr int kRotC = kS * kRotD;  // 576 floats per channel
constexpr int kH1Row = 36;
constexpr int kW1Pitch = 34;         // transposed W1 rows padded 32 -> 34 floats: coalesced staging, conflict-free float2 reads

struct Fp32Smem {
  float vol[kLines * kC];
  float w1t[kK * kW1Pitch];
  float rotA[kC * kRotC];
  float rotT[kC * kRotC];
  float h1s[kP * kH1Row];
  float w2s[kO * kH1Row];
  float base[8];
  float red[8];
  float Rcur[12];
};

// ---- staging -------------------------------------------------------------
__device__ __forceinline__ void stage_weights(Fp32Smem& sm, const float* __restrict__ W1,
                                              const float* __restrict__ W2,
                                              const float* __restrict__ base) {
  for (int i = threadIdx.x; i < kO * kK; i += kThreads) {
    const int o = i / kK, k = i - o * kK;  // coalesced read of W1[o][k]; store banks (2k + o) mod 32: 2-way at worst
    sm.w1t[k * kW1Pitch + o] = __ldg(W1 + i);
  }
  for (int i = threadIdx.x; i < kO * kO; i += kThreads) {
    int o = i / kO, c = i % kO;
    sm.w2s[((o % 8) * 4 + o / 8) * kH1Row + c] = W2[i];
  }
  if (threadIdx.x < 8) sm.base[threadIdx.x] = base ? base[threadIdx.x] : 0.0f;
}

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

// vol_g: [16][512] NCDHW -> halo'd, channel-innermost lines
template <typename T>
__device__ __forceinline__ void stage_volume(float* __restrict__ vol, const T* __restrict__ vol_g) {
  for (int i = threadIdx.x; i < kLines * kC; i += kThreads) vol[i] = 0.0f;
  __syncthreads();
  for (int i = threadIdx.x; i < kC * kVox; i += kThreads) {
    int c = i >> 9, v = i & 511;
    int z = v >> 6, y = (v >> 3) & 7, x = v & 7;
    int line = ((z + 1) * kHalo + (y + 1)) * kHalo + (x + 1);
    vol[line * kC + c] = to_f32<T>(vol_g[i]);
  }
}

// plain (un-rotated) volume [16][512] -> rotA / rotT (forward_3d2d on its own)
template <typename T>
__device__ __forceinline__ void load_plain_volume(Fp32Smem& sm, const T* __restrict__ vol_g) {
  for (int i = threadIdx.x; i < kC * kVox; i += kThreads) {
    int c = i >> 9, v = i & 511;
    int d = v >> 6, h = (v >> 3) & 7, w = v & 7;
    float x = to_f32<T>(vol_g[i]);
    sm.rotA[c * kRotC + d * kRotD + h * 8 + w] = x;
    sm.rotT[c * kRotC + d * kRotD + w * 8 + h] = x;
  }
}

// ---- phase G: trilinear gather of one hypothesis into rotA / rotT ---------
// 4 lanes per output voxel (4 channels each), 8 voxels per warp step.
// kRecord: lane j==0 of every voxel also stores the voxel's tap (corner line, fractions) to taps[v] - the
// backward kernel's adjoint gather re-uses them so that its weights are the forward's bit for bit.
template <bool kRecord>
__device__ __forceinline__ void gather_hypothesis(Fp32Smem& sm, const float* R, float4* taps) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = lane & 3, q = lane >> 2;
#pragma unroll 1
  for (int it = 0; it < 8; ++it) {
    const int s = it * 8 + warp;  // (d,h) slab
    const int d = s >> 3, h = s & 7, w = q;
    Tap t = make_tap(R, sm.base[w], sm.base[h], sm.base[d]);
    if (kRecord && j == 0) taps[d * 64 + h * 8 + w] = make_float4(__int_as_float(t.line), t.fx, t.fy, t.fz);
    // Two voxels share a 128-bit shared-memory phase (8 lanes).  Their x-taps
    // sit in adjacent 64 B lines of opposite bank halves; issuing them in
    // parity order makes every phase conflict-free.
    const int swap = (t.line ^ q) & 1;
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
    const int oa = d * kRotD + h * 8 + w, ot = d * kRotD + w * 8 + h;
    const int c0 = j * 4;
    sm.rotA[(c0 + 0) * kRotC + oa] = acc.x; sm.rotT[(c0 + 0) * kRotC + ot] = acc.x;
    sm.rotA[(c0 + 1) * kRotC + oa] = acc.y; sm.rotT[(c0 + 1) * kRotC + ot] = acc.y;
    sm.rotA[(c0 + 2) * kRotC + oa] = acc.z; sm.rotT[(c0 + 2) * kRotC + ot] = acc.z;
    sm.rotA[(c0 + 3) * kRotC + oa] = acc.w; sm.rotT[(c0 + 3) * kRotC + ot] = acc.w;
  }
}

// ---- phase C1: tri-plane conv 384->32 + ReLU -> h1s ------------------------
// h1[o,p,q] = sum_{c,k} W1[o,c*8+k] V[c,p,q,k] + W1[o,128+c*8+k] V[c,p,k,q]
//                     + W1[o,256+c*8+k] V[c,k,p,q]      (modules/modules.py:115-118)
// thread tile: 4 positions (p, q0..q0+3) x 2 channels.
__device__ __forceinline__ void conv1_relu(Fp32Smem& sm) {
  const int cg = threadIdx.x & 15, pg = threadIdx.x >> 4;
  const int p = pg >> 1, q0 = (pg & 1) * 4;
  float acc[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = 0.0f;
  const float* wbase = sm.w1t + 2 * cg;
#pragma unroll 1
  for (int view = 0; view < 3; ++view) {
    const float* a0 = (view == 0 ? sm.rotT : sm.rotA) + (view == 2 ? p * 8 + q0 : p * kRotD + q0);
    const int kstride = (view == 2) ? kRotD : 8;
#pragma unroll 2
    for (int c = 0; c < kC; ++c) {
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const float4 a = *reinterpret_cast<const float4*>(a0 + c * kRotC + kk * kstride);
        const float2 w = *reinterpret_cast<const float2*>(wbase + (view * 128 + c * 8 + kk) * kW1Pitch);
        acc[0][0] = fmaf(a.x, w.x, acc[0][0]); acc[0][1] = fmaf(a.x, w.y, acc[0][1]);
        acc[1][0] = fmaf(a.y, w.x, acc[1][0]); acc[1][1] = fmaf(a.y, w.y, acc[1][1]);
        acc[2][0] = fmaf(a.z, w.x, acc[2][0]); acc[2][1] = fmaf(a.z, w.y, acc[2][1]);
        acc[3][0] = fmaf(a.w, w.x, acc[3][0]); acc[3][1] = fmaf(a.w, w.y, acc[3][1]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 r = make_float2(fmaxf(acc[i][0], 0.0f), fmaxf(acc[i][1], 0.0f));
    *reinterpret_cast<float2*>(sm.h1s + (p * 8 + q0 + i) * kH1Row + 2 * cg) = r;
  }
}

// ---- phase C2: conv 32->32 + bias; thread = (position, 8 output channels) --
__device__ __forceinline__ void conv2_bias(const Fp32Smem& sm, const float* b2r, float* v) {
  const int pos = threadIdx.x >> 2, cg2 = threadIdx.x & 3;
  float h[kO];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float4 t = *reinterpret_cast<const float4*>(sm.h1s + pos * kH1Row + 4 * i);
    h[4 * i] = t.x; h[4 * i + 1] = t.y; h[4 * i + 2] = t.z; h[4 * i + 3] = t.w;
  }
#pragma unroll
  for (int oo = 0; oo < 8; ++oo) {
    const float* wr = sm.w2s + (oo * 4 + cg2) * kH1Row;
    float a = 0.0f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float4 w = *reinterpret_cast<const float4*>(wr + 4 * i);
      a = fmaf(w.x, h[4 * i], a); a = fmaf(w.y, h[4 * i + 1], a);
      a = fmaf(w.z, h[4 * i + 2], a); a = fmaf(w.w, h[4 * i + 3], a);
    }
    v[oo] = a + b2r[oo];
  }
}

// ---- rotation gradient of the trilinear resampling (utils.py:113-131 differentiated in its grid) -----------
// Output voxel X[c] = trilinear(V[c], i) at i = (ix, iy, iz) = 4 (R b) + 3.5 (sample_coords), b = (base[w], base[h],
// base[d]).  Given the upstream gradient gx4 = dL/dX[4j .. 4j+3] this adds sum_c dL/dX[c] dX[c]/di (x) b to G (3x3,
// row-major); dL/dR = 4 G once summed over voxels and channel quads.  ATen's grid_sampler_3d_backward convention: the
// corner is floor(i) (forward difference at an exact integer), a tap outside the volume reads the zero halo, and the
// derivative along an axis is zero unless -1 <= i < 8 on that axis, tested on the unclamped coordinate (tap_at clamps
// to [-1, 8] and caps the corner at 7, which would otherwise turn it into -V[7] or V[0]).  `vol` is the halo'd
// shared-memory volume of stage_volume.
__device__ __forceinline__ void rot_grad_accum(const float* vol, const float* R, float bx, float by, float bz, int j,
                                               float4 gx4, float (&G)[9]) {
  const float3 u = sample_coords(R, bx, by, bz);
  const Tap t = tap_at(u);
  const float* p = vol + t.line * kC + j * 4;
  float dx = 0.0f, dy = 0.0f, dz = 0.0f;
#pragma unroll
  for (int k = 0; k < 8; ++k) {  // corner (ex, ey, ez) = (k & 1, (k >> 1) & 1, k >> 2)
    const int ex = k & 1, ey = (k >> 1) & 1, ez = k >> 2;
    const float4 a = *reinterpret_cast<const float4*>(p + (ez * kHalo * kHalo + ey * kHalo + ex) * kC);
    const float cv = fmaf(gx4.w, a.w, fmaf(gx4.z, a.z, fmaf(gx4.y, a.y, gx4.x * a.x)));   // <dL/dX, V[corner]>
    const float wx = ex ? t.fx : 1.0f - t.fx, wy = ey ? t.fy : 1.0f - t.fy, wz = ez ? t.fz : 1.0f - t.fz;
    dx = fmaf(ex ? cv : -cv, wy * wz, dx);
    dy = fmaf(ey ? cv : -cv, wx * wz, dy);
    dz = fmaf(ez ? cv : -cv, wx * wy, dz);
  }
  dx = (u.x >= -1.0f && u.x < 8.0f) ? dx : 0.0f;
  dy = (u.y >= -1.0f && u.y < 8.0f) ? dy : 0.0f;
  dz = (u.z >= -1.0f && u.z < 8.0f) ? dz : 0.0f;
  G[0] = fmaf(dx, bx, G[0]); G[1] = fmaf(dx, by, G[1]); G[2] = fmaf(dx, bz, G[2]);
  G[3] = fmaf(dy, bx, G[3]); G[4] = fmaf(dy, by, G[4]); G[5] = fmaf(dy, bz, G[5]);
  G[6] = fmaf(dz, bx, G[6]); G[7] = fmaf(dz, by, G[7]); G[8] = fmaf(dz, bz, G[8]);
}

// CTA-wide sum of the 9 accumulators, times `scale`, returned in threads 0..8 (element threadIdx.x); red: 72 floats of
// shared memory.  One __syncthreads; the caller synchronises before red is written again.
__device__ __forceinline__ float block_sum9(float (&G)[9], float* red, float scale) {
#pragma unroll
  for (int e = 0; e < 9; ++e) G[e] = warp_sum(G[e]);
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int e = 0; e < 9; ++e) red[(threadIdx.x >> 5) * 9 + e] = G[e];
  }
  __syncthreads();
  float s = 0.0f;
  if (threadIdx.x < 9) {
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) s += red[w * 9 + threadIdx.x];
  }
  return s * scale;
}

__device__ __forceinline__ float quad_sum(float x) {
  x += __shfl_xor_sync(0xffffffffu, x, 1);
  x += __shfl_xor_sync(0xffffffffu, x, 2);
  return x;
}

// ---- the score of one hypothesis: mean over the 64 positions of <F_p, T_p>, F = H2 / max(|H2|, 1e-12) --------
// ss = |H2_p|^2 and dt = <H2_p, T_p> over the 32 channels of this thread's position (the 4 lanes of its quad), from
// conv2_bias' v and the thread's target features tg.
__device__ __forceinline__ void head_dots(const float (&v)[8], const float (&tg)[8], float& ss, float& dt) {
  ss = 0.0f;
  dt = 0.0f;
#pragma unroll
  for (int oo = 0; oo < 8; ++oo) { ss = fmaf(v[oo], v[oo], ss); dt = fmaf(v[oo], tg[oo], dt); }
  ss = quad_sum(ss);
  dt = quad_sum(dt);
}

// F.normalize: v / max(||v||, 1e-12); then <.,tgt> summed over channels, .mean(dim=-1) over the 64 positions.  Thread 0
// stores the score to *out; red: the 8 floats of sm.red.  One __syncthreads.  The fp32 scorer and the gradient ascent
// both score through here, so their scores agree bit for bit.
__device__ __forceinline__ void mean_cosine(float ss, float dt, float* red, float* out) {
  float cosv = ((threadIdx.x & 3) == 0) ? dt / fmaxf(sqrtf(ss), 1e-12f) : 0.0f;
  cosv = warp_sum(cosv);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = cosv;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.0f;
#pragma unroll
    for (int w = 0; w < 8; ++w) tot += red[w];
    *out = tot * (1.0f / 64.0f);
  }
}


// One volume -> normalised features [32][64] (feat[o*64 + pos]); all 256 threads of the CTA.
// Caller has staged the weights (stage_weights) and synchronised.
template <typename T>
__device__ __forceinline__ void forward_3d2d_block(Fp32Smem& sm, const T* __restrict__ vol_g,
                                                   const float* b2r, float* __restrict__ feat_out) {
  const int pos = threadIdx.x >> 2, cg2 = threadIdx.x & 3;
  __syncthreads();
  load_plain_volume<T>(sm, vol_g);
  __syncthreads();
  conv1_relu(sm);
  __syncthreads();
  float v[8];
  conv2_bias(sm, b2r, v);
  float ss = 0.0f;
#pragma unroll
  for (int oo = 0; oo < 8; ++oo) ss = fmaf(v[oo], v[oo], ss);
  ss = quad_sum(ss);
  const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);  // F.normalize eps (modules/modules.py:122)
#pragma unroll
  for (int oo = 0; oo < 8; ++oo) feat_out[(cg2 * 8 + oo) * kP + pos] = v[oo] * inv;
}

}  // namespace ahv
