// fp32 CUDA-core backward half of the verification head, shared by the fused backward (score_bwd_kernel) and the
// gradient ascent (ascent_fp32_kernel): from H2 of the hypothesis just scored back to dX = dL/d(rotated volume), and the
// rotation gradient dL/dR.  Shared-memory layout: Fp32Smem (ahv_score_fp32.cu) plus the caller's dH2 buffer
// [64 pos][kH1Row].
#pragma once
#include <cstddef>

#include "ahv_head_fp32.cuh"

namespace ahv {

// dX (gradient w.r.t. the rotated volume) overlays rotA / rotT once nothing reads the rotated volume any more,
// voxel-major with the 16 channels innermost: element (d, h, w, c) at d*kDxD + h*kDxH + w*kDxW + c floats - the
// backward's adjoint reads a voxel's record as four LDS.128.  The pitches are 4*odd mod 32: the fold's lanes (which
// run over h or over w) meet distinct bank groups.
constexpr int kDxW = 20, kDxH = 164, kDxD = 1312, kDxFloats = 8 * kDxD;
static_assert(offsetof(Fp32Smem, rotT) == offsetof(Fp32Smem, rotA) + sizeof(float) * kC * kRotC &&
              offsetof(Fp32Smem, h1s) == offsetof(Fp32Smem, rotT) + sizeof(float) * kC * kRotC, "rotA, rotT, h1s are contiguous");
static_assert(kDxFloats <= 2 * kC * kRotC, "dX fits rotA / rotT and leaves h1s (dH1) alone");

// dH2 = g64 (T - F <F,T>) / |v| at this thread's (position, 8 channels) into its dh2 row [pos][kH1Row], from
// conv2_bias' v and head_dots' ss = |v|^2, ft = <v,T>; g64 = dL/dscore / 64 (d mean over the 64 positions).
// F = v / max(|v|, eps) (modules/modules.py:122): d<F,T>/dv = (T - F <F,T>) / |v| above the clamp, T / eps below.
// acc(oo, F, dH2) runs for every channel (the fused backward's dT and db2 accumulators).  v is overwritten with dH2.
template <class Acc>
__device__ __forceinline__ void head_dh2(float (&v)[8], const float (&tg)[8], float ss, float ft, float g64, float* dh2,
                                         Acc&& acc) {
  const int pos = threadIdx.x >> 2, cg2 = threadIdx.x & 3;
  const float nraw = sqrtf(ss), nr = fmaxf(nraw, 1e-12f), inv = 1.0f / nr;
  const float fdot = ft * inv;  // <F, T>
  const bool clamped = nraw < 1e-12f;
#pragma unroll
  for (int oo = 0; oo < 8; ++oo) {
    const float F = v[oo] * inv;
    const float d2 = g64 * inv * (clamped ? tg[oo] : tg[oo] - F * fdot);
    acc(oo, F, d2);
    v[oo] = d2;
  }
  float* dst = dh2 + pos * kH1Row + cg2 * 8;
  *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
}

// dH1 = (dH2 W2) * [H1 > 0], written over H1 in sm.h1s; pos = threadIdx.x >> 2, cg2 = threadIdx.x & 3.  The caller
// has synchronised after the dH2 stores and after anything else that still reads H1; ends with a __syncthreads.
__device__ __forceinline__ void head_dh1(Fp32Smem& sm, const float* dh2, int pos, int cg2) {
  float dh1[8];
  {
    const int ig = cg2;  // input channels ig*8 .. +7 of position `pos`
#pragma unroll
    for (int j = 0; j < 8; ++j) dh1[j] = 0.0f;
#pragma unroll 4
    for (int o = 0; o < kO; ++o) {
      const float d = dh2[pos * kH1Row + o];
      const float* wr = sm.w2s + ((o % 8) * 4 + o / 8) * kH1Row + ig * 8;  // W2[o][ig*8 ..]
      const float4 w0 = *reinterpret_cast<const float4*>(wr), w1 = *reinterpret_cast<const float4*>(wr + 4);
      dh1[0] = fmaf(d, w0.x, dh1[0]); dh1[1] = fmaf(d, w0.y, dh1[1]);
      dh1[2] = fmaf(d, w0.z, dh1[2]); dh1[3] = fmaf(d, w0.w, dh1[3]);
      dh1[4] = fmaf(d, w1.x, dh1[4]); dh1[5] = fmaf(d, w1.y, dh1[5]);
      dh1[6] = fmaf(d, w1.z, dh1[6]); dh1[7] = fmaf(d, w1.w, dh1[7]);
    }
    const float* hp = sm.h1s + pos * kH1Row + ig * 8;  // ReLU mask (modules/modules.py:68)
#pragma unroll
    for (int j = 0; j < 8; ++j) dh1[j] = hp[j] > 0.0f ? dh1[j] : 0.0f;
  }
  __syncthreads();  // every read of h1s is done: overwrite it in place with dH1
  {
    float* hp = sm.h1s + pos * kH1Row + cg2 * 8;
    *reinterpret_cast<float4*>(hp) = make_float4(dh1[0], dh1[1], dh1[2], dh1[3]);
    *reinterpret_cast<float4*>(hp + 4) = make_float4(dh1[4], dh1[5], dh1[6], dh1[7]);
  }
  __syncthreads();
}

// dA = dH1 W1, folded view by view into dX (sm.rotA, layout above); t = threadIdx.x.  The caller has synchronised
// after the last read of rotA / rotT; every view ends with a __syncthreads.
__device__ __forceinline__ void fold_dA(Fp32Smem& sm, int t) {
  const int pl = t & 15, c = t >> 4;  // positions pl + 16 j, channel c, all (view, kk)
  float* dX = sm.rotA + c;            // element (d, h, w, c) at d*kDxD + h*kDxH + w*kDxW + c
#pragma unroll 1
  for (int view = 0; view < 3; ++view) {
    float acc[4][8];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) acc[j][kk] = 0.0f;
    const float* wv = sm.w1t + (view * 128 + c * 8) * kW1Pitch;
#pragma unroll 2
    for (int iq = 0; iq < 8; ++iq) {
      float4 d[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) d[j] = *reinterpret_cast<const float4*>(sm.h1s + (pl + 16 * j) * kH1Row + iq * 4);
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const float2 wa = *reinterpret_cast<const float2*>(wv + kk * kW1Pitch + iq * 4);
        const float2 wb = *reinterpret_cast<const float2*>(wv + kk * kW1Pitch + iq * 4 + 2);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          acc[j][kk] = fmaf(d[j].x, wa.x, fmaf(d[j].y, wa.y, fmaf(d[j].z, wb.x, fmaf(d[j].w, wb.y, acc[j][kk]))));
      }
    }
    // fold: every dX element gets exactly one contribution per view, so no races inside a view
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ps = pl + 16 * j, p = ps >> 3, q = ps & 7;
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        if (view == 0) dX[p * kDxD + q * kDxH + kk * kDxW] = acc[j][kk];          // V'[c, d=p, h=q, w=kk]
        else if (view == 1) dX[p * kDxD + kk * kDxH + q * kDxW] += acc[j][kk];    // V'[c, d=p, h=kk, w=q]
        else dX[kk * kDxD + p * kDxH + q * kDxW] += acc[j][kk];                   // V'[c, d=kk, h=p, w=q]
      }
    }
    __syncthreads();
  }
}

// dL/dR of the hypothesis whose dX fold_dA left in sm.rotA: the resampling differentiated in its grid (rot_grad_accum)
// over the halo'd source volume (sm.vol) at R = sm.Rcur (read from shared memory: the fused backward runs at the register
// limit).  Mapping of gather_hypothesis: 4 lanes per output voxel, 4 channels each.  Returns element threadIdx.x in
// threads 0..8 (block_sum9; red: 72 floats of shared memory); t = threadIdx.x.
__device__ __forceinline__ float rotation_grad(Fp32Smem& sm, float* red, int t) {
  float G[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) G[e] = 0.0f;
  const int lane = t & 31, warp = t >> 5, j = lane & 3, w = lane >> 2;
#pragma unroll 1
  for (int pass = 0; pass < 8; ++pass) {
    const int s = pass * 8 + warp, d = s >> 3, h = s & 7;
    const float4 gx4 = *reinterpret_cast<const float4*>(sm.rotA + d * kDxD + h * kDxH + w * kDxW + 4 * j);
    rot_grad_accum(sm.vol, sm.Rcur, sm.base[w], sm.base[h], sm.base[d], j, gx4, G);
  }
  return block_sum9(G, red, 4.0f);
}

}  // namespace ahv
