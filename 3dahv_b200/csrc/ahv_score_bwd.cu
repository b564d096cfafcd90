// Fused backward of the verification scores (training variant, SURVEY.md §8a-8 / §8f-3).
//
// The reference trains through `infoNCE_loss` (modules/model.py:43-63) with PyTorch autograd over
// rotate_volume -> forward_3d2d -> similarity, saving ~420 KB of activations per hypothesis.  Here one
// kernel recomputes the forward per (pair, hypothesis) in shared memory and pushes the upstream gradient
// g = dL/dscore[b,n] back to everything the score depends on, materialising nothing:
//
//   forward (as score_fp32_kernel)   X = rotate(V_b, R_n);  A = tri-plane(X);  H1 = relu(A W1^T);
//                                    H2 = H1 W2^T + b2;  F = H2 / max(|H2|, eps);  s = mean_p <F_p, T_p>
//   backward                         dH2 = (g/64) (T - F <F,T>) / |H2|          (per position p)
//                                    dT_b += (g/64) F;   db2 += sum_p dH2;   dW2 += dH2^T H1
//                                    dH1 = (dH2 W2) * [H1 > 0];   dW1 += dH1^T A;   dA = dH1 W1
//                                    dX = fold(dA)  (three views onto the rotated volume)
//                                    dV_b += rotate^T(dX, R_n)   (adjoint of the trilinear resampling)
//                                    dR_n += 4 sum_v (sum_c dX[c,v] dX[c,v]/di) b_v^T   (ahv_score_backward_ex only:
//                                    the resampling differentiated in its grid, i = 4 R b + 3.5; DESIGN.md §4.4)
//
// fp32 FFMA throughout (gradients match fp64 autograd of the oracle to ~1e-6 of their maximum).
// One CTA = 256 threads, 1 CTA / SM, contiguous range of (pair, hypothesis) items.  Persistent
// per-thread accumulators: dW1 (48), dW2 (4), db2 (8), dT (8, flushed per pair), dV (32, flushed per
// pair); they leave the CTA through global atomics (caller zero-initialises the outputs).
//
// The adjoint of the resampling is a GATHER, not a scatter (floating-point shared-memory atomics would cost
// ~130k cycles per hypothesis): every INPUT voxel gets the list of the (output voxel, weight) contributions that reach
// it (counting sort over the <= 4096 contributions with integer shared-memory atomics and prefix sums), and every
// thread walks the lists of its two input voxels - exactly the output voxels that touch them, whatever the matrix R
// is - reading dX, which lies voxel-major with the channels innermost, as four LDS.128 per contribution.
#include "ahv_bwd_fp32.cuh"

namespace ahv {

struct BwdSmem {
  Fp32Smem f;
  float dh2[kP * kH1Row];  // dL/dH2 [pos][36]
  float4 taps[kVox];       // (corner line, fx, fy, fz) of every output voxel of the current hypothesis
};
static_assert(sizeof(BwdSmem) <= 232448, "shared memory budget");

// dX (ahv_bwd_fp32.cuh) overlays rotA / rotT once dW1 is done.  The adjoint's work list (<= 4096 entries of 8 bytes)
// follows it, into the dH1 buffer, which is dead by then as well.
static_assert((kDxFloats + 2 * kVox * 8) <= 2 * kC * kRotC + kP * kH1Row, "dX and the work list fit the dead buffers");
static_assert(2 * kVox * sizeof(int) <= sizeof(float) * kP * kH1Row, "counters fit the dH2 buffer");
static_assert((2 * kVox + 9 * kThreads / 32) * sizeof(float) <= sizeof(float) * kP * kH1Row,
              "the rotation phase's partial sums fit behind the counters");

// output voxel (z*64 + y*8 + x) a thread lists for the adjoint: lane bits -> x2 x1 y2 y1 z2, warp bits and j -> the rest
__device__ __forceinline__ int adjoint_out_voxel(int t, int j) {
  const int x = ((t & 3) << 1) | ((t >> 5) & 1), y = (((t >> 2) & 3) << 1) | ((t >> 6) & 1);
  const int z = (((t >> 4) & 1) << 2) | (((t >> 7) & 1) << 1) | j;
  return z * 64 + y * 8 + x;
}

// kEx (ahv_score_backward_ex): every gradient output may be NULL - its accumulation and, for g_vol / g_W1 / g_R, its
// phase are skipped - and the rotation-gradient phase (dS/dR into g_R) is compiled in.  kEx = false is the plain
// backward of ahv_score_backward / ahv_score_backward_saved, which writes all five.
// kDet (ahv_score_backward_det): no float atomics.  g_W1 / g_W2 / g_b2 point at the weight slots and g_vol / g_tgt at
// the segment slots of the workspace (DetBwdWs, ahv_common.cuh), g_R at [B*N][9] for a shared R; every input voxel's
// adjoint list is summed in increasing output-voxel order.
template <bool kEx, bool kDet>
__global__ void __launch_bounds__(kThreads, 1)
score_bwd_kernel(const float* __restrict__ vol_src, const float* __restrict__ tgt_feat,
                 const float* __restrict__ R, int r_per_pair, const float* __restrict__ W1,
                 const float* __restrict__ W2, const float* __restrict__ b2, const float* __restrict__ base,
                 const float* __restrict__ grad_scores, float* __restrict__ g_vol, float* __restrict__ g_tgt,
                 float* __restrict__ g_W1, float* __restrict__ g_W2, float* __restrict__ g_b2, int B, int64_t N,
                 const __half* __restrict__ h1_saved, const float* __restrict__ pair_inv, float* __restrict__ g_R) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  BwdSmem& bs = *reinterpret_cast<BwdSmem*>(smem_raw);
  Fp32Smem& sm = bs.f;
  const int64_t total = (int64_t)B * N;
  const int64_t lo = total * blockIdx.x / gridDim.x, hi = total * (blockIdx.x + 1) / gridDim.x;
  if (lo >= hi) return;
  const int t = threadIdx.x;
  const bool want_vol = !kEx || g_vol, want_tgt = !kEx || g_tgt, want_W1 = !kEx || g_W1;
  const bool want_W2 = !kEx || g_W2, want_b2 = !kEx || g_b2, want_R = kEx && g_R;
  stage_weights(sm, W1, W2, base);
  // conv2 / normalise mapping: thread = (position, 8 output channels cg2*8 ..)
  const int pos = t >> 2, cg2 = t & 3;
  float b2r[8], tg[8];
#pragma unroll
  for (int oo = 0; oo < 8; ++oo) b2r[oo] = b2[cg2 * 8 + oo];
  // persistent accumulators
  float aW1[3][8][2];  // dW1[o = 2cg (+1)][k = view*128 + c*8 + kk], cg = t & 15, c = t >> 4
  float aW2[4];        // dW2[o = t >> 3][i = (t & 7) * 4 ..]
  float ab2[8];        // db2[cg2*8 + oo] (this thread's position only)
  float aT[8];         // dT_b[cg2*8 + oo][pos]
  float aV[2][kC];     // dV_b[c][voxel t + 256 j]
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) aW1[v][kk][0] = aW1[v][kk][1] = 0.0f;
#pragma unroll
  for (int i = 0; i < 4; ++i) aW2[i] = 0.0f;
#pragma unroll
  for (int i = 0; i < 8; ++i) ab2[i] = aT[i] = 0.0f;
#pragma unroll
  for (int j = 0; j < 2; ++j)
#pragma unroll
    for (int c = 0; c < kC; ++c) aV[j][c] = 0.0f;

  auto flush_pair = [&](int b) {  // dT and dV of pair b leave the CTA
    if constexpr (kDet) {   // the whole segment, zeros included, into slot blockIdx.x + b
      const size_t slot = (size_t)(blockIdx.x + b) * kDetSegSlot;
#pragma unroll
      for (int oo = 0; oo < 8; ++oo) {
        if (want_tgt) g_tgt[slot + (cg2 * 8 + oo) * kP + pos] = aT[oo];
        aT[oo] = 0.0f;
      }
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int c = 0; c < kC; ++c) {
          if (want_vol) g_vol[slot + c * kVox + t + 256 * j] = aV[j][c];
          aV[j][c] = 0.0f;
        }
    } else {
#pragma unroll
    for (int oo = 0; oo < 8; ++oo) {
      if (want_tgt && aT[oo] != 0.0f) atomicAdd(g_tgt + ((size_t)b * kO + cg2 * 8 + oo) * kP + pos, aT[oo]);
      aT[oo] = 0.0f;
    }
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int c = 0; c < kC; ++c) {
        if (want_vol && aV[j][c] != 0.0f) atomicAdd(g_vol + ((size_t)b * kC + c) * kVox + t + 256 * j, aV[j][c]);
        aV[j][c] = 0.0f;
      }
    }
  };

  int cur_b = -1;
  for (int64_t it = lo; it < hi; ++it) {
    const int b = (int)(it / N);
    const int64_t n = it - (int64_t)b * N;
    if (b != cur_b) {
      if (cur_b >= 0) flush_pair(cur_b);
      __syncthreads();
      stage_volume<float>(sm.vol, vol_src + (size_t)b * kC * kVox);
#pragma unroll
      for (int oo = 0; oo < 8; ++oo) tg[oo] = tgt_feat[((size_t)b * kO + cg2 * 8 + oo) * kP + pos];
      cur_b = b;
    }
    if (t < 9) sm.Rcur[t] = R[(r_per_pair ? (size_t)it : (size_t)n) * 9 + t];
    __syncthreads();
    float Rr[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) Rr[e] = sm.Rcur[e];
    const float g64 = grad_scores[it] * (1.0f / 64.0f);  // d mean over the 64 positions

    // ---------------- forward recompute ----------------
    gather_hypothesis<true>(sm, Rr, bs.taps);
    if (h1_saved) {
      // saved-activation form: H1 = relu(conv1(A)) of this item was kept by the training forward (fp16, in the pair's
      // scaled units) - 4 KB read instead of 786 k FMA recomputed; A itself is still needed (dW1) and was just gathered
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(h1_saved + ((size_t)it * kP + pos) * kO + cg2 * 8));
      const float inv = __ldg(pair_inv + b);
      const __half2* hp = reinterpret_cast<const __half2*>(&q);
      float* dst = sm.h1s + pos * kH1Row + cg2 * 8;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 f2 = __half22float2(hp[e]);
        dst[2 * e] = f2.x * inv;
        dst[2 * e + 1] = f2.y * inv;
      }
      __syncthreads();
    } else {
      __syncthreads();
      conv1_relu(sm);
      __syncthreads();
    }
    float v[8];
    conv2_bias(sm, b2r, v);
    float ss, ft;
    head_dots(v, tg, ss, ft);
    head_dh2(v, tg, ss, ft, g64, bs.dh2, [&](int oo, float F, float d2) {
      aT[oo] = fmaf(g64, F, aT[oo]);
      ab2[oo] += d2;
    });
    __syncthreads();

    // ---------------- dW2 += dH2^T H1 ; dH1 = (dH2 W2) * [H1 > 0] (head_dh1) ----------------
    {
      const int o = t >> 3, i0 = (t & 7) * 4;
#pragma unroll 8
      for (int p = 0; p < kP; ++p) {
        const float d = bs.dh2[p * kH1Row + o];
        const float4 h = *reinterpret_cast<const float4*>(sm.h1s + p * kH1Row + i0);
        aW2[0] = fmaf(d, h.x, aW2[0]); aW2[1] = fmaf(d, h.y, aW2[1]);
        aW2[2] = fmaf(d, h.z, aW2[2]); aW2[3] = fmaf(d, h.w, aW2[3]);
      }
    }
    head_dh1(sm, bs.dh2, pos, cg2);

    // ---------------- dW1 += dH1^T A  (A = tri-plane views of the rotated volume) ----------------
    if (want_W1) {
      const int cg = t & 15, c = t >> 4;
#pragma unroll 1
      for (int pq = 0; pq < 16; ++pq) {
        const int p = pq >> 1, q0 = (pq & 1) * 4;
        float2 d[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) d[j] = *reinterpret_cast<const float2*>(sm.h1s + (p * 8 + q0 + j) * kH1Row + 2 * cg);
#pragma unroll
        for (int view = 0; view < 3; ++view) {
          const float* a0 = (view == 0 ? sm.rotT : sm.rotA) + c * kRotC + (view == 2 ? p * 8 + q0 : p * kRotD + q0);
          const int kstride = (view == 2) ? kRotD : 8;
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(a0 + kk * kstride);
            float s0 = aW1[view][kk][0], s1 = aW1[view][kk][1];
            s0 = fmaf(a.x, d[0].x, s0); s1 = fmaf(a.x, d[0].y, s1);
            s0 = fmaf(a.y, d[1].x, s0); s1 = fmaf(a.y, d[1].y, s1);
            s0 = fmaf(a.z, d[2].x, s0); s1 = fmaf(a.z, d[2].y, s1);
            s0 = fmaf(a.w, d[3].x, s0); s1 = fmaf(a.w, d[3].y, s1);
            aW1[view][kk][0] = s0; aW1[view][kk][1] = s1;
          }
        }
      }
    }
    __syncthreads();  // rotA / rotT are free: they become dX, voxel-major with the channels innermost

    // ---------------- dA = dH1 W1, folded view by view into dX ----------------
    fold_dA(sm, t);

    // ---------------- dS/dR: the resampling differentiated in its grid (rotation_grad) ----------------
    // The 9 partial sums meet in the dead dH2 buffer behind the adjoint's counters.
    if (want_R) {
      const float sR = rotation_grad(sm, bs.dh2 + 2 * kVox, t);
      if (t < 9) {
        if (r_per_pair) g_R[(size_t)it * 9 + t] += sR;   // the item is this CTA's alone
        else if constexpr (kDet) g_R[(size_t)it * 9 + t] = sR;   // summed over the pairs by score_bwd_det_reduce
        else atomicAdd(g_R + (size_t)n * 9 + t, sR);
      }
    }

    // ---------------- dV_b += rotate^T(dX): adjoint of utils.py:113-131 as a gather ----------------
    // Output voxel vo feeds the 8 input voxels of its tap, corner(vo) + {0,1}^3, with the forward's weights.  Turned round:
    // every INPUT voxel gets the list of its (vo, weight) contributions - a counting sort over the <= 4096 contributions
    // that land inside the volume (shared-memory integer atomics whose return value is the place in the list, prefix
    // sums, 8-byte entries behind dX in the dead rotated-volume / dH1 buffers) - and the adjoint is one flat loop per
    // input voxel: exactly the contributing voxels, no geometry test, valid for any matrix R, fp32 weights recomputed from
    // the taps the forward gather recorded.
    if (want_vol) {
      int* cnt = reinterpret_cast<int*>(bs.dh2);   // [512] contributions per input voxel
      int* start = cnt + kVox;                     // [512] exclusive prefix sum
      uint2* ent = reinterpret_cast<uint2*>(smem_raw + offsetof(BwdSmem, f) + offsetof(Fp32Smem, rotA) + sizeof(float) * kDxFloats);   // [<= 4096] (offset of dX[vo], weight), behind dX
      cnt[t] = 0;
      cnt[t + 256] = 0;
      __syncthreads();
      // the thread's two output voxels: two apart in x and y, four in z across the lanes of a warp, so that the taps of one
      // warp's voxels rarely meet in the same counter
      int tgt0[2];
      uint32_t inside[2], rank[2][4];
      float fx[2], fy[2], fz[2];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int vo = adjoint_out_voxel(t, j);
        const float4 tp = bs.taps[vo];
        const int line = __float_as_int(tp.x);   // ((z0+1)*10 + (y0+1))*10 + (x0+1), corner in [-1, 7]^3
        const int zl = line / (kHalo * kHalo), rl = line - zl * (kHalo * kHalo), yl = rl / kHalo, xl = rl - yl * kHalo;
        const int x0 = xl - 1, y0 = yl - 1, z0 = zl - 1;
        fx[j] = tp.y; fy[j] = tp.z; fz[j] = tp.w;
        tgt0[j] = z0 * 64 + y0 * 8 + x0;
        uint32_t m = 0;
        rank[j][0] = rank[j][1] = rank[j][2] = rank[j][3] = 0;
#pragma unroll
        for (int dlt = 0; dlt < 8; ++dlt) {
          const int x = x0 + (dlt & 1), y = y0 + ((dlt >> 1) & 1), z = z0 + (dlt >> 2);
          if ((unsigned)x < 8u && (unsigned)y < 8u && (unsigned)z < 8u) {
            m |= 1u << dlt;   // the atomic's return value is this contribution's place in its list (<= 511: 16 bits)
            rank[j][dlt >> 1] |= (uint32_t)atomicAdd(&cnt[tgt0[j] + (dlt >> 2) * 64 + ((dlt >> 1) & 1) * 8 + (dlt & 1)], 1) << (16 * (dlt & 1));
          }
        }
        inside[j] = m;
      }
      __syncthreads();
      {  // exclusive scan of the 512 counters: 2 per thread, warp scan, then the 8 warp totals
        const int c0 = cnt[2 * t], c1 = cnt[2 * t + 1];
        const int local = c0 + c1;
        int incl = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int up = __shfl_up_sync(0xffffffffu, incl, o);
          if ((t & 31) >= o) incl += up;
        }
        int* wtot = reinterpret_cast<int*>(sm.red);          // 8 warp totals (sm.red is free outside volume staging)
        if ((t & 31) == 31) wtot[t >> 5] = incl;
        __syncthreads();
        int basep = incl - local;
        for (int w = 0; w < (t >> 5); ++w) basep += wtot[w];
        start[2 * t] = basep;
        start[2 * t + 1] = basep + c0;
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int vo = adjoint_out_voxel(t, j);
        const uint32_t off = (uint32_t)((vo >> 6) * kDxD + ((vo >> 3) & 7) * kDxH + (vo & 7) * kDxW);
#pragma unroll
        for (int dlt = 0; dlt < 8; ++dlt)
          if ((inside[j] >> dlt) & 1u) {
            const int dx = dlt & 1, dy = (dlt >> 1) & 1, dz = dlt >> 2;
            const float w = (dx ? fx[j] : 1.0f - fx[j]) * (dy ? fy[j] : 1.0f - fy[j]) * (dz ? fz[j] : 1.0f - fz[j]);
            const int v = tgt0[j] + dz * 64 + dy * 8 + dx;
            ent[start[v] + ((rank[j][dlt >> 1] >> (16 * (dlt & 1))) & 0xffffu)] = make_uint2(off, __float_as_uint(w));
          }
      }
      __syncthreads();
      if constexpr (kDet) {
        // The atomics ranked each list in arrival order; it is summed in increasing dX offset instead.  Up to 16 entries
        // (a rotation puts at most ~12 on a voxel) the keys (offset, place) are sorted in registers by a network and the
        // entries read in that order; longer lists (matrices that crowd the samples) are sorted in place first.
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int vi = t + 256 * j;
          const int nn = cnt[vi];
          uint2* e = ent + start[vi];
          int nmax = nn;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, o));
          if (nmax <= 16) {
            uint32_t key[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) key[i] = i < nn ? (e[i].x << 4) | (uint32_t)i : 0xffffffffu;
            sort_row(key, nmax);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              if (i >= nmax) break;   // warp-uniform
              if (i < nn) {
                const uint2 en = e[key[i] & 15u];
                const float w = __uint_as_float(en.y);
                const float* src = sm.rotA + en.x;
#pragma unroll
                for (int c4 = 0; c4 < 4; ++c4) {
                  const float4 x = *reinterpret_cast<const float4*>(src + 4 * c4);
                  aV[j][4 * c4] = fmaf(w, x.x, aV[j][4 * c4]); aV[j][4 * c4 + 1] = fmaf(w, x.y, aV[j][4 * c4 + 1]);
                  aV[j][4 * c4 + 2] = fmaf(w, x.z, aV[j][4 * c4 + 2]); aV[j][4 * c4 + 3] = fmaf(w, x.w, aV[j][4 * c4 + 3]);
                }
              }
            }
            continue;
          }
          sort_list(e, nn);
#pragma unroll 2
          for (int i = 0; i < nn; ++i) {
            const uint2 en = e[i];
            const float w = __uint_as_float(en.y);
            const float* src = sm.rotA + en.x;
#pragma unroll
            for (int c4 = 0; c4 < 4; ++c4) {
              const float4 x = *reinterpret_cast<const float4*>(src + 4 * c4);
              aV[j][4 * c4] = fmaf(w, x.x, aV[j][4 * c4]); aV[j][4 * c4 + 1] = fmaf(w, x.y, aV[j][4 * c4 + 1]);
              aV[j][4 * c4 + 2] = fmaf(w, x.z, aV[j][4 * c4 + 2]); aV[j][4 * c4 + 3] = fmaf(w, x.w, aV[j][4 * c4 + 3]);
            }
          }
        }
      } else {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int vi = t + 256 * j;
        const int nn = cnt[vi];
        const uint2* e = ent + start[vi];
#pragma unroll 2
        for (int i = 0; i < nn; ++i) {
          const uint2 en = e[i];
          const float w = __uint_as_float(en.y);
          const float* src = sm.rotA + en.x;
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const float4 x = *reinterpret_cast<const float4*>(src + 4 * c4);
            aV[j][4 * c4] = fmaf(w, x.x, aV[j][4 * c4]); aV[j][4 * c4 + 1] = fmaf(w, x.y, aV[j][4 * c4 + 1]);
            aV[j][4 * c4 + 2] = fmaf(w, x.z, aV[j][4 * c4 + 2]); aV[j][4 * c4 + 3] = fmaf(w, x.w, aV[j][4 * c4 + 3]);
          }
        }
      }
      }
    }
    __syncthreads();  // dX, the work list and the taps are re-used by the next hypothesis
  }
  flush_pair(cur_b);
  // weight gradients: one atomic per accumulator and CTA
  {
    const int cg = t & 15, c = t >> 4;
#pragma unroll
    for (int view = 0; view < 3; ++view)
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const int k = view * 128 + c * 8 + kk;
        if constexpr (kDet) {
          if (want_W1) {
            g_W1[(size_t)blockIdx.x * kDetWSlot + (2 * cg) * kK + k] = aW1[view][kk][0];
            g_W1[(size_t)blockIdx.x * kDetWSlot + (2 * cg + 1) * kK + k] = aW1[view][kk][1];
          }
        } else if (want_W1) {
          atomicAdd(g_W1 + (2 * cg) * kK + k, aW1[view][kk][0]);
          atomicAdd(g_W1 + (2 * cg + 1) * kK + k, aW1[view][kk][1]);
        }
      }
    const int o = t >> 3, i0 = (t & 7) * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if constexpr (kDet) {
        if (want_W2) g_W2[(size_t)blockIdx.x * kDetWSlot + o * kO + i0 + i] = aW2[i];
      } else if (want_W2) atomicAdd(g_W2 + o * kO + i0 + i, aW2[i]);
    }
    // db2: sum over the 64 positions inside the CTA first (threads with equal cg2 = t & 3)
    __syncthreads();
    float* red = sm.h1s;  // [4 cg2][8 oo][64 pos]
#pragma unroll
    for (int oo = 0; oo < 8; ++oo) red[(cg2 * 8 + oo) * kP + pos] = ab2[oo];
    __syncthreads();
    if (want_b2 && t < kO) {
      float s = 0.0f;
      for (int p = 0; p < kP; ++p) s += red[t * kP + p];
      if constexpr (kDet) g_b2[(size_t)blockIdx.x * kDetWSlot + t] = s;
      else atomicAdd(g_b2 + t, s);
    }
  }
}

int launch_score_bwd(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                     const float* W1, const float* W2, const float* b2, const float* base,
                     const float* grad_scores, float* g_vol, float* g_tgt, float* g_W1, float* g_W2,
                     float* g_b2, int B, int64_t N, cudaStream_t s, const void* h1_saved, const float* pair_inv,
                     float* g_R) {
  const int64_t total = (int64_t)B * N;
  if (total == 0) return AHV_OK;
  int dev = 0, sms = 0;
  AHV_CUDA_OK(cudaGetDevice(&dev));
  AHV_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const unsigned grid = (unsigned)(total < sms ? total : sms);
  const size_t smem = sizeof(BwdSmem);
  const __half* h1 = static_cast<const __half*>(h1_saved);
  if (g_R || !g_vol || !g_tgt || !g_W1 || !g_W2 || !g_b2) {
    AHV_CUDA_OK(cudaFuncSetAttribute(score_bwd_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    score_bwd_kernel<true, false><<<grid, kThreads, smem, s>>>(vol_src, tgt_feat, R, r_per_pair, W1, W2, b2, base, grad_scores,
                                                        g_vol, g_tgt, g_W1, g_W2, g_b2, B, N, h1, pair_inv, g_R);
  } else {
    AHV_CUDA_OK(cudaFuncSetAttribute(score_bwd_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    score_bwd_kernel<false, false><<<grid, kThreads, smem, s>>>(vol_src, tgt_feat, R, r_per_pair, W1, W2, b2, base, grad_scores,
                                                         g_vol, g_tgt, g_W1, g_W2, g_b2, B, N, h1, pair_inv, nullptr);
  }
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

// Largest CTA c of a grid over `total` items whose first item, total * c / grid, is at or before item i.
__device__ __forceinline__ int cta_of(int64_t i, int64_t total, int grid) {
  int c = (int)(i * grid / total);
  while (c + 1 < grid && total * (c + 1) / grid <= i) ++c;
  return c;
}

// The deterministic backward's fixed-order reduction: one thread per output element adds the element's partials in
// increasing slot order - the weight slots of CTAs 0 .. grid-1, the segment slots c + b of the CTAs c that hold items of
// pair b, a shared R's per-item values over b = 0 .. B-1 - and adds the sum into the output with one plain add.
// Index space: [W1 | W2 | b2] (kDetWSlot), then B segments [dV_b | dT_b] (kDetSegSlot each), then grad_R [N][9] when a
// shared R's gradient is asked for.  NULL outputs are skipped.
__global__ void __launch_bounds__(256)
score_bwd_det_reduce(const float* __restrict__ ws, size_t seg_off, size_t rot_off, int grid, int B, int64_t N,
                     float* __restrict__ g_vol, float* __restrict__ g_tgt, float* __restrict__ g_W1,
                     float* __restrict__ g_W2, float* __restrict__ g_b2, float* __restrict__ g_R_shared) {
  const int64_t total = (int64_t)B * N;
  const int64_t n_w = kDetWSlot, n_seg = (int64_t)B * kDetSegSlot, n_all = n_w + n_seg + (g_R_shared ? N * 9 : 0);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_all; i += (int64_t)gridDim.x * blockDim.x) {
    if (i < n_w) {
      const int e = (int)i;
      float* out = e < kO * kK ? (g_W1 ? g_W1 + e : nullptr)
                 : e < kO * kK + kO * kO ? (g_W2 ? g_W2 + (e - kO * kK) : nullptr)
                 : (g_b2 ? g_b2 + (e - kO * kK - kO * kO) : nullptr);
      if (!out) continue;
      float s = ws[e];
      for (int c = 1; c < grid; ++c) s += ws[(size_t)c * kDetWSlot + e];
      *out += s;
    } else if (i < n_w + n_seg) {
      const int64_t j = i - n_w;
      const int b = (int)(j / kDetSegSlot), f = (int)(j - (int64_t)b * kDetSegSlot);
      float* out = f < kC * kVox ? (g_vol ? g_vol + (size_t)b * kC * kVox + f : nullptr)
                                 : (g_tgt ? g_tgt + (size_t)b * kO * kP + (f - kC * kVox) : nullptr);
      if (!out) continue;
      const int c0 = cta_of((int64_t)b * N, total, grid), c1 = cta_of((int64_t)(b + 1) * N - 1, total, grid);
      const float* p = ws + seg_off + f;
      float s = p[(size_t)(c0 + b) * kDetSegSlot];
      for (int c = c0 + 1; c <= c1; ++c) s += p[(size_t)(c + b) * kDetSegSlot];
      *out += s;
    } else {
      const int64_t j = i - n_w - n_seg;   // n * 9 + e
      const float* p = ws + rot_off + j;
      float s = p[0];
      for (int b = 1; b < B; ++b) s += p[(size_t)b * N * 9];
      g_R_shared[j] += s;
    }
  }
}

int launch_score_bwd_det(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                         const float* W1, const float* W2, const float* b2, const float* base, const float* grad_scores,
                         const void* h1_saved, const float* pair_inv, float* g_vol, float* g_tgt, float* g_W1,
                         float* g_W2, float* g_b2, float* g_R, int B, int64_t N, bool tc, float* ws, cudaStream_t s) {
  const int64_t total = (int64_t)B * N;
  if (total == 0) return AHV_OK;
  int dev = 0, sms = 0;
  AHV_CUDA_OK(cudaGetDevice(&dev));
  AHV_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int grid = (int)std::min<int64_t>(total, std::min(sms, kDetGridCap));
  const bool shared_R = g_R && !r_per_pair;
  const DetBwdWs w(B, N, shared_R);
  float* ws_w = ws;
  float* ws_seg = ws + w.seg;
  if (tc) {
    const int st = launch_score_bwd_tc_det(vol_src, tgt_feat, R, r_per_pair, W1, W2, b2, base, grad_scores, h1_saved,
                                           pair_inv, ws_w, ws_seg, B, N, (unsigned)grid, s);
    if (st != AHV_OK) return st;
  } else {
    // the kernel's outputs are the workspace slots (NULL where the caller's output is NULL); a per-pair R's gradient
    // has one writer per element and goes straight to the caller's buffer
    float* k_vol = g_vol ? ws_seg : nullptr;
    float* k_tgt = g_tgt ? ws_seg + kC * kVox : nullptr;
    float* k_W1 = g_W1 ? ws_w : nullptr;
    float* k_W2 = g_W2 ? ws_w + kO * kK : nullptr;
    float* k_b2 = g_b2 ? ws_w + kO * kK + kO * kO : nullptr;
    float* k_R = g_R ? (r_per_pair ? g_R : ws + w.rot) : nullptr;
    const size_t smem = sizeof(BwdSmem);
    const __half* h1 = static_cast<const __half*>(h1_saved);
    if (g_R || !g_vol || !g_tgt || !g_W1 || !g_W2 || !g_b2) {
      AHV_CUDA_OK(cudaFuncSetAttribute(score_bwd_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      score_bwd_kernel<true, true><<<grid, kThreads, smem, s>>>(vol_src, tgt_feat, R, r_per_pair, W1, W2, b2, base,
                                                                grad_scores, k_vol, k_tgt, k_W1, k_W2, k_b2, B, N, h1,
                                                                pair_inv, k_R);
    } else {
      AHV_CUDA_OK(cudaFuncSetAttribute(score_bwd_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      score_bwd_kernel<false, true><<<grid, kThreads, smem, s>>>(vol_src, tgt_feat, R, r_per_pair, W1, W2, b2, base,
                                                                 grad_scores, k_vol, k_tgt, k_W1, k_W2, k_b2, B, N, h1,
                                                                 pair_inv, nullptr);
    }
    AHV_CUDA_OK(cudaGetLastError());
  }
  const int64_t n_all = kDetWSlot + (int64_t)B * kDetSegSlot + (shared_R ? N * 9 : 0);
  const unsigned blocks = (unsigned)std::min<int64_t>((n_all + 255) / 256, 8 * (int64_t)sms);
  score_bwd_det_reduce<<<blocks, 256, 0, s>>>(ws, w.seg, w.rot, grid, B, N, g_vol, g_tgt, g_W1, g_W2, g_b2,
                                              shared_R ? g_R : nullptr);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

}  // namespace ahv
