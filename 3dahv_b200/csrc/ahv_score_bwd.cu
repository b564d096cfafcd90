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
// is - reading dX, which lies voxel-major with the channels innermost, as four LDS.128 per contribution.  The work
// list, the orders the deterministic form sums it in and the flushes of the gradients are shared with the tcgen05
// backward (ahv_adjoint.cuh).
#include "ahv_adjoint.cuh"
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

  auto flush = [&](int b) { flush_pair<kDet>(g_tgt, g_vol, b, aT, aV, cg2, pos, want_tgt, want_vol); };

  int cur_b = -1;
  for (int64_t it = lo; it < hi; ++it) {
    const int b = (int)(it / N);
    const int64_t n = it - (int64_t)b * N;
    if (b != cur_b) {
      if (cur_b >= 0) flush(cur_b);
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
    // Every INPUT voxel gets the list of its (output voxel, weight) contributions (build_exact_list, ahv_adjoint.cuh: 8-byte
    // entries behind dX in the dead rotated-volume / dH1 buffers), and the adjoint is one flat loop per input voxel:
    // exactly the contributing voxels, no geometry test, valid for any matrix R, fp32 weights recomputed from the taps
    // the forward gather recorded.
    if (want_vol) {
      int* cnt = reinterpret_cast<int*>(bs.dh2);   // [512] contributions per input voxel
      int* start = cnt + kVox;                     // [512] exclusive prefix sum
      uint2* ent = reinterpret_cast<uint2*>(smem_raw + offsetof(BwdSmem, f) + offsetof(Fp32Smem, rotA) + sizeof(float) * kDxFloats);   // [<= 4096] (offset of dX[vo], weight), behind dX
      // sm.red is free outside volume staging: the scan's 8 warp totals
      build_exact_list<kDxD, kDxH, kDxW>(bs.taps, cnt, start, ent, reinterpret_cast<int*>(sm.red));
      __syncthreads();
      // acc[0..15] += w * dX[vo][0..15]: four LDS.128 per contribution
      auto axpy = [&](float* acc, uint2 en) {
        const float w = __uint_as_float(en.y);
        const float* src = sm.rotA + en.x;
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
          const float4 x = *reinterpret_cast<const float4*>(src + 4 * c4);
          acc[4 * c4] = fmaf(w, x.x, acc[4 * c4]); acc[4 * c4 + 1] = fmaf(w, x.y, acc[4 * c4 + 1]);
          acc[4 * c4 + 2] = fmaf(w, x.z, acc[4 * c4 + 2]); acc[4 * c4 + 3] = fmaf(w, x.w, acc[4 * c4 + 3]);
        }
      };
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int vi = t + 256 * j;
        const int nn = cnt[vi];
        uint2* e = ent + start[vi];
        if constexpr (kDet) {
          // The atomics ranked each list in arrival order; it is summed in increasing dX offset instead.  Up to 16
          // entries (a rotation puts at most ~12 on a voxel) the keys (offset, place) are sorted in registers by a
          // network and the entries read in that order; longer lists (matrices that crowd the samples) are sorted in
          // place first.
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
              if (i < nn) axpy(aV[j], e[key[i] & 15u]);
            }
            continue;
          }
          sort_list(e, nn);
        }
        walk_list(e, nn, [&](uint2 en) { axpy(aV[j], en); });
      }
    }
    __syncthreads();  // dX, the work list and the taps are re-used by the next hypothesis
  }
  flush(cur_b);
  // weight gradients: one atomic per accumulator and CTA (kDet: one store into the CTA's weight slot)
  {
    const int cg = t & 15, c = t >> 4;
#pragma unroll
    for (int view = 0; view < 3; ++view)
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const int k = view * 128 + c * 8 + kk;
        if (want_W1) {
          flush_weight<kDet>(g_W1 + (2 * cg) * kK + k, aW1[view][kk][0]);
          flush_weight<kDet>(g_W1 + (2 * cg + 1) * kK + k, aW1[view][kk][1]);
        }
      }
    const int o = t >> 3, i0 = (t & 7) * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (want_W2) flush_weight<kDet>(g_W2 + o * kO + i0 + i, aW2[i]);
    flush_b2<kDet>(sm.h1s, ab2, cg2, pos, g_b2, want_b2);   // sm.h1s: [4 cg2][8 oo][64 pos]
  }
}

int launch_score_bwd(const Scored& p, const float* tgt_feat, const float* grad_scores, float* g_vol, float* g_tgt,
                     float* g_W1, float* g_W2, float* g_b2, cudaStream_t s, const void* h1_saved, const float* pair_inv,
                     float* g_R, unsigned grid, bool det) {
  const int64_t total = (int64_t)p.B * p.N;
  if (total == 0) return AHV_OK;
  if (grid == 0) {
    const int sms = sm_count();
    if (sms <= 0) return AHV_ECUDA;
    grid = (unsigned)(total < sms ? total : sms);
  }
  const bool ex = g_R || !g_vol || !g_tgt || !g_W1 || !g_W2 || !g_b2;
  const auto kernel = ex ? (det ? score_bwd_kernel<true, true> : score_bwd_kernel<true, false>)
                         : (det ? score_bwd_kernel<false, true> : score_bwd_kernel<false, false>);
  const size_t smem = sizeof(BwdSmem);
  AHV_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<grid, kThreads, smem, s>>>(p.vol_f32(), tgt_feat, p.R, p.r_per_pair, p.W1, p.W2, p.b2, p.base, grad_scores,
                                      g_vol, g_tgt, g_W1, g_W2, g_b2, p.B, p.N, static_cast<const __half*>(h1_saved),
                                      pair_inv, g_R);
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

int launch_score_bwd_det(const Scored& p, const float* tgt_feat, const float* grad_scores, const void* h1_saved,
                         const float* pair_inv, float* g_vol, float* g_tgt, float* g_W1, float* g_W2, float* g_b2,
                         float* g_R, bool tc, const DetBwdWs& w, cudaStream_t s) {
  const int B = p.B;
  const int64_t N = p.N, total = (int64_t)B * N;
  if (total == 0) return AHV_OK;
  const int sms = sm_count();
  if (sms <= 0) return AHV_ECUDA;
  const int grid = (int)std::min<int64_t>(total, std::min(sms, kDetGridCap));
  const bool shared_R = g_R && !p.r_per_pair;
  // the kernel's outputs are the workspace slots (NULL where the caller's output is NULL); a per-pair R's gradient
  // has one writer per element and goes straight to the caller's buffer
  float* k_vol = g_vol ? w.seg : nullptr;
  float* k_tgt = g_tgt ? w.seg + kC * kVox : nullptr;
  float* k_W1 = g_W1 ? w.w : nullptr;
  float* k_W2 = g_W2 ? w.w + kO * kK : nullptr;
  float* k_b2 = g_b2 ? w.w + kO * kK + kO * kO : nullptr;
  float* k_R = g_R ? (p.r_per_pair ? g_R : w.rot) : nullptr;
  const int st = tc ? launch_score_bwd_tc(p, tgt_feat, grad_scores, h1_saved, pair_inv, k_vol, k_tgt, k_W1, k_W2, k_b2, s,
                                          (unsigned)grid, true)
                    : launch_score_bwd(p, tgt_feat, grad_scores, k_vol, k_tgt, k_W1, k_W2, k_b2, s, h1_saved, pair_inv, k_R,
                                       (unsigned)grid, true);
  if (st != AHV_OK) return st;
  const int64_t n_all = kDetWSlot + (int64_t)B * kDetSegSlot + (shared_R ? N * 9 : 0);
  const unsigned blocks = (unsigned)std::min<int64_t>((n_all + 255) / 256, 8 * (int64_t)sms);
  score_bwd_det_reduce<<<blocks, 256, 0, s>>>(w.w, w.seg - w.w, w.rot - w.w, grid, B, N, g_vol, g_tgt, g_W1, g_W2, g_b2,
                                              shared_R ? g_R : nullptr);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

}  // namespace ahv
