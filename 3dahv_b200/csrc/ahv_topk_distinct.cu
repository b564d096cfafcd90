// Top-k of distinct rotations (ahv_topk_distinct; extension, DESIGN.md §4.6): greedy geodesic non-maximum suppression
// on SO(3) over the score-sorted hypotheses of each pair.
//
//   key(n)   = make_key(score, n)                       (ahv_topk's order: score descending, ties -> lowest index)
//   t(a, b)  = trace(R_a R_b^T), nine __fmul_rn products summed left to right with __fadd_rn (no contraction)
//   w_0      = argmax key;  w_j = argmax { key(n) : key(n) < key(w_{j-1}),  t(n, w_i) < c for every i < j }
//   c        = fp32(1 + 2 cos(min_sep)), rounded once on the host from double; min_sep = 0 tests nothing (the result is
//              ahv_topk's) and min_sep = 180 keeps w_0 alone (every rotation lies within 180 degrees of it).
//
// One thread-block cluster of 8 CTAs per pair (clusters walk pairs blockIdx.y, +gridDim.y, ...); CTA r owns the r-th
// eighth of the N hypotheses and stages its scores in shared memory once when they fit (N up to ~370 000), otherwise
// it re-reads them from L2 every round.  Round j: each thread keeps its best eligible key; a hypothesis's rotation is
// read and tested against the winners only when its key lies below the ceiling and above the thread's running best,
// so almost every hypothesis costs one 4-byte read per round.  One byte per hypothesis in shared memory (N up to
// ~1 800 000) remembers the outcome: a suppressed hypothesis is never tested again, and a kept one is tested only
// against the winners chosen since.  warp -> CTA -> cluster max: every CTA publishes its
// best in its own shared memory, double-buffered by round parity, so one cluster.sync() per round suffices; then
// every CTA reads the 8 partials through DSMEM, finds the same winner and appends its rotation to a local list.
// No workspace, no atomics, no host synchronisation: deterministic and CUDA-graph capturable.
#include <cooperative_groups.h>

#include <algorithm>
#include <cmath>

#include "ahv_topk.cuh"

namespace ahv {
namespace cg = cooperative_groups;

namespace distinct {
constexpr int kCtas = 8;  // portable cluster size
constexpr int kThreads = 1024;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxSmemBytes = 227 * 1024;
constexpr int kStaticSmemBytes = kMaxK * 9 * 4 + kWarps * 8 + 2 * 8 + 8;
constexpr int64_t kDynSmemBytes = kMaxSmemBytes - kStaticSmemBytes - 1024;
constexpr uint8_t kDead = 0xFF;

__device__ __forceinline__ u64 warp_max64(u64 v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const u64 w = __shfl_xor_sync(0xffffffffu, v, o);
    v = w > v ? w : v;
  }
  return v;
}

// t(a, w) = trace(R_a R_w^T): nine __fmul_rn products summed left to right with __fadd_rn (no contraction).  The one
// definition of the trace that the distinct selection and the posterior mass (ahv_posterior_mass) both test.
__device__ __forceinline__ float trace_rn(const float (&a)[9], const float* w) {
  float t = __fmul_rn(a[0], w[0]);
#pragma unroll
  for (int e = 1; e < 9; ++e) t = __fadd_rn(t, __fmul_rn(a[e], w[e]));
  return t;
}

// t(n, w_i) < c for every winner i in [from, to)
__device__ __forceinline__ bool separated(const float* __restrict__ Rn, const float (*win)[9], int from, int to, float c) {
  float a[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) a[e] = __ldg(Rn + e);
#pragma unroll 1
  for (int i = from; i < to; ++i) {
    if (!(trace_rn(a, win[i]) < c)) return false;
  }
  return true;
}

__global__ void __cluster_dims__(kCtas, 1, 1) __launch_bounds__(kThreads, 1)
topk_distinct_kernel(const float* __restrict__ scores, const float* __restrict__ R, int r_per_pair, int B, int64_t N,
                     int k, int rounds, bool suppress, float c, bool staged, bool tracked, float* __restrict__ val,
                     int64_t* __restrict__ idx, float* __restrict__ R_best) {
  // dynamic shared memory: [the CTA's slice of one pair's scores (staged)][one byte per hypothesis of the slice
  // (tracked): how many winners it is known to lie more than min_sep from, or kDead once one suppressed it]
  extern __shared__ __align__(16) unsigned char s_dyn[];
  float* s_scores = reinterpret_cast<float*>(s_dyn);
  __shared__ float s_win[kMaxK][9];                   // the winners' rotations, in selection order
  __shared__ u64 s_warp[kWarps];
  __shared__ u64 s_part[2];                           // this CTA's best of the round, by round parity (read via DSMEM)
  __shared__ u64 s_key;                               // the round's winner
  cg::cluster_group cluster = cg::this_cluster();
  const int r = (int)cluster.block_rank();
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int64_t lo = N * r / kCtas, hi = N * (r + 1) / kCtas;
  uint8_t* s_chk = s_dyn + (staged ? (size_t)((N + kCtas - 1) / kCtas) * sizeof(float) : 0);
  unsigned rnd = 0;
  for (int b = blockIdx.y; b < B; b += gridDim.y) {
    const float* row = scores + (size_t)b * N;
    const float* Rp = R + (r_per_pair ? (size_t)b * N * 9 : 0);
    if (staged || tracked) {  // the previous pair's last scan ended before that round's cluster.sync
      for (int64_t i = lo + t; i < hi; i += kThreads) {
        if (staged) s_scores[i - lo] = row[i];
        if (tracked) s_chk[i - lo] = 0;
      }
      __syncthreads();
    }
    u64 ceiling = ~0ull;
    int j = 0;
    for (; j < rounds; ++j, ++rnd) {
      u64 best = 0;
#pragma unroll 4
      for (int64_t i = lo + t; i < hi; i += kThreads) {
        const u64 key = make_key(staged ? s_scores[i - lo] : __ldg(row + i), (uint32_t)i);
        if (key < ceiling && key > best) {
          if (!suppress) {
            best = key;
          } else if (tracked) {  // a suppressed hypothesis is never tested again, a kept one only against new winners
            const int from = s_chk[i - lo];
            if (from != kDead) {
              const bool keep = separated(Rp + i * 9, s_win, from, j, c);
              s_chk[i - lo] = keep ? (uint8_t)j : kDead;
              if (keep) best = key;
            }
          } else if (separated(Rp + i * 9, s_win, 0, j, c)) {
            best = key;
          }
        }
      }
      best = warp_max64(best);
      if (lane == 0) s_warp[warp] = best;
      __syncthreads();
      if (warp == 0) {
        best = warp_max64(s_warp[lane]);
        if (lane == 0) s_part[rnd & 1] = best;
      }
      cluster.sync();
      if (warp == 0) {
        u64 w = lane < kCtas ? *cluster.map_shared_rank(&s_part[rnd & 1], lane) : 0ull;
        w = warp_max64(w);
        if (w != 0ull && lane < 9) {
          const float v = __ldg(Rp + (size_t)key_index(w) * 9 + lane);
          s_win[j][lane] = v;
          if (r == 0 && R_best) R_best[((size_t)b * k + j) * 9 + lane] = v;
        }
        if (lane == 0) {
          s_key = w;
          if (r == 0 && w != 0ull) {
            val[(size_t)b * k + j] = key_score(w);
            idx[(size_t)b * k + j] = (int64_t)key_index(w);
          }
        }
      }
      __syncthreads();
      ceiling = s_key;
      if (ceiling == 0ull) break;  // nothing qualifies: the same decision in every CTA of the cluster
    }
    if (r == 0) {  // empty slots, as topk_final_kernel and gather_rotations_kernel write them
      for (int e = j * 9 + t; e < k * 9; e += kThreads) {
        if (e % 9 == 0) {
          val[(size_t)b * k + e / 9] = -INFINITY;
          idx[(size_t)b * k + e / 9] = -1;
        }
        if (R_best) R_best[(size_t)b * k * 9 + e] = nanf("");
      }
    }
    if (j < rounds) ++rnd;  // the round that found nothing used a parity slot too
  }
  cluster.sync();  // no CTA leaves while another may still read its partials
}
// c = fp32(1 + 2 cos(theta)), evaluated in double and rounded once: t(a, b) >= c <=> the rotations lie within theta
// of each other (up to the rounding of t).  theta >= 180 gives -inf: every rotation lies within 180 degrees (the
// distinct selection does not test then, it keeps w_0 alone).
inline float trace_threshold(float theta_deg) {
  if (theta_deg >= 180.0f) return -INFINITY;
  return (float)(1.0 + 2.0 * std::cos((double)theta_deg * 3.14159265358979323846 / 180.0));
}
}  // namespace distinct

int launch_topk_distinct(const float* scores, const float* R, int r_per_pair, int B, int64_t N, int k, float min_sep_deg,
                         float* val, int64_t* idx, float* R_best, cudaStream_t s) {
  using namespace distinct;
  if (B == 0) return AHV_OK;
  const bool suppress = min_sep_deg > 0.0f;
  const float c = trace_threshold(min_sep_deg);
  const int rounds = min_sep_deg >= 180.0f ? 1 : k;
  const int64_t slice = (N + kCtas - 1) / kCtas;
  const bool staged = slice * (int64_t)(sizeof(float) + 1) <= kDynSmemBytes;  // N up to ~370 000
  const bool tracked = slice <= kDynSmemBytes;                                 // N up to ~1 800 000
  const size_t smem = (staged ? (size_t)slice * sizeof(float) : 0) + (tracked ? (size_t)slice : 0);
  AHV_CUDA_OK(cudaFuncSetAttribute(topk_distinct_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned clusters = (unsigned)(B < 65535 ? B : 65535);
  topk_distinct_kernel<<<dim3(kCtas, clusters), kThreads, smem, s>>>(scores, R, r_per_pair, B, N, k, rounds, suppress, c,
                                                                     staged, tracked, val, idx, R_best);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

// Posterior mass of the selected rotations (ahv_posterior_mass; DESIGN.md §4.7) under p_b(n) = e^{s[b,n]/T} / Z_b:
//   log_z[b]   = m/T + log sum_n exp((s[b,n] - m)/T),  m = max_n s[b,n]
//   mass[b,j]  = sum_{n -> j} exp((s - m)/T) / sum_n exp((s - m)/T),
// where n -> j for the lowest slot j with t(n, c_j) >= c (trace_rn and trace_threshold above, so with the distinct
// winners as centres and theta = min_sep, slot j holds the winner and exactly the hypotheses it suppressed).
//
// Two launches, deterministic: the hypotheses of a pair are cut into chunks of kChunk (a constant, so the summation
// order depends on N alone, not on B or on the SM count).  Pass 1, grid (chunk, pair): the chunk's maximum m_c and,
// in double, S_c = sum exp((s - m_c)/T) and each slot's share, per thread in index order, then warp butterflies and
// warps in order; a chunk holding a NaN or +inf score records m_c = NaN.  Pass 2, one CTA per pair: m = max m_c
// (exact), then every sum rescaled by exp((m_c - m)/T) and added over the chunks in a fixed tree, each cast to fp32
// once.  Workspace: [the chunk sums, B*chunks*(k+1) doubles | the chunk maxima, B*chunks floats].
//
// With kMoments (ahv_posterior_moments; DESIGN.md §4.7.1) the same two launches also form each slot's first moment
// M_j = sum_{n -> j} e_n R_n / W_j (W_j = the mass's own unnormalised sum) and project it onto SO(3).  Pass 1: every
// thread remembers the slot of each of its kPer hypotheses (a byte); per slot that some lane of the warp holds, each
// lane sums e_n R_n over its own hits in index order (re-reading R_n through L1/L2), a butterfly adds the lanes, and
// the warps are added in order into the chunk's record of k*9 doubles.  Pass 2: one warp per slot rescales the records
// with the mass's factors exp((m_c - m)/T) and adds them over the chunks (lane-strided, then the butterfly), divides by
// W_j, and slot j's thread projects M_j (q-method, project_so3).  Workspace: the mass's, then B*chunks*k*9 doubles.
namespace posterior {
constexpr int kThreads = 128;
constexpr int kWarps = kThreads / 32;
constexpr int kPer = 16;                      // hypotheses per thread of a chunk
constexpr int64_t kChunk = kThreads * kPer;   // 2048
constexpr int kFinalThreads = 256;

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Slot j's record of the chunk, out[j*9 + q] = sum_{n -> j} e_n R_n[q]: per lane over its own hits in index order (s_n
// and R_n re-read through L1/L2, e_n recomputed as the mass formed it), then the warp butterfly, then the warps in
// order.  A slot no lane of the warp holds adds zeros.
__device__ __forceinline__ void chunk_moments(const uint8_t (&slot)[kPer], unsigned held, float mx, double T,
                                              const float* __restrict__ row, const float* __restrict__ Rp, int64_t first,
                                              int k, double* __restrict__ out) {
  __shared__ double s_mom[kMaxK][kWarps][9];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const unsigned warp_held = __reduce_or_sync(0xffffffffu, held);
  for (int j = 0; j < k; ++j) {
    double a[9];
#pragma unroll
    for (int q = 0; q < 9; ++q) a[q] = 0.0;
    if ((warp_held >> j) & 1u) {
      unsigned hits = 0u;  // bit i: the thread's i-th hypothesis is in slot j
#pragma unroll
      for (int i = 0; i < kPer; ++i) hits |= (unsigned)(slot[i] == j) << i;
      while (hits) {
        const int i = __ffs(hits) - 1;
        hits &= hits - 1;
        const int64_t n = first + i * kThreads + t;
        const double e = exp(((double)__ldg(row + n) - (double)mx) / T);
        const float* Rn = Rp + (size_t)n * 9;
#pragma unroll
        for (int q = 0; q < 9; ++q) a[q] += e * (double)__ldg(Rn + q);
      }
#pragma unroll
      for (int q = 0; q < 9; ++q) a[q] = warp_sum_d(a[q]);
    }
    if (lane == 0) {
#pragma unroll
      for (int q = 0; q < 9; ++q) s_mom[j][warp][q] = a[q];
    }
  }
  __syncthreads();
  for (int v = t; v < k * 9; v += kThreads) {
    const int j = v / 9, q = v % 9;
    double x = s_mom[j][0][q];
#pragma unroll
    for (int w = 1; w < kWarps; ++w) x += s_mom[j][w][q];
    out[v] = x;
  }
}

template <bool kMoments>
__global__ void __launch_bounds__(kThreads)
posterior_chunk_kernel(const float* __restrict__ scores, const float* __restrict__ R, int r_per_pair,
                       const float* __restrict__ centers, int B, int64_t N, int k, float c, double T, int chunks,
                       double* __restrict__ ws_sum, float* __restrict__ ws_max, double* __restrict__ ws_mom) {
  __shared__ double s_acc[kMaxK * kThreads];  // slot j of thread t at [j][t]: each thread adds into its own column
  __shared__ double s_red[kMaxK + 1][kWarps];
  __shared__ float s_cen[kMaxK][9];
  __shared__ float s_wmax[kWarps];
  __shared__ int s_wbad[kWarps];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int64_t first = (int64_t)blockIdx.x * kChunk;
  for (int b = blockIdx.y; b < B; b += gridDim.y) {
    const float* row = scores + (size_t)b * N;
    const float* Rp = R + (r_per_pair ? (size_t)b * N * 9 : 0);
    float s[kPer];
    float mx = -INFINITY;
    bool bad = false;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      const int64_t n = first + i * kThreads + t;
      s[i] = n < N ? __ldg(row + n) : -INFINITY;
      bad |= isnan(s[i]) || s[i] == INFINITY;
      mx = fmaxf(mx, s[i]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    bad = __any_sync(0xffffffffu, bad);
    if (lane == 0) {
      s_wmax[warp] = mx;
      s_wbad[warp] = bad;
    }
    for (int e = t; e < k * 9; e += kThreads) s_cen[e / 9][e % 9] = __ldg(centers + (size_t)b * k * 9 + e);
    for (int j = 0; j < k; ++j) s_acc[j * kThreads + t] = 0.0;
    __syncthreads();
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
      mx = fmaxf(mx, s_wmax[w]);
      bad |= s_wbad[w] != 0;
    }
    double tot = 0.0;
    [[maybe_unused]] uint8_t slot[kPer];  // kMoments: the slot of each of the thread's hypotheses (0xFF: none)
    [[maybe_unused]] unsigned held = 0u;  // kMoments: bit j set when the thread holds a hypothesis of slot j
    if constexpr (kMoments) {
#pragma unroll
      for (int i = 0; i < kPer; ++i) slot[i] = 0xFF;
    }
    if (!bad) {
#pragma unroll
      for (int i = 0; i < kPer; ++i) {
        if (s[i] == -INFINITY) continue;  // contributes 0 (and every score of the chunk may be -inf: no inf - inf)
        const double e = exp(((double)s[i] - (double)mx) / T);
        tot += e;
        if (k > 0) {
          const float* Rn = Rp + (size_t)(first + i * kThreads + t) * 9;
          float a[9];
#pragma unroll
          for (int q = 0; q < 9; ++q) a[q] = __ldg(Rn + q);
#pragma unroll 1
          for (int j = 0; j < k; ++j) {
            if (distinct::trace_rn(a, s_cen[j]) >= c) {  // a NaN trace (empty slot) never passes
              s_acc[j * kThreads + t] += e;
              if constexpr (kMoments) {
                slot[i] = (uint8_t)j;
                held |= 1u << j;
              }
              break;
            }
          }
        }
      }
    }
    for (int v = 0; v <= k; ++v) {
      const double x = warp_sum_d(v == 0 ? tot : s_acc[(v - 1) * kThreads + t]);
      if (lane == 0) s_red[v][warp] = x;
    }
    __syncthreads();
    const size_t rec = (size_t)b * chunks + blockIdx.x;
    if (t <= k) {
      double x = s_red[t][0];
#pragma unroll
      for (int w = 1; w < kWarps; ++w) x += s_red[t][w];
      ws_sum[rec * (k + 1) + t] = x;
    }
    if (t == 0) ws_max[rec] = bad ? NAN : mx;
    if constexpr (kMoments) chunk_moments(slot, held, mx, T, row, Rp, first, k, ws_mom + rec * k * 9);
    __syncthreads();  // the next pair reuses the shared arrays
  }
}

constexpr int kFinalW = kFinalThreads / 32;
constexpr int kJacobiSweeps = 8;  // at most; 4-5 cyclic sweeps bring a 4x4 to diagonal in double

// R = argmax_{R in SO(3)} tr(R^T M) by the q-method (Horn 1987, Davenport): for R = R(w, x, y, z), tr(R^T M) = q^T K q
// with K below, so R's unit quaternion is K's eigenvector of the largest eigenvalue (any of them on a tie) and
// R(q) is a proper rotation by construction.  K is diagonalised by cyclic Jacobi in double, at most kJacobiSweeps
// sweeps, stopping once the off-diagonal squares sum to at most 1e-32 of the diagonal's: the result depends on M
// alone.  Returns tr(R^T M).  Row-major 3x3.
__host__ __device__ inline double project_so3(const double (&M)[9], double (&Rout)[9]) {
  double a[4][4] = {{M[0] + M[4] + M[8], M[7] - M[5], M[2] - M[6], M[3] - M[1]},
                    {M[7] - M[5], M[0] - M[4] - M[8], M[1] + M[3], M[2] + M[6]},
                    {M[2] - M[6], M[1] + M[3], -M[0] + M[4] - M[8], M[5] + M[7]},
                    {M[3] - M[1], M[2] + M[6], M[5] + M[7], -M[0] - M[4] + M[8]}};
  double v[4][4] = {{1, 0, 0, 0}, {0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1}};
#pragma unroll 1
  for (int sweep = 0; sweep < kJacobiSweeps; ++sweep) {
    double off = 0.0, diag = 0.0;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      diag += a[p][p] * a[p][p];
#pragma unroll
      for (int q = p + 1; q < 4; ++q) off += a[p][q] * a[p][q];
    }
    if (off <= 1e-32 * diag) break;
#pragma unroll
    for (int p = 0; p < 3; ++p) {
#pragma unroll
      for (int q = p + 1; q < 4; ++q) {
        if (a[p][q] == 0.0) continue;
        // Golub & Van Loan, sym.schur2: J = [c s; -s c] on (p, q) zeroes a[p][q] of J^T A J
        const double tau = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
        const double cs = 1.0 / sqrt(1.0 + t * t), sn = t * cs;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const double ap = a[r][p], aq = a[r][q];
          a[r][p] = cs * ap - sn * aq;
          a[r][q] = sn * ap + cs * aq;
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const double ap = a[p][r], aq = a[q][r];
          a[p][r] = cs * ap - sn * aq;
          a[q][r] = sn * ap + cs * aq;
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const double vp = v[r][p], vq = v[r][q];
          v[r][p] = cs * vp - sn * vq;
          v[r][q] = sn * vp + cs * vq;
        }
      }
    }
  }
  double best = a[0][0], w = v[0][0], x = v[1][0], y = v[2][0], z = v[3][0];
#pragma unroll
  for (int e = 1; e < 4; ++e) {
    if (a[e][e] > best) {
      best = a[e][e];
      w = v[0][e], x = v[1][e], y = v[2][e], z = v[3][e];
    }
  }
  const double inv = 1.0 / sqrt(w * w + x * x + y * y + z * z);
  w *= inv, x *= inv, y *= inv, z *= inv;
  Rout[0] = w * w + x * x - y * y - z * z, Rout[1] = 2.0 * (x * y - w * z), Rout[2] = 2.0 * (x * z + w * y);
  Rout[3] = 2.0 * (x * y + w * z), Rout[4] = w * w - x * x + y * y - z * z, Rout[5] = 2.0 * (y * z - w * x);
  Rout[6] = 2.0 * (x * z - w * y), Rout[7] = 2.0 * (y * z + w * x), Rout[8] = w * w - x * x - y * y + z * z;
  double tr = 0.0;
#pragma unroll
  for (int e = 0; e < 9; ++e) tr += Rout[e] * M[e];
  return tr;
}

// Pass 2 of the moments, after the mass.  Warp w takes slots w, w + 8, ...: each lane adds the slot's records of chunks
// lane, lane + 32, ... in index order, rescaled by the mass's factors exp((m_c - m)/T), then the butterfly; the sums are
// divided by W_j (the mass's own sum of slot j, re-added from s_red in the mass's order).  Then slot j's thread projects
// M_j.  A pair with a NaN or +inf score, and a slot with W_j = 0, get NaN.
__device__ __forceinline__ void final_moments(const double* __restrict__ rec, const float* __restrict__ mc, int chunks, int k,
                                              double T, float m, bool live, bool bad, const double (*s_red)[kFinalW],
                                              float* __restrict__ mean_R, float* __restrict__ mean_cos,
                                              float* __restrict__ moment) {
  __shared__ double s_M[kMaxK][9];
  const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  for (int j = warp; j < k; j += kFinalW) {
    double a[9];
#pragma unroll
    for (int q = 0; q < 9; ++q) a[q] = 0.0;
    if (live) {
      for (int i = lane; i < chunks; i += 32) {
        const float mi = mc[i];
        if (mi == -INFINITY) continue;  // the chunk holds nothing (its records are 0)
        const double f = exp(((double)mi - (double)m) / T);
        const double* r = rec + ((size_t)i * k + j) * 9;
#pragma unroll
        for (int q = 0; q < 9; ++q) a[q] += r[q] * f;
      }
    }
#pragma unroll
    for (int q = 0; q < 9; ++q) a[q] = warp_sum_d(a[q]);
    if (lane == 0) {
      double W = s_red[j + 1][0];
#pragma unroll
      for (int w = 1; w < kFinalW; ++w) W += s_red[j + 1][w];
#pragma unroll
      for (int q = 0; q < 9; ++q) {
        const double M = !bad && W > 0.0 ? a[q] / W : (double)NAN;
        s_M[j][q] = M;
        moment[((size_t)b * k + j) * 9 + q] = (float)M;
      }
    }
  }
  __syncthreads();
  if (t < k) {
    double M[9], Rb[9];
    bool nan = false;
#pragma unroll
    for (int e = 0; e < 9; ++e) {
      M[e] = s_M[t][e];
      nan |= isnan(M[e]);
    }
    const double tr = project_so3(M, Rb);
    float* out = mean_R + ((size_t)b * k + t) * 9;
#pragma unroll
    for (int e = 0; e < 9; ++e) out[e] = nan ? NAN : (float)Rb[e];
    mean_cos[(size_t)b * k + t] = nan ? NAN : (float)fmin(fmax((tr - 1.0) * 0.5, -1.0), 1.0);
  }
}

template <bool kMoments>
__global__ void __launch_bounds__(kFinalThreads)
posterior_final_kernel(const double* __restrict__ ws_sum, const float* __restrict__ ws_max, int chunks, int k, double T,
                       float* __restrict__ log_z, float* __restrict__ mass, const double* __restrict__ ws_mom,
                       float* __restrict__ mean_R, float* __restrict__ mean_cos, float* __restrict__ moment) {
  constexpr int kW = kFinalW;
  __shared__ float s_wmax[kW];
  __shared__ int s_wbad[kW];
  __shared__ double s_red[kMaxK + 1][kW];
  const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const float* mc = ws_max + (size_t)b * chunks;
  const double* sc = ws_sum + (size_t)b * chunks * (k + 1);
  float m = -INFINITY;
  bool bad = false;
  for (int i = t; i < chunks; i += kFinalThreads) {
    const float x = mc[i];
    bad |= isnan(x);
    m = fmaxf(m, x);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  bad = __any_sync(0xffffffffu, bad);
  if (lane == 0) {
    s_wmax[warp] = m;
    s_wbad[warp] = bad;
  }
  __syncthreads();
#pragma unroll
  for (int w = 0; w < kW; ++w) {
    m = fmaxf(m, s_wmax[w]);
    bad |= s_wbad[w] != 0;
  }
  // every score -inf: Z = 0, log_z = -inf and the masses 0/0 = NaN
  const bool live = !bad && m != -INFINITY;
  for (int v = 0; v <= k; ++v) {
    double x = 0.0;
    if (live) {
      for (int i = t; i < chunks; i += kFinalThreads) {
        const float mi = mc[i];
        if (mi != -INFINITY) x += sc[(size_t)i * (k + 1) + v] * exp(((double)mi - (double)m) / T);
      }
    }
    x = warp_sum_d(x);
    if (lane == 0) s_red[v][warp] = x;
  }
  __syncthreads();
  if (t <= k) {
    double S = s_red[t][0], Z = s_red[0][0];
#pragma unroll
    for (int w = 1; w < kW; ++w) {
      S += s_red[t][w];
      Z += s_red[0][w];
    }
    if (t == 0) log_z[b] = bad ? NAN : (float)((double)m / T + log(S));
    else mass[(size_t)b * k + t - 1] = bad ? NAN : (float)(S / Z);
  }
  if constexpr (kMoments)
    final_moments(ws_mom + (size_t)b * chunks * k * 9, mc, chunks, k, T, m, live, bad, s_red, mean_R, mean_cos, moment);
}

struct Ws {  // [sums | maxima | moment records (moments)], each 256-byte aligned
  int chunks;
  double* sum;
  float* max;
  double* mom;
  Ws(Carve& c, int B, int64_t N, int k, bool moments)
      : chunks((int)((N + kChunk - 1) / kChunk)),
        sum(c.take<double>((size_t)B * chunks * (k + 1), 256)),
        max(c.take<float>((size_t)B * chunks, 256)),
        mom(c.take<double>(moments ? (size_t)B * chunks * k * 9 : 0, 256)) {}
};
}  // namespace posterior

size_t posterior_workspace_bytes(int B, int64_t N, int k, bool moments) {
  Carve c;
  (void)posterior::Ws(c, B, N, k, moments);
  return c.off;
}

int launch_posterior(const float* scores, const float* R, int r_per_pair, const float* centers, int B, int64_t N, int k,
                     float radius_deg, float temperature, float* log_z, float* mass, float* mean_R, float* mean_cos,
                     float* moment, void* ws, cudaStream_t s) {
  using namespace posterior;
  if (B == 0) return AHV_OK;
  const bool moments = moment != nullptr;
  Carve cur(ws);
  const Ws w(cur, B, N, k, moments);
  const dim3 grid1((unsigned)w.chunks, (unsigned)(B < 65535 ? B : 65535));
  const float c = distinct::trace_threshold(radius_deg);
  const double T = (double)temperature;
  if (moments) {
    posterior_chunk_kernel<true><<<grid1, kThreads, 0, s>>>(scores, R, r_per_pair, centers, B, N, k, c, T, w.chunks, w.sum,
                                                            w.max, w.mom);
  } else {
    posterior_chunk_kernel<false><<<grid1, kThreads, 0, s>>>(scores, R, r_per_pair, centers, B, N, k, c, T, w.chunks,
                                                             w.sum, w.max, nullptr);
  }
  AHV_CUDA_OK(cudaGetLastError());
  if (moments) {
    posterior_final_kernel<true><<<(unsigned)B, kFinalThreads, 0, s>>>(w.sum, w.max, w.chunks, k, T, log_z, mass, w.mom,
                                                                       mean_R, mean_cos, moment);
  } else {
    posterior_final_kernel<false><<<(unsigned)B, kFinalThreads, 0, s>>>(w.sum, w.max, w.chunks, k, T, log_z, mass,
                                                                        nullptr, nullptr, nullptr, nullptr);
  }
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

// Coarse-to-fine search that keeps k distinct modes (ahv_search_modes; DESIGN.md §4.8.1).  With the distinct winners
// c_j of the base level (ahv_topk_distinct) as centres, base cell n belongs to slot j when n = c_j, else to the lowest
// slot j with t(n, c_j) >= c (the posterior mass's rule, trace_rn and trace_threshold above): slot j holds its winner and
// the cells that winner suppressed, and c_j is the slot's largest key.  Each slot keeps a beam of w <= 8 cells of the
// current level, ascending in grid index and padded with -1 at the end; a level scores the 8 children of every beam cell
// as one per-pair set [B, 8kw], slot j's children being the segment [8wj, 8w(j+1)), and keeps the top-w of each
// segment.  One CTA per pair, warp j serving slot j, keeps every selection in ahv_topk's key order.
namespace modes {
constexpr int kSlotThreads = 256;
constexpr int kBeamBatch = 4;  // cells per lane whose loads a beam warp issues at once
constexpr uint8_t kNoSlot = 0xFF;

// slot[b, n] of every base cell, grid (cells / kSlotThreads, pairs)
__global__ void __launch_bounds__(kSlotThreads)
modes_slot_kernel(const float* __restrict__ G, int64_t n0, const int64_t* __restrict__ first_idx,
                  const float* __restrict__ first_R, int B, int k, float c, uint8_t* __restrict__ slot) {
  __shared__ float s_cen[kMaxK][9];
  __shared__ int64_t s_win[kMaxK];
  for (int b = blockIdx.y; b < B; b += gridDim.y) {
    __syncthreads();  // the previous pair's centres are no longer read
    for (int e = threadIdx.x; e < k * 9; e += kSlotThreads) s_cen[e / 9][e % 9] = __ldg(first_R + (size_t)b * k * 9 + e);
    for (int j = threadIdx.x; j < k; j += kSlotThreads) s_win[j] = __ldg(first_idx + (size_t)b * k + j);
    __syncthreads();
    for (int64_t n = (int64_t)blockIdx.x * kSlotThreads + threadIdx.x; n < n0; n += (int64_t)gridDim.x * kSlotThreads) {
      float a[9];
#pragma unroll
      for (int e = 0; e < 9; ++e) a[e] = __ldg(G + n * 9 + e);
      int s = kNoSlot;
      for (int j = 0; j < k; ++j) {
        if (s_win[j] == n) {
          s = j;
          break;
        }
      }
      if (s == kNoSlot) {
#pragma unroll 1
        for (int j = 0; j < k; ++j) {
          if (distinct::trace_rn(a, s_cen[j]) >= c) {  // a NaN centre (empty slot) never passes
            s = j;
            break;
          }
        }
      }
      slot[(size_t)b * n0 + n] = (uint8_t)s;
    }
  }
}

// The w best keys of a warp's sorted list (lanes < w) as cells, written ascending with -1 last to par and, with the -1
// replaced by cell 0 of the level (a valid rotation for the children generator), to gen.
__device__ __forceinline__ void write_beam(u64 best, const int64_t* cells, int w, int lane, int64_t* par, int64_t* gen) {
  int64_t v = -1;
  if (lane < w && best != 0ull) v = cells ? cells[key_index(best)] : (int64_t)key_index(best);
  const uint64_t ord = (uint64_t)v;  // -1 sorts after every cell
  int pos = 0;
  for (int i = 0; i < w; ++i) {
    const uint64_t u = (uint64_t)__shfl_sync(0xffffffffu, v, i);
    pos += (u < ord) || (u == ord && i < lane);
  }
  if (lane < w) {
    par[pos] = v;
    gen[pos] = v < 0 ? 0 : v;
  }
}

// The initial beams: warp j keeps the top-w keys of slot j's cells.  Block (pair), k warps.
__global__ void __launch_bounds__(kMaxK * 32)
modes_beam_kernel(const float* __restrict__ S0, const uint8_t* __restrict__ slot, int64_t n0, int k, int w,
                  int64_t* __restrict__ par, int64_t* __restrict__ gen) {
  const int b = blockIdx.x, j = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* row = S0 + (size_t)b * n0;
  const uint8_t* sl = slot + (size_t)b * n0;
  u64 best = 0ull;
  for (int64_t i = 0; i < n0; i += 32 * kBeamBatch) {  // a batch's loads in flight together: the scan is latency-bound
    u64 cand[kBeamBatch];
#pragma unroll
    for (int u = 0; u < kBeamBatch; ++u) {
      const int64_t n = i + u * 32 + lane;
      cand[u] = n < n0 && __ldg(sl + n) == j ? make_key(__ldg(row + n), (uint32_t)n) : 0ull;
    }
#pragma unroll
    for (int u = 0; u < kBeamBatch; ++u) best = warp_offer(best, cand[u], lane);
  }
  const size_t at = ((size_t)b * k + j) * w;
  write_beam(best, nullptr, w, lane, par + at, gen + at);
}

// One level: warp j keeps the top-w of segment j of the pair's scored children (a -1 parent's 8 children never
// qualify).  Not the last level: the beams of the next.  The last: each slot's best, then warp 0 orders the k modes by
// key (score descending, ties to the lower grid index; empty modes last, in slot order) into val, idx and R_out.
__global__ void __launch_bounds__(kMaxK * 32)
modes_level_kernel(const float* __restrict__ sc, const int64_t* __restrict__ kids, const float* __restrict__ kids_R, int k,
                   int w, bool last, int64_t* __restrict__ par, int64_t* __restrict__ gen, float* __restrict__ val,
                   int64_t* __restrict__ idx, float* __restrict__ R_out) {
  __shared__ u64 s_key[kMaxK];
  __shared__ int64_t s_cell[kMaxK];
  const int b = blockIdx.x, j = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nc = 8 * w;
  const size_t seg = ((size_t)b * k + j) * nc, at = ((size_t)b * k + j) * w;
  u64 best = 0ull;
#pragma unroll
  for (int h = 0; h < 64; h += 32) {
    const int t = h + lane;
    const bool real = t < nc && par[at + (t >> 3)] >= 0;
    best = warp_offer(best, real ? make_key(__ldg(sc + seg + t), (uint32_t)t) : 0ull, lane);
  }
  if (!last) {  // a warp overwrites only the parents it has read
    write_beam(best, kids + seg, w, lane, par + at, gen + at);
    return;
  }
  if (lane == 0) {
    s_key[j] = best;
    s_cell[j] = best != 0ull ? kids[seg + key_index(best)] : -1;
  }
  __syncthreads();
  if (j != 0) return;
  const u64 key = lane < k ? s_key[lane] : 0ull;
  const uint32_t hi = (uint32_t)(key >> 32);
  const uint64_t tie = key != 0ull ? (uint64_t)s_cell[lane] : (uint64_t)lane;  // empty: hi == 0, in slot order
  int pos = 0;
  for (int i = 0; i < k; ++i) {
    const uint32_t hi_i = __shfl_sync(0xffffffffu, hi, i);
    const uint64_t tie_i = __shfl_sync(0xffffffffu, tie, i);
    pos += hi_i > hi || (hi_i == hi && tie_i < tie);
  }
  if (lane >= k) return;
  const size_t o = (size_t)b * k + pos;
  idx[o] = s_cell[lane];
  if (key == 0ull) {
    val[o] = -INFINITY;
#pragma unroll
    for (int e = 0; e < 9; ++e) R_out[o * 9 + e] = nanf("");
    return;
  }
  val[o] = key_score(key);
  const float* src = kids_R + (((size_t)b * k + lane) * nc + key_index(key)) * 9;
#pragma unroll
  for (int e = 0; e < 9; ++e) R_out[o * 9 + e] = src[e];
}
}  // namespace modes

int launch_modes_beams(const float* S0, const float* G, int64_t n0, const int64_t* first_idx, const float* first_R, int B,
                       int k, int w, float min_sep_deg, uint8_t* slot, int64_t* par, int64_t* gen, cudaStream_t s) {
  using namespace modes;
  if (B == 0) return AHV_OK;
  const unsigned gx = (unsigned)std::min<int64_t>((n0 + kSlotThreads - 1) / kSlotThreads, 1 << 16);
  modes_slot_kernel<<<dim3(gx, (unsigned)(B < 65535 ? B : 65535)), kSlotThreads, 0, s>>>(
      G, n0, first_idx, first_R, B, k, distinct::trace_threshold(min_sep_deg), slot);
  AHV_CUDA_OK(cudaGetLastError());
  modes_beam_kernel<<<(unsigned)B, 32 * k, 0, s>>>(S0, slot, n0, k, w, par, gen);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

int launch_modes_level(const float* sc, const int64_t* kids, const float* kids_R, int B, int k, int w, bool last,
                       int64_t* par, int64_t* gen, float* val, int64_t* idx, float* R_out, cudaStream_t s) {
  if (B == 0) return AHV_OK;
  modes::modes_level_kernel<<<(unsigned)B, 32 * k, 0, s>>>(sc, kids, kids_R, k, w, last, par, gen, val, idx, R_out);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

}  // namespace ahv
