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

#include <cmath>

#include "ahv_common.cuh"

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

// t(n, w_i) < c for every winner i in [from, to)
__device__ __forceinline__ bool separated(const float* __restrict__ Rn, const float (*win)[9], int from, int to, float c) {
  float a[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) a[e] = __ldg(Rn + e);
#pragma unroll 1
  for (int i = from; i < to; ++i) {
    float t = __fmul_rn(a[0], win[i][0]);
#pragma unroll
    for (int e = 1; e < 9; ++e) t = __fadd_rn(t, __fmul_rn(a[e], win[i][e]));
    if (!(t < c)) return false;
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
}  // namespace distinct

int launch_topk_distinct(const float* scores, const float* R, int r_per_pair, int B, int64_t N, int k, float min_sep_deg,
                         float* val, int64_t* idx, float* R_best, cudaStream_t s) {
  using namespace distinct;
  if (B == 0) return AHV_OK;
  const bool suppress = min_sep_deg > 0.0f;
  const float c = (float)(1.0 + 2.0 * std::cos((double)min_sep_deg * 3.14159265358979323846 / 180.0));
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

}  // namespace ahv
