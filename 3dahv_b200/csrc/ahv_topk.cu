// Selection: torch.max(pred_sim, dim=1) (modules/model.py:195) generalised to
// top-k (k <= 32), plus the merge of per-shard lists and sampled_R[pred_index]
// (modules/model.py:196).
//
// Ordering rule everywhere: score descending, ties -> lowest hypothesis index
// (torch.max on CPU returns the first maximal index).  Implemented by packing
// (score, index) into one 64-bit key — high word: the fp32 score mapped to an
// order-preserving uint32 (-0.0 canonicalised to +0.0), low word: ~index — and
// keeping, per warp, a sorted list of 32 keys distributed one per lane that is
// updated with a shuffle-based bitonic sort + bitonic merge.
#include "ahv_topk.cuh"

namespace ahv {

constexpr int kTopkThreads = 256;

// stage 1: grid (S, B); each CTA reduces its slice of one pair to 32 keys
__global__ void __launch_bounds__(kTopkThreads)
topk_slice_kernel(const float* __restrict__ scores, int64_t N, u64* __restrict__ partial) {
  __shared__ u64 lists[kTopkThreads / 32][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int S = gridDim.x, b = blockIdx.y;
  const int64_t lo = N * blockIdx.x / S, hi = N * (blockIdx.x + 1) / S;
  const float* row = scores + (size_t)b * N;
  u64 best = 0;
  for (int64_t i = lo + warp * 32; i < hi; i += kTopkThreads) {
    const int64_t n = i + lane;
    const u64 cand = (n < hi) ? make_key(row[n], (uint32_t)n) : 0ull;
    best = warp_offer(best, cand, lane);
  }
  lists[warp][lane] = best;
  __syncthreads();
  if (warp == 0) {
    for (int w = 1; w < kTopkThreads / 32; ++w) best = warp_merge_sorted(best, lists[w][lane], lane);
    partial[((size_t)b * S + blockIdx.x) * 32 + lane] = best;
  }
}

// stage 2: one warp per pair merges the S slice lists and decodes
__global__ void __launch_bounds__(32)
topk_final_kernel(const u64* __restrict__ partial, int S, int k, int64_t idx_offset,
                  float* __restrict__ val, int64_t* __restrict__ idx) {
  const int lane = threadIdx.x, b = blockIdx.x;
  u64 best = partial[(size_t)b * S * 32 + lane];
  for (int s = 1; s < S; ++s)
    best = warp_merge_sorted(best, partial[((size_t)b * S + s) * 32 + lane], lane);
  if (lane < k) {
    const bool valid = best != 0ull;
    val[(size_t)b * k + lane] = valid ? key_score(best) : -INFINITY;
    idx[(size_t)b * k + lane] = valid ? (int64_t)key_index(best) + idx_offset : (int64_t)-1;
  }
}

// merge [parts,B,k] lists of (value, global index).  Keys order by (score, low 32 bits of the index); the
// full 64-bit index is then read back from the winning entry, so global indices >= 2^32 are reported intact
// (only the tie order between equal scores whose indices agree in the low 32 bits is unspecified).
__global__ void __launch_bounds__(32)
topk_merge_kernel(const float* __restrict__ vals, const int64_t* __restrict__ idx, int parts, int B,
                  int k, float* __restrict__ out_val, int64_t* __restrict__ out_idx) {
  const int lane = threadIdx.x, b = blockIdx.x;
  const int total = parts * k;
  auto key_at = [&](int e) -> u64 {
    const int p = e / k, j = e % k;
    const size_t at = ((size_t)p * B + b) * k + j;
    const int64_t gi = idx[at];
    return gi >= 0 ? make_key(vals[at], (uint32_t)gi) : 0ull;
  };
  u64 best = 0;
  for (int i = 0; i < total; i += 32) {
    const int e = i + lane;
    best = warp_offer(best, e < total ? key_at(e) : 0ull, lane);
  }
  if (lane < k) {
    float v = -INFINITY;
    int64_t gi = -1;
    if (best != 0ull) {
      v = key_score(best);
      gi = (int64_t)key_index(best);
      for (int e = 0; e < total; ++e)
        if (key_at(e) == best) { gi = idx[((size_t)(e / k) * B + b) * k + e % k]; break; }
    }
    out_val[(size_t)b * k + lane] = v;
    out_idx[(size_t)b * k + lane] = gi;
  }
}

__global__ void gather_rotations_kernel(const float* __restrict__ R, int r_per_pair,
                                        const int64_t* __restrict__ idx, int64_t idx_offset, int B,
                                        int64_t N, int k, float* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * k * 9) return;
  const int e = t % 9, bj = t / 9, b = bj / k;
  const int64_t n = idx[bj] - idx_offset;
  float v = nanf("");
  if (n >= 0 && n < N) v = R[((r_per_pair ? (size_t)b * N : 0) + (size_t)n) * 9 + e];
  out[t] = v;
}

// ---- screened arg-max of ahv_verify (see launch_verify_tc_screened in ahv_score_tc.cu) --------------------------
// select: one CTA per pair collects the contenders {n : s16[b,n] >= m_b - 2 tau}, m_b = the pair's screened maximum
// (its arg-max key), in no particular order; pads to kScreenCap with the first; appends the strided probes.
constexpr int kSelectThreads = 512;
__global__ void __launch_bounds__(kSelectThreads)
screen_select_kernel(const float* __restrict__ s16, const u64* __restrict__ keys, int N, ScreenLists L) {
  __shared__ int cnt;
  __shared__ int sidx[kScreenCap];
  __shared__ float sval[kScreenCap];
  const int b = blockIdx.x, t = threadIdx.x;
  if (t == 0) {
    cnt = 0;
    if (b == 0) L.flagged[0] = 0;
  }
  __syncthreads();
  const float* row = s16 + (size_t)b * N;
  const float lo = key_score(keys[b]) - 2.0f * kScreenTau;  // NaN maximum: no contender, the pair is flagged
#pragma unroll 8
  for (int n = t; n < N; n += kSelectThreads) {
    const float v = row[n];
    if (v >= lo) {
      const int p = atomicAdd(&cnt, 1);
      if (p < kScreenCap) { sidx[p] = n; sval[p] = v; }
    }
  }
  __syncthreads();
  const int c = min(cnt, kScreenCap);
  for (int i = t; i < kScreenList; i += kSelectThreads) {
    int n;
    float v;
    if (i < c) {
      n = sidx[i]; v = sval[i];
    } else if (i < kScreenCap && c > 0) {
      n = sidx[0]; v = sval[0];
    } else {
      n = (int)((int64_t)(i < kScreenCap ? 0 : i - kScreenCap) * N / kScreenProbes);
      v = row[n];
    }
    L.idx[(size_t)b * kScreenList + i] = n;
    L.s16[(size_t)b * kScreenList + i] = v;
  }
  if (t == 0) L.count[b] = cnt;
}

// the rotations of every list entry, [B][kScreenList][9]: the fp32 pass scores them as per-pair rotation sets
__global__ void __launch_bounds__(kScreenList)
screen_gather_kernel(const float* __restrict__ R, int r_per_pair, int64_t N, ScreenLists L, float* __restrict__ R_list) {
  const size_t at = (size_t)blockIdx.x * kScreenList + threadIdx.x;
  const float* src = R + ((r_per_pair ? (size_t)blockIdx.x * N : 0) + (size_t)L.idx[at]) * 9;
#pragma unroll
  for (int e = 0; e < 9; ++e) R_list[at * 9 + e] = __ldg(src + e);
}

// guard: the list's fp32 arg-max key (original indices) replaces the pair's screened key; the pair is flagged for the
// exact pass when a realised |s32 - s16| on its list exceeds tau / 4 (or is NaN), or it had no or too many contenders
__global__ void __launch_bounds__(kScreenList)
screen_guard_kernel(const float* __restrict__ s32, ScreenLists L, u64* __restrict__ keys) {
  __shared__ u64 wkey[kScreenList / 32];
  __shared__ float werr[kScreenList / 32];
  const int b = blockIdx.x, t = threadIdx.x, lane = t & 31;
  const size_t at = (size_t)b * kScreenList + t;
  const float v = s32[at];
  float e = fabsf(v - L.s16[at]);
  const bool bad = !(e <= 0.25f * kScreenTau);
  u64 key = make_key(v, (uint32_t)L.idx[at]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    key = umax64(key, __shfl_xor_sync(0xffffffffu, key, o));
    e = fmaxf(e, __shfl_xor_sync(0xffffffffu, e, o));
  }
  if (lane == 0) { wkey[t >> 5] = key; werr[t >> 5] = e; }
  const int any_bad = __syncthreads_or(bad);
  if (t == 0) {
    for (int w = 1; w < kScreenList / 32; ++w) { key = umax64(key, wkey[w]); e = fmaxf(e, werr[w]); }
    keys[b] = key;
    L.err[b] = e;  // fmaxf skips NaN errors; they flag the pair all the same
    const int c = L.count[b];
    if (any_bad || c < 1 || c > kScreenCap) L.flagged[1 + atomicAdd(L.flagged, 1)] = b;
  }
}

int launch_screen_select(const float* s16, const u64* keys, int B, int64_t N, const float* R, int r_per_pair,
                         const ScreenLists& L, float* R_list, cudaStream_t s) {
  screen_select_kernel<<<B, kSelectThreads, 0, s>>>(s16, keys, (int)N, L);
  AHV_CUDA_OK(cudaGetLastError());
  // R_list overwrites s16: launched after every pair's selection
  screen_gather_kernel<<<B, kScreenList, 0, s>>>(R, r_per_pair, N, L, R_list);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

int launch_screen_guard(const float* s32, const ScreenLists& L, int B, u64* keys, cudaStream_t s) {
  screen_guard_kernel<<<B, kScreenList, 0, s>>>(s32, L, keys);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

static int slices_for(int64_t N) {
  int64_t s = N / 4096;
  if (s < 1) s = 1;
  if (s > 64) s = 64;
  return (int)s;
}

size_t topk_workspace_bytes(int B, int64_t N, int k) {
  (void)k;
  return (size_t)B * slices_for(N) * 32 * sizeof(u64);
}

int launch_topk(const float* scores, int B, int64_t N, int k, int64_t idx_offset, float* val,
                int64_t* idx, void* ws, size_t ws_bytes, cudaStream_t s) {
  if (B == 0) return AHV_OK;
  if (ws_bytes < topk_workspace_bytes(B, N, k)) return AHV_EWORKSPACE;
  const int S = slices_for(N);
  u64* partial = reinterpret_cast<u64*>(ws);
  topk_slice_kernel<<<dim3(S, B), kTopkThreads, 0, s>>>(scores, N, partial);
  AHV_CUDA_OK(cudaGetLastError());
  topk_final_kernel<<<B, 32, 0, s>>>(partial, S, k, idx_offset, val, idx);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

int launch_topk_merge(const float* vals, const int64_t* idx, int parts, int B, int k, float* out_val,
                      int64_t* out_idx, cudaStream_t s) {
  if (B == 0) return AHV_OK;
  topk_merge_kernel<<<B, 32, 0, s>>>(vals, idx, parts, B, k, out_val, out_idx);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

int launch_gather_rotations(const float* R, int r_per_pair, const int64_t* idx, int64_t idx_offset,
                            int B, int64_t N, int k, float* R_out, cudaStream_t s) {
  const int total = B * k * 9;
  if (total == 0) return AHV_OK;
  gather_rotations_kernel<<<(total + 255) / 256, 256, 0, s>>>(R, r_per_pair, idx, idx_offset, B, N, k,
                                                             R_out);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

}  // namespace ahv
