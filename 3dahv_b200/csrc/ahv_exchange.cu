// Top-k exchange of a hypothesis set sharded over the GPUs of one NVSwitch node (SURVEY.md §8e; the reference
// runs one GPU, batch 1): every rank holds the top-k of ITS shard per pair; this kernel writes them - score,
// global index and the rotation itself - into every peer's exchange buffer over NVLink, announces them with a
// sequence-numbered flag, waits for the peers' flags and merges (score descending, ties -> lowest global index),
// so that every rank ends with the bit-identical top-k over the WHOLE set and sampled_R[pred_index]
// (modules/model.py:195-196) without an NCCL call, a merge launch or a gather launch.  For k == 1 the scoring
// kernel does the same inside its own epilogue (ahv_tc_common.cuh::peer_exchange_and_merge); both share one
// buffer and one sequence counter (ahv_peer.cuh), so fused and top-k steps may alternate freely.
//
// One CTA: the payload is B*k*64 B per peer (256 KB at B=128, k=32) and the step is latency-bound.
#include <algorithm>

#include "ahv_peer.cuh"
#include "ahv_topk.cuh"

namespace ahv {

constexpr int kXchgThreads = 512, kXchgWarps = kXchgThreads / 32;

__global__ void __launch_bounds__(kXchgThreads)
topk_exchange_kernel(const float* __restrict__ val, const int64_t* __restrict__ idx, const float* __restrict__ R,
                     int r_per_pair, int64_t idx_offset, int64_t N, int B, int k, float* __restrict__ out_val,
                     int64_t* __restrict__ out_idx, float* __restrict__ R_best, peer::Args pa) {
  __shared__ u64 skeys[kXchgWarps][peer::kMaxPeers * kMaxK];
  __shared__ int s_ok;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned char* mine = pa.bufs[pa.rank];
  uint32_t* hdr = reinterpret_cast<uint32_t*>(mine);
  const uint32_t seq = *reinterpret_cast<volatile uint32_t*>(hdr) + 1u;  // every thread, before thread 0 updates it
  const int par = (int)(seq & 1u);
  if (tid == 0) s_ok = 1;
  // 1. this shard's lists -> every rank's buffer (NVLink peer stores; own buffer: local)
  for (int e = tid; e < B * k; e += kXchgThreads) {
    const int b = e / k, j = e - b * k;
    const int64_t gi = idx[e];
    const int64_t n = gi - idx_offset;
    float r9[9];
    const bool valid = gi >= 0 && n >= 0 && n < N;
    const float* src = R + ((r_per_pair ? (size_t)b * N : 0) + (size_t)(valid ? n : 0)) * 9;
#pragma unroll
    for (int q = 0; q < 9; ++q) r9[q] = valid ? __ldg(src + q) : 0.0f;
    const peer::Entry ent = peer::pack_entry(valid ? gi : -1, val[e], r9);
    for (int p = 0; p < pa.world; ++p)
      peer::store_entry(pa.bufs[p] + peer::entry_off(par, pa.rank, pa.cap_pairs, pa.cap_k, b, j), ent);
  }
  __threadfence_system();  // entries before the flag, system scope
  __syncthreads();
  // 2. announce, wait for the peers
  if (warp == 0) {
    peer::publish_flags(pa, seq, par, lane);
    if (!__all_sync(0xffffffffu, peer::wait_flags(pa, seq, par, lane)) && lane == 0) s_ok = 0;
  }
  __syncthreads();
  __threadfence_system();
  const bool ok = s_ok != 0;
  // 3. merge: one warp per pair
  const int total = pa.world * k;
  const float nanv = __int_as_float(0x7fc00000);
  for (int b = warp; b < B; b += kXchgWarps) {
    for (int e = lane; e < total; e += 32) {
      const int p = e / k, j = e - p * k;
      const uint4 q0 = __ldcv(reinterpret_cast<const uint4*>(mine + peer::entry_off(par, p, pa.cap_pairs, pa.cap_k, b, j)));
      const int64_t gi = peer::entry_index(q0);
      skeys[warp][e] = gi >= 0 ? make_key(__uint_as_float(q0.z), (uint32_t)gi) : 0ull;
    }
    __syncwarp();
    u64 best = 0;
    for (int i = 0; i < total; i += 32) best = warp_offer(best, i + lane < total ? skeys[warp][i + lane] : 0ull, lane);
    if (lane < k) {
      float v = -INFINITY;
      int64_t gi = -1;
      float o9[9];
#pragma unroll
      for (int q = 0; q < 9; ++q) o9[q] = nanv;
      if (best != 0ull) {
        int e = 0;
        while (e < total - 1 && skeys[warp][e] != best) ++e;  // the entry this key came from (payload lookup)
        const uint4* src = reinterpret_cast<const uint4*>(mine + peer::entry_off(par, e / k, pa.cap_pairs, pa.cap_k, b, e % k));
        const uint4 q0 = __ldcv(src), q1 = __ldcv(src + 1), q2 = __ldcv(src + 2);
        v = __uint_as_float(q0.z);
        gi = peer::entry_index(q0);
        peer::unpack_rotation(q0, q1, q2, o9);
      }
      out_val[(size_t)b * k + lane] = ok ? v : nanv;
      out_idx[(size_t)b * k + lane] = ok ? gi : -1;
      if (R_best) {
#pragma unroll
        for (int q = 0; q < 9; ++q) R_best[((size_t)b * k + lane) * 9 + q] = ok ? o9[q] : nanv;
      }
    }
    __syncwarp();
  }
  __syncthreads();
  if (tid == 0) {
    hdr[0] = seq;
    if (!ok) hdr[1] = 1u;
  }
}

int launch_topk_exchange(const float* val, const int64_t* idx, const float* R, int r_per_pair, int64_t idx_offset,
                         int64_t N, int B, int k, float* out_val, int64_t* out_idx, float* R_best,
                         const peer::Args& pa, cudaStream_t s) {
  if (pa.world < 2 || pa.world > peer::kMaxPeers || pa.rank < 0 || pa.rank >= pa.world) return AHV_EINVAL;
  if (B < 1 || k < 1 || k > kMaxK || B > pa.cap_pairs || k > pa.cap_k) return AHV_EINVAL;
  for (int r = 0; r < pa.world; ++r)
    if (!pa.bufs[r]) return AHV_EINVAL;
  topk_exchange_kernel<<<1, kXchgThreads, 0, s>>>(val, idx, R, r_per_pair, idx_offset, N, B, k, out_val, out_idx, R_best, pa);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

// ---- all-gather of a score matrix sliced by hypothesis (ahv_scores_exchange) ----------------------------------
// Every rank holds part = scores[:, lo:hi) of [B,N] (lo, hi = its shard_bounds) and stores it into every rank's
// score region (ahv_peer.cuh).  The payload (B*(hi-lo)*4 B per peer, 3.2 MB at 128 x 50 000 over 8 ranks) is spread
// over a grid; each CTA fences its stores and takes a ticket, and only the CTA that takes the last ticket announces
// the exchange and spins on the peers' flags - so at most one CTA per rank waits, and the grids of two ranks sharing
// one GPU need not be co-resident.  score_copyout_kernel, the next launch on the stream, moves the matrix out.
constexpr int kScoreXchgThreads = 256;

__global__ void __launch_bounds__(kScoreXchgThreads)
scores_exchange_kernel(const float* __restrict__ part, int64_t lo, int64_t width, int B, peer::Args pa, int64_t cap_hyps) {
  __shared__ int s_last;
  const int tid = threadIdx.x;
  unsigned char* mine = pa.bufs[pa.rank];
  uint32_t* hdr = reinterpret_cast<uint32_t*>(mine);
  const uint32_t seq = *reinterpret_cast<volatile uint32_t*>(hdr) + 1u;  // read before this CTA takes its ticket
  const int par = (int)(seq & 1u);
  const int64_t total = (int64_t)B * width;
  for (int64_t e = (int64_t)blockIdx.x * kScoreXchgThreads + tid; e < total; e += (int64_t)gridDim.x * kScoreXchgThreads) {
    const int b = (int)(e / width);
    const int64_t n = e - (int64_t)b * width;
    const float v = __ldg(part + e);
    for (int p = 0; p < pa.world; ++p)
      *reinterpret_cast<float*>(pa.bufs[p] + peer::score_off(par, pa.cap_pairs, pa.cap_k, cap_hyps, b, lo + n)) = v;
  }
  __threadfence_system();  // this CTA's stores before its ticket, system scope
  __syncthreads();
  if (tid == 0) s_last = atomicAdd(hdr + peer::kHdrTicket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last || tid >= 32) return;
  __threadfence_system();  // every CTA's stores (seen through the tickets) before the flags
  peer::publish_flags(pa, seq, par, tid);
  const bool ok = __all_sync(0xffffffffu, peer::wait_flags(pa, seq, par, tid));
  __threadfence_system();
  if (tid == 0) {
    hdr[peer::kHdrTicket] = 0u;
    hdr[peer::kHdrScoresStatus] = ok ? 0u : 1u;
    if (!ok) hdr[1] = 1u;
    hdr[0] = seq;
  }
}

// The exchange just completed (header word 0) -> out [B,N]; NaN everywhere if it timed out.
__global__ void __launch_bounds__(kScoreXchgThreads)
score_copyout_kernel(const unsigned char* __restrict__ mine, int cap_pairs, int cap_k, int64_t cap_hyps, int B, int64_t N,
                     float* __restrict__ out) {
  const volatile uint32_t* hdr = reinterpret_cast<const volatile uint32_t*>(mine);
  const int par = (int)(hdr[0] & 1u);
  const bool ok = hdr[peer::kHdrScoresStatus] == 0u;
  const float nanv = __int_as_float(0x7fc00000);
  const int64_t total = (int64_t)B * N;
  for (int64_t e = (int64_t)blockIdx.x * kScoreXchgThreads + threadIdx.x; e < total; e += (int64_t)gridDim.x * kScoreXchgThreads) {
    const int b = (int)(e / N);
    const int64_t n = e - (int64_t)b * N;
    out[e] = ok ? __ldcv(reinterpret_cast<const float*>(mine + peer::score_off(par, cap_pairs, cap_k, cap_hyps, b, n))) : nanv;
  }
}

static unsigned grid_for(int64_t total, int max_ctas) {
  const int64_t want = (total + kScoreXchgThreads * 8 - 1) / (kScoreXchgThreads * 8);  // ~8 elements per thread
  return (unsigned)(want < 1 ? 1 : (want > max_ctas ? max_ctas : want));
}

int launch_scores_exchange(const float* part, int B, int64_t N, float* out, const peer::Args& pa, int64_t cap_hyps,
                           cudaStream_t s) {
  if (pa.world < 2 || pa.world > peer::kMaxPeers || pa.rank < 0 || pa.rank >= pa.world) return AHV_EINVAL;
  if (B < 1 || N < 1 || B > pa.cap_pairs || N > cap_hyps) return AHV_EINVAL;
  for (int r = 0; r < pa.world; ++r)
    if (!pa.bufs[r]) return AHV_EINVAL;
  const int64_t per = (N + pa.world - 1) / pa.world;  // dist.shard_bounds
  const int64_t lo = std::min(N, (int64_t)pa.rank * per), hi = std::min(N, lo + per);
  int dev = 0, sms = 0;
  AHV_CUDA_OK(cudaGetDevice(&dev));
  AHV_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  scores_exchange_kernel<<<grid_for((int64_t)B * (hi - lo), 2 * sms), kScoreXchgThreads, 0, s>>>(part, lo, hi - lo, B, pa,
                                                                                                  cap_hyps);
  AHV_CUDA_OK(cudaGetLastError());
  score_copyout_kernel<<<grid_for((int64_t)B * N, 4 * sms), kScoreXchgThreads, 0, s>>>(pa.bufs[pa.rank], pa.cap_pairs, pa.cap_k,
                                                                                        cap_hyps, B, N, out);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

// ---- gather of ascended slots (ahv_refine_gradient_sharded) ---------------------------------------------------
// Rank r has ascended items [item_lo, item_hi) of the B*k (pair, slot) items, in R_all / score_all; the others hold
// the rest.  Each item travels as the 64-byte entry {item, score, R[9]} to every rank's entries region, at (b, j) of
// rank plane 0 (the item ranges are disjoint, so no two ranks write one entry), and is copied back into R_all /
// score_all on every rank: bits, not keys, so NaN rotations and -inf scores of empty slots arrive unchanged.  One CTA:
// B*k*64 B in all (256 KB at B = 128, k = 32).
__global__ void __launch_bounds__(kXchgThreads)
slot_gather_kernel(float* __restrict__ R_all, float* __restrict__ score_all, int64_t item_lo, int64_t item_hi, int B, int k,
                   peer::Args pa) {
  __shared__ int s_ok;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned char* mine = pa.bufs[pa.rank];
  uint32_t* hdr = reinterpret_cast<uint32_t*>(mine);
  const uint32_t seq = *reinterpret_cast<volatile uint32_t*>(hdr) + 1u;
  const int par = (int)(seq & 1u);
  if (tid == 0) s_ok = 1;
  for (int64_t it = item_lo + tid; it < item_hi; it += kXchgThreads) {
    const int b = (int)(it / k), j = (int)(it - (int64_t)b * k);
    float r9[9];
#pragma unroll
    for (int q = 0; q < 9; ++q) r9[q] = R_all[it * 9 + q];
    const peer::Entry ent = peer::pack_entry(it, score_all[it], r9);
    for (int p = 0; p < pa.world; ++p)
      peer::store_entry(pa.bufs[p] + peer::entry_off(par, 0, pa.cap_pairs, pa.cap_k, b, j), ent);
  }
  __threadfence_system();
  __syncthreads();
  if (warp == 0) {
    peer::publish_flags(pa, seq, par, lane);
    if (!__all_sync(0xffffffffu, peer::wait_flags(pa, seq, par, lane)) && lane == 0) s_ok = 0;
  }
  __syncthreads();
  __threadfence_system();
  const bool ok = s_ok != 0;
  const float nanv = __int_as_float(0x7fc00000);
  for (int e = tid; e < B * k; e += kXchgThreads) {
    const int b = e / k, j = e - b * k;
    const uint4* src = reinterpret_cast<const uint4*>(mine + peer::entry_off(par, 0, pa.cap_pairs, pa.cap_k, b, j));
    const uint4 q0 = __ldcv(src), q1 = __ldcv(src + 1), q2 = __ldcv(src + 2);
    float o9[9];
    peer::unpack_rotation(q0, q1, q2, o9);
    score_all[e] = ok ? __uint_as_float(q0.z) : nanv;
#pragma unroll
    for (int q = 0; q < 9; ++q) R_all[(size_t)e * 9 + q] = ok ? o9[q] : nanv;
  }
  __syncthreads();
  if (tid == 0) {
    hdr[0] = seq;
    if (!ok) hdr[1] = 1u;
  }
}

int launch_slot_gather(float* R_all, float* score_all, int64_t item_lo, int64_t item_hi, int B, int k, const peer::Args& pa,
                       cudaStream_t s) {
  if (pa.world < 2 || pa.world > peer::kMaxPeers || pa.rank < 0 || pa.rank >= pa.world) return AHV_EINVAL;
  if (B < 1 || k < 1 || k > kMaxK || B > pa.cap_pairs || k > pa.cap_k) return AHV_EINVAL;
  if (item_lo < 0 || item_hi < item_lo || item_hi > (int64_t)B * k) return AHV_EINVAL;
  for (int r = 0; r < pa.world; ++r)
    if (!pa.bufs[r]) return AHV_EINVAL;
  slot_gather_kernel<<<1, kXchgThreads, 0, s>>>(R_all, score_all, item_lo, item_hi, B, k, pa);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

// With lazy module loading (the CUDA default) a kernel is loaded at its first launch, and loading synchronises the
// context.  A rank whose first exchanging call is enqueued while another stream of the same device spins on it (ranks
// that share a GPU in one process) would then wait for that spin to time out.  ahv_peer_alloc_ex loads the
// exchanging kernels, and the ascent's ranged instances that run between two exchanges, up front.
int preload_exchange_kernels() {
  cudaFuncAttributes a;
  AHV_CUDA_OK(cudaFuncGetAttributes(&a, topk_exchange_kernel));
  AHV_CUDA_OK(cudaFuncGetAttributes(&a, scores_exchange_kernel));
  AHV_CUDA_OK(cudaFuncGetAttributes(&a, score_copyout_kernel));
  AHV_CUDA_OK(cudaFuncGetAttributes(&a, slot_gather_kernel));
  return preload_ranged_ascent();
}

}  // namespace ahv
