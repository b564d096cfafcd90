// Peer-exchange buffer shared by the sharded verification step (SURVEY.md §8e; the reference is single GPU):
// one buffer per rank (ahv_peer_alloc, a zeroed cudaMalloc), IPC-mapped into every peer of the node.
//   [0,256)    header: uint32 seq (exchanges this rank has completed), uint32 err, uint32 cap_pairs, uint32 cap_k
//   [256,512)  flags[2 parity][8 ranks] uint32: flags[par][r] == s  <=>  rank r's entries of exchange s are here
//   [512,...)  entries[2 parity][8 ranks][cap_pairs][cap_k] x 64 B: {int64 global index, float score, float R[9], pad}
// The entry stride depends only on the CAPACITY the buffer was allocated with, never on the B or k of a call, so
// exchanges of different sizes may follow one another.  Exchange s uses parity s & 1.  A rank stores the entries of
// exchange s+2 into the plane of s only after it has finished exchange s+1, which needs every peer's flag s+1, and a
// peer announces s+1 only after it has read exchange s, so two parities suffice; sequence numbers make the flags
// self-cleaning (CUDA-graph replay needs no host-side reset).
//
// Every exchanging kernel takes one step of the protocol below: open (seq, par), store_to_all (its entries into
// every rank's buffer), announce_and_wait (fence, flags, spin on the peers' flags, fence), load_head / load_entry (the
// peers' entries, from its own buffer), close (header word 0 = seq, and the error word on a timeout).
//
// Optional score region (ahv_peer_alloc_ex with max_hyps > 0; cap_hyps is header word 4, 0 = none):
//   [entries end, ...)  scores[2 parity][cap_pairs][cap_hyps] fp32: exchange s of ahv_scores_exchange leaves the
//                       whole [B,N] matrix in every rank's parity s & 1 plane (each rank stores its columns [lo,hi))
// Header words 5 and 6 are private to the owning rank: the CTA ticket of a scores exchange (back to 0 when the
// exchange ends) and that exchange's outcome (0 = complete, 1 = a peer never arrived), read by the copy-out.
// The stride again depends on the capacity only.  Two parities suffice here as well, because the matrix is read
// out of the region by a SECOND, stream-ordered launch (score_copyout_kernel) that precedes the rank's next
// exchanging launch: rank q announces exchange s+1 only after it has copied exchange s out, so a peer that sees
// q's flag s+1 (which it must before it completes s+1 and starts s+2, the next user of the plane) can no longer
// overwrite anything q has still to read.  A caller that inserted another exchanging launch between the two would
// break this; the entry points never do.
#pragma once
#include <algorithm>

#include "ahv_common.cuh"

namespace ahv {
namespace peer {

constexpr int kMaxPeers = 8;  // GPUs of one NVSwitch node
constexpr int kFlagsOff = 256, kEntriesOff = 512, kEntryBytes = 64;
constexpr long long kSpinTimeoutClocks = 40000000000LL;  // ~20 s at 2 GHz

struct Args {  // by-value kernel argument
  int rank = 0, world = 1;
  int cap_pairs = 0, cap_k = 0;
  unsigned char* bufs[kMaxPeers] = {};  // bufs[r] = rank r's buffer as mapped in this process

  // rank of a group of 2 to kMaxPeers ranks, every buffer mapped, room for 1 to kMaxK entries per pair
  __host__ bool valid() const {
    if (world < 2 || world > kMaxPeers || rank < 0 || rank >= world) return false;
    for (int r = 0; r < world; ++r)
      if (!bufs[r]) return false;
    return cap_pairs >= 1 && cap_k >= 1 && cap_k <= kMaxK;
  }
  // a valid group whose buffers hold a call of B pairs: k entries per pair and, unless hyps == 0, hyps scores per pair
  // in a score region of cap_hyps (header word 4)
  __host__ bool fits(int B, int k, int64_t hyps = 0, int64_t cap_hyps = 0) const {
    return valid() && B >= 1 && B <= cap_pairs && k >= 0 && k <= cap_k && (hyps == 0 || hyps <= cap_hyps);
  }
};

// dist.shard_bounds: rank's contiguous share [lo, hi) of n items
__host__ inline void shard_bounds(int64_t n, int rank, int world, int64_t* lo, int64_t* hi) {
  const int64_t per = (n + world - 1) / world;
  *lo = std::min(n, (int64_t)rank * per);
  *hi = std::min(n, *lo + per);
}

__host__ __device__ inline size_t entry_off(int par, int r, int cap_pairs, int cap_k, int b, int j) {
  return (size_t)kEntriesOff + ((((size_t)par * kMaxPeers + r) * cap_pairs + b) * cap_k + j) * kEntryBytes;
}
__host__ inline size_t buffer_bytes(int cap_pairs, int cap_k) { return entry_off(2, 0, cap_pairs, cap_k, 0, 0); }
constexpr int kHdrCapHyps = 4, kHdrTicket = 5, kHdrScoresStatus = 6;  // uint32 header words of the score region
__host__ __device__ inline size_t score_off(int par, int cap_pairs, int cap_k, int64_t cap_hyps, int b, int64_t n) {
  return entry_off(2, 0, cap_pairs, cap_k, 0, 0) + (((size_t)par * cap_pairs + b) * (size_t)cap_hyps + (size_t)n) * sizeof(float);
}
__host__ inline size_t buffer_bytes_ex(int cap_pairs, int cap_k, int64_t cap_hyps) {
  return score_off(2, cap_pairs, cap_k, cap_hyps, 0, 0);
}

// one 64-byte entry as three 16-byte words
struct Entry {
  uint4 q0, q1, q2;
};
__device__ __forceinline__ Entry pack_entry(int64_t gidx, float score, const float* r9) {
  Entry e;
  e.q0 = make_uint4((uint32_t)gidx, (uint32_t)((u64)gidx >> 32), __float_as_uint(score), __float_as_uint(r9[0]));
  e.q1 = make_uint4(__float_as_uint(r9[1]), __float_as_uint(r9[2]), __float_as_uint(r9[3]), __float_as_uint(r9[4]));
  e.q2 = make_uint4(__float_as_uint(r9[5]), __float_as_uint(r9[6]), __float_as_uint(r9[7]), __float_as_uint(r9[8]));
  return e;
}
__device__ __forceinline__ int64_t entry_index(const uint4& q0) { return (int64_t)(((u64)q0.y << 32) | q0.x); }
__device__ __forceinline__ float entry_score(const uint4& q0) { return __uint_as_float(q0.z); }
__device__ __forceinline__ void unpack_rotation(const Entry& e, float* o9) {
  o9[0] = __uint_as_float(e.q0.w);
  o9[1] = __uint_as_float(e.q1.x); o9[2] = __uint_as_float(e.q1.y); o9[3] = __uint_as_float(e.q1.z); o9[4] = __uint_as_float(e.q1.w);
  o9[5] = __uint_as_float(e.q2.x); o9[6] = __uint_as_float(e.q2.y); o9[7] = __uint_as_float(e.q2.z); o9[8] = __uint_as_float(e.q2.w);
}

// ---- one exchange step ----------------------------------------------------------------------------------------
struct Step {
  uint32_t seq;  // this exchange: one more than the exchanges this rank has completed (header word 0)
  int par;       // its plane, seq & 1
};

// Read before this launch's close can advance the header: in a one-CTA kernel (or the scoring kernel's one warp) by
// every thread, ahead of the barrier that precedes close; in the score exchange by each CTA before it takes its
// ticket, since the CTA that takes the last one closes.
__device__ __forceinline__ Step open(const Args& pa) {
  const uint32_t seq = *reinterpret_cast<volatile uint32_t*>(pa.bufs[pa.rank]) + 1u;
  return {seq, (int)(seq & 1u)};
}

// In a launch that follows this rank's last close on its stream: the plane of the exchange that close completed.
__device__ __forceinline__ int closed_par(const unsigned char* mine) {
  return (int)(*reinterpret_cast<const volatile uint32_t*>(mine) & 1u);
}

// Into every rank's buffer (NVLink peer stores; our own buffer: local): entry e as entry (b, j) of rank plane r, or
// score v as score (b, n) of a score region of cap_hyps.
__device__ __forceinline__ void store_to_all(const Args& pa, Step st, int r, int b, int j, const Entry& e) {
  for (int p = 0; p < pa.world; ++p) {
    uint4* d = reinterpret_cast<uint4*>(pa.bufs[p] + entry_off(st.par, r, pa.cap_pairs, pa.cap_k, b, j));
    d[0] = e.q0; d[1] = e.q1; d[2] = e.q2;
  }
}
__device__ __forceinline__ void store_to_all(const Args& pa, Step st, int64_t cap_hyps, int b, int64_t n, float v) {
  for (int p = 0; p < pa.world; ++p)
    *reinterpret_cast<float*>(pa.bufs[p] + score_off(st.par, pa.cap_pairs, pa.cap_k, cap_hyps, b, n)) = v;
}

// One warp, once every store of this rank's exchange is ordered before it: the warp's own, the rest of its CTA's
// through a __syncthreads before the call (the barrier orders them before this warp's fence, which is cumulative),
// and the other CTAs' of a score exchange through their fenced tickets.  Lanes < world announce exchange st.seq to
// peer `lane`, then wait until that peer has announced it in OUR buffer.  The fence after the wait orders the reads
// of the peers' entries after their flags, for the whole CTA when a __syncthreads follows.  False on every lane when
// a peer did not arrive within kSpinTimeoutClocks: ranks may reach a step seconds apart (host-side skew), and only a
// peer that never arrives is turned into an error (NaN results, index -1, header error word) instead of a GPU that
// hangs forever.
__device__ __forceinline__ bool announce_and_wait(const Args& pa, Step st, int lane) {
  __threadfence_system();  // the entries before the flags, system scope
  __syncwarp();
  if (lane < pa.world)
    *(reinterpret_cast<volatile uint32_t*>(pa.bufs[lane] + kFlagsOff) + st.par * kMaxPeers + pa.rank) = st.seq;
  bool ok = true;
  if (lane < pa.world) {
    const volatile uint32_t* flag = reinterpret_cast<const volatile uint32_t*>(pa.bufs[pa.rank] + kFlagsOff) + st.par * kMaxPeers + lane;
    const long long t0 = clock64();
    while (*flag != st.seq) {
      if (clock64() - t0 > kSpinTimeoutClocks) { ok = false; break; }
    }
  }
  ok = __all_sync(0xffffffffu, ok);
  __threadfence_system();
  return ok;
}

// The peers' entries in our own buffer, written by other GPUs: read past the caches (__ldcv).  load_head reads the
// first 16 bytes, the index and the score.
__device__ __forceinline__ uint4 load_head(const unsigned char* p) { return __ldcv(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ Entry load_entry(const unsigned char* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  return {__ldcv(q), __ldcv(q + 1), __ldcv(q + 2)};
}

// One thread, after every read of the exchange from our buffer: exchange st.seq is complete; a timeout also sets
// the error word.
__device__ __forceinline__ void close(const Args& pa, Step st, bool ok) {
  uint32_t* hdr = reinterpret_cast<uint32_t*>(pa.bufs[pa.rank]);
  hdr[0] = st.seq;
  if (!ok) hdr[1] = 1u;
}

}  // namespace peer
}  // namespace ahv
