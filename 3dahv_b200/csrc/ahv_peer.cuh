// Peer-exchange buffer shared by the sharded verification step (SURVEY.md §8e; the reference is single GPU):
// one buffer per rank (ahv_peer_alloc, a zeroed cudaMalloc), IPC-mapped into every peer of the node.
//   [0,256)    header: uint32 seq (exchanges this rank has completed), uint32 err, uint32 cap_pairs, uint32 cap_k
//   [256,512)  flags[2 parity][8 ranks] uint32: flags[par][r] == s  <=>  rank r's entries of exchange s are here
//   [512,...)  entries[2 parity][8 ranks][cap_pairs][cap_k] x 64 B: {int64 global index, float score, float R[9], pad}
// The entry stride depends only on the CAPACITY the buffer was allocated with, never on the B or k of a call, so
// exchanges of different sizes may follow one another.  Exchange s uses parity s & 1.  A rank can only finish
// exchange s+1 after every peer has sent s+1, i.e. after every peer is done reading exchange s, so two parities
// suffice; sequence numbers make the flags self-cleaning (CUDA-graph replay needs no host-side reset).
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
};

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

__device__ __forceinline__ uint32_t ordered_bits(float score) {  // same order as make_key()
  uint32_t u = __float_as_uint(score + 0.0f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
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
__device__ __forceinline__ void store_entry(unsigned char* dst, const Entry& e) {
  uint4* d = reinterpret_cast<uint4*>(dst);
  d[0] = e.q0; d[1] = e.q1; d[2] = e.q2;
}
__device__ __forceinline__ int64_t entry_index(const uint4& q0) { return (int64_t)(((u64)q0.y << 32) | q0.x); }
__device__ __forceinline__ void unpack_rotation(const uint4& q0, const uint4& q1, const uint4& q2, float* o9) {
  o9[0] = __uint_as_float(q0.w);
  o9[1] = __uint_as_float(q1.x); o9[2] = __uint_as_float(q1.y); o9[3] = __uint_as_float(q1.z); o9[4] = __uint_as_float(q1.w);
  o9[5] = __uint_as_float(q2.x); o9[6] = __uint_as_float(q2.y); o9[7] = __uint_as_float(q2.z); o9[8] = __uint_as_float(q2.w);
}

// lanes < world: announce exchange `seq` to peer `lane` (after the entries, which the caller fenced)
__device__ __forceinline__ void publish_flags(const Args& pa, uint32_t seq, int par, int lane) {
  if (lane < pa.world) {
    volatile uint32_t* flag = reinterpret_cast<volatile uint32_t*>(pa.bufs[lane] + kFlagsOff) + par * kMaxPeers + pa.rank;
    *flag = seq;
  }
}
// lanes < world: wait until peer `lane` has announced exchange `seq` in OUR buffer; false on timeout.
// Ranks may reach a step seconds apart (host-side skew); only a peer that never arrives is turned into an
// error (NaN results, index -1, header error word) instead of a GPU that hangs forever.
__device__ __forceinline__ bool wait_flags(const Args& pa, uint32_t seq, int par, int lane) {
  bool ok = true;
  if (lane < pa.world) {
    const volatile uint32_t* flag = reinterpret_cast<const volatile uint32_t*>(pa.bufs[pa.rank] + kFlagsOff) + par * kMaxPeers + lane;
    const long long t0 = clock64();
    while (*flag != seq) {
      if (clock64() - t0 > kSpinTimeoutClocks) { ok = false; break; }
    }
  }
  return ok;
}

}  // namespace peer
}  // namespace ahv
