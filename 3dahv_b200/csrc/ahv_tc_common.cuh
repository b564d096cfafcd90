// Building blocks of the tensor-core scoring kernel (see ahv_score_tc.cu for the overview):
// warp roles and pipeline barriers, the per-CTA work range and 32-bit tile iterator, in-kernel weight
// packing and pair-volume staging (power-of-two pre-scale), and the epilogue role (ReLU -> conv2 operand,
// normalise -> correlate -> mean -> score, running arg-max, fused winner decode).
#pragma once
#include "ahv_peer.cuh"
#include "ahv_tc_ptx.cuh"

namespace ahv {
namespace tc {

// Optional in-kernel timeline (build with -DAHV_TIMELINE, read with ahv_diag_timeline): globaltimer stamps
// of the TS kernel's setup / first-tile milestones per CTA, used to attribute the fixed cost of a launch.
#ifdef AHV_TIMELINE
__device__ unsigned long long g_timeline[160][16];
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define AHV_TL(i) g_timeline[blockIdx.x][i] = gtimer()
#else
#define AHV_TL(i) ((void)0)
#endif

constexpr int kGatherWarps = 8;
constexpr int kEpiWarp0 = 8;
constexpr int kMmaWarp = 12;
constexpr int kThreadsTC = 13 * 32;
#ifndef AHV_STAGES
#define AHV_STAGES 3
#endif
constexpr int kStages = AHV_STAGES;  // A-operand pipeline depth (a stage = one tile = two hypotheses)

// ---- shared memory map (bytes) ----
constexpr int kW1Bytes = 24 * 1024;  // 24 MMA slices x [2 chalf][4 ngroup][8][8] fp16
constexpr int kW2Bytes = 2 * 1024;

enum Bar { kFull = 0, kEmpty = 3, kD1Full = 6, kD1Empty = 8, kA2Full = 10, kD2Full = 12, kVolFull = 14 };

// 1.0f the compiler cannot fold.  The rotation prefetch is loop-carried in registers; multiplying the
// values loaded BEFORE the loop by this makes every loop-entry value ALU-defined, so the first use at
// the loop top carries no scoreboard wait - otherwise that wait (on the scoreboard the just-issued
// prefetch of the NEXT tile also uses) stalls the warp for a full L2 round trip per tile.
__device__ __forceinline__ float opaque_one(int flag01) { return __uint_as_float(0x3f800000u + ((uint32_t)flag01 >> 8)); }

// Fused selection epilogue (modules/model.py:195-196): the last CTA to finish decodes the arg-max keys
// into (score, global index, sampled_R[pred_index]) per pair.  val == nullptr disables it.
struct Finalize {
  float* val = nullptr;
  int64_t* idx = nullptr;
  float* R_best = nullptr;
  int64_t idx_offset = 0;
  unsigned* counter = nullptr;  // zero at kernel start (cleared with the keys), reset by the last CTA
  // training forward (kSave instantiation only): conv1's ReLU'd output of every item, fp16 in the units the kernel
  // computed it in (pair scale s, normalised W1) [B*N][64 positions][32 channels], and per pair the factor that turns
  // it back into conv1's output, 2^e1 / s - the fused backward reads them instead of recomputing conv1 (4 KB per
  // item; the reference's autograd saves ~420 KB per hypothesis)
  __half* h1_out = nullptr;
  float* pair_inv_out = nullptr;
  // hypothesis set sharded over `peers.world` GPUs (SURVEY.md §8e): the winners are exchanged through peer
  // memory by this kernel itself (no NCCL call, no merge kernel); see ahv_peer.cuh for the buffer
  peer::Args peers;
};

// Last CTA of rank `rank`: publish this shard's winners to every peer, wait for theirs, merge
// (higher score wins, ties -> lowest global index, like torch.max on the unsharded set; every rank computes
// the same result).  One warp.  A step that timed out waiting for a peer returns NaN score, index -1 and a NaN
// rotation, and sets the header's error word.
__device__ __forceinline__ void peer_exchange_and_merge(const Finalize& fin, const u64* best_keys, const float* R,
                                                        int r_per_pair, int64_t N, int B, int lane) {
  const peer::Args& pa = fin.peers;
  const unsigned char* mine = pa.bufs[pa.rank];
  const peer::Step st = peer::open(pa);
  for (int b = lane; b < B; b += 32) {
    const u64 key = __ldcg(best_keys + b);
    const uint32_t n = key_index(key);
    const float* src = R + ((r_per_pair ? (size_t)b * N : 0) + (size_t)n) * 9;
    float r9[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) r9[e] = __ldg(src + e);
    const peer::Entry ent = peer::pack_entry((int64_t)n + fin.idx_offset, key_score(key), r9);
    peer::store_to_all(pa, st, pa.rank, b, 0, ent);
  }
  const bool ok = peer::announce_and_wait(pa, st, lane);
  for (int b = lane; b < B; b += 32) {
    uint32_t bo = 0;
    int64_t bi = -1;
    peer::Entry be = {};
    for (int r = 0; r < pa.world; ++r) {
      const unsigned char* e = mine + peer::entry_off(st.par, r, pa.cap_pairs, pa.cap_k, b, 0);
      const uint4 q0 = peer::load_head(e);
      const int64_t gi = peer::entry_index(q0);
      const uint32_t o = score_bits(peer::entry_score(q0));
      if (bi < 0 || o > bo || (o == bo && gi < bi)) {
        bo = o; bi = gi; be = peer::load_entry(e);
      }
    }
    const float nanv = __int_as_float(0x7fc00000);
    fin.val[b] = ok ? peer::entry_score(be.q0) : nanv;
    fin.idx[b] = ok ? bi : -1;
    if (fin.R_best) {
      float o9[9];
      peer::unpack_rotation(be, o9);
#pragma unroll
      for (int e = 0; e < 9; ++e) fin.R_best[b * 9 + e] = ok ? o9[e] : nanv;
    }
  }
  __syncwarp();
  if (lane == 0) peer::close(pa, st, ok);
}

struct Work {  // contiguous range of (pair, hypothesis) items of this CTA
  int64_t lo, hi, N;
  // pairs of the item range are the listed ones when set (the fallback pass of the screened arg-max scores only the
  // pairs it flagged): item pair b is pair map[b].  The ring of pair scales stays indexed by the item pair.
  const int* map = nullptr;
  __device__ __forceinline__ int pair(int b) const { return map ? __ldg(map + b) : b; }
};

// Ticket of a CTA whose keys are published: the last CTA of the grid decodes the arg-max keys into (score, index,
// rotation), or exchanges and merges them with the peers' when the set is sharded.  One warp.
__device__ __forceinline__ void finalize_ticket(const Finalize& fin, const u64* best_keys, const float* R, int r_per_pair,
                                                int64_t N, int B, int lane) {
  __syncwarp();
  unsigned last = 0;
  if (lane == 0) {
    __threadfence();  // this CTA's keys before its ticket
    last = atomicAdd(fin.counter, 1u) == gridDim.x - 1;
  }
  last = __shfl_sync(0xffffffffu, last, 0);
  if (last && fin.peers.world > 1) {
    __threadfence();
    peer_exchange_and_merge(fin, best_keys, R, r_per_pair, N, B, lane);
    if (lane == 0) *fin.counter = 0u;
  } else if (last) {  // every other CTA has published its keys
    __threadfence();
    for (int b = lane; b < B; b += 32) {
      const u64 key = __ldcg(best_keys + b);
      const uint32_t n = key_index(key);
      fin.val[b] = key_score(key);
      fin.idx[b] = (int64_t)n + fin.idx_offset;
      if (fin.R_best) {
        const float* src = R + ((r_per_pair ? (size_t)b * N : 0) + (size_t)n) * 9;
#pragma unroll
        for (int e = 0; e < 9; ++e) fin.R_best[b * 9 + e] = __ldg(src + e);
      }
    }
    if (lane == 0) *fin.counter = 0u;
  }
}

// tile = two consecutive hypotheses of one pair; advance() returns false when exhausted.  All per-tile
// state is 32-bit (N <= 2^31-1 and the CTA's share of B*N < 2^32 are checked on the host): the iterator
// runs once per tile in every role.
struct TileIter {
  uint32_t n, N, left;  // next hypothesis within the pair, hypotheses per pair, items left for this CTA
  int b;
  uint32_t n0;  // first hypothesis of the tile
  int cnt;      // 1 or 2 valid hypotheses
  __device__ __forceinline__ TileIter(const Work& w) : N((uint32_t)w.N), left((uint32_t)(w.hi - w.lo)), n0(0), cnt(0) {
    b = (int)(w.lo / w.N);
    n = (uint32_t)(w.lo - (int64_t)b * w.N);
  }
  __device__ __forceinline__ bool advance() {
    if (left == 0) return false;
    if (n == N) { ++b; n = 0; }
    n0 = n;
    const uint32_t room = min(N - n, left);
    cnt = room >= 2 ? 2 : 1;
    n += cnt;
    left -= cnt;
    return true;
  }
  // (pair, first hypothesis, count) of the tile the next advance() will produce; at the very end the
  // current tile again (a harmless, valid address for the rotation prefetch)
  __device__ __forceinline__ void peek_tile(int& pb, uint32_t& pn, int& pc) const {
    if (left == 0) { pb = b; pn = n0; pc = cnt > 0 ? cnt : 1; return; }
    pb = b; pn = n;
    if (n == N) { ++pb; pn = 0; }
    pc = min(N - pn, left) >= 2 ? 2 : 1;
  }
  // Looking two tiles ahead (after advance() produced tile t): does tile t+2 exist and start a new pair?  pb2 = that
  // pair.  (Tiles never straddle pairs; tile t+1 = {pair b or b+1, 1 or 2 hypotheses}.)
  __device__ __forceinline__ bool second_next_starts_pair(int& pb2, uint32_t& left2) const {
    if (left == 0) return false;
    int b1 = b;
    uint32_t n1 = n;
    if (n1 == N) { ++b1; n1 = 0; }
    const uint32_t c1 = min(N - n1, left) >= 2 ? 2u : 1u;
    n1 += c1;
    left2 = left - c1;
    pb2 = b1 + 1;
    return left2 > 0 && n1 == N;
  }
  // (pair, hypothesis) of the item following this tile, or the tile's own first item at the very end
  __device__ __forceinline__ void peek(int& pb, uint32_t& pn) const {
    if (left == 0) { pb = b; pn = n0; }
    else if (n == N) { pb = b + 1; pn = 0; }
    else { pb = b; pn = n; }
  }
};

// What undoes the normalisation: 2^e1 (conv1's output = its normalised form * w1) and 2^(e1+e2) (conv2's)
struct WeightScale {
  float w1 = 1.0f, w12 = 1.0f;
};

// ---- one-time per CTA: W1/W2 (fp32, global) -> normalised fp16 UMMA B-operand layouts in shared memory ------------
// conv1: 24 slices j = (view, kk), each [chalf][ngroup][n%8][c%8]; conv2: [kc][ngroup][8][8] behind them.
// Every CTA does this itself (52 KB of L2 reads, twice) so that the scoring kernel depends on no preparation kernel.
// It runs on the 5 non-gather warps (MMA + epilogue, tid = 0..159) while the gather warps already stage the first
// volume and resample the first tile; the MMA warp is released by named barrier 3.  l1max_bits[2] (zero on entry)
// collects the row-norm maxima of W1 and W2 (a non-negative float's bit pattern orders like the float).
constexpr int kPackThreads = kThreadsTC - kGatherWarps * 32;  // 160
__device__ __forceinline__ WeightScale pack_weights(unsigned char* wsm, const float* __restrict__ W1,
                                                    const float* __restrict__ W2, uint32_t* l1max_bits, int tid) {
  {
    const int warp = tid >> 5, lane = tid & 31;
    const float m1 = row_l1max<kK, kPackThreads / 32>(W1, warp, lane), m2 = row_l1max<kO, kPackThreads / 32>(W2, warp, lane);
    if (lane == 0) {
      atomicMax(l1max_bits, __float_as_uint(m1));
      atomicMax(l1max_bits + 1, __float_as_uint(m2));
    }
    named_bar_sync(3, kPackThreads);
  }
  const int e1 = weight_exponent(__uint_as_float(l1max_bits[0]), kW1NormTarget);
  const int e2 = weight_exponent(__uint_as_float(l1max_bits[1]), kW2NormTarget);
  const float n1 = scalbnf(1.0f, -e1), n2 = scalbnf(1.0f, -e2);
  __half* w1h = reinterpret_cast<__half*>(wsm);
  constexpr int kV4 = kO * kK / 4;  // float4 = 4 consecutive kk of one (row, view, channel)
#pragma unroll 10
  for (int i = tid; i < kV4; i += kPackThreads) {
    const float4 w4 = __ldg(reinterpret_cast<const float4*>(W1) + i);
    const int n = i / (kK / 4), k = (i - n * (kK / 4)) * 4;
    const int view = k >> 7, c = (k >> 3) & 15, kk = k & 7;
    __half* dst = w1h + (view * 8 + kk) * 512 + (c >> 3) * 256 + (n >> 3) * 64 + (n & 7) * 8 + (c & 7);
    dst[0] = __float2half_rn(w4.x * n1); dst[512] = __float2half_rn(w4.y * n1);
    dst[1024] = __float2half_rn(w4.z * n1); dst[1536] = __float2half_rn(w4.w * n1);
  }
  for (int i = tid; i < kO * kO; i += kPackThreads) {
    const int n = i / kO, k = i % kO;
    w1h[kW1Bytes / 2 + (k >> 3) * 256 + (n >> 3) * 64 + (n & 7) * 8 + (k & 7)] = __float2half_rn(__ldg(W2 + i) * n2);
  }
  WeightScale ws;
  ws.w1 = scalbnf(1.0f, e1);
  ws.w12 = scalbnf(1.0f, e1 + e2);
  return ws;
}

// ---- per pair: stage the source volume, pre-scaled by the pair's power-of-two scale -------------------
// Called by the 256 gather threads between two named barriers.  `raw` is the pair's volume as it lies in HBM
// ([16 ch][512 voxels], fp32 or bf16), brought into shared memory by TMA (a 3-D tensor-map copy issued one tile
// before the pair switch, landing in the A-operand stage the next tile will use; completion on mbarrier
// `bar_vol`, phase `parity`).  The volume is read once into registers, its
// max |V| reduced over the 8 warps, the scale s = 2^e chosen so that max|V|*s lies in (b/2, b] (exact, undone after
// conv2), b = 2^15 / L1n with L1n the largest row L1 norm of the normalised W1 (in [4, 8), see pack_weights): conv1's
// output |H1| <= max|V|*s*L1n then lies in (2^14, 2^15] for the pair's largest voxel - as far above fp16's subnormals as
// its maximum (65504) allows - and b in (2^12, 2^13] depends on W1's mantissa only, not on its magnitude.  (It used to
// be min(2^12, 2^14 / L1max) of the raw W1, which cost the volume a bit of headroom per factor of 2 in W1.)  W1's row
// norms are summed here too (the same sums as pack_weights', which runs concurrently), folded into *l1max_bits (a
// non-negative float's bit pattern orders like the float).  Then the scaled values are written in
// the gather's layout: fp32 lines [halo voxel][16 ch], or for 16-bit "x-pair lines" (every voxel is tap 0 of
// pair xh and tap 1 of pair xh-1).  Returns 1/s.
template <typename T>
__device__ __forceinline__ float ld_raw(const T* p);
template <>
__device__ __forceinline__ float ld_raw<float>(const float* p) { return *p; }
template <>
__device__ __forceinline__ float ld_raw<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }

#ifndef AHV_STAGE_INLINE
#define AHV_STAGE_INLINE __forceinline__
#endif
template <typename T, bool K16>
__device__ AHV_STAGE_INLINE float stage_pair_volume(unsigned char* vsm, const T* raw, uint32_t bar_vol, uint32_t parity,
                                                   uint32_t* l1max_bits, const float* __restrict__ W1, bool first,
                                                   float* red, int gtid) {
  float wnorm = 0.0f;
  if (first) wnorm = row_l1max<kK, kGatherWarps>(W1, gtid >> 5, gtid & 31);  // W1 row norms: in flight while the TMA lands
  mbar_wait(bar_vol, parity);                                                  // the pair's volume is in shared memory
  float val[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    // fp32: task = gtid + 256*(i>>2) -> (voxel, 4-channel group jj), channel jj*4 + (i&3)
    // 16-bit: task = gtid + 256*(i>>3) -> (voxel, channel half), channel chalf*8 + (i&7)
    const int task = gtid + 256 * (K16 ? (i >> 3) : (i >> 2));
    const int v = task & 511, grp = task >> 9;
    const int ch = K16 ? grp * 8 + (i & 7) : grp * 4 + (i & 3);
    val[i] = ld_raw<T>(raw + ch * kVox + v);   // lanes = consecutive voxels of one channel: conflict-free
  }
  if (first && (gtid & 31) == 0) atomicMax(l1max_bits, __float_as_uint(wnorm));
  float mx = 0.0f;
#pragma unroll
  for (int i = 0; i < 32; ++i) mx = fmaxf(mx, fabsf(val[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((gtid & 31) == 0) red[gtid >> 5] = mx;
  named_bar_sync(1, kGatherWarps * 32);
  const float l1max = __uint_as_float(*l1max_bits);
  float m = red[0];
#pragma unroll
  for (int w = 1; w < kGatherWarps; ++w) m = fmaxf(m, red[w]);
  float sc = 1.0f;
  if (m > 0.0f && isfinite(m)) {
    const float l1n = scalbnf(l1max, -weight_exponent(l1max, kW1NormTarget));
    const float bound = fminf(8192.0f, 32768.0f / fmaxf(l1n, 1e-20f));
    int e = ilogbf(bound / m);  // floor(log2)
    e = max(-100, min(100, e));
    sc = scalbnf(1.0f, e);
  }
  if constexpr (!K16) {
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int task = gtid + 256 * it;
      const int v = task & 511, jj = task >> 9;
      const int z = v >> 6, y = (v >> 3) & 7, x = v & 7;
      const int line = ((z + 1) * kHalo + (y + 1)) * kHalo + (x + 1);
      *reinterpret_cast<float4*>(vsm + (line * kC + jj * 4) * 4) =
          make_float4(val[4 * it] * sc, val[4 * it + 1] * sc, val[4 * it + 2] * sc, val[4 * it + 3] * sc);
    }
  } else {
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int task = gtid + 256 * it;
      const int v = task & 511, chalf = task >> 9;
      const int zh = (v >> 6) + 1, yh = ((v >> 3) & 7) + 1, xh = (v & 7) + 1;
      uint32_t pk[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {  // bf16 inputs (8-bit mantissa) x power-of-two scale -> fp16 exactly; fp32 inputs are rounded
        const __half2 two = __floats2half2_rn(val[8 * it + 2 * e] * sc, val[8 * it + 2 * e + 1] * sc);
        pk[e] = *reinterpret_cast<const uint32_t*>(&two);
      }
      const uint4 q4 = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      unsigned char* row = vsm + ((zh * kHalo + yh) * 9) * 64;
      *reinterpret_cast<uint4*>(row + xh * 64 + chalf * 16) = q4;              // tap 0 of pair xh (xh <= 8)
      *reinterpret_cast<uint4*>(row + (xh - 1) * 64 + 32 + chalf * 16) = q4;   // tap 1 of pair xh-1
    }
  }
  return 1.0f / sc;
}

// ---- epilogue role ---------------------------------------------------
// 4 warps, warp s = TMEM sub-partition s.  Per hypothesis pair (tile):
//   phase A: tcgen05.ld D1 -> ReLU (modules/modules.py:68) -> fp16 -> conv2's A operand, straight into TMEM
//            (tcgen05.st; conv2 runs in the TS form);
//   phase B (one tile later, after conv2): tcgen05.ld D2 -> undo the pair and weight scales, + bias -> L2 norm with
//            F.normalize's eps (:122) -> dot with the target features (registers) -> mean over the 64
//            positions (modules/model.py:193) -> score, and the running arg-max key (:195).
template <bool kSave = false>
__device__ __forceinline__ void epilogue_role(const Work& work, int s, int lane, uint32_t tmem, uint32_t bar0,
                                              uint32_t tmem_a2, float* partial,
                                              const float* __restrict__ tgt_feat, const float* __restrict__ b2,
                                              const float* inv_ring, WeightScale ws, float* __restrict__ scores,
                                              u64* __restrict__ best_keys, int64_t N, int B,
                                              const float* __restrict__ R, int r_per_pair, const Finalize& fin) {
  const int slot = lane >> 4;            // which hypothesis of the tile
  const int pos = 16 * s + (lane & 15);  // position p*8+q of the folded plane
  float b2r[kO], tg[kO];
#pragma unroll
  for (int o = 0; o < kO; ++o) b2r[o] = __ldg(b2 + o);
  // the target features and the cleared arg-max keys come from the prologue grid; every other role of this
  // kernel is independent of it (no-op when the kernel was not launched programmatically dependent)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (s == 0 && lane == 0) AHV_TL(7);
  TileIter it(work);
  int cur_b = -1;
  float inv_s = 1.0f;
  uint32_t g = 0;
  int prev_b = 0, prev_cnt = 0;
  uint32_t prev_n0 = 0;
  float prev_inv = 1.0f;
  // arg-max fused into the epilogue (torch.max, modules/model.py:195): the two score-writing lanes keep a
  // running best key for the pair they are in and publish it with one atomicMax per (CTA, pair) - keys
  // order by score, ties by lowest index
  int key_b = -1;
  u64 key_best = 0;
  auto phase_b = [&](uint32_t gg, int pb, uint32_t pn0, int pcnt, float pinv) {
    const uint32_t gb = gg & 1, u = gg >> 1;
    mbar_wait(bar0 + (kD2Full + gb) * 8, u & 1);
    tc_fence_after();
    uint32_t r[32];
    tmem_ld32(tmem + ((uint32_t)(32 * s) << 16) + 64 + gb * 32, r);
    tmem_ld_wait();
    float ss = 0.0f, dt = 0.0f;
#pragma unroll
    for (int o = 0; o < kO; ++o) {
      const float v = fmaf(__uint_as_float(r[o]), pinv, b2r[o]);  // undo the pair and weight scales, add bias
      ss = fmaf(v, v, ss);
      dt = fmaf(v, tg[o], dt);
    }
    float cosv = dt / fmaxf(sqrtf(ss), 1e-12f);  // F.normalize eps (modules/modules.py:122)
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) cosv += __shfl_xor_sync(0xffffffffu, cosv, o);  // 16 positions of this slot
    if ((lane & 15) == 0) partial[(gb * 2 + slot) * 4 + s] = cosv;
    tc_fence_before();
    named_bar_sync(2, 128);
    if (s == 0 && lane < pcnt) {
      const float* pp = partial + (gb * 2 + lane) * 4;
      const float tot = ((pp[0] + pp[1]) + pp[2]) + pp[3];  // fixed order: deterministic
      const float sc = tot * (1.0f / 64.0f);                // .mean(dim=-1)
      const int rb = work.pair(pb);
      if (scores) scores[(size_t)rb * N + pn0 + lane] = sc;
      if (best_keys) {
        const u64 key = make_key(sc, (uint32_t)(pn0 + lane));
        if (rb != key_b) {
          if (key_b >= 0) atomicMax(best_keys + key_b, key_best);
          key_b = rb;
          key_best = key;
        } else if (key > key_best) {
          key_best = key;
        }
      }
    }
  };
  while (it.advance()) {
    const uint32_t gb = g & 1, u = g >> 1;
    // ---- phase A ----
    mbar_wait(bar0 + (kD1Full + gb) * 8, u & 1);
    tc_fence_after();
    uint32_t r[32];
    tmem_ld32(tmem + ((uint32_t)(32 * s) << 16) + gb * 32, r);
    tmem_ld_wait();
    uint32_t wq[16];  // ReLU -> fp16: the 32 channels of this thread's row
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const __half2 hh = __floats2half2_rn(fmaxf(__uint_as_float(r[2 * e]), 0.0f), fmaxf(__uint_as_float(r[2 * e + 1]), 0.0f));
      wq[e] = *reinterpret_cast<const uint32_t*>(&hh);
    }
    tmem_st16(tmem + ((uint32_t)(32 * s) << 16) + tmem_a2 + gb * 16, wq);  // 16 TMEM columns of conv2's A operand
    if constexpr (kSave) {  // training forward: keep this row of H1 (64 B) for the backward pass
      if (slot < it.cnt) {
        uint4* dst = reinterpret_cast<uint4*>(fin.h1_out + (((size_t)it.b * N + it.n0 + slot) * kP + pos) * kO);
#pragma unroll
        for (int e = 0; e < 4; ++e) dst[e] = make_uint4(wq[4 * e], wq[4 * e + 1], wq[4 * e + 2], wq[4 * e + 3]);
      }
    }
    tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      mbar_arrive(bar0 + (kA2Full + gb) * 8);
      mbar_arrive(bar0 + (kD1Empty + gb) * 8);
    }
    if (s == 0 && lane == 0 && g == 0) AHV_TL(8);
    // ---- phase B of the previous tile ----
    if (g > 0) phase_b(g - 1, prev_b, prev_n0, prev_cnt, prev_inv);
    if (it.b != cur_b) {  // target features / scale of the tile just handed to conv2
      cur_b = it.b;
      const float inv_pair = inv_ring[cur_b & 7];  // 1/s, written by the gather role when it staged this pair
      inv_s = inv_pair * ws.w12;                   // conv2's output = D2 * 2^(e1+e2) / s (powers of two: exact)
      if constexpr (kSave) {                       // the same value from every CTA that scores this pair
        if (s == 0 && lane == 0) fin.pair_inv_out[cur_b] = inv_pair * ws.w1;
      }
#pragma unroll
      for (int o = 0; o < kO; ++o) tg[o] = __ldg(tgt_feat + ((size_t)work.pair(cur_b) * kO + o) * kP + pos);
    }
    prev_b = it.b; prev_n0 = it.n0; prev_cnt = it.cnt; prev_inv = inv_s;
    ++g;
  }
  phase_b(g - 1, prev_b, prev_n0, prev_cnt, prev_inv);
  if (s == 0 && lane == 0) AHV_TL(9);
  if (best_keys && key_b >= 0) atomicMax(best_keys + key_b, key_best);
  if (best_keys && fin.val && s == 0) finalize_ticket(fin, best_keys, R, r_per_pair, N, B, lane);
}

}  // namespace tc
}  // namespace ahv
