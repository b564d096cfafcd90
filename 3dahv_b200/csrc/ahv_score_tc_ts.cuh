// The scoring kernel: view x of conv1 and conv2's A operand go register -> TMEM (tcgen05.st) and are consumed in
// the TS form of tcgen05.mma; only the YZ operand copy lives in shared memory; a pipeline stage is a tile of two
// hypotheses; the source volumes arrive by TMA.  Overview, roles and precision notes: ahv_score_tc.cu.
#pragma once
#include "ahv_tc_common.cuh"

namespace ahv {
namespace tc {

// ==============================================================================================
// View x of conv1 never touches shared memory.  Each gather lane owns one
// accumulator row (slot, d, h) - i.e. one TMEM lane - walks the 8 voxels along w, and writes the
// fp16 channels of every voxel (a) once into the YZ copy (views y and z, K-major core matrices,
// 144-byte row pitch so the STS.64 are conflict-free for this lane map) and (b) with tcgen05.st
// straight into TMEM as the A operand of view x, which the MMA warp consumes in the TS form
// (tcgen05.mma [d], [a_tmem], b_desc).  A and D of one M=64 tile share the lane offset (0 or 16),
// verified by experiments/ts_mma_probe.cu.  Compared with keeping a second operand copy in shared memory this
// removes 16 KB of stores and 16 KB of tensor-core reads per hypothesis from the shared-memory pipe.
struct MapTS {
  // YZ operand copy of one tile (two hypotheses = slots), fp16, K-major core matrices [8 w rows][8 channels]:
  //   address = chalf*yz_ch + (d>>1)*yz_dhi + slot*yz_slot + (d&1)*yz_dlo + h*yz_h + w*16   (yz_h = 144: 16 B pad
  //   per core matrix keeps the operand stores conflict-free for the gather's lane map).
  // The slot sits BETWEEN the two halves of d so that 8-row group g = (d>>1)*4 + slot*2 + (d&1) of view y advances
  // by one constant stride: view y of BOTH hypotheses is then one M=128 MMA per K slice whose row i is TMEM lane i -
  // exactly the rows the interleaved M=64 tiles of view z accumulate into (halves view y's W1 operand reads).
  static constexpr int yz_h = 144, yz_dlo = 8 * yz_h, yz_slot = 2 * yz_dlo, yz_dhi = 2 * yz_slot, yz_ch = 4 * yz_dhi;
  static constexpr int tile_bytes = 2 * yz_ch;  // 36864
  static constexpr int off_vol = 0;
  static constexpr int off_w1 = off_vol + kVolSmemBytes;
  static constexpr int off_w2 = off_w1 + kW1Bytes;
  static constexpr int off_a = off_w2 + kW2Bytes;
  static constexpr int off_bar = off_a + kStages * tile_bytes;
  static constexpr int off_misc = off_bar + 16 * 8;
  static constexpr int smem_bytes = off_misc + 256;
  static constexpr int tmem_cols = 512;      // D1[2] 0..63, D2[2] 64..127, A_x[3] 128 + 64*stage, A2[2] 448 + 16*buf
  static constexpr int tmem_ax = 128;
  static constexpr int tmem_a2 = 448;
  static_assert(off_a % 128 == 0 && off_bar % 8 == 0, "align");
  static_assert(smem_bytes <= 232448, "shared memory budget");
};

template <typename T, bool K16, bool kSave = false>
__global__ void __launch_bounds__(kThreadsTC, 1)
score_tc_ts_kernel(const __grid_constant__ CUtensorMap vol_map, const float* __restrict__ tgt_feat,
                   const float* __restrict__ R, int r_per_pair, const float* __restrict__ b2,
                   const float* __restrict__ base, const float* __restrict__ W1,
                   const float* __restrict__ W2, float* __restrict__ scores,
                   u64* __restrict__ best_keys, int B, int64_t N, Finalize fin, int late_ctas,
                   const int* __restrict__ pair_list) {
  extern __shared__ __align__(128) unsigned char smem[];
  using M = MapTS;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // provably warp-uniform
  Work work;
  {
    // pair_list = [count, pair...]: score the `count` listed pairs only (their number is known on the device alone)
    const int64_t total = (pair_list ? (int64_t)min(__ldg(pair_list), B) : (int64_t)B) * N;
    if (pair_list) work.map = pair_list + 1;
    // Contiguous, near-equal item ranges.  When the target-feature prologue of a SMALL batch precedes this kernel
    // (programmatic dependent launch), the last `late_ctas` CTAs - the ones that get the SMs the prologue's CTAs
    // occupy - start about one tile time late (in-kernel timeline: +2.4 us at B = 1); they are given one tile
    // (two items) less and the others share the difference, which shortens the B = 1 makespan by a tile.
    constexpr int64_t kLateItems = 2;
    const int64_t first_late = (int64_t)gridDim.x - late_ctas;
    auto cut = [&](int64_t i) {
      return (total + kLateItems * late_ctas) * i / gridDim.x - kLateItems * (i > first_late ? i - first_late : 0);
    };
    work.lo = cut(blockIdx.x);
    work.hi = cut((int64_t)blockIdx.x + 1);
    work.N = N;
  }
  if (work.lo >= work.hi) {  // no items: the fused selection still needs this CTA's ticket
    if (best_keys && fin.val && warp == 0) finalize_ticket(fin, best_keys, R, r_per_pair, N, B, lane);
    return;
  }
  if (threadIdx.x == 0) AHV_TL(0);

  float* vol = reinterpret_cast<float*>(smem + M::off_vol);
  const uint32_t s_base = smem_u32(smem);
  const uint32_t bar0 = s_base + M::off_bar;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + M::off_misc);
  float* partial = reinterpret_cast<float*>(smem + M::off_misc + 16);  // [2 tilebuf][2 slot][4 warps]
  float* sbase = reinterpret_cast<float*>(smem + M::off_misc + 96);    // 8 base coordinates
  uint32_t* l1max_bits = reinterpret_cast<uint32_t*>(smem + M::off_misc + 128);  // max L1 row norms (float bits): W1, W2 for
                                                                                 // pack_weights, W1 for the gather's pair scale
  float* red = reinterpret_cast<float*>(smem + M::off_misc + 144);        // 8 per-warp maxima (volume staging)
  float* inv_ring = reinterpret_cast<float*>(smem + M::off_misc + 176);   // 1/scale of pair b at [b & 7] (gather -> epilogue)

  for (int i = threadIdx.x; i < kVolSmemBytes / 16; i += kThreadsTC)
    reinterpret_cast<uint4*>(vol)[i] = make_uint4(0, 0, 0, 0);  // halo stays zero for the whole kernel
  if (threadIdx.x < 8) sbase[threadIdx.x] = base[threadIdx.x];
  if (threadIdx.x >= 8 && threadIdx.x < 11) l1max_bits[threadIdx.x - 8] = 0u;
  // ---- source volumes by TMA (cp.async.bulk.tensor, 3-D map over [B*16 ch][8 d][64 hw]; one box = one pair's
  // volume, 32 KB fp32 / 16 KB bf16).  The box of the pair that starts at tile t lands in A-operand stage buffer
  // t % kStages - idle at that moment: the tensor core finished reading it with tile t-3 and the gather fills it only
  // after it has turned the box into its own layout (stage_pair_volume).  Requests are made by the MMA warp, which
  // sees every tile one tile-time before the gather reaches it plus one: after issuing tile t it looks two tiles
  // ahead, so a pair switch never waits for HBM/L2 and the gather's loop carries no TMA code.  At most two boxes
  // are in flight (a new pair every tile, N <= 2), hence two mbarriers used alternately.
  uint32_t vol_req = 0;  // MMA warp: boxes requested so far
  auto request_volume = [&](int pair, uint32_t stage_buf) {
    const uint32_t bar = bar0 + (kVolFull + (vol_req & 1)) * 8;
    if (elect_one()) {
      mbar_arrive_expect_tx(bar, kC * kVox * (uint32_t)sizeof(T));
      tma_load_3d(s_base + M::off_a + stage_buf * M::tile_bytes, &vol_map, bar, 0, 0, work.pair(pair) * kC);
    }
    ++vol_req;
  };
  if (warp == kMmaWarp) {
    if (lane == 0) {
      for (int i = 0; i < 3; ++i) { mbar_init(bar0 + (kFull + i) * 8, kGatherWarps); mbar_init(bar0 + (kEmpty + i) * 8, 1); }
      for (int i = 0; i < 2; ++i) {
        mbar_init(bar0 + (kD1Full + i) * 8, 1);
        mbar_init(bar0 + (kD1Empty + i) * 8, 4);
        mbar_init(bar0 + (kA2Full + i) * 8, 4);
        mbar_init(bar0 + (kD2Full + i) * 8, 1);
      }
      mbar_init(bar0 + kVolFull * 8, 1);
      mbar_init(bar0 + (kVolFull + 1) * 8, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    {  // the first tile's pair, and the second tile's if it is another pair - before anything else in this CTA (the
       // barriers were initialised by this warp; nobody else touches the stage buffers yet)
      TileIter it0(work);
      it0.advance();
      request_volume(it0.b, 0);
      int b1, c1; uint32_t n1;
      it0.peek_tile(b1, n1, c1);
      if (it0.left > 0 && b1 != it0.b) request_volume(b1, 1 % kStages);
    }
    tmem_alloc(smem_u32(tmem_slot), M::tmem_cols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (threadIdx.x == 0) AHV_TL(1);
  WeightScale wscale;
  if (warp >= kGatherWarps) {  // MMA + epilogue warps: weights -> fp16 operand layouts, then release the MMA warp
    wscale = pack_weights(smem + M::off_w1, W1, W2, l1max_bits, threadIdx.x - kGatherWarps * 32);
    fence_proxy_async();  // written through the generic proxy, UMMA reads through the async proxy
    named_bar_sync(3, kPackThreads);
    if (threadIdx.x == 256) AHV_TL(5);
  }

  if (warp < kGatherWarps) {
    // =========================== GATHER ===========================
    // lane -> accumulator row: slot = lane>>4 (hypothesis of the tile), d = 2*sub + ((lane>>3)&1), h = lane&7;
    // the warp's TMEM sub-partition is warp&3, warps w and w+4 split the w axis
    const int sub = warp & 3, whalf = warp >> 2;
    const int slot = lane >> 4, dlo = (lane >> 3) & 1, h_ = lane & 7, d = 2 * sub + dlo;
    const int pf = (lane >> 2) & 1;            // bank parity this lane reads first
    const int rot = ((lane & 3) + dlo) & 3;    // chunk rotation
    const float by = sbase[h_], bz = sbase[d];
    // fp32 gather: this warp's four x base coordinates live in registers (rotated once per voxel).  Read from shared
    // memory inside the voxel loop, the value queued behind the gather's own LDS.128 and sat at the head of every
    // voxel's coordinate -> address -> load chain: 3.8 % of the kernel's stall samples, +2.1 % throughput once gone.
    // (The 16-bit gather computes its coordinates one step ahead of their use and keeps the shared-memory read.)
    [[maybe_unused]] float bxr[4];
    if constexpr (!K16) {
#pragma unroll
      for (int i = 0; i < 4; ++i) bxr[i] = sbase[whalf * 4 + i];
    }
    uint32_t koff[4], syz[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      // chunk visited at step t: a rotation for fp32, an XOR swizzle for 16-bit lines (chunk = tap*2 + chalf, so
      // the tap of step t is (t>>1)^(rot>>1): steps 0,1 share one x tap, steps 2,3 the other - compile-time)
      const int ck = K16 ? (rot ^ t) : ((rot + t) & 3);
      koff[t] = ck * 16;
      const uint32_t row_off = sub * M::yz_dhi + slot * M::yz_slot + dlo * M::yz_dlo + h_ * M::yz_h;
      if constexpr (!K16)  // fp32: chunk ck = channels 4ck..4ck+3 (8 B of fp16)
        syz[t] = (ck >> 1) * M::yz_ch + (ck & 1) * 8 + row_off;
      else                 // 16-bit: accumulator t&1 holds channel half (rot^t)&1 (16 B of fp16); t < 2 used
        syz[t] = ((rot ^ t) & 1) * M::yz_ch + row_off;
    }
    const unsigned char* volb = smem + M::off_vol;
    const int gtid = threadIdx.x;
    TileIter it(work);
    int cur_b = -1;
    uint32_t g = 0;
    // Pair volumes arrive by TMA, requested by the MMA warp two tiles ahead of the pair switch (see there); the
    // volume of the pair that starts at tile g sits in A-operand stage buffer g % kStages, completion on mbarrier
    // kVolFull + (ordinal & 1) where ordinal counts the pairs this CTA has staged.
    uint32_t vol_uses = 0;
    // Rotation prefetch, one tile ahead, 9 loads per lane (all lanes of a slot read the same 36 bytes).  A coalesced
    // variant - one load per warp + 9 shuffles - removes 70 LSU wavefronts per hypothesis but was 3-7 % SLOWER:
    // the shuffles queue behind the gather's LDS.128 in the same pipe and sit on the coordinate critical path.  Three
    // aligned 16-byte loads of the row's 48-byte window + selects: 13 % (fp32) / 30 % (16-bit) slower still.
    float Rn[9];
    auto fetch_R = [&](int fb, uint32_t fn) {
      const float* Rg = R + (r_per_pair ? ((size_t)work.pair(fb) * N + fn) : (size_t)fn) * 9;
#pragma unroll
      for (int e = 0; e < 9; ++e) Rn[e] = __ldg(Rg + e);
    };
    {
      int fb; uint32_t fn; int fc;
      it.peek_tile(fb, fn, fc);
      fetch_R(fb, fn + (slot < fc ? slot : 0));
      // first pair of this CTA: its volume (and the W1 row norms) ride the same memory round trip as the
      // first rotations
      cur_b = fb;
      const float inv = stage_pair_volume<T, K16>(smem + M::off_vol, reinterpret_cast<const T*>(smem + M::off_a),
                                                  bar0 + kVolFull * 8, 0, l1max_bits + 2, W1, true, red, gtid);
      ++vol_uses;
      if (gtid == 0) inv_ring[fb & 7] = inv;
      named_bar_sync(1, kGatherWarps * 32);
      if (threadIdx.x == 0) AHV_TL(3);
#pragma unroll
      for (int e = 0; e < 9; ++e) Rn[e] *= opaque_one(r_per_pair);
    }
    // ---- 16-bit path: coordinates/weights of a voxel pair (w0, w0+1), computed one step AHEAD of its loads
    // (software pipeline across voxel pairs and across tiles) so that the serial coordinate chains of one
    // pair overlap the shared-memory traffic of the previous one ----
    struct VoxPair16 {
      const unsigned char* pa[2];
      const unsigned char* pb[2];
      __half2 wg[2][2][4];  // [voxel][x tap of steps {0,1} / {2,3}][y-z corner]
    };
    auto coords16 = [&](const float (&Rq)[9], int w0, VoxPair16& o) {
      // grid = R @ (x, y, z): y and z are fixed per lane, x walks with w
      const float pgx = fmaf(Rq[2], bz, Rq[1] * by), pgy = fmaf(Rq[5], bz, Rq[4] * by), pgz = fmaf(Rq[8], bz, Rq[7] * by);
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        const float bx = sbase[w0 + v];
        float ix = unnorm(fmaf(Rq[0], bx, pgx)), iy = unnorm(fmaf(Rq[3], bx, pgy)), iz = unnorm(fmaf(Rq[6], bx, pgz));
        ix = fminf(fmaxf(ix, -1.0f), 8.0f); iy = fminf(fmaxf(iy, -1.0f), 8.0f); iz = fminf(fmaxf(iz, -1.0f), 8.0f);
        const float x0 = fminf(floorf(ix), 7.0f), y0 = fminf(floorf(iy), 7.0f), z0 = fminf(floorf(iz), 7.0f);
        const float fx = ix - x0, fy = iy - y0, fz = iz - z0;
        const int pline = (((int)z0 + 1) * kHalo + ((int)y0 + 1)) * 9 + ((int)x0 + 1);
        const int swapy = (pline ^ pf) & 1;  // first y tap = the one whose line has bank parity pf (9 is odd)
        o.pa[v] = volb + (pline + swapy * 9) * 64;
        o.pb[v] = volb + (pline + (1 - swapy) * 9) * 64;
        const float wya = swapy ? fy : 1.0f - fy, wyb = swapy ? 1.0f - fy : fy;
        const __half2 wy2[2] = {__float2half2_rn(wya), __float2half2_rn(wyb)};
        const __half2 wz2[2] = {__float2half2_rn(1.0f - fz), __float2half2_rn(fz)};
        // x tap read at steps {0,1} is (rot>>1), at steps {2,3} the other one
        const __half2 wxf = __float2half2_rn((rot & 2) ? fx : 1.0f - fx), wxs = __float2half2_rn((rot & 2) ? 1.0f - fx : fx);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const __half2 w4 = __hmul2(wy2[c >> 1], wz2[c & 1]);
          o.wg[v][0][c] = __hmul2(wxf, w4);
          o.wg[v][1][c] = __hmul2(wxs, w4);
        }
      }
    };
    // trilinear taps of the pair (16 LDS.128 per voxel, packed HFMA2), then the operand stores
    auto sample16 = [&](const VoxPair16& q, int w0, unsigned char* st, uint32_t ax) {
      constexpr int kDz = kHalo * 9 * 64;
      __half2 acc[2][2][4];
#pragma unroll
      for (int v = 0; v < 2; ++v)
#pragma unroll
        for (int e2 = 0; e2 < 4; ++e2) acc[v][0][e2] = acc[v][1][e2] = __float2half2_rn(0.0f);
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        uint4 buf[2][4];
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          buf[v][0] = *reinterpret_cast<const uint4*>(q.pa[v] + koff[t]);
          buf[v][1] = *reinterpret_cast<const uint4*>(q.pa[v] + koff[t] + kDz);
          buf[v][2] = *reinterpret_cast<const uint4*>(q.pb[v] + koff[t]);
          buf[v][3] = *reinterpret_cast<const uint4*>(q.pb[v] + koff[t] + kDz);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int v = 0; v < 2; ++v) {
            const __half2 wg = q.wg[v][t >> 1][c];
            const uint4 q4 = buf[v][c];
            const uint32_t wd[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
            for (int k2 = 0; k2 < 4; ++k2)
              acc[v][t & 1][k2] = __hfma2(wg, *reinterpret_cast<const __half2*>(&wd[k2]), acc[v][t & 1][k2]);
          }
      }
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        const int w = w0 + v;
        uint32_t a0[4], a1[4];
#pragma unroll
        for (int k2 = 0; k2 < 4; ++k2) {
          a0[k2] = *reinterpret_cast<const uint32_t*>(&acc[v][0][k2]);
          a1[k2] = *reinterpret_cast<const uint32_t*>(&acc[v][1][k2]);
        }
        *reinterpret_cast<uint4*>(st + syz[0] + w * 16) = make_uint4(a0[0], a0[1], a0[2], a0[3]);
        *reinterpret_cast<uint4*>(st + syz[1] + w * 16) = make_uint4(a1[0], a1[1], a1[2], a1[3]);
        // view x: acc[.][0] holds channel half (rot&1); put the halves in channel order and store to TMEM
        const bool sw = rot & 1;
        uint32_t regs[8];
#pragma unroll
        for (int k2 = 0; k2 < 4; ++k2) {
          regs[k2] = sw ? a1[k2] : a0[k2];
          regs[4 + k2] = sw ? a0[k2] : a1[k2];
        }
        tmem_st8(ax + w * 8, regs);
      }
    };
    VoxPair16 vp_a, vp_b;
    if constexpr (K16) coords16(Rn, whalf * 4, vp_a);  // first pair of the first tile
    while (it.advance()) {
      if (it.b != cur_b) {
        named_bar_sync(1, kGatherWarps * 32);
        // requested two tiles ago, into the stage buffer THIS tile is about to fill
        const float inv = stage_pair_volume<T, K16>(smem + M::off_vol, reinterpret_cast<const T*>(smem + M::off_a + (g % kStages) * M::tile_bytes),
                                                    bar0 + (kVolFull + (vol_uses & 1)) * 8, (vol_uses >> 1) & 1, l1max_bits + 2, W1, false,
                                                    red, gtid);
        ++vol_uses;
        if (gtid == 0) inv_ring[it.b & 7] = inv;
        named_bar_sync(1, kGatherWarps * 32);
        cur_b = it.b;
      }
      float Rr[9];
#pragma unroll
      for (int e = 0; e < 9; ++e) Rr[e] = Rn[e];
      {  // prefetch this lane's rotation of the next tile
        int nb; uint32_t nn; int nc;
        it.peek_tile(nb, nn, nc);
        fetch_R(nb, nn + (slot < nc ? slot : 0));
      }
      const uint32_t stage = g % kStages, use = g / kStages;
      if (use > 0) mbar_wait(bar0 + (kEmpty + stage) * 8, (use - 1) & 1);
      unsigned char* st = smem + M::off_a + stage * M::tile_bytes;
      const uint32_t ax = tmem + ((uint32_t)(32 * sub) << 16) + M::tmem_ax + stage * 64;
      if constexpr (!K16) {
        // grid = R @ (x, y, z): y and z are fixed per lane, x walks with w
        const float pgx = fmaf(Rr[2], bz, Rr[1] * by), pgy = fmaf(Rr[5], bz, Rr[4] * by), pgz = fmaf(Rr[8], bz, Rr[7] * by);
#pragma unroll 1
        for (int wi = 0; wi < 4; ++wi) {
          const int w = whalf * 4 + wi;
          const float bx = bxr[0];
          { const float t0 = bxr[0]; bxr[0] = bxr[1]; bxr[1] = bxr[2]; bxr[2] = bxr[3]; bxr[3] = t0; }  // rotate: wi + 1 next
          float ix = unnorm(fmaf(Rr[0], bx, pgx)), iy = unnorm(fmaf(Rr[3], bx, pgy)), iz = unnorm(fmaf(Rr[6], bx, pgz));
          ix = fminf(fmaxf(ix, -1.0f), 8.0f); iy = fminf(fmaxf(iy, -1.0f), 8.0f); iz = fminf(fmaxf(iz, -1.0f), 8.0f);
          const float x0 = fminf(floorf(ix), 7.0f), y0 = fminf(floorf(iy), 7.0f), z0 = fminf(floorf(iz), 7.0f);
          const float fx = ix - x0, fy = iy - y0, fz = iz - z0;
          const int line = (((int)z0 + 1) * kHalo + ((int)y0 + 1)) * kHalo + ((int)x0 + 1);
          const int swap = (line ^ pf) & 1;
          const float wxa = swap ? fx : 1.0f - fx, wxb = swap ? 1.0f - fx : fx;
          const unsigned char* pa = volb + (line + swap) * 64;
          const unsigned char* pb = volb + (line + 1 - swap) * 64;
          float wa[4], wb[4];
  #pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float wyz = ((c & 1) ? fy : 1.0f - fy) * ((c >> 1) ? fz : 1.0f - fz);
            wa[c] = wyz * wxa;
            wb[c] = wyz * wxb;
          }
          float4 buf[2][8];
  #pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int off = ((c >> 1) * kHalo * kHalo + (c & 1) * kHalo) * 64;
            buf[0][2 * c] = *reinterpret_cast<const float4*>(pa + koff[0] + off);
            buf[0][2 * c + 1] = *reinterpret_cast<const float4*>(pb + koff[0] + off);
          }
          uint2 pk[4];
  #pragma unroll
          for (int t = 0; t < 4; ++t) {
            if (t < 3) {
  #pragma unroll
              for (int c = 0; c < 4; ++c) {
                const int off = ((c >> 1) * kHalo * kHalo + (c & 1) * kHalo) * 64;
                buf[(t + 1) & 1][2 * c] = *reinterpret_cast<const float4*>(pa + koff[t + 1] + off);
                buf[(t + 1) & 1][2 * c + 1] = *reinterpret_cast<const float4*>(pb + koff[t + 1] + off);
              }
            }
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  #pragma unroll
            for (int c = 0; c < 4; ++c) {
              const float4 a = buf[t & 1][2 * c], q = buf[t & 1][2 * c + 1];
              acc.x = fmaf(wa[c], a.x, acc.x); acc.y = fmaf(wa[c], a.y, acc.y);
              acc.z = fmaf(wa[c], a.z, acc.z); acc.w = fmaf(wa[c], a.w, acc.w);
              acc.x = fmaf(wb[c], q.x, acc.x); acc.y = fmaf(wb[c], q.y, acc.y);
              acc.z = fmaf(wb[c], q.z, acc.z); acc.w = fmaf(wb[c], q.w, acc.w);
            }
            const __half2 lo = __floats2half2_rn(acc.x, acc.y), hi2 = __floats2half2_rn(acc.z, acc.w);
            pk[t].x = *reinterpret_cast<const uint32_t*>(&lo);
            pk[t].y = *reinterpret_cast<const uint32_t*>(&hi2);
            *reinterpret_cast<uint2*>(st + syz[t] + w * 16) = pk[t];  // YZ copy: row w of core matrix (d,h,chalf)
          }
          // view x: un-rotate the chunks (chunk c was produced at step (c - rot) & 3) and store the 16 channels
          // of this voxel as K slice w of this lane's accumulator row in TMEM
          uint2 s1[4], o4[4];
          const bool r1 = rot & 1, r2 = rot & 2;
  #pragma unroll
          for (int c = 0; c < 4; ++c) {
            s1[c].x = r1 ? pk[(c + 3) & 3].x : pk[c].x;
            s1[c].y = r1 ? pk[(c + 3) & 3].y : pk[c].y;
          }
  #pragma unroll
          for (int c = 0; c < 4; ++c) {
            o4[c].x = r2 ? s1[(c + 2) & 3].x : s1[c].x;
            o4[c].y = r2 ? s1[(c + 2) & 3].y : s1[c].y;
          }
          const uint32_t regs[8] = {o4[0].x, o4[0].y, o4[1].x, o4[1].y, o4[2].x, o4[2].y, o4[3].x, o4[3].y};
          tmem_st8(ax + w * 8, regs);
        }
      } else {
        // 16-bit staged volume (x-pair lines, packed HFMA2): pair 0 was prepared during the previous tile
        sample16(vp_a, whalf * 4, st, ax);
        coords16(Rr, whalf * 4 + 2, vp_b);   // overlaps the loads of pair 0
        sample16(vp_b, whalf * 4 + 2, st, ax);
        coords16(Rn, whalf * 4, vp_a);       // next tile's pair 0 (Rn = its prefetched rotation) overlaps pair 1
      }
      tmem_st_wait();
      fence_proxy_async();  // YZ stores -> async proxy
      tc_fence_before();    // TMEM stores -> tensor core
      __syncwarp();
      if (lane == 0) mbar_arrive(bar0 + (kFull + stage) * 8);
      if (threadIdx.x == 0 && g == 0) AHV_TL(4);
      ++g;
    }
  } else if (warp == kMmaWarp) {
    // =========================== MMA ISSUER (converged warp) ===========================
    {
      constexpr uint32_t idesc1 = instr_desc(64, 32), idesc2 = instr_desc(128, 32);
      const uint32_t w1s = s_base + M::off_w1, w2s = s_base + M::off_w2;
      TileIter it(work);
      uint32_t g = 0;
      auto conv2 = [&](uint32_t gg) {
        const uint32_t gb = gg & 1, u = gg >> 1;
        mbar_wait(bar0 + (kA2Full + gb) * 8, u & 1);
        tc_fence_after();
#pragma unroll
        for (int i = 0; i < 2; ++i)  // conv2: A = ReLU(conv1) rows in TMEM (written by the epilogue), M = 128
          umma_f16_ts(tmem + 64 + gb * 32, tmem + M::tmem_a2 + gb * 16 + i * 8, smem_desc(w2s + i * 1024, 512, 128), idesc2, i);
        umma_commit(bar0 + (kD2Full + gb) * 8);
      };
      while (it.advance()) {
        const uint32_t gb = g & 1, u = g >> 1;
        if (u > 0) mbar_wait(bar0 + (kD1Empty + gb) * 8, (u - 1) & 1);
        const uint32_t stage = g % kStages, use = g / kStages;
        mbar_wait(bar0 + (kFull + stage) * 8, use & 1);
        tc_fence_after();
        // view x from TMEM, both hypotheses of the tile in one M=128 MMA per K slice (w=kk, c): A and D of a
        // TS-form MMA share the lane, so row i of the M=128 tile is TMEM lane i - exactly the rows the
        // two interleaved M=64 tiles below accumulate into.  Halves view x's W1 (B operand) reads.
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
          umma_f16_ts(tmem + gb * 32, tmem + M::tmem_ax + stage * 64 + kk * 8, smem_desc(w1s + kk * 1024, 512, 128), idesc2, kk);
        const uint32_t a_tile = s_base + M::off_a + stage * M::tile_bytes;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)  // view y, both hypotheses: rows (d,slot,w) in 16 groups of 8, K slice = (h=kk, c)
          umma_f16(tmem + gb * 32, smem_desc(a_tile + kk * M::yz_h, M::yz_ch, M::yz_dlo), smem_desc(w1s + (8 + kk) * 1024, 512, 128), idesc2, 1);
#pragma unroll
        for (int sl = 0; sl < 2; ++sl) {
          const uint32_t d1 = tmem + ((uint32_t)(16 * sl) << 16) + gb * 32;
          const uint32_t a = a_tile + sl * M::yz_slot;
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)  // view z: rows (h,w), K slice = (d=kk, c)
            umma_f16(d1, smem_desc(a + (kk >> 1) * M::yz_dhi + (kk & 1) * M::yz_dlo, M::yz_ch, M::yz_h),
                     smem_desc(w1s + (16 + kk) * 1024, 512, 128), idesc1, 1);
        }
        umma_commit(bar0 + (kEmpty + stage) * 8);
        umma_commit(bar0 + (kD1Full + gb) * 8);
        if (lane == 0 && g == 0) AHV_TL(6);
        {  // two tiles ahead: does tile g+2 start a new pair?  then request its volume into stage (g+2) % kStages
          int pb2; uint32_t left2;
          if (it.second_next_starts_pair(pb2, left2)) {
            const uint32_t nstage = (g + 2) % kStages, nuse = (g + 2) / kStages;
            if (nuse > 0) mbar_wait(bar0 + (kEmpty + nstage) * 8, (nuse - 1) & 1);  // tile g-1's MMAs are done with it
            request_volume(pb2, nstage);
          }
        }
        if (g > 0) conv2(g - 1);
        ++g;
      }
      conv2(g - 1);
    }
    __syncwarp();
  } else {
    // =========================== EPILOGUE ===========================
    epilogue_role<kSave>(work, warp - kEpiWarp0, lane, tmem, bar0, M::tmem_a2, partial, tgt_feat, b2, inv_ring, wscale,
                        scores, best_keys, N, B, R, r_per_pair, fin);
  }

  if (threadIdx.x == 0) AHV_TL(10);
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem, M::tmem_cols);
  }
  if (threadIdx.x == 0) AHV_TL(11);
}

}  // namespace tc
}  // namespace ahv
