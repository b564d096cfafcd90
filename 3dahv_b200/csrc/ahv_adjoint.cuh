// Pieces of the fused backward shared by the exact fp32 kernel (ahv_score_bwd.cu) and the tcgen05 one
// (ahv_score_bwd_tc.cu): the adjoint of the trilinear resampling as a gather over per-input-voxel work lists, the
// orders the deterministic form sums those lists in, and the way the gradients leave a CTA (kDet: stores into the
// workspace slots of DetBwdWs, ahv_common.cuh; else float atomics).  256 threads; thread t owns input voxels t, t + 256.
#pragma once
#include "ahv_common.cuh"

namespace ahv {

// output voxel (z*64 + y*8 + x) a thread lists for the adjoint: lane bits -> x2 x1 y2 y1 z2, warp bits and j -> the rest
__device__ __forceinline__ int adjoint_out_voxel(int t, int j) {
  const int x = ((t & 3) << 1) | ((t >> 5) & 1), y = (((t >> 2) & 3) << 1) | ((t >> 6) & 1);
  const int z = (((t >> 4) & 1) << 2) | (((t >> 7) & 1) << 1) | j;
  return z * 64 + y * 8 + x;
}

// Ascending sort of a[0 .. kM) in registers (kM <= kN, kN a power of two; a[kM .. kN) hold 0xffffffff): Batcher's
// odd-even merge network for kN inputs, fully unrolled, without the comparators that touch a place >= kM.  Every
// comparator puts the smaller value at the lower place, so those places keep the largest value and their comparators
// are no-ops.  19, 42 and 63 comparators for (8, 8), (16, 12) and (16, 16) (each checked on all 0-1 inputs).
template <int kN, int kM>
__device__ __forceinline__ void oddeven_sort(uint32_t* a) {
#pragma unroll
  for (int p = 1; p < kN; p <<= 1)
#pragma unroll
    for (int k = p; k >= 1; k >>= 1)
#pragma unroll
      for (int x = 0; x < kN; ++x)   // comparator (x, x + k): x = j + i, j = k % p (mod 2k), i < k, same 2p-block
        if (x + k < kM && x >= k % p && (x - k % p) % (2 * k) < k && x / (2 * p) == (x + k) / (2 * p)) {
          const uint32_t lo = min(a[x], a[x + k]);
          a[x + k] = max(a[x], a[x + k]);
          a[x] = lo;
        }
}
// the n <= 16 register values of a warp whose largest count is nmax (warp-uniform)
__device__ __forceinline__ void sort_row(uint32_t* a, int nmax) {
  if (nmax <= 8) oddeven_sort<8, 8>(a);
  else if (nmax <= 12) oddeven_sort<16, 12>(a);
  else oddeven_sort<16, 16>(a);
}

// Insertion sort of one adjoint work list (offset of dX[vo], weight) by offset, which is unique per output voxel vo:
// the deterministic backward sums every input voxel's contributions in this order, not in the order shared-memory
// atomics handed out the places.  A rotation puts about 8 (at most ~12) entries on a voxel.
__device__ __forceinline__ void sort_list(uint2* e, int n) {
  for (int i = 1; i < n; ++i) {
    const uint2 x = e[i];
    int k = i;
    for (; k > 0 && e[k - 1].x > x.x; --k) e[k] = e[k - 1];
    e[k] = x;
  }
}

// The exact work list of the adjoint: output voxel vo feeds the 8 input voxels of its tap, corner(vo) + {0,1}^3, with the
// forward's weights; turned round, every INPUT voxel v gets the list ent[start[v] .. start[v] + cnt[v]) of its
// (offset of dX[vo], fp32 weight) contributions - a counting sort over the <= 4096 that land inside the volume (shared-
// memory integer atomics whose return value is the place in the list, then an exclusive scan), valid for any matrix R.
// dX element (d, h, w, 0) lies at d*kD + h*kH + w*kW.  taps: the forward's (corner line, fx, fy, fz) per output voxel;
// cnt, start: [512]; ent: [<= 4096]; wtot: 8 ints.  The caller puts a barrier before the call (nothing may still read
// cnt, start or ent) and after it.
template <int kD, int kH, int kW>
__device__ __forceinline__ void build_exact_list(const float4* taps, int* cnt, int* start, uint2* ent, int* wtot) {
  const int t = threadIdx.x;
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
    const float4 tp = taps[vo];
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
    const uint32_t off = (uint32_t)((vo >> 6) * kD + ((vo >> 3) & 7) * kH + (vo & 7) * kW);
#pragma unroll
    for (int dlt = 0; dlt < 8; ++dlt)
      if ((inside[j] >> dlt) & 1u) {
        const int dx = dlt & 1, dy = (dlt >> 1) & 1, dz = dlt >> 2;
        const float w = (dx ? fx[j] : 1.0f - fx[j]) * (dy ? fy[j] : 1.0f - fy[j]) * (dz ? fz[j] : 1.0f - fz[j]);
        const int v = tgt0[j] + dz * 64 + dy * 8 + dx;
        ent[start[v] + ((rank[j][dlt >> 1] >> (16 * (dlt & 1))) & 0xffffu)] = make_uint2(off, __float_as_uint(w));
      }
  }
}

// acc(e[i]) for the n entries of a work list, in list order
template <class Acc>
__device__ __forceinline__ void walk_list(const uint2* e, int n, Acc&& acc) {
#pragma unroll 2
  for (int i = 0; i < n; ++i) acc(e[i]);
}

// dT and dV of pair b leave the CTA and the accumulators restart at zero: aT[oo] is dT_b[cg2*8 + oo][pos], aV[j][c] is
// dV_b[c][voxel t + 256 j].  kDet: the whole segment, zeros included, into slot blockIdx.x + b (g_tgt, g_vol point at
// the segment slots' dT and dV); else atomics into pair b, zeros skipped.
template <bool kDet>
__device__ __forceinline__ void flush_pair(float* g_tgt, float* g_vol, int b, float (&aT)[8], float (&aV)[2][kC], int cg2,
                                           int pos, bool want_tgt, bool want_vol) {
  const int t = threadIdx.x;
  if constexpr (kDet) {
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
}

// one element of a weight gradient leaves the CTA: kDet into the CTA's weight slot (dst: the element in slot 0), else
// one atomic
template <bool kDet>
__device__ __forceinline__ void flush_weight(float* dst, float v) {
  if constexpr (kDet) dst[(size_t)blockIdx.x * kDetWSlot] = v;
  else atomicAdd(dst, v);
}

// db2: ab2[oo] is this thread's share of db2[cg2*8 + oo] (position pos); the 64 positions are summed inside the CTA
// first, in `red` ([32][64] floats of dead shared memory), then leave it through flush_weight
template <bool kDet>
__device__ __forceinline__ void flush_b2(float* red, const float (&ab2)[8], int cg2, int pos, float* g_b2, bool want) {
  const int t = threadIdx.x;
  __syncthreads();
#pragma unroll
  for (int oo = 0; oo < 8; ++oo) red[(cg2 * 8 + oo) * kP + pos] = ab2[oo];
  __syncthreads();
  if (want && t < kO) {
    float s = 0.0f;
    for (int p = 0; p < kP; ++p) s += red[t * kP + p];
    flush_weight<kDet>(g_b2 + t, s);
  }
}

}  // namespace ahv
