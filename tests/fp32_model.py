"""numpy model of the fp32 CUDA-core kernels' arithmetic: the AHV_MATH_FP32 scorer, the target-feature kernel and
rotate_volume, plus the reference its backward is held to.

TEST INFRASTRUCTURE ONLY.  It restates, rounding for rounding and in the kernels' order, what csrc/ahv_common.cuh,
csrc/ahv_head_fp32.cuh, csrc/ahv_score_fp32.cu and csrc/ahv_score_tc.cu compute, so that the suite can hold those
kernels bit for bit instead of to a distance from fp64:

  taps              make_tap (kernel_arith.sample_coords, tap_at): g = fmaf(R2, z, fmaf(R1, y, R0 x)).
  score_fp32_kernel gather_hypothesis: kernel_arith.gather32 with make_tap's coordinates and the x taps in bank-parity
                    order swap = (line ^ w) & 1 (parity="w").  conv1_relu: one fmaf chain over k = 0 .. 383 in tri-plane
                    order from 0, fmaxf(., 0).  conv2_bias: a chain over the 32 inputs from 0, then + b2.
                    kernel_arith.head_dots, then dt / fmaxf(sqrtf(ss), 1e-12).  mean_cosine: warp_sum's xor butterfly
                    16 .. 1, the 8 warp partials added in order from 0, times 1/64.  bf16 volumes are staged exactly, so
                    they are modelled as their fp32 values.
  tc_tgt_feat_kernel conv1: lane l sums the 12 terms k = l + 32 j, j = 0 .. 11, in an fmaf chain from 0, then the xor
                    butterfly 16 .. 1 (every lane ends with the same tree), fmaxf(., 0).  conv2: a chain from b2 over
                    the 32 inputs.  ss = warp_sum(v * v) over the 32 channels; v * (1 / fmaxf(sqrtf(ss), 1e-12)).
  rotate_volume     weights (wx wy) wz with each product rounded; FMAs in the (dz, dy, dx) nesting order from 0.

Contractions (--fmad=true): the SASS of both kernels shows none at the sites where one could happen.  v * v in the
target-feature kernel's warp_sum is an FMUL followed by SHFL.BFLY / FADD; the tap-weight products are FMULs that feed
FFMA multiplicands; 1.0f - t.fx is an FADD; conv2's + b2 in the scorer is an FADD after the FFMA chain.  sqrtf and /
are IEEE (no --use_fast_math), as numpy's float32 sqrt and division are.

The fp32 FMA, the taps, the gathers and the butterfly are kernel_arith's.  `rounding=False` evaluates every step in
fp64 (the function the kernels approximate).  Switches restate a kernel in another order, to show what the bit-exact
tests can see: `swap` (x taps without the parity swap), `coords="tc"` (the tensor-core gather's coordinate order),
`b2_first` (the scorer's conv2 chain starting from b2) and `divide` (the target features divided by the norm instead of
multiplied by its reciprocal).

rotate_volume_bwd_kernel sums with shared-memory and global float atomics in no fixed order, so it has no bit-exact
model: `rotate_volume_adjoint` returns the exact sum of the kernel's own rounded terms RN(w g), the number of terms
and CTA flushes that meet at each element, and the bound gamma_(n+1) sum |w g| that any order of those additions obeys.
"""
from __future__ import annotations

import numpy as np

from kernel_arith import (C, HALO, KTRI, NPOS, OCH, S, VOX, butterfly, fma32, gather32, gather64, halo, head_dots,
                          run_chunks, sample_coords, tap_at)
from oracle import ahv_oracle as oracle

f32, f64 = np.float32, np.float64
U32 = 2.0 ** -24                                           # unit roundoff of fp32


# ---- rotate_volume --------------------------------------------------------------------------------------------------
def rotate_volume(vol, R, base=None, rounding: bool = True) -> np.ndarray:
    """rotate_volume_kernel: vol [16,8,8,8] (shared) or [n,16,8,8,8] (one per rotation), R [n,3,3] -> [n,16,8,8,8]
    fp32 (fp64 with rounding=False)."""
    R = np.asarray(R, f32).reshape(-1, 9)
    n = len(R)
    vol = np.asarray(vol, f32)
    pair = np.arange(n) if vol.ndim == 5 else None
    if not rounding:
        return gather64(vol, R, base, pair).reshape(n, C, S, S, S)
    _, (fx, fy, fz), line = tap_at(sample_coords(R, base))
    V, off = halo(vol, f32, pair, n)
    line = line + off
    one = f32(1.0)
    acc = np.zeros((C, n, VOX), f32)
    for dz in (0, 1):
        for dy in (0, 1):
            for dx in (0, 1):
                wgt = ((fx if dx else one - fx) * (fy if dy else one - fy)) * (fz if dz else one - fz)
                acc = fma32(wgt, V[:, line + dz * HALO * HALO + dy * HALO + dx], acc)
    return acc.transpose(1, 0, 2).reshape(n, C, S, S, S)


def rotate_volume_adjoint(grad_out, R, per_rotation: bool, base=None, rot_per_cta: int = 8):
    """The reference rotate_volume_bwd_kernel is held to: (exact [n|1,16,8,8,8] fp64, count, bound).

    exact: the sum in fp64 of the kernel's terms RN(w g) (w the fp32 weights of rotate_volume) that land on each
    interior element.  count: the nonzero terms that meet there, plus, for a shared volume, the CTAs (rot_per_cta
    rotations each) that flush a value to it.  bound: gamma_(count+1) sum |RN(w g)|, gamma_m = m u / (1 - m u), which
    bounds the error of adding those values in any order."""
    R = np.asarray(R, f32).reshape(-1, 9)
    n = len(R)
    g = np.asarray(grad_out, f32).reshape(n, C, VOX)
    _, (fx, fy, fz), line = tap_at(sample_coords(R, base))
    one = f32(1.0)
    slots = n if per_rotation else 1
    size = slots * HALO ** 3 * C
    exact, mag, cnt = np.zeros(size), np.zeros(size), np.zeros(size, np.int64)
    flushes = np.zeros(size, np.int64)
    ch = np.arange(C)[None, :, None]
    for i0 in range(0, n, rot_per_cta):
        sl = slice(i0, min(i0 + rot_per_cta, n))
        cta_cnt = np.zeros(size, np.int64)
        for dz in (0, 1):
            for dy in (0, 1):
                for dx in (0, 1):
                    wgt = ((fx[sl] if dx else one - fx[sl]) * (fy[sl] if dy else one - fy[sl])) * \
                        (fz[sl] if dz else one - fz[sl])
                    term = (wgt[:, None, :] * g[sl]).astype(f64)          # RN(w g), [r,16,512]
                    ln = line[sl] + dz * HALO * HALO + dy * HALO + dx
                    slot = np.arange(sl.start, sl.stop)[:, None, None] if per_rotation else 0
                    idx = ((slot * HALO ** 3 + ln[:, None, :]) * C + ch).ravel()
                    exact += np.bincount(idx, term.ravel(), size)
                    mag += np.bincount(idx, np.abs(term).ravel(), size)
                    cta_cnt += np.bincount(idx, (term != 0).ravel(), size).astype(np.int64)
        cnt += cta_cnt
        flushes += cta_cnt > 0
    if not per_rotation:
        cnt = cnt + flushes

    def interior(a):
        a = a.reshape(slots, HALO, HALO, HALO, C)[:, 1:9, 1:9, 1:9]
        return a.transpose(0, 4, 1, 2, 3).reshape((n,) * per_rotation + (C, S, S, S))

    m = interior(cnt).astype(f64) + 1
    gamma = m * U32 / (1 - m * U32)
    return interior(exact), interior(cnt), gamma * interior(mag)


# ---- the scorer -----------------------------------------------------------------------------------------------------
def _conv1_chain(tri: np.ndarray, W1: np.ndarray) -> np.ndarray:
    """conv1_relu's accumulation: [n,384,64] fp32 operand -> [n,32,64] fp32, one fmaf chain over k from 0."""
    acc = np.zeros((tri.shape[0], OCH, NPOS), f32)
    for k in range(KTRI):
        acc = fma32(tri[:, None, k, :], W1[None, :, k, None], acc)
    return acc


def score(vol_src, tgt_feat, R, W1, W2, b2, *, rounding: bool = True, swap: bool = True, coords: str = "make_tap",
          b2_first: bool = False, base=None, items=None, chunk: int = 8) -> np.ndarray:
    """score_fp32_kernel: scores [B,N] fp32 (fp64 with rounding=False).

    vol_src [B,16,8,8,8] (bf16 volumes as their float32 values), tgt_feat [B,32,64], R [N,3,3] shared or [B,N,3,3] per
    pair.  items: flat item indices b N + n to score; the result is then [len(items)]."""
    vs = np.asarray(vol_src, f32).reshape(-1, C, S, S, S)
    B = vs.shape[0]
    R = np.asarray(R, f32)
    per_pair = R.ndim == 4
    N = R.shape[1] if per_pair else R.shape[0]
    Rall = R.reshape(-1, 9)
    W1 = np.asarray(W1, f32).reshape(OCH, KTRI)
    W2 = np.asarray(W2, f32).reshape(OCH, OCH)
    b2 = np.asarray(b2, f32).reshape(OCH)
    tg = np.asarray(tgt_feat, f32).reshape(B, OCH, NPOS)
    whole = items is None
    items = np.arange(B * N) if whole else np.asarray(items, np.int64).reshape(-1)
    out = np.zeros(len(items), f32 if rounding else f64)

    def run(i0):
        it = items[i0 : i0 + chunk]
        pair = it // N
        Rc = Rall[it if per_pair else it % N]
        used, slot = np.unique(pair, return_inverse=True)
        n = len(it)
        if not rounding:
            A = gather64(vs[used], Rc, base, slot)
            tri = oracle.triplane_np(A.reshape(n, C, S, S, S)).reshape(n, KTRI, NPOS)
            v = W2.astype(f64) @ np.maximum(W1.astype(f64) @ tri, 0.0) + b2.astype(f64)[:, None]
            nrm = np.maximum(np.sqrt((v * v).sum(axis=1, keepdims=True)), 1e-12)
            out[i0 : i0 + n] = ((v / nrm) * tg[pair].astype(f64)).sum(axis=1).mean(axis=-1)
            return
        A = gather32(vs[used], Rc, base, slot, parity="w" if swap else None, coords=coords)
        tri = oracle.triplane_np(A.reshape(n, C, S, S, S)).reshape(n, KTRI, NPOS)
        h1 = np.fmax(_conv1_chain(tri, W1), f32(0.0))       # fmaxf(acc, 0): NaN -> 0
        a = np.broadcast_to(b2[None, :, None], h1.shape).astype(f32) if b2_first else np.zeros_like(h1)
        for i in range(OCH):
            a = fma32(W2[None, :, i, None], h1[:, None, i, :], a)
        v = a if b2_first else a + b2[None, :, None]
        ss, dt = head_dots(v, tg[pair], axis=1)             # quad_sum as lane 0 of position pos sees it
        cosv = dt / np.fmax(np.sqrt(ss), f32(1e-12))        # [n,64]
        # warp w holds positions 8w .. 8w + 7 in lanes 0, 4, .., 28; the other lanes add 0
        lanes = np.zeros((n, 8, 32), f32)
        lanes[:, :, 0::4] = cosv.reshape(n, 8, 8)
        red = butterfly(lanes)
        tot = np.zeros(n, f32)
        for w in range(8):
            tot = tot + red[:, w]
        out[i0 : i0 + n] = tot * f32(1.0 / 64.0)

    run_chunks(run, range(0, len(items), chunk))
    return out.reshape(B, N) if whole else out


# ---- target features ------------------------------------------------------------------------------------------------
def target_features(vol, W1, W2, b2, *, rounding: bool = True, divide: bool = False, chunk: int = 4) -> np.ndarray:
    """tc_tgt_feat_kernel: vol [m,16,8,8,8] -> normalised features [m,32,64] fp32 (fp64 with rounding=False)."""
    vol = np.asarray(vol, f32).reshape(-1, C, S, S, S)
    m = vol.shape[0]
    W1 = np.asarray(W1, f32).reshape(OCH, KTRI)
    W2 = np.asarray(W2, f32).reshape(OCH, OCH)
    b2 = np.asarray(b2, f32).reshape(OCH)
    out = np.zeros((m, OCH, NPOS), f32 if rounding else f64)
    W1r = W1.reshape(OCH, 12, 32)                          # W1[o, lane + 32 j] = W1r[o, j, lane]

    def run(i0):
        tri = oracle.triplane_np(vol[i0 : i0 + chunk]).reshape(-1, KTRI, NPOS)
        n = tri.shape[0]
        if not rounding:
            v = W2.astype(f64) @ np.maximum(W1.astype(f64) @ tri.astype(f64), 0.0) + b2.astype(f64)[:, None]
            out[i0 : i0 + n] = v / np.maximum(np.sqrt((v * v).sum(axis=1, keepdims=True)), 1e-12)
            return
        Ar = tri.reshape(n, 12, 32, NPOS)
        acc = np.zeros((n, OCH, 32, NPOS), f32)              # [item, o, lane, position]
        for j in range(12):
            acc = fma32(W1r[None, :, j, :, None], Ar[:, None, j], acc)
        h1 = np.fmax(butterfly(acc, axis=2), f32(0.0))       # [n,32,64]
        v = np.broadcast_to(b2[None, :, None], h1.shape).astype(f32)
        for o in range(OCH):
            v = fma32(W2[None, :, o, None], h1[:, None, o, :], v)
        nrm = np.fmax(np.sqrt(butterfly(v * v, axis=1)), f32(1e-12))[:, None, :]
        out[i0 : i0 + n] = v / nrm if divide else v * (f32(1.0) / nrm)

    run_chunks(run, range(0, m, chunk))
    return out


# ---- helpers for the tests ------------------------------------------------------------------------------------------
def sample_items(B: int, N: int, cap: int, seed: int = 0) -> np.ndarray:
    """At most `cap` flat items of a [B,N] problem: every item when that fits, else the first and last item of the
    first and last pair and a seeded uniform draw of the rest, ascending."""
    total = B * N
    if total <= cap:
        return np.arange(total)
    ends = np.unique([0, N - 1, (B - 1) * N, total - 1])
    rest = np.setdiff1d(np.arange(total), ends)
    return np.union1d(ends, np.random.default_rng(seed).choice(rest, cap - len(ends), replace=False))


def case_items(name: str, B: int, N: int, cap: int = 300) -> np.ndarray:
    """The items the GPU test compares: the golden set's first 200 hypotheses of each pair, else sample_items."""
    if name == "golden":
        return (np.arange(B)[:, None] * N + np.arange(200)[None]).reshape(-1)
    return sample_items(B, N, cap, seed=sum(map(ord, name)))
