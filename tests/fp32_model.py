"""numpy model of the fp32 CUDA-core kernels' arithmetic: the AHV_MATH_FP32 scorer, the target-feature kernel and
rotate_volume, plus the reference its backward is held to.

TEST INFRASTRUCTURE ONLY.  It restates, rounding for rounding and in the kernels' order, what csrc/ahv_common.cuh,
csrc/ahv_head_fp32.cuh, csrc/ahv_score_fp32.cu and csrc/ahv_score_tc.cu compute, so that the suite can hold those
kernels bit for bit instead of to a distance from fp64:

  taps              sample_coords / unnorm / tap_at: g = fmaf(R2, z, fmaf(R1, y, R0 x)), u = fmaf(g + 1, 4, -0.5),
                    clamp to [-1, 8] (NaN-dropping), corner floor(u) capped at 7, fraction u - corner.
  score_fp32_kernel gather_hypothesis: the x taps in bank-parity order (swap = (line ^ w) & 1), the (dz, dy) corners
                    (0,0) (0,1) (1,0) (1,1), wyz = wy wz, wa = wyz wx_first, wb = wyz wx_second each rounded, two FMAs
                    per corner pair.  conv1_relu: one fmaf chain over k = 0 .. 383 in tri-plane order from 0, fmaxf(., 0).
                    conv2_bias: a chain over the 32 inputs from 0, then + b2.  head_dots: an 8-term chain per lane of a
                    quad, quad_sum (x0 + x1) + (x2 + x3), dt / fmaxf(sqrtf(ss), 1e-12).  mean_cosine: warp_sum's xor
                    butterfly 16 .. 1, the 8 warp partials added in order from 0, times 1/64.  bf16 volumes are staged
                    exactly, so they are modelled as their fp32 values.
  tc_tgt_feat_kernel conv1: lane l sums the 12 terms k = l + 32 j, j = 0 .. 11, in an fmaf chain from 0, then the xor
                    butterfly 16 .. 1 (every lane ends with the same tree), fmaxf(., 0).  conv2: a chain from b2 over
                    the 32 inputs.  ss = warp_sum(v * v) over the 32 channels; v * (1 / fmaxf(sqrtf(ss), 1e-12)).
  rotate_volume     weights (wx wy) wz with each product rounded; FMAs in the (dz, dy, dx) nesting order from 0.

Contractions (--fmad=true): the SASS of both kernels shows none at the sites where one could happen.  v * v in the
target-feature kernel's warp_sum is an FMUL followed by SHFL.BFLY / FADD; the tap-weight products are FMULs that feed
FFMA multiplicands; 1.0f - t.fx is an FADD; conv2's + b2 in the scorer is an FADD after the FFMA chain.  sqrtf and /
are IEEE (no --use_fast_math), as numpy's float32 sqrt and division are.

The fp32 FMA is tc_model.fma32 (correctly rounded).  `rounding=False` evaluates every step in fp64 (the function the
kernels approximate).  Switches restate a kernel in another order, to show what the bit-exact tests can see: `swap`
(x taps without the parity swap), `coords="tc"` (the tensor-core gather's coordinate order), `b2_first` (the scorer's
conv2 chain starting from b2) and `divide` (the target features divided by the norm instead of multiplied by its
reciprocal).

rotate_volume_bwd_kernel sums with shared-memory and global float atomics in no fixed order, so it has no bit-exact
model: `rotate_volume_adjoint` returns the exact sum of the kernel's own rounded terms RN(w g), the number of terms
and CTA flushes that meet at each element, and the bound gamma_(n+1) sum |w g| that any order of those additions obeys.
"""
from __future__ import annotations

import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from oracle import ahv_oracle as oracle
from tc_model import CASES, _halo, _voxels, bf16_round, fma32, lattice_rotations, make_case  # noqa: F401
import tc_model as T

C, S, VOX, OCH, KTRI, NPOS, HALO = 16, 8, 512, 32, 384, 64, 10
f32, f64 = np.float32, np.float64
U32 = 2.0 ** -24                                           # unit roundoff of fp32
LANE = np.arange(32)


def _pool_map(fn, starts):
    # numpy releases the GIL in its loops: chunks of items run on all cores
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as pool:
        for fut in [pool.submit(fn, i0) for i0 in starts]:
            fut.result()


def butterfly(x, axis=-1) -> np.ndarray:
    """warp_sum over a 32-long axis in fp32: x + shfl_xor(x, o) for o = 16, 8, 4, 2, 1.  The adds are commutative, so
    every lane ends with the same tree; lane 0's value is returned."""
    x = np.moveaxis(np.asarray(x, f32), axis, -1)
    for o in (16, 8, 4, 2, 1):
        x = x + x[..., LANE ^ o]
    return x[..., 0]


# ---- taps -----------------------------------------------------------------------------------------------------------
def coords32(R, base=None, coords: str = "fp32"):
    """Unclamped sample positions (ux, uy, uz) [n,512] fp32 of the output voxels under R [n,9]: sample_coords and
    unnorm (ahv_common.cuh).  coords="tc": the tensor-core gather's order fmaf(R0, x, fmaf(R2, z, R1 y))."""
    base = oracle.base_coords_np() if base is None else np.asarray(base, f32)
    R = np.asarray(R, f32).reshape(-1, 9)
    d, h, w = _voxels()
    bx, by, bz = base[w][None], base[h][None], base[d][None]
    out = []
    for r in range(3):
        R0, R1, R2 = (R[:, 3 * r + i, None] for i in range(3))
        if coords == "tc":
            g = fma32(R0, bx, fma32(R2, bz, R1 * by))
        else:
            g = fma32(R2, bz, fma32(R1, by, R0 * bx))
        out.append(fma32(g + f32(1.0), f32(4.0), f32(-0.5)))
    return out


def taps32(R, base=None, coords: str = "fp32"):
    """tap_at of every output voxel: (line [n,512] halo line of the (x0, y0, z0) corner, fx, fy, fz fp32)."""
    corner, frac = [], []
    for u in coords32(R, base, coords):
        i = np.fmin(np.fmax(u, f32(-1.0)), f32(8.0))         # fminf / fmaxf drop NaN
        i0 = np.fmin(np.floor(i), f32(7.0))
        corner.append(i0.astype(np.int64))
        frac.append(i - i0)
    x0, y0, z0 = corner
    return ((z0 + 1) * HALO + (y0 + 1)) * HALO + (x0 + 1), frac[0], frac[1], frac[2]


# ---- the gathers ----------------------------------------------------------------------------------------------------
def gather(vs, R, base=None, pair=None, swap: bool = True, coords: str = "fp32") -> np.ndarray:
    """gather_hypothesis of the fp32 scorer: [n,16,512] fp32 from volumes vs [P,16,8,8,8] (hypothesis i samples
    volume pair[i]; one volume [16,8,8,8] when pair is None)."""
    line, fx, fy, fz = taps32(R, base, coords)
    n = len(line)
    w = _voxels()[2][None]
    sw = (line ^ w) & 1 if swap else np.zeros_like(line)
    one = f32(1.0)
    wx_first = np.where(sw == 1, fx, one - fx)
    wx_second = np.where(sw == 1, one - fx, fx)
    V, off = _halo(vs, f32, pair, n)
    line = line + off
    acc = np.zeros((C, n, VOX), f32)
    for dz in (0, 1):
        for dy in (0, 1):
            wyz = (fy if dy else one - fy) * (fz if dz else one - fz)
            la = line + dz * HALO * HALO + dy * HALO
            acc = fma32(wyz * wx_first, V[:, la + sw], acc)
            acc = fma32(wyz * wx_second, V[:, la + 1 - sw], acc)
    return acc.transpose(1, 0, 2)


def rotate_volume(vol, R, base=None, rounding: bool = True) -> np.ndarray:
    """rotate_volume_kernel: vol [16,8,8,8] (shared) or [n,16,8,8,8] (one per rotation), R [n,3,3] -> [n,16,8,8,8]
    fp32 (fp64 with rounding=False)."""
    R = np.asarray(R, f32).reshape(-1, 9)
    n = len(R)
    vol = np.asarray(vol, f32)
    pair = np.arange(n) if vol.ndim == 5 else None
    if not rounding:
        return T.gather_f64(vol, R, base, pair).reshape(n, C, S, S, S)
    line, fx, fy, fz = taps32(R, base)
    V, off = _halo(vol, f32, pair, n)
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
    line, fx, fy, fz = taps32(R, base)
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


def score(vol_src, tgt_feat, R, W1, W2, b2, *, rounding: bool = True, swap: bool = True, coords: str = "fp32",
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
            A = T.gather_f64(vs[used], Rc, base, slot)
            tri = oracle.triplane_np(A.reshape(n, C, S, S, S)).reshape(n, KTRI, NPOS)
            v = W2.astype(f64) @ np.maximum(W1.astype(f64) @ tri, 0.0) + b2.astype(f64)[:, None]
            nrm = np.maximum(np.sqrt((v * v).sum(axis=1, keepdims=True)), 1e-12)
            out[i0 : i0 + n] = ((v / nrm) * tg[pair].astype(f64)).sum(axis=1).mean(axis=-1)
            return
        A = gather(vs[used], Rc, base, slot, swap=swap, coords=coords)
        tri = oracle.triplane_np(A.reshape(n, C, S, S, S)).reshape(n, KTRI, NPOS)
        h1 = np.fmax(_conv1_chain(tri, W1), f32(0.0))       # fmaxf(acc, 0): NaN -> 0
        a = np.broadcast_to(b2[None, :, None], h1.shape).astype(f32) if b2_first else np.zeros_like(h1)
        for i in range(OCH):
            a = fma32(W2[None, :, i, None], h1[:, None, i, :], a)
        v = a if b2_first else a + b2[None, :, None]
        # thread (pos, cg2) holds channels cg2 * 8 .. cg2 * 8 + 7 of its position
        vq, tq = v.reshape(n, 4, 8, NPOS), tg[pair].reshape(n, 4, 8, NPOS)
        ss = np.zeros((n, 4, NPOS), f32)
        dt = np.zeros((n, 4, NPOS), f32)
        for oo in range(8):
            ss = fma32(vq[:, :, oo], vq[:, :, oo], ss)
            dt = fma32(vq[:, :, oo], tq[:, :, oo], dt)
        ss = (ss[:, 0] + ss[:, 1]) + (ss[:, 2] + ss[:, 3])    # quad_sum as lane 0 sees it
        dt = (dt[:, 0] + dt[:, 1]) + (dt[:, 2] + dt[:, 3])
        cosv = dt / np.fmax(np.sqrt(ss), f32(1e-12))        # [n,64]
        # warp w holds positions 8w .. 8w + 7 in lanes 0, 4, .., 28; the other lanes add 0
        lanes = np.zeros((n, 8, 32), f32)
        lanes[:, :, 0::4] = cosv.reshape(n, 8, 8)
        red = butterfly(lanes)
        tot = np.zeros(n, f32)
        for w in range(8):
            tot = tot + red[:, w]
        out[i0 : i0 + n] = tot * f32(1.0 / 64.0)

    _pool_map(run, range(0, len(items), chunk))
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

    _pool_map(run, range(0, m, chunk))
    return out


# ---- helpers for the tests ------------------------------------------------------------------------------------------
def ulp_distance(a, b) -> np.ndarray:
    """Distance in fp32 ulps (steps of the ordered integer line; +0 and -0 are 0 apart)."""
    def ordered(x):
        u = np.ascontiguousarray(x, f32).view(np.int32).astype(np.int64)
        return np.where(u < 0, -(u & 0x7FFFFFFF), u)
    return np.abs(ordered(a) - ordered(b))


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
