"""numpy restatements of the kernel arithmetic that several kernels share, one per device function.

TEST INFRASTRUCTURE ONLY.  The kernel models (tc_model.py: the tensor-core scorer, tc_bwd_model.py: the tensor-core
backward, fp32_model.py: the fp32 CUDA-core kernels) build on these; each takes the kernel-specific choices as
parameters:

  roundings        rn16, rz16 (cvt.rn / cvt.rz .f16), fma32 (fmaf, correctly rounded), fma16 (HFMA2), ilogb32,
                   exp_bits (the fp32 exponent field), bf16_round, ulp_distance.
  butterfly        warp_sum (ahv_common.cuh): x + shfl_xor(x, o) for o = 16, 8, 4, 2, 1.
  coordinates      sample_coords / unnorm (ahv_common.cuh): g = fmaf(R2, z, fmaf(R1, y, R0 x)),
                   u = fmaf(g + 1, 4, -0.5); coords="tc": the tensor-core gather's order fmaf(R0, x, fmaf(R2, z, R1 y)).
                   sample_coords64 is the exact form, from fp32 base coordinates or the fp64 linspace of fp64 autograd.
  taps             tap_at: clamp to [-1, 8] with fminf / fmaxf (NaN-dropping), corner floor(u) capped at 7, fraction
                   u - corner, halo line of the corner; in the precision of its input.
  volume layout    voxels (the (d, h, w) of output voxel v) and halo (the zero-halo layout, 10^3 lines per volume).
  gathers          gather32: the fp32 trilinear gather of gather_hypothesis, gather_rotated and the tensor-core scorer's
                   fp32 gather; gather64: trilinear resampling in fp64.
  head_dots        |v|^2 and <v, t> as four 8-channel fmaf chains, added as quad_sum does (0 + 1) + (2 + 3).
  chunks           run_chunks: chunks of items on all cores, results in chunk order.
  cases            the rotations, volumes and head weights the models' case lists draw.
"""
from __future__ import annotations

import itertools
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from oracle import ahv_oracle as oracle
from oracle.ahv_oracle import C, KTRI, NPOS, OCH, VOX  # noqa: F401  (the models take their sizes from here)

S = oracle.D                                                   # edge of a volume
HALO = S + 2                                                   # kHalo: edge of a volume with its zero halo
f16, f32, f64 = np.float16, np.float32, np.float64


# ---- roundings ------------------------------------------------------------------------------------------------------
def rn16(x) -> np.ndarray:
    """Round to fp16, to nearest even, subnormals and overflow to inf included (cvt.rn.f16)."""
    with np.errstate(over="ignore"):
        return np.asarray(x).astype(f16)


def rz16(x) -> np.ndarray:
    """Round to fp16 toward zero (cvt.rz.f16): finite inputs never become inf."""
    x = np.asarray(x, dtype=f64)
    with np.errstate(over="ignore"):
        h = x.astype(f16)
    over = np.abs(h.astype(f64)) > np.abs(x)
    return np.where(over, np.nextafter(h, f16(0)), h)


def fma32(a, b, c) -> np.ndarray:
    """fp32 fused multiply-add, correctly rounded.  The product of two fp32 values is exact in fp64; the sum s =
    fl64(p + c) is made round-to-odd (TwoSum gives its error e; when e != 0 and s has an even last bit, s moves one
    fp64 ulp towards p + c), and round-to-odd at 53 >= 2 * 24 + 2 bits followed by round-to-nearest at 24 bits is the
    correctly rounded result (Boldo & Melquiond).  fp32 subnormal results included.

    Every fp32 midpoint is an fp64 value, so RN64 cannot carry p + c across one: RN32(s) differs from RN32(p + c) only
    when s is itself a midpoint.  Only those elements (low 29 bits 1 << 28 in the normal range) and the nonzero ones of
    fp32's subnormal range take the round-to-odd path."""
    p = np.asarray(a, f32).astype(f64) * np.asarray(b, f32).astype(f64)
    c = np.asarray(c, f32).astype(f64)
    shape = np.broadcast(p, c).shape
    s = np.atleast_1d(p + c)
    r = s.astype(f32)
    u = s.view(np.int64)
    risky = ((u & 0x1FFFFFFF) == 0x10000000) | ((np.abs(s) < 2.0 ** -126) & (s != 0))
    if risky.any():
        i = np.nonzero(risky)
        pi, ci, si = np.broadcast_to(p, s.shape)[i], np.broadcast_to(c, s.shape)[i], s[i]
        t = si - pi
        e = (pi - (si - t)) + (ci - t)                       # TwoSum: si + e == pi + ci exactly
        ui = si.view(np.int64)
        fix = (e != 0) & ((ui & 1) == 0)
        ui = ui + fix * (np.sign(e) * np.sign(si)).astype(np.int64)  # towards p + c: away from zero when e, s agree
        r[i] = ui.view(f64).astype(f32)
    return r.reshape(shape)


def fma16(a, b, c) -> np.ndarray:
    """fp16 fused multiply-add (HFMA2): exact in fp64, rounded once to fp16."""
    return rn16(np.asarray(a, f64) * np.asarray(b, f64) + np.asarray(c, f64))


def ilogb32(x) -> np.ndarray:
    """ilogbf of positive float32 values: floor(log2 x), subnormals included, INT_MAX for inf."""
    x = np.asarray(x, f32)
    return np.where(np.isinf(x), 2**31 - 1, np.frexp(x)[1].astype(np.int64) - 1)


def exp_bits(x) -> np.ndarray:
    """((float_as_int(x) >> 23) & 0xff) - 127: floor(log2 x) of a normal positive fp32, -127 for zero and subnormals."""
    return ((np.asarray(x, f32).view(np.uint32) >> 23) & 0xFF).astype(np.int64) - 127


def bf16_round(x: np.ndarray) -> np.ndarray:
    """float32 -> the float32 value of its bf16 rounding (to nearest even), as torch's .bfloat16() makes it."""
    u = np.ascontiguousarray(x, f32).view(np.uint32).astype(np.uint64)
    u = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return u.astype(np.uint32).view(f32)


def ulp_distance(a, b) -> np.ndarray:
    """Distance in fp32 ulps (steps of the ordered integer line; +0 and -0 are 0 apart)."""
    def ordered(x):
        u = np.ascontiguousarray(x, f32).view(np.int32).astype(np.int64)
        return np.where(u < 0, -(u & 0x7FFFFFFF), u)
    return np.abs(ordered(a) - ordered(b))


def butterfly(x, axis=-1) -> np.ndarray:
    """warp_sum over a 32-long axis in fp32: x + shfl_xor(x, o) for o = 16, 8, 4, 2, 1.  The adds are commutative, so
    every lane ends with the same tree; lane 0's value is returned."""
    x = np.moveaxis(np.asarray(x, f32), axis, -1)
    lane = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        x = x + x[..., lane ^ o]
    return x[..., 0]


# ---- coordinates and taps -------------------------------------------------------------------------------------------
def voxels():
    v = np.arange(VOX)
    return v >> 6, (v >> 3) & 7, v & 7                       # (d, h, w) of the output voxel


def sample_coords(R, base=None, coords: str = "make_tap"):
    """Unclamped sample positions (ux, uy, uz) [n,512] fp32 of the output voxels under R [n,9] (or [...,3,3]):
    sample_coords and unnorm.  coords="tc": the tensor-core gather's order fmaf(R0, x, fmaf(R2, z, R1 y))."""
    base = oracle.base_coords_np() if base is None else np.asarray(base, f32)
    R = np.asarray(R, f32).reshape(-1, 9)
    d, h, w = voxels()
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


def sample_coords64(R, base=None):
    """The same positions in fp64 (no rounding anywhere) from base coordinates taken as given: the kernels' fp32 values
    (the default), or the fp64 linspace that fp64 autograd samples."""
    b = np.asarray(oracle.base_coords_np() if base is None else base, f64)
    d, h, w = voxels()
    g = np.asarray(R, f64).reshape(-1, 3, 3) @ np.stack([b[w], b[h], b[d]])
    u = (g + 1.0) * 4.0 - 0.5
    return [u[:, i] for i in range(3)]


def tap_at(u):
    """tap_at of positions u = (ux, uy, uz) in their precision: ((x0, y0, z0) int [n,512], (fx, fy, fz), line [n,512]
    the halo line of the (x0, y0, z0) corner)."""
    corner, frac = [], []
    for t in u:
        i = np.fmin(np.fmax(t, -1.0), 8.0)                   # fminf / fmaxf drop NaN
        i0 = np.fmin(np.floor(i), 7.0)
        corner.append(i0.astype(np.int64))
        frac.append(i - i0)
    x0, y0, z0 = corner
    return corner, frac, ((z0 + 1) * HALO + (y0 + 1)) * HALO + (x0 + 1)


def halo(vol: np.ndarray, dtype, pair, n: int):
    """[P,16,8,8,8] or [16,8,8,8] -> ([16, P*1000] with the zero halo: line ((z+1)*10 + (y+1))*10 + (x+1) of volume p
    at p*1000 + line, the line offset [n,1] of each hypothesis' volume)."""
    vol = np.asarray(vol).reshape(-1, C, S, S, S)
    out = np.zeros((vol.shape[0], C, HALO, HALO, HALO), dtype)
    out[:, :, 1:9, 1:9, 1:9] = vol
    off = np.zeros((n, 1), np.int64) if pair is None else np.asarray(pair, np.int64).reshape(n, 1) * HALO ** 3
    return out.transpose(1, 0, 2, 3, 4).reshape(C, -1), off


# ---- gathers --------------------------------------------------------------------------------------------------------
def gather32(vol, R, base=None, pair=None, parity: str | None = "w", coords: str = "make_tap") -> np.ndarray:
    """The fp32 trilinear gather of vol [16,8,8,8] under R [n,3,3]: [n,16,512] fp32.  With volumes [P,16,8,8,8],
    hypothesis i samples volume pair[i].

    Corners (dy, dz) in the order (0,0) (1,0) (0,1) (1,1); wyz = wy wz and each tap weight wyz wx rounded, one FMA per
    tap.  The x taps of a corner go in the order of the lane's bank parity p, swapped when (line ^ p) & 1: p = w for
    gather_hypothesis and gather_rotated ("w"), (h >> 2) & 1 for the tensor-core scorer's gather ("h"); None: x0
    first."""
    _, (fx, fy, fz), line = tap_at(sample_coords(R, base, coords))
    _, h, w = voxels()
    swap = np.zeros_like(line) if parity is None else (line ^ {"w": w, "h": (h >> 2) & 1}[parity][None]) & 1
    one = f32(1.0)
    wxa = np.where(swap == 1, fx, one - fx)
    wxb = np.where(swap == 1, one - fx, fx)
    V, off = halo(vol, f32, pair, len(line))
    line = line + off
    acc = np.zeros((C,) + line.shape, f32)
    for c in range(4):
        wyz = (fy if c & 1 else one - fy) * (fz if c >> 1 else one - fz)
        la = line + (c >> 1) * HALO * HALO + (c & 1) * HALO
        acc = fma32(wyz * wxa, V[:, la + swap], acc)
        acc = fma32(wyz * wxb, V[:, la + 1 - swap], acc)
    return acc.transpose(1, 0, 2)


def gather64(vol, R, base=None, pair=None) -> np.ndarray:
    """Trilinear resampling with zero padding in fp64 (no rounding anywhere): [n,16,512] fp64, base coordinates as
    sample_coords64 takes them, volumes as gather32."""
    _, (fx, fy, fz), line = tap_at(sample_coords64(R, base))
    V, off = halo(np.asarray(vol, f64), f64, pair, len(line))
    line = line + off
    acc = np.zeros((C,) + line.shape, f64)
    for dz in (0, 1):
        for dy in (0, 1):
            for dx in (0, 1):
                wgt = (fx if dx else 1 - fx) * (fy if dy else 1 - fy) * (fz if dz else 1 - fz)
                acc += wgt * V[:, line + dz * HALO * HALO + dy * HALO + dx]
    return acc.transpose(1, 0, 2)


# ---- the head -------------------------------------------------------------------------------------------------------
def head_dots(v, t, axis: int = -1):
    """head_dots and quad_sum over the 32 channels on `axis`: lane q of a quad chains channels 8q .. 8q + 7 in fmaf
    from 0 (v v and v t), then (q0 + q1) + (q2 + q3).  Returns (ss, dt) fp32 without that axis."""
    v, t = (np.moveaxis(np.asarray(a, f32), axis, -1) for a in (v, t))
    vq, tq = v.reshape(v.shape[:-1] + (4, 8)), t.reshape(t.shape[:-1] + (4, 8))
    ss = np.zeros(vq.shape[:-1], f32)
    dt = np.zeros(vq.shape[:-1], f32)
    for o in range(8):
        ss = fma32(vq[..., o], vq[..., o], ss)
        dt = fma32(vq[..., o], tq[..., o], dt)
    return (ss[..., 0] + ss[..., 1]) + (ss[..., 2] + ss[..., 3]), (dt[..., 0] + dt[..., 1]) + (dt[..., 2] + dt[..., 3])


# ---- chunks ---------------------------------------------------------------------------------------------------------
def run_chunks(fn, starts) -> list:
    """fn(i0) for every chunk start, on all cores (numpy releases the GIL in its loops); the results in chunk order."""
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as pool:
        return list(pool.map(fn, starts))


# ---- case helpers ---------------------------------------------------------------------------------------------------
def random_rotations(rng, *shape) -> np.ndarray:
    """Rotations [*shape,3,3] fp32 from rng's normal quaternions."""
    n = int(np.prod(shape))
    return oracle.rotations_from_normals_np(rng.normal(size=(n, 4)).astype(f32)).reshape(*shape, 3, 3)


def random_volumes(rng, B):
    """A source and a target batch [B,16,8,8,8] fp32 of normal(-0.2, 1.1) voxels."""
    return [(rng.normal(size=(B, C, S, S, S)) * 1.1 - 0.2).astype(f32) for _ in range(2)]


def trained_like(W1, W2, kind, seed):
    """tests/test_gpu_weight_range.py's kinds of trained-looking head weights, drawn with numpy."""
    rng = np.random.default_rng(seed)
    if kind == "row_scales":                                 # log-uniform row scales over 2^0 .. 2^6
        W1 = W1 * np.exp2(rng.random((OCH, 1)) * 6)
    elif kind == "student_t":                                # heavy-tailed entries (df = 3), about 10 % exact zeros
        def draw(shape, scale):
            t = rng.normal(size=shape) / np.sqrt((rng.normal(size=(3,) + shape) ** 2).sum(0) / 3)
            return np.where(rng.random(shape) < 0.1, 0.0, t * scale)
        W1, W2 = draw((OCH, KTRI), 1 / np.sqrt(KTRI)), draw((OCH, OCH), 1 / np.sqrt(OCH))
    elif kind == "zero_rows":                                # two dead conv1 channels
        W1 = W1.copy()
        W1[[5, 22]] = 0.0
    return W1.astype(f32), W2.astype(f32)


def lattice_rotations() -> np.ndarray:
    """The 24 proper signed permutation matrices [24,3,3]: every sample lands on a lattice point."""
    out = []
    for p in itertools.permutations(range(3)):
        for sg in itertools.product((1, -1), repeat=3):
            R = np.zeros((3, 3), f32)
            R[[0, 1, 2], list(p)] = sg
            if np.linalg.det(R) > 0:
                out.append(R)
    return np.stack(out)


def axis_rotation(axis, deg) -> np.ndarray:
    a = np.asarray(axis, f64) / np.linalg.norm(axis)
    t = np.deg2rad(deg)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return (np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * K @ K).astype(f32)


def outside_rotations() -> np.ndarray:
    """Rotations that send samples outside [-1, 8): 45 degrees about z, 30 about a face diagonal, and three more (the
    set of tests/test_gpu_rotation_grad.py)."""
    return np.stack([axis_rotation((0, 0, 1), 45), axis_rotation((1, 1, 0), 30), axis_rotation((1, 0, 0), 45),
                     axis_rotation((0, 1, 1), 60), axis_rotation((1, -2, 0.5), 135)])
