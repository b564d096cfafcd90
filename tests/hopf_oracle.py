"""CPU restatements of the nested Hopf x HEALPix SO(3) grid (ahv_so3_hopf_grid, ahv_so3_hopf_children): numpy here and plain C
in tests/hopf_oracle.c, both written from Yershova et al. (2010) and the HEALPix nested scheme of Gorski et al. (2005),
not from the CUDA source.  Test infrastructure only: nothing in the product path imports it.

Level L: Nside = 2^L, 12*4^L pixels p, 6*2^L psi-intervals j (centres psi_j = 2 pi (j + 1/2) / (6*2^L)), 72*8^L cells.
Cell i = 6 p0 + j0 at level 0; the children of cell i are 8i + 2a + b (p' = 4p + a, j' = 2j + b)."""
from __future__ import annotations

import ctypes
import math
import os
import subprocess
import tempfile

import numpy as np

from oracle.ahv_oracle import rotations_from_normals_np

_JRLL = np.array([2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4], dtype=np.int64)
_JPLL = np.array([1, 3, 5, 7, 0, 2, 4, 6, 1, 3, 5, 7], dtype=np.int64)


def cells(level: int) -> int:
    return 72 * 8 ** level


def decode(level: int, idx) -> tuple[np.ndarray, np.ndarray]:
    """Cell indices of `level` -> (HEALPix nested pixel p at Nside 2^level, psi interval j)."""
    idx = np.asarray(idx, dtype=np.int64)
    top = idx >> (3 * level)
    p, j = top // 6, top % 6
    for l in range(level - 1, -1, -1):
        d = (idx >> (3 * l)) & 7
        p, j = 4 * p + (d >> 1), 2 * j + (d & 1)
    return p, j


def _even_bits(x: np.ndarray) -> np.ndarray:
    out = np.zeros_like(x)
    for b in range(32):
        out |= ((x >> (2 * b)) & 1) << b
    return out


def _interleave(ix: np.ndarray, iy: np.ndarray) -> np.ndarray:
    out = np.zeros_like(ix)
    for b in range(32):
        out |= (((ix >> b) & 1) << (2 * b)) | (((iy >> b) & 1) << (2 * b + 1))
    return out


def pix2ang_parts(level: int, p):
    """HEALPix nested pix2ang at Nside 2^level, in the exact form the grid uses: (cos^2(theta/2), sin^2(theta/2), phi / pi),
    fp64."""
    p = np.asarray(p, dtype=np.int64)
    nside = 1 << level
    npface = nside * nside
    face = p >> (2 * level)
    ipf = p & (npface - 1)
    ix, iy = _even_bits(ipf), _even_bits(ipf >> 1)
    jr = _JRLL[face] * nside - ix - iy - 1
    north, south = jr < nside, jr > 3 * nside
    nr = np.where(north, jr, np.where(south, 4 * nside - jr, nside))
    t = (nr * nr).astype(np.float64) / (3.0 * float(npface))
    hz = (2 * nside - jr).astype(np.float64) / (3.0 * float(nside))
    c2 = np.where(north, 1.0 - 0.5 * t, np.where(south, 0.5 * t, 0.5 + hz))
    s2 = np.where(north, 0.5 * t, np.where(south, 1.0 - 0.5 * t, 0.5 - hz))
    tp = _JPLL[face] * nr + ix - iy
    tp = np.where(tp < 0, tp + 8 * nr, tp)
    return c2, s2, tp.astype(np.float64) / (4.0 * nr.astype(np.float64))


def pix2ang(level: int, p):
    """(z = cos theta, phi) of the centres of nested pixels p at Nside 2^level."""
    c2, s2, ph = pix2ang_parts(level, p)
    return c2 - s2, ph * math.pi


def ang2pix(level: int, z, phi) -> np.ndarray:
    """HEALPix nested ang2pix at Nside 2^level (Gorski et al. 2005): the pixel holding (z = cos theta, phi)."""
    z, phi = np.asarray(z, dtype=np.float64), np.asarray(phi, dtype=np.float64)
    nside = 1 << level
    za = np.abs(z)
    tt = np.mod(phi * (2.0 / math.pi), 4.0)
    # equatorial zone
    t1, t2 = nside * (0.5 + tt), nside * (z * 0.75)
    jp, jm = (t1 - t2).astype(np.int64), (t1 + t2).astype(np.int64)
    ifp, ifm = jp >> level, jm >> level
    face_eq = np.where(ifp == ifm, ifp | 4, np.where(ifp < ifm, ifp, ifm + 8))
    ix_eq, iy_eq = jm & (nside - 1), nside - (jp & (nside - 1)) - 1
    # polar caps
    ntt = np.minimum(tt.astype(np.int64), 3)
    tp = tt - ntt
    tmp = nside * np.sqrt(3.0 * (1.0 - za))
    jpc = np.minimum((tp * tmp).astype(np.int64), nside - 1)
    jmc = np.minimum(((1.0 - tp) * tmp).astype(np.int64), nside - 1)
    face_c = np.where(z >= 0, ntt, ntt + 8)
    ix_c = np.where(z >= 0, nside - jmc - 1, jpc)
    iy_c = np.where(z >= 0, nside - jpc - 1, jmc)
    eq = za <= 2.0 / 3.0
    face = np.where(eq, face_eq, face_c)
    ix, iy = np.where(eq, ix_eq, ix_c), np.where(eq, iy_eq, iy_c)
    return face * nside * nside + _interleave(ix, iy)


def psi_half(level: int, j) -> np.ndarray:
    """psi_j / 2 in units of pi: (2j + 1) / (12 * 2^level)."""
    return (2 * np.asarray(j, dtype=np.int64) + 1).astype(np.float64) / (3.0 * float(4 << level))


def quaternions(level: int, idx) -> np.ndarray:
    """The fp32 quaternions of cells `idx` of `level`, evaluated in fp64 and rounded once."""
    p, j = decode(level, idx)
    c2, s2, ph = pix2ang_parts(level, p)
    h = psi_half(level, j)
    a = ph + h
    a = np.where(a >= 2.0, a - 2.0, a)
    c, s = np.sqrt(c2), np.sqrt(s2)
    q = np.stack((c * np.cos(math.pi * h), c * np.sin(math.pi * h), s * np.cos(math.pi * a), s * np.sin(math.pi * a)), -1)
    return q.astype(np.float32)


def hopf_grid_np(level: int, first: int = 0, count: int | None = None) -> np.ndarray:
    """Cells [first, first + count) of `level` as rotations [count,3,3] fp32."""
    count = cells(level) - first if count is None else count
    return rotations_from_normals_np(quaternions(level, np.arange(first, first + count, dtype=np.int64)))


def hopf_rotations_np(level: int, idx) -> np.ndarray:
    idx = np.asarray(idx, dtype=np.int64)
    return rotations_from_normals_np(quaternions(level, idx.reshape(-1))).reshape(*idx.shape, 3, 3)


def hopf_children_np(parent_idx) -> np.ndarray:
    """The 8 children [...,8] of cells parent_idx [...]: 8 * parent + c."""
    return 8 * np.asarray(parent_idx, dtype=np.int64)[..., None] + np.arange(8, dtype=np.int64)


def nn_angle_ratio(R: np.ndarray) -> float:
    """Largest over smallest nearest-neighbour geodesic angle of a rotation set [N,3,3] (brute force)."""
    f = R.reshape(-1, 9).astype(np.float64)
    best = np.empty(len(f))
    for lo in range(0, len(f), 2048):
        tr = f[lo:lo + 2048] @ f.T                      # trace(R_a R_b^T) = 1 + 2 cos(angle)
        tr[np.arange(tr.shape[0]), np.arange(lo, lo + tr.shape[0])] = -np.inf
        best[lo:lo + 2048] = tr.max(1)
    nn = np.arccos(np.clip((best - 1.0) / 2.0, -1.0, 1.0))
    return float(nn.max() / nn.min())


# ---- the plain-C restatement (tests/hopf_oracle.c), compiled on first use into a temporary directory ----------------
_C = None


def c_lib():
    global _C
    if _C is None:
        src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hopf_oracle.c")
        so = os.path.join(tempfile.mkdtemp(prefix="ahv_hopf_oracle_"), "libhopf_oracle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", so, src, "-lm"])
        lib = ctypes.CDLL(so)
        lib.hopf_oracle_grid.argtypes = [ctypes.c_int, ctypes.c_int64, ctypes.c_int64, ctypes.POINTER(ctypes.c_float)]
        lib.hopf_oracle_grid.restype = None
        lib.hopf_oracle_ang2pix.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.c_double]
        lib.hopf_oracle_ang2pix.restype = ctypes.c_int64
        _C = lib
    return _C


def hopf_grid_c(level: int, first: int = 0, count: int | None = None) -> np.ndarray:
    count = cells(level) - first if count is None else count
    R = np.empty((count, 9), dtype=np.float32)
    c_lib().hopf_oracle_grid(level, first, count, R.ctypes.data_as(ctypes.POINTER(ctypes.c_float)))
    return R.reshape(-1, 3, 3)


def ang2pix_c(level: int, z, phi) -> np.ndarray:
    fn = c_lib().hopf_oracle_ang2pix
    return np.array([fn(level, float(a), float(b)) for a, b in zip(np.ravel(z), np.ravel(phi))], dtype=np.int64)
