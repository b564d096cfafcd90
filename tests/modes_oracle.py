"""CPU restatement of the selection steps of ahv_search_modes (coarse-to-fine search that keeps k distinct modes), given the
scores: the slot of every base cell, the initial beams, each level's segmented top-w and the final ordering of the modes.
The trace test is posterior_mass_np's (tests/posterior_oracle.py): nine float32 products summed left to right, against
c = fp32(1 + 2 cos(theta)).  Keys are ahv_topk's (tests/distinct_oracle.py).  Test infrastructure only: nothing in the
product path imports it."""
from __future__ import annotations

import numpy as np

from distinct_oracle import _topk_keys_np
from posterior_oracle import trace_threshold_np


def trace_np(Rs: np.ndarray, c: np.ndarray) -> np.ndarray:
    """t(n, c) = trace(R_n c^T) for Rs [N,9] and one centre c [9]: nine float32 products summed left to right."""
    t = Rs[:, 0] * c[0]
    for q in range(1, 9):
        t = t + Rs[:, q] * c[q]
    return t


def slots_np(G: np.ndarray, first_idx: np.ndarray, first_R: np.ndarray, min_sep_deg: float) -> np.ndarray:
    """slot [B,n0] of every base cell: j for the winner first_idx[b,j] itself, else the lowest slot j with t(n, c_j) >= c
    (a NaN centre, an empty slot, never passes), else -1."""
    f = np.float32
    B, k = first_idx.shape
    Gs = np.asarray(G, dtype=f).reshape(-1, 9)
    c = trace_threshold_np(min_sep_deg)
    slot = np.full((B, len(Gs)), -1, dtype=np.int64)
    for b in range(B):
        for j in range(k):
            t = trace_np(Gs, np.asarray(first_R[b, j], dtype=f).reshape(9))
            slot[b, (slot[b] < 0) & (t >= c)] = j
        for j in range(k):
            if first_idx[b, j] >= 0:
                slot[b, first_idx[b, j]] = j
    return slot


def _sorted_beam(cells, w: int) -> np.ndarray:
    """w cells ascending, padded with -1 at the end."""
    out = np.full(w, -1, dtype=np.int64)
    cells = np.sort(np.asarray(cells, dtype=np.int64))
    out[: len(cells)] = cells
    return out


def _top_keys(keys: np.ndarray, mask: np.ndarray, w: int) -> np.ndarray:
    """The positions of the (at most) w largest keys where mask holds, largest first."""
    pos = np.flatnonzero(mask)
    return pos[np.argsort(keys[pos], kind="stable")[::-1][:w]]


def beams_np(S0: np.ndarray, slot: np.ndarray, k: int, w: int) -> np.ndarray:
    """The initial beams [B,k,w]: slot j's top-w cells in ahv_topk's key order, then sorted ascending, -1 padded."""
    B = S0.shape[0]
    par = np.full((B, k, w), -1, dtype=np.int64)
    for b in range(B):
        keys = _topk_keys_np(np.asarray(S0[b], dtype=np.float32))
        for j in range(k):
            par[b, j] = _sorted_beam(_top_keys(keys, slot[b] == j, w), w)
    return par


def generator_parents_np(par: np.ndarray) -> np.ndarray:
    """The parents handed to the children generator: a -1 pad becomes cell 0, whose children never qualify."""
    return np.where(par >= 0, par, 0)


def level_np(scores: np.ndarray, kids: np.ndarray, par: np.ndarray, last: bool):
    """One level, given the scores [B, 8kw] of the children kids [B, 8kw] of the beams par [B,k,w] (slot j's children the
    segment [8wj, 8w(j+1))).  Not last: the next beams [B,k,w].  Last: (val [B,k], idx [B,k], pos [B,k]) - each slot's
    best child (its score, grid index and position in the pair's set, -1 for an empty slot), ordered by score
    descending, ties to the lower grid index, empty modes last in slot order."""
    f = np.float32
    B, k, w = par.shape
    nc = 8 * w
    nxt = np.full((B, k, w), -1, dtype=np.int64)
    val = np.full((B, k), -np.inf, dtype=f)
    idx = np.full((B, k), -1, dtype=np.int64)
    pos = np.full((B, k), -1, dtype=np.int64)
    for b in range(B):
        modes = []
        for j in range(k):
            seg = np.asarray(scores[b, nc * j: nc * (j + 1)], dtype=f)
            real = np.repeat(par[b, j] >= 0, 8)
            top = _top_keys(_topk_keys_np(seg), real, w)
            if not last:
                nxt[b, j] = _sorted_beam(kids[b, nc * j + top], w)
            elif len(top):
                t = nc * j + top[0]
                hi = int(_topk_keys_np(seg)[top[0]] >> np.uint64(32))
                modes.append((-hi, int(kids[b, t]), f(seg[top[0]] + f(0)), t))
        for o, (_, cell, v, t) in enumerate(sorted(modes)):
            val[b, o], idx[b, o], pos[b, o] = v, cell, t
    return nxt if not last else (val, idx, pos)


def search_modes_np(S0, G, first_val, first_idx, first_R, min_sep_deg: float, w: int, levels: int, children, score):
    """Steps 3-5 of the search from the base scores S0 [B,n0] of grid G [n0,3,3] and the distinct winners first_*:
    children(level, gen [B,k,w]) -> (kids [B,8kw], R [B,8kw,3,3]) and score(R [B,8kw,3,3]) -> [B,8kw] are the caller's.
    Returns (val [B,k], idx [B,k], R [B,k,3,3]); levels = 0 gives first_* as they are."""
    B, k = first_idx.shape
    if levels == 0:
        return first_val, first_idx, first_R
    par = beams_np(S0, slots_np(G, first_idx, first_R, min_sep_deg), k, w)
    for lev in range(levels):
        kids, kR = children(lev, generator_parents_np(par))
        res = level_np(score(kR), kids, par, lev == levels - 1)
        if lev < levels - 1:
            par = res
    val, idx, pos = res
    R = np.full((B, k, 3, 3), np.nan, dtype=np.float32)
    for b in range(B):
        for o in range(k):
            if pos[b, o] >= 0:
                R[b, o] = kR[b, pos[b, o]]
    return val, idx, R
