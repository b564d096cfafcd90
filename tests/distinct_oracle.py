"""CPU restatement of ahv_topk_distinct (top-k of distinct rotations), the definition the GPU kernel is checked against bit
for bit.  Test infrastructure only: nothing in the product path imports it."""
from __future__ import annotations

import math

import numpy as np


def _topk_keys_np(scores: np.ndarray) -> np.ndarray:
    """ahv_topk's 64-bit keys (make_key, csrc/ahv_common.cuh): the device adds +0.0, which turns -0.0 into +0.0 and every
    NaN into the canonical 0x7fffffff, then maps the bits to an order-preserving uint32 above ~index."""
    u = scores.astype(np.float32).view(np.uint32).copy()
    u[np.isnan(scores)] = np.uint32(0x7FFFFFFF)
    u[u == np.uint32(0x80000000)] = np.uint32(0)
    u = np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint64)
    n = np.arange(scores.shape[-1], dtype=np.uint64)
    return (u << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - n)


def select_distinct_np(scores: np.ndarray, R: np.ndarray, k: int, min_sep_deg: float):
    """Top-k of distinct rotations, the definition ahv_topk_distinct computes bit for bit: greedy non-maximum
    suppression over the hypotheses in ahv_topk's order, where n is suppressed by an earlier winner w unless
    t(n, w) = trace(R_n R_w^T) < c = fp32(1 + 2 cos(min_sep_deg)).  t is nine float32 products summed left to right;
    min_sep_deg = 0 suppresses nothing, 180 keeps the top-1 alone.  scores [B,N]; R [N,3,3] or [B,N,3,3].
    Returns (val [B,k] f32, idx [B,k] int64, R_best [B,k,3,3] f32); empty slots are (-inf, -1, NaN)."""
    f = np.float32
    scores = np.asarray(scores, dtype=f)
    B, N = scores.shape
    per_pair = R.ndim == 4
    c = f(1.0 + 2.0 * math.cos(float(f(min_sep_deg)) * math.pi / 180.0))
    rounds = 1 if min_sep_deg >= 180 else k
    val = np.full((B, k), -np.inf, dtype=f)
    idx = np.full((B, k), -1, dtype=np.int64)
    Rb = np.full((B, k, 3, 3), np.nan, dtype=f)
    keys = _topk_keys_np(scores)
    for b in range(B):
        order = np.argsort(keys[b], kind="stable")[::-1]           # keys are distinct: descending key order
        Rs = np.asarray(R[b] if per_pair else R, dtype=f).reshape(N, 9)[order]
        alive = np.ones(N, dtype=bool)
        pos = 0
        for j in range(min(rounds, N)):
            while pos < N and not alive[pos]:
                pos += 1
            if pos == N:
                break
            n = order[pos]
            val[b, j], idx[b, j], Rb[b, j] = f(scores[b, n] + f(0)), n, Rs[pos].reshape(3, 3)
            alive[pos] = False                                      # the key ceiling: nothing at or above the winner
            if min_sep_deg > 0:
                t = Rs[:, 0] * Rs[pos, 0]                           # float32, each product and sum rounded on its own
                for e in range(1, 9):
                    t = t + Rs[:, e] * Rs[pos, e]
                alive &= t < c
    return val, idx, Rb
