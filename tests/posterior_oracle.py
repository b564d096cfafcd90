"""CPU restatement of ahv_posterior_mass (posterior mass of selected rotations), the definition the GPU kernels are
checked against.  The trace test is select_distinct_np's (tests/distinct_oracle.py): nine float32 products summed left to
right, against c = fp32(1 + 2 cos(theta)).  Test infrastructure only: nothing in the product path imports it."""
from __future__ import annotations

import math

import numpy as np


def trace_threshold_np(theta_deg: float) -> np.float32:
    """c = fp32(1 + 2 cos(theta)) from double, as ahv_topk_distinct and ahv_posterior_mass round it; -inf at 180 degrees
    (every rotation lies within 180 degrees)."""
    if theta_deg >= 180:
        return np.float32(-np.inf)
    return np.float32(1.0 + 2.0 * math.cos(float(np.float32(theta_deg)) * math.pi / 180.0))


def posterior_mass_np(scores: np.ndarray, R: np.ndarray, centers, radius_deg: float, temperature: float = 0.1):
    """ahv_posterior_mass restated: log_z [B] = m/T + log sum_n exp((s - m)/T), and mass [B,k], where hypothesis n goes to
    the lowest slot j with t(n, c_j) >= c (the fp32 trace of select_distinct_np; a NaN centre never passes).  Sums are
    math.fsum of float64 terms.  A -inf score contributes 0; a pair with a NaN or +inf score gets NaN; a pair whose
    scores are all -inf gets log_z = -inf and NaN masses.  centers [B,k,3,3] or None (k = 0)."""
    f = np.float32
    scores = np.asarray(scores, dtype=f)
    B, N = scores.shape
    per_pair = R.ndim == 4
    k = 0 if centers is None else centers.shape[1]
    T = float(f(temperature))
    c = trace_threshold_np(radius_deg)
    log_z = np.empty(B, dtype=f)
    mass = np.zeros((B, k), dtype=f)
    for b in range(B):
        s = scores[b].astype(np.float64)
        if np.isnan(s).any() or np.isposinf(s).any():
            log_z[b], mass[b] = np.nan, np.nan
            continue
        m = s.max()
        if m == -np.inf:
            log_z[b], mass[b] = -np.inf, np.nan
            continue
        e = np.where(np.isneginf(s), 0.0, np.exp((s - m) / T))
        Z = math.fsum(e)
        log_z[b] = f(m / T + math.log(Z))
        Rs = np.asarray(R[b] if per_pair else R, dtype=f).reshape(N, 9)
        slot = np.full(N, -1)
        for j in range(k):
            cj = np.asarray(centers[b, j], dtype=f).reshape(9)
            t = Rs[:, 0] * cj[0]
            for q in range(1, 9):
                t = t + Rs[:, q] * cj[q]
            slot[(slot < 0) & (t >= c)] = j
        for j in range(k):
            mass[b, j] = f(math.fsum(e[slot == j]) / Z)
    return log_z, mass
