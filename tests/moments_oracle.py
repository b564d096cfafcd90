"""CPU restatement of ahv_posterior_moments (first moment of the posterior over each slot), the definition the GPU
kernels are checked against.  Slots come from posterior_mass_np's fp32 trace rule (tests/posterior_oracle.py), weights
and sums are math.fsum of float64 terms, and the mean rotation comes from numpy.linalg.svd with the determinant fixed.
Test infrastructure only: nothing in the product path imports it."""
from __future__ import annotations

import math

import numpy as np

from posterior_oracle import posterior_mass_np, trace_threshold_np


def slots_np(R: np.ndarray, centers: np.ndarray, radius_deg: float) -> np.ndarray:
    """[N] lowest slot j with the fp32 trace t(n, c_j) >= c, or -1 (posterior_mass_np's rule).  R [N,3,3], centers [k,3,3]."""
    f = np.float32
    c = trace_threshold_np(radius_deg)
    Rs = np.asarray(R, dtype=f).reshape(-1, 9)
    slot = np.full(Rs.shape[0], -1)
    for j in range(centers.shape[0]):
        cj = np.asarray(centers[j], dtype=f).reshape(9)
        t = Rs[:, 0] * cj[0]
        for q in range(1, 9):
            t = t + Rs[:, q] * cj[q]
        slot[(slot < 0) & (t >= c)] = j
    return slot


def project_so3_np(M: np.ndarray):
    """(argmax over SO(3) of tr(R^T M), the top-two eigenvalue gap of the q-method's 4x4 matrix): the SVD U S V^T with
    the last singular direction flipped when det(U V^T) < 0.  The gap is 2 (s2 + d s3)."""
    U, S, Vt = np.linalg.svd(M)
    d = 1.0 if np.linalg.det(U @ Vt) > 0 else -1.0
    return U @ np.diag([1.0, 1.0, d]) @ Vt, 2.0 * (S[1] + d * S[2])


def posterior_moments_np(scores: np.ndarray, R: np.ndarray, centers: np.ndarray, radius_deg: float,
                         temperature: float = 0.1):
    """ahv_posterior_moments restated: (log_z [B], mass [B,k], mean_R [B,k,3,3], mean_cos [B,k], moment [B,k,3,3],
    gap [B,k]) in float64 but for log_z and mass (posterior_mass_np's float32).  moment[b,j] = fsum(e_n R_n) / W_j with
    e_n = exp((s_n - m)/T) and W_j = fsum(e_n) over the slot; mean_R from the SVD; mean_cos = (tr(mean_R^T M) - 1)/2
    clamped to [-1, 1].  NaN moments for a pair with a NaN or +inf score and for a slot with W_j == 0."""
    f = np.float32
    scores = np.asarray(scores, dtype=f)
    B, N = scores.shape
    k = centers.shape[1]
    per_pair = R.ndim == 4
    T = float(f(temperature))
    log_z, mass = posterior_mass_np(scores, R, centers, radius_deg, temperature)
    moment = np.full((B, k, 3, 3), np.nan)
    mean_R = np.full((B, k, 3, 3), np.nan)
    mean_cos = np.full((B, k), np.nan)
    gap = np.full((B, k), np.nan)
    for b in range(B):
        s = scores[b].astype(np.float64)
        if np.isnan(s).any() or np.isposinf(s).any() or s.max() == -np.inf:
            continue
        m = s.max()
        e = np.where(np.isneginf(s), 0.0, np.exp((s - m) / T))
        Rb = np.asarray(R[b] if per_pair else R, dtype=f).astype(np.float64).reshape(N, 9)
        slot = slots_np(Rb.astype(f).reshape(N, 3, 3), np.asarray(centers[b]), radius_deg)
        for j in range(k):
            sel = slot == j
            W = math.fsum(e[sel])
            if W == 0.0:
                continue
            M = np.array([math.fsum(e[sel] * Rb[sel, q]) for q in range(9)]).reshape(3, 3) / W
            Rm, g = project_so3_np(M)
            moment[b, j], mean_R[b, j], gap[b, j] = M, Rm, g
            mean_cos[b, j] = min(max((float(np.sum(Rm * M)) - 1.0) / 2.0, -1.0), 1.0)
    return log_z, mass, mean_R, mean_cos, moment, gap
