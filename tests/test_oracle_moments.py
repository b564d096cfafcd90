"""CPU: moments_oracle.posterior_moments_np, the definition ahv_posterior_moments is checked against, on cases whose answer
is known without it."""
import math
import os
import sys

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import moments_oracle  # noqa: E402  (tests/moments_oracle.py)
import posterior_oracle  # noqa: E402  (tests/posterior_oracle.py)

# a signed permutation with det +1: exact in fp32, and its products with fp32 matrices are exact
R_LATTICE = np.array([[0, -1, 0], [0, 0, 1], [-1, 0, 0]], dtype=np.float32)


def _rotations(n, seed):
    return Rotation.random(n, random_state=seed).as_matrix().astype(np.float32)


def _cos_angle(A, B):
    return (float(np.sum(A.astype(np.float64) * B.astype(np.float64))) - 1.0) / 2.0


def test_single_hypothesis_slot():
    R = np.concatenate([R_LATTICE[None], _rotations(1, 3)])                       # an exact and a rounded rotation
    s = np.array([[0.3, -0.2]], dtype=np.float32)
    for n in range(2):
        centers = R[n][None, None]
        _, mass, mean_R, mean_cos, moment, _ = moments_oracle.posterior_moments_np(s, R, centers, 1.0)
        w = np.exp((s[0].astype(np.float64) - 0.3) / np.float64(np.float32(0.1)))
        assert abs(mass[0, 0] - w[n] / w.sum()) < 1e-6
        assert np.abs(moment[0, 0] - R[n]).max() <= 1e-15                        # e R / e, rounded twice
        tol = 1e-15 if n == 0 else 1e-6                                           # fp32 R[1] is orthonormal to ~1e-7
        assert np.abs(mean_R[0, 0] - R[n]).max() <= tol and abs(np.linalg.det(mean_R[0, 0]) - 1) < 1e-12
        assert mean_cos[0, 0] <= 1.0 and 1.0 - mean_cos[0, 0] <= (1e-15 if n == 0 else 1e-7)


@pytest.mark.parametrize("theta_deg", [0.5, 5.0, 14.0])
@pytest.mark.parametrize("axis", [0, 1, 2])
def test_equal_weight_pairs_around_a_rotation(axis, theta_deg):
    """R0 exp(+-theta e_i): the fp32 pair is R0 A and R0 A^T exactly, so M = R0 (A + A^T)/2, mean_R = R0 and mean_cos =
    cos(theta) of the fp32 matrices."""
    v = np.zeros(3)
    v[axis] = math.radians(theta_deg)
    A = Rotation.from_rotvec(v).as_matrix().astype(np.float32)
    R = np.stack([R_LATTICE @ A, R_LATTICE @ A.T, _rotations(1, 5)[0]]).astype(np.float32)
    assert np.array_equal(R[1], (R_LATTICE @ A.T).astype(np.float32))
    s = np.array([[0.25, 0.25, 0.9]], dtype=np.float32)                         # the outsider holds most of p
    _, _, mean_R, mean_cos, moment, gap = moments_oracle.posterior_moments_np(s, R, R_LATTICE[None, None], 20.0)
    cos_fp32 = (float(np.trace(A.astype(np.float64))) - 1.0) / 2.0
    assert np.abs(mean_R[0, 0] - R_LATTICE).max() <= 1e-12
    assert abs(mean_cos[0, 0] - cos_fp32) <= 1e-12 and abs(mean_cos[0, 0] - math.cos(math.radians(theta_deg))) < 1e-7
    assert np.abs(moment[0, 0] - R_LATTICE @ (A.astype(np.float64) + A.T.astype(np.float64)) / 2).max() <= 1e-15
    assert gap[0, 0] > 1.0


def test_trace_identity():
    """mean_cos = E_j[cos theta(R_n, mean_R)]: tr(R^T M) is linear in M."""
    rng = np.random.default_rng(1)
    C = _rotations(3, 11)
    near = np.concatenate([(C[j] @ Rotation.from_rotvec(rng.normal(size=(300, 3)) * 0.12).as_matrix()).astype(np.float32)
                           for j in range(3)])
    R = np.concatenate([near, _rotations(2000, 12)])
    s = rng.uniform(-1, 1, (2, R.shape[0])).astype(np.float32)
    T = 0.3
    _, _, mean_R, mean_cos, _, _ = moments_oracle.posterior_moments_np(s, R, np.stack([C, C[::-1]]), 25.0, T)
    for b in range(2):
        cen = C if b == 0 else C[::-1]
        slot = moments_oracle.slots_np(R, cen, 25.0)
        e = np.exp((s[b].astype(np.float64) - s[b].max()) / np.float64(np.float32(T)))
        for j in range(3):
            sel = np.nonzero(slot == j)[0]
            assert len(sel) > 100
            want = math.fsum(e[n] * _cos_angle(R[n], mean_R[b, j]) for n in sel) / math.fsum(e[sel])
            assert abs(mean_cos[b, j] - want) <= 1e-12 and 0.9 < mean_cos[b, j] < 1.0, (b, j)


def test_mass_and_slots_match_posterior_mass():
    rng = np.random.default_rng(2)
    R = _rotations(3000, 21)
    s = rng.uniform(-1, 1, (3, 3000)).astype(np.float32)
    centers = np.stack([R[rng.choice(3000, 6, replace=False)] for _ in range(3)])
    centers[1, 2] = np.nan                                                       # an empty slot
    lz, mass, mean_R, mean_cos, moment, _ = moments_oracle.posterior_moments_np(s, R, centers, 30.0, 0.05)
    o_lz, o_mass = posterior_oracle.posterior_mass_np(s, R, centers, 30.0, 0.05)
    assert np.array_equal(lz, o_lz) and np.array_equal(mass, o_mass)
    for b in range(3):
        slot = moments_oracle.slots_np(R, centers[b], 30.0)
        e = np.exp((s[b].astype(np.float64) - s[b].max()) / np.float64(np.float32(0.05)))
        for j in range(6):
            assert np.float32(math.fsum(e[slot == j]) / math.fsum(e)) == mass[b, j], (b, j)
    assert np.isnan(moment[1, 2]).all() and np.isnan(mean_R[1, 2]).all() and np.isnan(mean_cos[1, 2])
    ok = ~np.isnan(mean_cos)
    assert ok.sum() == 17 and (np.abs(mean_cos[ok]) <= 1).all()
    dets = np.linalg.det(mean_R[ok])
    assert np.abs(dets - 1).max() < 1e-12


def test_value_rules():
    R = _rotations(400, 31)
    s = np.random.default_rng(3).uniform(-1, 1, (4, 400)).astype(np.float32)
    C = np.stack([R[:2]] * 4)
    s[:, 0] = 1.0                                                                # slot 0's centre holds the maximum
    s[1, 7] = np.nan
    s[2] = -np.inf
    # T = 1e-3: slot 1's scores all lie more than 0.75 below the maximum, so exp((s - m)/T) underflows in double
    slot = moments_oracle.slots_np(R, C[3], 20.0)
    s[3, slot == 1] = s[3].max() - 0.8
    lz, mass, mean_R, mean_cos, moment, _ = moments_oracle.posterior_moments_np(s, R, C, 20.0, 1e-3)
    assert np.isnan(moment[1]).all() and np.isnan(mean_cos[1]).all() and np.isnan(lz[1])
    assert np.isnan(moment[2]).all() and np.isnan(mean_cos[2]).all() and lz[2] == -np.inf
    assert mass[3, 1] == 0 and np.isnan(moment[3, 1]).all() and np.isnan(mean_R[3, 1]).all() and np.isnan(mean_cos[3, 1])
    assert np.isfinite(moment[3, 0]).all() and np.isfinite(moment[0, 0]).all() and np.isfinite(mean_cos[[0, 3], 0]).all()
