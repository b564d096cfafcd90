"""CPU: posterior_oracle.posterior_mass_np, the definition ahv_posterior_mass is checked against, on cases whose answer is
known without it."""
import math
import os
import sys

import numpy as np
import pytest
import torch
from scipy.spatial.transform import Rotation

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import distinct_oracle  # noqa: E402  (tests/distinct_oracle.py)
import posterior_oracle  # noqa: E402  (tests/posterior_oracle.py)


def _rotations(n, seed):
    return Rotation.random(n, random_state=seed).as_matrix().astype(np.float32)


def _geodesic_deg(R, C):
    t = np.einsum("nij,ij->n", R.astype(np.float64), C.astype(np.float64))
    return np.degrees(np.arccos(np.clip((t - 1) / 2, -1, 1)))


def test_half_turn_gives_slot_zero_everything():
    rng = np.random.default_rng(0)
    R = _rotations(500, 1)
    s = rng.uniform(-1, 1, (3, 500)).astype(np.float32)
    _, _, Rb = distinct_oracle.select_distinct_np(s, R, 4, 20.0)
    log_z, mass = posterior_oracle.posterior_mass_np(s, R, Rb, 180.0)
    assert np.all(mass[:, 0] == 1.0) and np.all(mass[:, 1:] == 0.0)
    want = [s[b].max() / np.float32(0.1) + math.log(math.fsum(np.exp((s[b].astype(np.float64) - s[b].max()) / 0.1)))
            for b in range(3)]
    assert np.allclose(log_z, want, rtol=1e-6)


def test_large_temperature_gives_counts_over_n():
    rng = np.random.default_rng(1)
    R = _rotations(2000, 2)
    s = rng.uniform(-1, 1, (2, 2000)).astype(np.float32)
    _, _, Rb = distinct_oracle.select_distinct_np(s, R, 5, 40.0)
    _, mass = posterior_oracle.posterior_mass_np(s, R, Rb, 40.0, temperature=1e7)
    for b in range(2):
        taken = np.zeros(2000, dtype=bool)
        for j in range(5):
            if np.isnan(Rb[b, j]).any():
                assert mass[b, j] == 0.0
                continue
            near = (_geodesic_deg(R, Rb[b, j]) < 40.0 - 1e-3) & ~taken
            far = _geodesic_deg(R, Rb[b, j]) > 40.0 + 1e-3
            taken |= ~far
            # away from the boundary the count is exact; allow the few hypotheses within 1e-3 degree of it
            assert abs(mass[b, j] - near.sum() / 2000) <= ((~near & ~far).sum() + 1) / 2000, (b, j)


@pytest.mark.parametrize("k,theta", [(1, 5.0), (8, 15.0), (32, 30.0), (32, 90.0)])
def test_mass_sums_to_at_most_one(k, theta):
    rng = np.random.default_rng(k)
    R = _rotations(3000, k)
    s = (rng.standard_normal((4, 3000)) * 0.3).astype(np.float32)
    _, _, Rb = distinct_oracle.select_distinct_np(s, R, k, theta)
    _, mass = posterior_oracle.posterior_mass_np(s, R, Rb, theta)
    assert np.all(mass >= 0) and np.all(mass.sum(1) <= 1 + 1e-6)
    filled = ~np.isnan(Rb).any((2, 3))
    assert np.all(mass[~filled] == 0) and np.all(mass[filled] > 0)


def test_empty_slots_neg_inf_and_nan_scores():
    R = _rotations(100, 3)
    s = np.random.default_rng(3).standard_normal((3, 100)).astype(np.float32)
    C = np.full((3, 2, 3, 3), np.nan, dtype=np.float32)
    C[:, 0] = R[0]
    s[1, 50:] = -np.inf
    s[2, 7] = np.nan
    log_z, mass = posterior_oracle.posterior_mass_np(s, R, C, 30.0)
    assert np.all(mass[:2, 1] == 0) and np.isfinite(log_z[:2]).all()
    ref_log_z, _ = posterior_oracle.posterior_mass_np(s[1:2, :50], R[:50], C[1:2], 30.0)
    assert np.isclose(log_z[1], ref_log_z[0], rtol=1e-7)                  # -inf scores contribute nothing
    assert np.isnan(log_z[2]) and np.isnan(mass[2]).all()
    s[2] = -np.inf
    log_z, mass = posterior_oracle.posterior_mass_np(s, R, C, 30.0)
    assert log_z[2] == -np.inf and np.isnan(mass[2]).all()


def test_single_gt_centre_is_infonce():
    """k = 1, centre = the ground truth, radius = ACC_THR: -log mass is the InfoNCE loss of training.infonce_loss_torch,
    on sets with no hypothesis within 0.5 degree of the radius (where the arccos test and the trace test agree)."""
    import importlib

    training = importlib.import_module("3dahv_b200.training")
    rng = np.random.default_rng(4)
    thr = 15.0
    B, N = 4, 4000
    G = _rotations(B, 5)
    R = np.stack([_rotations(N, 10 + b) for b in range(B)])
    for b in range(B):                                                   # a few hypotheses near the GT
        R[b, :40] = (Rotation.from_matrix(G[b]) * Rotation.from_rotvec(rng.normal(size=(40, 3)) * 0.1)).as_matrix()
        R[b, np.abs(_geodesic_deg(R[b], G[b]) - thr) < 0.5] = G[b]        # nothing within 0.5 degree of the radius
    assert all((np.abs(_geodesic_deg(R[b], G[b]) - thr) >= 0.5).all() for b in range(B))
    s = (rng.standard_normal((B, N)) * 0.2).astype(np.float32)
    s[:, :40] += 0.5
    _, mass = posterior_oracle.posterior_mass_np(s, R, G[:, None], thr)
    loss = training.infonce_loss_torch(torch.from_numpy(s).double(), torch.from_numpy(R).double(),
                                       torch.from_numpy(G).double(), thr).numpy()
    assert np.allclose(-np.log(mass[:, 0].astype(np.float64)), loss, rtol=1e-6, atol=1e-7)
