"""CPU: the numpy and C restatements of the nested Hopf x HEALPix SO(3) grid (tests/hopf_oracle.py, tests/hopf_oracle.c)
agree, and the grid has the properties its definition promises at levels 0-3."""
import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import hopf_oracle as h  # noqa: E402  (tests/hopf_oracle.py)

LEVELS = (0, 1, 2, 3)


@pytest.fixture(scope="module")
def grids():
    return {L: h.hopf_grid_np(L) for L in LEVELS}


def test_level0_healpix_centres_are_the_known_values():
    z, phi = h.pix2ang(0, np.arange(12))
    m = np.arange(4)
    np.testing.assert_allclose(z[:4], 2 / 3, rtol=0, atol=1e-15)                    # north cap
    np.testing.assert_allclose(z[4:8], 0.0, rtol=0, atol=1e-15)                     # equator
    np.testing.assert_allclose(z[8:], -2 / 3, rtol=0, atol=1e-15)                   # south cap
    np.testing.assert_allclose(phi[:4], math.pi / 4 + m * math.pi / 2, rtol=0, atol=1e-14)
    np.testing.assert_allclose(phi[4:8], m * math.pi / 2, rtol=0, atol=1e-14)
    np.testing.assert_allclose(phi[8:], math.pi / 4 + m * math.pi / 2, rtol=0, atol=1e-14)


@pytest.mark.parametrize("level", LEVELS)
def test_numpy_and_c_restatements_agree_bit_for_bit(level, grids):
    assert np.array_equal(grids[level], h.hopf_grid_c(level))
    first, count = h.cells(level) // 3, min(100, h.cells(level) // 3)                # a range, not only the whole level
    assert np.array_equal(h.hopf_grid_c(level, first, count), grids[level][first:first + count])


@pytest.mark.parametrize("level", LEVELS)
def test_counts_and_proper_rotations(level, grids):
    R = grids[level]
    assert R.shape == (72 * 8 ** level, 3, 3) and R.dtype == np.float32
    Rd = R.astype(np.float64)
    assert np.abs(Rd @ Rd.transpose(0, 2, 1) - np.eye(3)).max() < 2e-6
    assert np.abs(np.linalg.det(Rd) - 1.0).max() < 2e-6
    # distinct cells give distinct rotations (q and -q would collide)
    assert len(np.unique(np.round(R.reshape(-1, 9), 5), axis=0)) == len(R)


@pytest.mark.parametrize("level", LEVELS)
def test_ang2pix_inverts_pix2ang_in_numpy_and_c(level):
    p = np.arange(12 * 4 ** level)
    z, phi = h.pix2ang(level, p)
    assert np.array_equal(h.ang2pix(level, z, phi), p)
    sel = p[:: max(1, len(p) // 97)]
    assert np.array_equal(h.ang2pix_c(level, z[sel], phi[sel]), sel)


@pytest.mark.parametrize("level", LEVELS)
def test_children_lie_inside_their_parent(level):
    parents = np.arange(h.cells(level))
    kids = h.hopf_children_np(parents)                                              # [n,8] = 8i .. 8i+7
    assert np.array_equal(kids.reshape(-1), np.arange(h.cells(level + 1)))
    pp, pj = h.decode(level, parents)
    kp, kj = h.decode(level + 1, kids)
    # S^2: the child's pixel centre, located at the parent's Nside, is the parent's pixel
    z, phi = h.pix2ang(level + 1, kp.reshape(-1))
    assert np.array_equal(h.ang2pix(level, z, phi).reshape(kp.shape), np.broadcast_to(pp[:, None], kp.shape))
    # S^1: the child's psi centre lies inside the parent's interval [2 pi j / n, 2 pi (j + 1) / n), n = 6 * 2^level
    psi = 2.0 * h.psi_half(level + 1, kj)                                            # psi / pi
    n = 6 * 2 ** level
    lo, hi = 2.0 * pj[:, None] / n, 2.0 * (pj[:, None] + 1) / n
    assert ((psi > lo) & (psi < hi)).all()


# Largest over smallest nearest-neighbour angle, measured on CPU with this restatement (equal-volume cells; the ratio
# grows slowly with the level as the HEALPix pixels near the caps and the face corners deform).
NN_RATIO = {0: 1.0298035906512264, 1: 1.0777317071931927, 2: 1.1838534210187994, 3: 1.231543312160427}


@pytest.mark.parametrize("level", LEVELS)
def test_nearest_neighbour_ratio_is_pinned(level, grids):
    assert h.nn_angle_ratio(grids[level]) == pytest.approx(NN_RATIO[level], rel=1e-9)
