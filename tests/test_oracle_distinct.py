"""CPU: distinct_oracle.select_distinct_np, the definition ahv_topk_distinct is checked against, on hand-worked cases."""
import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import distinct_oracle  # noqa: E402  (tests/distinct_oracle.py)


def _rot_z(deg):
    a = math.radians(deg)
    c, s = math.cos(a), math.sin(a)
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]], dtype=np.float32)


@pytest.mark.parametrize("per_pair", [False, True])
@pytest.mark.parametrize("k", [1, 5, 32])
def test_zero_separation_is_select_np(oracle, per_pair, k):
    rng = np.random.default_rng(3)
    B, N = 3, 57
    scores = np.round(rng.standard_normal((B, N)).astype(np.float32), 1)      # many ties
    R = rng.standard_normal((B, N, 3, 3) if per_pair else (N, 3, 3)).astype(np.float32)
    val, idx, Rb = distinct_oracle.select_distinct_np(scores, R, k, 0.0)
    v0, i0 = oracle.select_np(scores, k)
    assert np.array_equal(val[:, : min(k, N)], v0) and np.array_equal(idx[:, : min(k, N)], i0)
    for b in range(B):
        src = R[b] if per_pair else R
        assert np.array_equal(Rb[b, : min(k, N)], src[i0[b]])


def test_rotations_about_one_axis():
    # angles about z, scores descending with the angle list; two ties at 0.5 (index 3 before index 4)
    ang = [0.0, 3.0, 40.0, 180.0, 25.0, 75.0, 41.0, 110.0]
    sc = np.array([[0.9, 0.8, 0.7, 0.5, 0.5, 0.4, 0.3, 0.2]], dtype=np.float32)
    R = np.stack([_rot_z(a) for a in ang])
    # 10 degrees: 0 | 3 is within 10 of 0 | 40 | 180 | 25 | 75 | 41 is within 10 of 40 | 110
    val, idx, _ = distinct_oracle.select_distinct_np(sc, R, 8, 10.0)
    assert idx[0].tolist() == [0, 2, 3, 4, 5, 7, -1, -1]
    assert val[0, 6] == -np.inf and val[0, 0] == np.float32(0.9)
    # 30 degrees: 0 | 40 | 180 | 25 is within 30 of 0 | 75 | 41 is within 30 of 40 | 110
    _, idx, _ = distinct_oracle.select_distinct_np(sc, R, 8, 30.0)
    assert idx[0].tolist() == [0, 2, 3, 5, 7, -1, -1, -1]
    # k stops the selection
    _, idx, _ = distinct_oracle.select_distinct_np(sc, R, 2, 30.0)
    assert idx[0].tolist() == [0, 2]
    # ties go to the lower index: indices 3 and 4 tie at 0.5; moved within 10 degrees of index 2, index 3 is suppressed
    # and index 4 takes its place
    R2 = R.copy()
    R2[3] = _rot_z(38.0)
    _, idx, _ = distinct_oracle.select_distinct_np(sc, R2, 8, 10.0)
    assert idx[0].tolist() == [0, 2, 4, 5, 7, -1, -1, -1]


def test_edge_separations():
    rng = np.random.default_rng(0)
    R = np.stack([_rot_z(a) for a in rng.uniform(0, 360, 40)])
    sc = rng.standard_normal((2, 40)).astype(np.float32)
    val, idx, Rb = distinct_oracle.select_distinct_np(sc, R, 6, 180.0)              # the top-1 alone
    assert (idx[:, 1:] == -1).all() and np.isnan(Rb[:, 1:]).all() and (val[:, 1:] == -np.inf).all()
    assert np.array_equal(idx[:, 0], sc.argmax(1))
    val, idx, _ = distinct_oracle.select_distinct_np(sc[:, :3], R[:3], 5, 1.0)      # N < k: empty tail
    assert (idx[:, 3:] == -1).all() and sorted(idx[0, :3].tolist()) == [0, 1, 2]
    dup = np.repeat(R[:1], 4, axis=0)                                       # duplicated rotations collapse to one
    _, idx, _ = distinct_oracle.select_distinct_np(np.float32([[1.0, 2.0, 3.0, 4.0]]), dup, 4, 0.5)
    assert idx[0].tolist() == [3, -1, -1, -1]
    _, idx, _ = distinct_oracle.select_distinct_np(np.float32([[1.0, 2.0, 3.0, 4.0]]), dup, 4, 0.0)
    assert idx[0].tolist() == [3, 2, 1, 0]
