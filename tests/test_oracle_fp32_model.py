"""CPU: the numpy model of the fp32 CUDA-core kernels (tests/fp32_model.py) - its exact FMA against rational arithmetic,
its fp64 form against the oracles, its fp32 rotate_volume against oracle.rotate_volume_np on the lattice, and the power
of the bit-exact tests of tests/test_gpu_fp32_model.py to see reorderings that the suite's distance gates cannot."""
import os
import sys
from fractions import Fraction

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import fp32_model as F  # noqa: E402  (tests/fp32_model.py)
import kernel_arith as K  # noqa: E402

f32, f64 = np.float32, np.float64


def _relerr(a, b):
    return float(np.max(np.abs(np.asarray(a, f64) - b) / np.maximum(np.abs(b), 1e-6)))


def _rn32(x: Fraction) -> f32:
    """x rounded to the nearest fp32, ties to an even significand, from exact rational arithmetic."""
    r = f32(float(x))
    cands = [r, np.nextafter(r, f32(np.inf)), np.nextafter(r, f32(-np.inf))]
    dist = [abs(Fraction(float(c)) - x) for c in cands]
    best = min(dist)
    ties = [c for c, d in zip(cands, dist) if d == best]
    return min(ties, key=lambda c: int(np.asarray(c, f32).view(np.int32)) & 1)


def _fma_exact(a, b, c) -> f32:
    return _rn32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


# ---- the exact fp32 FMA ---------------------------------------------------------------------------------------------
def test_fma32_equals_rational_arithmetic_on_random_inputs():
    """Random operands over many binades, fp32 subnormal results and exact cancellations included."""
    rng = np.random.default_rng(3)
    n = 3000
    a = (rng.normal(size=n) * np.exp2(rng.integers(-70, 40, n))).astype(f32)
    b = (rng.normal(size=n) * np.exp2(rng.integers(-70, 40, n))).astype(f32)
    c = (rng.normal(size=n) * np.exp2(rng.integers(-140, 60, n))).astype(f32)
    c[:300] = (-(a[:300].astype(f64) * b[:300]).astype(f32))       # near-cancellation: the product's low bits decide
    a[300:400], b[300:400] = f32(2.0 ** -75), f32(1.5)              # results in fp32's subnormal range
    got = K.fma32(a, b, c)
    want = np.array([_fma_exact(*t) for t in zip(a, b, c)], f32)
    assert np.array_equal(got.view(np.int32), want.view(np.int32)), np.argwhere(got != want)[:5].ravel().tolist()


# p + c lands within 2^-70 of an fp32 midpoint, so fl64(p + c) is the midpoint itself and a tie to even follows
_DOUBLE_ROUNDING = [
    # p = 2^-24 (1 + 2^-23)(1 - 2^-23) = 2^-24 - 2^-70; 1 + 2^-23 + p sits just below 1 + 3 2^-24
    (f32(2.0 ** -24 * (1 + 2.0 ** -23)), f32(1 - 2.0 ** -23), f32(1 + 2.0 ** -23)),
    (f32(-(2.0 ** -24) * (1 + 2.0 ** -23)), f32(1 - 2.0 ** -23), f32(-(1 + 2.0 ** -23))),
    (f32(2.0 ** -4 * (1 + 2.0 ** -23)), f32(1 - 2.0 ** -23), f32(2.0 ** 20 * (1 + 2.0 ** -23))),
    # (3 + 2^-22) - (2^-23 - 2^-69) sits just above the midpoint 3 + 2^-23, whose tie goes down to 3 (even)
    (f32(2.0 ** -23 * (1 + 2.0 ** -23)), f32(-(1 - 2.0 ** -23)), f32(3 + 2.0 ** -22)),
]


@pytest.mark.parametrize("case", range(len(_DOUBLE_ROUNDING)))
def test_fma32_rounds_once_where_fp64_rounds_twice(case):
    a, b, c = _DOUBLE_ROUNDING[case]
    want = _fma_exact(a, b, c)
    assert K.fma32(a, b, c) == want
    s = Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))
    mid = Fraction(float(f64(float(s))))                             # fl64(p + c) is an fp32 midpoint
    assert _rn32(mid) != want and mid != s


def test_fp64_route_double_rounds():
    """The fp64 route float32(a b + c) gets the constructed cases wrong: an fp32 scorer of about 10^6 FMAs per score
    would then be off by an ulp in about one score in 700."""
    wrong = [(f64(a) * f64(b) + f64(c)).astype(f32) != _fma_exact(a, b, c) for a, b, c in _DOUBLE_ROUNDING]
    assert all(wrong)


# ---- the fp64 form against the oracles ------------------------------------------------------------------------------
def test_exact_scorer_equals_the_c_oracle(golden, oracle):
    """rounding=False is the scorer's function in fp64: it equals the C oracle to 1e-6 (both are fp32 restatements of
    it), which checks the model's taps, tri-plane indexing and epilogue independently of its roundings."""
    g, w = golden["shared_n3000_b3"], golden["weights"]
    W = (w["W1"], w["W2"], w["b2"])
    R = g["R"][:200]
    tgt = oracle.forward_3d2d_np(g["vol_tgt"], *W)
    ref = oracle.score_c(g["vol_src"], g["vol_tgt"], R, *W)
    assert _relerr(F.score(g["vol_src"], tgt, R, *W, rounding=False), ref) <= 1e-6
    # and the fp32 model lies within 1e-6 of it too (the kernel's rounding error, DESIGN 4.2)
    assert _relerr(F.score(g["vol_src"], tgt, R[:48], *W), ref[:, :48]) <= 1e-6
    pp = golden["per_pair"]
    got = F.score(g["vol_src"], tgt, pp["R"], *W, rounding=False)
    assert _relerr(got, pp["scores"]) <= 1e-6


def test_exact_target_features_and_rotate_volume_equal_the_oracle(golden, oracle):
    g, w = golden["shared_n3000_b3"], golden["weights"]
    W = (w["W1"], w["W2"], w["b2"])
    vt = np.concatenate([g["vol_tgt"], g["vol_src"]])
    ref = oracle.forward_3d2d_np(vt, *W)
    assert np.abs(F.target_features(vt, *W, rounding=False) - ref).max() <= 1e-6
    assert np.abs(F.target_features(vt, *W) - ref).max() <= 1e-6
    vs = g["vol_src"][1]
    R = g["R"][:300]
    ref = oracle.rotate_volume_np(vs, R)
    scale = np.abs(vs).max()
    assert np.abs(F.rotate_volume(vs, R, rounding=False) - ref).max() <= 2e-6 * scale
    assert np.abs(F.rotate_volume(vs, R) - ref).max() <= 2e-6 * scale


def test_rotate_volume_is_bit_identical_to_the_oracle_on_the_lattice(golden, oracle):
    """On the 24 lattice rotations every sample lands on a lattice point (up to the two base coordinates ATen
    rounds, where both restatements round the same way): the fp32 model and the oracle agree bit for bit, shared and
    per rotation."""
    vs = golden["shared_n3000_b3"]["vol_src"]
    L = K.lattice_rotations()
    ref = oracle.rotate_volume_np(vs[1], L)
    assert np.array_equal(F.rotate_volume(vs[1], L), ref)
    per = np.stack([vs[i % 3] for i in range(len(L))])
    ref = np.stack([oracle.rotate_volume_np(per[i], L[i : i + 1])[0] for i in range(len(L))])
    assert np.array_equal(F.rotate_volume(per, L), ref)


def test_adjoint_reference_is_the_transpose_of_rotate_volume(golden):
    """<rotate_volume(x), g> = <x, adjoint(g)> in fp64, and the bound covers the reference's own terms."""
    R = golden["shared_n3000_b3"]["R"][:20]
    rng = np.random.default_rng(5)
    x = rng.normal(size=(16, 8, 8, 8)).astype(f32)
    g = rng.normal(size=(20, 16, 8, 8, 8)).astype(f32)
    fwd = F.rotate_volume(x, R, rounding=False)
    exact, cnt, bound = F.rotate_volume_adjoint(g, R, per_rotation=False)
    lhs, rhs = float((fwd * g.astype(f64)).sum()), float((x.astype(f64) * exact).sum())
    assert abs(lhs - rhs) <= 1e-5 * np.abs(fwd * g).sum()
    assert exact.shape == (16, 8, 8, 8) and cnt.max() > 0 and np.all(bound >= 0)
    # rotations 0 .. 7 and 8 .. 15 and 16 .. 19 are three CTAs: every element touched is flushed by at most three
    ex1, cnt1, _ = F.rotate_volume_adjoint(g, R, per_rotation=True)
    assert np.allclose(ex1.sum(0), exact, rtol=0, atol=1e-12)
    assert np.all(cnt - cnt1.sum(0) <= 3) and np.all(cnt >= cnt1.sum(0))


# ---- what the bit-exact tests see -----------------------------------------------------------------------------------
# Share of the golden subset's scores (3 pairs x the first 100 hypotheses) whose bits each reordering changes, measured
# with this model: about 29 % (no parity swap), 49 % (tensor-core coordinate order) and 27 % (b2 first), each by at most
# 3 ulps and within 2.1e-7 of fp64.  The suite's fp32 gates (2e-5 against the C oracle) cannot see any of them.
SWITCHES = {"no_parity_swap": (dict(swap=False), 0.2), "tc_coords": (dict(coords="tc"), 0.35),
            "b2_first": (dict(b2_first=True), 0.2)}


@pytest.fixture(scope="module")
def golden_subset(golden):
    g, w = golden["shared_n3000_b3"], golden["weights"]
    W = (w["W1"], w["W2"], w["b2"])
    items = (np.arange(3)[:, None] * 3000 + np.arange(100)[None]).reshape(-1)
    args = (g["vol_src"], g["tgt_feat"], g["R"]) + W
    return args, items, F.score(*args, items=items), F.score(*args, items=items, rounding=False)


@pytest.mark.parametrize("switch", list(SWITCHES))
def test_scorer_reordering_is_visible_to_bits_only(golden_subset, switch):
    args, items, base, exact = golden_subset
    kw, share = SWITCHES[switch]
    moved = F.score(*args, items=items, **kw)
    changed = float(np.mean(moved != base))
    assert changed >= share, (switch, changed)
    assert _relerr(moved, exact) <= 2e-5 and _relerr(base, exact) <= 2e-5


def test_target_feature_division_is_visible_to_bits_only(golden):
    """v / norm instead of v * (1 / norm) changes about 26 % of the target features (golden targets and 61 random
    volumes), each within 2e-7 of fp64: the suite's 2e-6 gate on the target features cannot see it."""
    g, w = golden["shared_n3000_b3"], golden["weights"]
    W = (w["W1"], w["W2"], w["b2"])
    vt = np.concatenate([g["vol_tgt"], (np.random.default_rng(1).normal(size=(61, 16, 8, 8, 8)) * 1.1 - 0.2).astype(f32)])
    base, moved = F.target_features(vt, *W), F.target_features(vt, *W, divide=True)
    exact = F.target_features(vt, *W, rounding=False)
    assert float(np.mean(moved != base)) >= 0.2
    assert np.abs(moved - exact).max() <= 2e-5 and np.abs(base - exact).max() <= 2e-5


def test_ulp_distance():
    one = f32(1.0)
    assert K.ulp_distance(one, np.nextafter(one, f32(2.0))) == 1
    assert K.ulp_distance(f32(0.0), f32(-0.0)) == 0
    assert K.ulp_distance(np.nextafter(f32(0.0), f32(1.0)), np.nextafter(f32(0.0), f32(-1.0))) == 2
    assert K.ulp_distance(f32(-1.0), f32(-1.0)) == 0
