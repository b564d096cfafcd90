"""CPU: the numpy model of the tensor-core scorer (tests/tc_model.py) - its exact form against the C oracle, its fp32
gather against oracle.rotate_volume_np, its rounding helpers against numpy's IEEE types, and the power of the score
gate of tests/test_gpu_tc_model.py to see conversion defects that the 1e-3 gate of the parity tests cannot."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import kernel_arith as K  # noqa: E402  (tests/kernel_arith.py)
import tc_model as M  # noqa: E402  (tests/tc_model.py)

f16, f32, f64 = np.float16, np.float32, np.float64


def _relerr(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-6)))


# ---- the exact form and the gather ----------------------------------------------------------------------------------
def test_exact_form_equals_the_c_oracle(golden, oracle):
    """rounding=False is the scorer's function in fp64: it equals the C oracle to 1e-6, which checks the model's
    coordinate, tap, tri-plane and epilogue indexing independently of its roundings."""
    g, w = golden["shared_n3000_b3"], golden["weights"]
    R = g["R"][:400]
    tgt = oracle.forward_3d2d_np(g["vol_tgt"], w["W1"], w["W2"], w["b2"])
    got = M.tc_forward(g["vol_src"], tgt, R, w["W1"], w["W2"], w["b2"], rounding=False)
    ref = oracle.score_c(g["vol_src"], g["vol_tgt"], R, w["W1"], w["W2"], w["b2"])
    assert _relerr(got, ref) <= 1e-6, _relerr(got, ref)
    # per-pair rotations take the same path
    pp = golden["per_pair"]
    got = M.tc_forward(g["vol_src"], tgt, pp["R"], w["W1"], w["W2"], w["b2"], rounding=False)
    assert _relerr(got, pp["scores"]) <= 1e-6


def test_fp32_gather_equals_rotate_volume_np(golden, oracle):
    """Bit-identical on lattice rotations (every weight is 0 or 1 up to the two base coordinates ATen rounds), within
    a few fp32 ulps of the volume's largest value otherwise (the kernel's FMAs against the oracle's rounded sums)."""
    vs = golden["shared_n3000_b3"]["vol_src"][1]
    L = K.lattice_rotations()
    assert np.array_equal(K.gather32(vs, L, parity="h", coords="tc"),
                          oracle.rotate_volume_np(vs, L).reshape(len(L), 16, 512))
    R = golden["shared_n3000_b3"]["R"][:300]
    got = K.gather32(vs, R, parity="h", coords="tc").astype(f64)
    ref = oracle.rotate_volume_np(vs, R).reshape(len(R), 16, 512)
    assert np.abs(got - ref).max() <= 8 * np.finfo(f32).eps * np.abs(vs).max()
    # and the 16-bit gather lies within fp16 interpolation error of the exact resampling
    vh = K.rn16(vs * f32(1024.0))
    got16 = M.gather_f16(vh, R).astype(f64) / 1024.0
    assert np.abs(got16 - K.gather64(vs, R)).max() <= 8 * 2.0 ** -11 * np.abs(vs).max()


# ---- helpers --------------------------------------------------------------------------------------------------------
def test_rn16_matches_ieee_half():
    """Ties to even, subnormals, the overflow threshold, against numpy's float16 (IEEE binary16)."""
    one_ulp = 2.0 ** -10
    cases = {
        1.0 + one_ulp / 2: 1.0,                          # tie -> even
        1.0 + 3 * one_ulp / 2: 1.0 + 2 * one_ulp,        # tie -> even (upwards)
        1.0 + one_ulp / 2 + 2.0 ** -30: 1.0 + one_ulp,   # just above the tie
        2.0 ** -25: 0.0,                                 # half the smallest subnormal: tie -> 0
        3 * 2.0 ** -25: 2.0 ** -23,                      # 1.5 subnormal ulps -> even (2 ulps)
        2.0 ** -24 * 5.5: 2.0 ** -24 * 6,
        65519.99: 65504.0,                               # below the overflow threshold
        65520.0: np.inf,                                 # the threshold itself rounds to inf
        -65520.0: -np.inf,
    }
    for x, want in cases.items():
        assert float(K.rn16(f64(x))) == want, x
    x = np.random.default_rng(0).normal(size=20000) * np.exp2(np.random.default_rng(1).integers(-28, 17, 20000))
    assert np.array_equal(K.rn16(x), x.astype(f16))
    assert np.array_equal(K.rn16(x.astype(f32)), x.astype(f32).astype(f16))


def test_rz16_truncates():
    x = np.array([1.0 + 2.0 ** -11, -(1.0 + 2.0 ** -11), 1.0 + 2.0 ** -10 - 2.0 ** -30, 65520.0, 1e6, -1e6,
                  2.0 ** -24 * 1.9, 2.0 ** -25, 3.0])
    want = np.array([1.0, -1.0, 1.0, 65504.0, 65504.0, -65504.0, 2.0 ** -24, 0.0, 3.0])
    assert np.array_equal(K.rz16(x).astype(f64), want)
    y = np.random.default_rng(2).normal(size=5000) * 100
    r = K.rz16(y).astype(f64)
    assert np.all(np.abs(r) <= np.abs(y)) and np.all(np.abs(y - r) < np.spacing(np.abs(r).astype(f16)).astype(f64))


def test_fma_is_fused():
    """Cases where a fused multiply-add and a rounded product followed by an add differ."""
    a = f32(1.0 + 2.0 ** -12)
    # a*a = 1 + 2^-11 + 2^-24: the rounded product loses 2^-24, the fused form keeps it
    assert float(K.fma32(a, a, f32(-1.0))) == 2.0 ** -11 + 2.0 ** -24
    assert float((a * a).astype(f32) - f32(1.0)) == 2.0 ** -11
    h = f16(1.0 + 2.0 ** -6)
    # h*h = 1 + 2^-5 + 2^-12: in fp16 the product rounds the 2^-12 away
    assert float(K.fma16(h, h, f16(-1.0))) == 2.0 ** -5 + 2.0 ** -12
    assert float(f16(h * h) - f16(1.0)) == 2.0 ** -5
    # a fused result that lands in fp16's subnormal range
    assert float(K.fma16(f16(2.0 ** -12), f16(2.0 ** -12), f16(0.0))) == 2.0 ** -24


@pytest.mark.parametrize("k", [-20, -7, -1, 1, 5, 13])
def test_weight_exponent_moves_by_k(golden, k):
    W1 = golden["weights"]["W1"].astype(f32)
    W2 = golden["weights"]["W2"].astype(f32)
    _, _, e1, e2 = M.packed_weights(W1, W2)
    W1h2, _, e1k, e2k = M.packed_weights(W1 * f32(2.0 ** k), W2)
    assert e1k == e1 + k and e2k == e2
    # the fp16 operand does not change
    assert np.array_equal(W1h2, M.packed_weights(W1, W2)[0])
    # the normalised row norm lies in [4, 8)
    l1 = float(M.row_l1max(W1h2.astype(f32)))
    assert 4.0 <= l1 < 8.0 * (1 + 2.0 ** -9)


def test_row_l1max_order():
    """The kernel's summation order, not numpy's: a row whose sum depends on the order."""
    W = np.zeros((32, 384), f32)
    W[0, 0] = 1.0
    W[0, 1:] = 2.0 ** -24                                # lost one at a time after 1.0, kept when summed first
    lane = np.arange(32)
    part = np.zeros(32, f32)
    for j in range(12):
        part = (part + W[0, 32 * j : 32 * j + 32]).astype(f32)
    for o in (16, 8, 4, 2, 1):
        part = (part + part[lane ^ o]).astype(f32)
    assert M.row_l1max(W) == part[0]
    assert M.row_l1max(W) != f32(np.sum(W[0].astype(f64)))


def test_pair_exponent_ilogb_boundary():
    """e = floor(log2(bound / max|V|)): exactly at a power of two the exponent is that power, one ulp below it is one
    less.  With l1max = 4 (l1n = 4) the bound is 8192 = 2^13."""
    l1 = f32(4.0)
    assert M.pair_exponent(l1, f32(1.0)) == 13
    assert M.pair_exponent(l1, np.nextafter(f32(1.0), f32(2.0))) == 12
    assert M.pair_exponent(l1, f32(2.0 ** -5)) == 18
    assert M.pair_exponent(l1, f32(3.0)) == 11
    assert M.pair_exponent(l1, f32(2.0 ** -120)) == 100                       # clamped
    assert M.pair_exponent(l1, f32(2.0 ** 120)) == -100
    assert M.pair_exponent(l1, f32(0.0)) is None and M.pair_exponent(l1, f32(np.inf)) is None
    # l1max = 6 * 2^10 -> l1n = 6, bound = fp32(32768 / 6): bound / m = 8 exactly gives 3, one ulp more of m gives 2
    bound = f32(32768.0) / f32(6.0)
    assert M.pair_exponent(f32(6.0 * 2.0 ** 10), bound / f32(8.0)) == 3
    assert M.pair_exponent(f32(6.0 * 2.0 ** 10), np.nextafter(bound / f32(8.0), f32(1e9))) == 2


def test_model_reproduces_the_kernels_scale_symmetry(golden):
    """W1 times a power of two leaves the model's scores and h1 bit-identical and moves pair_inv by that power, as the
    kernel does (tests/test_gpu_weight_range.py)."""
    g, w = golden["shared_n3000_b3"], golden["weights"]
    R = g["R"][:64]
    s0, h0, p0, _ = M.tc_forward(g["vol_src"], g["tgt_feat"], R, w["W1"], w["W2"], w["b2"], want_h1=True)
    s1, h1, p1, _ = M.tc_forward(g["vol_src"], g["tgt_feat"], R, w["W1"] * f32(2.0 ** 9), w["W2"], w["b2"] * f32(2.0 ** 9),
                                 want_h1=True)
    assert np.array_equal(s0, s1) and np.array_equal(h0, h1) and np.array_equal(p1, p0 * f32(2.0 ** 9))


# ---- power of the gate ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def golden_scores(golden):
    g, w = golden["shared_n3000_b3"], golden["weights"]
    return M.tc_forward(g["vol_src"], g["tgt_feat"], g["R"], w["W1"], w["W2"], w["b2"], gather="f32")


@pytest.mark.parametrize("site", ["A", "H1", "W1h"])
def test_gate_sees_round_toward_zero(golden, golden_scores, site):
    """On the GPU test's golden case (3 x 3 000, AHV_MATH_TC) round-toward-zero at one fp16 conversion moves the scores
    by at least 3x the score gate - and by less than the parity tests' 1e-3, which therefore cannot see it."""
    g, w = golden["shared_n3000_b3"], golden["weights"]
    bad = M.tc_forward(g["vol_src"], g["tgt_feat"], g["R"], w["W1"], w["W2"], w["b2"], gather="f32", rz=(site,))
    moved = _relerr(bad, golden_scores)
    assert moved >= 3 * M.GATE["tc"], (site, moved)
    assert moved < 1e-3, (site, moved)
