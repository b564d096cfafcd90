"""CPU: the numpy model of the tensor-core backward (tests/tc_bwd_model.py) - its exact form against fp64 autograd of
the function the training forward ran, its per-item scales and 16-bit adjoint weights at their edges, the adjoint's
choice between the work-list row and the exact path, and the power of the gates of tests/test_gpu_tc_bwd_model.py to
see single rounding defects that the 1e-3 gate of the training tests cannot."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import tc_bwd_model as BM  # noqa: E402  (tests/tc_bwd_model.py)
import kernel_arith as K  # noqa: E402
import tc_model as M  # noqa: E402

f32 = np.float32


# ---- the exact form -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("per_pair,shrink", [(False, 1.0), (True, 1.0), (False, 0.35)])
def test_exact_form_equals_fp64_autograd(golden, per_pair, shrink):
    """rounding=False is the gradient of the function the forward ran (kept H1, its ReLU mask) in fp64: it equals
    torch's fp64 autograd of that function to 1e-9 of each gradient's maximum, which pins the model's views, W1^T
    layout, fold and adjoint indexing independently of its roundings.  Upstream gradients over six decades, an outlier
    voxel in the second volume (pair scale); shrink 0.35 is not a rotation (the adjoint's exact path)."""
    g, w = golden["shared_n3000_b3"], golden["weights"]
    B, N = 2, 150
    vs = g["vol_src"][:B].copy()
    vs[1, 3, 2, 5, 1] = 4.0e3
    R = ((g["R"][: B * N].reshape(B, N, 3, 3) if per_pair else g["R"][:N]) * f32(shrink)).astype(f32)
    rng = np.random.default_rng(9)
    gs = (rng.normal(size=(B, N)) * np.logspace(-6, 0, N)[rng.permutation(N)][None]).astype(f32)
    tgt = g["tgt_feat"][:B]
    _, h1, pinv, _ = M.tc_forward(vs, tgt, R, w["W1"], w["W2"], w["b2"], want_h1=True)
    got = BM.tc_backward(vs, tgt, R, w["W1"], w["W2"], w["b2"], gs, h1, pinv, rounding=False)
    ref = BM.fp64_autograd(vs, tgt, R, w["W1"], w["W2"], w["b2"], gs, h1, pinv)
    for name, r in zip(BM.GRADS, ref):
        assert BM.residual(got[name], r)["elem"] <= 1e-9, (name, BM.residual(got[name], r))


# ---- scales, weights, paths -----------------------------------------------------------------------------------------
def test_item_scale_at_its_boundaries():
    """S = 2^(13 - floor(log2 m)): a power of two maps to 2^13 exactly, one ulp below it to just under 2^14; m = 0 gives
    S = 1 (exponent 13); the exponent is clamped to [-100, 100]."""
    for k in (-90, -20, -1, 0, 7, 40):
        m = f32(np.ldexp(1.0, k))
        S, inv = BM.item_scale(m)
        assert m * S == 2.0 ** 13 and S * inv == 1.0
        below = np.nextafter(m, f32(0))
        S2, _ = BM.item_scale(below)
        assert S2 == 2 * S and 2.0 ** 13 <= below * S2 < 2.0 ** 14
    assert BM.item_scale(f32(0.0)) == (1.0, 1.0)
    assert BM.item_scale(f32(2.0 ** -120))[0] == f32(2.0 ** 113)          # subnormal-range bound: clamped at -100
    # the dH2 bound 2 |g/64| / max(sqrt(min |H2|^2), 1e-12): exactly 2^-7, then one ulp below it; |H2| below 1e-12
    assert BM.dh2_bound(f32(2.0 ** -7), f32(4.0)) == f32(2.0 ** -7)
    assert BM.item_scale(BM.dh2_bound(f32(2.0 ** -7), f32(4.0)))[0] == 2.0 ** 20
    b = BM.dh2_bound(np.nextafter(f32(2.0 ** -7), f32(0)), f32(4.0))
    assert b == np.nextafter(f32(2.0 ** -7), f32(0)) and BM.item_scale(b)[0] == 2.0 ** 21
    assert BM.dh2_bound(f32(2.0 ** -20), f32(0.0)) == f32(2.0 ** -19) / f32(1e-12)
    assert BM.dh2_bound(f32(0.0), f32(0.0)) == 0.0 and BM.item_scale(BM.dh2_bound(f32(0.0), f32(0.0)))[0] == 1.0


def test_kappa_at_its_boundaries():
    """kappa = 2^floor(log2(2 / (3 c))): with c = fp32(2/3), 3c rounds to 2 and x = 1 exactly (kappa 1); one ulp more
    of c gives x just under 1 (kappa 1/2); inv_kappa carries 2^e1; all-zero W1 keeps kappa = 1."""
    W = np.zeros((32, 384), f32)
    W[0, 5] = f32(2.0 / 3.0)
    assert BM.kappa_of(W, 3) == (1.0, 8.0)
    W[0, 5] = np.nextafter(f32(2.0 / 3.0), f32(1.0))
    assert BM.kappa_of(W, 3) == (0.5, 16.0)
    W[0, 5], W[1, 5] = f32(2.0 ** 12), f32(2.0 ** 12)                  # c = 2^13: x = 2^-12 / 3 -> 2^-14
    assert BM.kappa_of(W, 0) == (2.0 ** -14, 2.0 ** 14)
    assert BM.kappa_of(np.zeros((32, 384), f32), -2) == (1.0, 0.25)


def test_unorm16_edges():
    """__float2uint_rn(w * 65535): 1 -> 65535, 0 -> 0, products at a half step round to even; _rz truncates."""
    assert BM.unorm16(f32(1.0)) == 65535 and BM.unorm16(f32(0.0)) == 0 and BM.unorm16(f32(1.0), rz=True) == 65535
    seen = set()
    for k in range(1, 4000):
        w = f32((k + 0.5) / 65535.0)
        if f32(w * f32(65535.0)) != k + 0.5:
            continue                                                  # the product is not exactly at the half step
        assert BM.unorm16(w) == (k if k % 2 == 0 else k + 1), k
        assert BM.unorm16(w, rz=True) == k
        seen.add(k % 2)
    assert seen == {0, 1}
    x = np.random.default_rng(0).random(10000).astype(f32)
    assert np.all(np.abs(BM.unorm16(x) - (x * f32(65535)).astype(np.float64)) <= 0.5)


def test_zero_gradient_item_keeps_every_scale_finite(golden):
    """An item with g = 0: both per-item exponents fall back to 13 (S = 1), and it contributes exactly nothing."""
    g, w = golden["shared_n3000_b3"], golden["weights"]
    R = g["R"][:3]
    _, h1, pinv, _ = M.tc_forward(g["vol_src"][:1], g["tgt_feat"][:1], R, w["W1"], w["W2"], w["b2"], want_h1=True)
    gs = np.array([[0.0, 0.0, 0.0]], f32)
    got = BM.tc_backward(g["vol_src"][:1], g["tgt_feat"][:1], R, w["W1"], w["W2"], w["b2"], gs, h1, pinv)
    for name in BM.GRADS:
        assert np.all(got[name] == 0.0), name
    gs[0, 1] = 1.0
    got = BM.tc_backward(g["vol_src"][:1], g["tgt_feat"][:1], R, w["W1"], w["W2"], w["b2"], gs, h1, pinv)
    one = BM.tc_backward(g["vol_src"][:1], g["tgt_feat"][:1], R[1:2], w["W1"], w["W2"], w["b2"], gs[:, 1:2], h1[1:2], pinv)
    for name in BM.GRADS:
        assert np.isfinite(got[name]).all() and np.array_equal(got[name], one[name]), name


def test_adjoint_path_choice(golden):
    """The work list's row holds 16 contributions per input voxel, zero weights included.  A rotation puts up to 17 on
    a voxel (0.6 % of the golden rotations; most stay at 16 or below): those items take the exact path, every other
    rotation the row.  Lattice rotations put at most 8.  Matrices shrunk by 0.35 always overflow the row; in a set with
    every fifth matrix shrunk the path changes per item."""
    R = golden["shared_n3000_b3"]["R"]
    cnt = BM.contributions(R)
    assert cnt.max() == 17 and 0 < (cnt > 16).mean() < 0.02
    assert np.bincount(cnt)[:9].sum() == 0                            # every rotation sends 9 or more to some voxel
    assert BM.contributions(K.lattice_rotations()).max() == 8
    assert (BM.contributions(R[:300] * f32(0.35)) > 16).all()
    mixed = R[:300].copy()
    mixed[::5] *= f32(0.35)
    c = BM.contributions(mixed)
    shrunk = np.zeros(300, bool)
    shrunk[::5] = True
    assert (c[shrunk] > 16).all() and (c[~shrunk] <= 16).mean() > 0.98
    # the model takes the path the counts ask for, item by item
    g, w = golden["shared_n3000_b3"], golden["weights"]
    Rm = mixed[:60].reshape(2, 30, 3, 3)
    _, h1, pinv, _ = M.tc_forward(g["vol_src"][:2], g["tgt_feat"][:2], Rm, w["W1"], w["W2"], w["b2"], want_h1=True)
    gs = np.ones((2, 30), f32)
    _, info = BM.tc_backward(g["vol_src"][:2], g["tgt_feat"][:2], Rm, w["W1"], w["W2"], w["b2"], gs, h1, pinv, info=True)
    assert np.array_equal(info["exact"], c[:60] > 16) and np.array_equal(info["count"], c[:60])


# ---- power of the gates ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def golden_model(golden):
    case = BM.make_case("golden", golden)
    _, h1, pinv, _ = M.tc_forward(case["vs"], case["tgt"], case["R"], case["W1"], case["W2"], case["b2"], want_h1=True)
    return case, h1, pinv, BM.case_model(case, h1, pinv)


def _shift(bad, good):
    """For each gradient: the larger of (per-element shift / its gate, L2 shift / its gate), and the per-element shift."""
    out = {}
    for name in BM.GRADS:
        r = BM.residual(bad[name], good[name])
        out[name] = (max(r["elem"] / BM.GATE[name]["elem"], r["l2"] / BM.GATE[name]["l2"]), r["elem"])
    return out


@pytest.mark.parametrize("defect", ["AT", "W1t", "dH2", "dH1", "dX"])
def test_gates_see_each_rounding_defect(golden_model, defect):
    """On the GPU test's golden case (3 x 700) one fp16 conversion rounding toward zero moves at least one gradient by
    3x its gate or more - and no gradient by 1e-3 of its maximum, the gate of the training tests, which therefore
    cannot see it."""
    case, h1, pinv, good = golden_model
    shift = _shift(BM.case_model(case, h1, pinv, rz=(defect,)), good)
    assert max(s for s, _ in shift.values()) >= 3, (defect, shift)
    assert max(e for _, e in shift.values()) < 1e-3, (defect, shift)


@pytest.mark.parametrize("defect", ["w16", "fold_yxz"])
def test_defects_inside_the_residual(golden_model, defect):
    """Truncating the adjoint's unorm16 weights (5e-5 of vol_src's norm) and folding the views in the order y, x, z
    (2.7e-4) move only vol_src, by less than 3x its L2 gate: the tensor core's accumulation already turns a few fp16
    roundings of dX per item (4.7e-5 of the norm at most), so these two are not separable from the residual at 3x.  This
    pins that statement: if the model or the gates change so that they become separable, they belong in the test above."""
    case, h1, pinv, good = golden_model
    kw = {"fold": "yxz"} if defect == "fold_yxz" else {"rz": (defect,)}
    shift = _shift(BM.case_model(case, h1, pinv, **kw), good)
    assert all(s == 0 for name, (s, _) in shift.items() if name != "vol_src"), (defect, shift)
    assert 0 < shift["vol_src"][0] < 3, (defect, shift)
