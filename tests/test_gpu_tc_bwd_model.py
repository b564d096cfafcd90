"""GPU (B200): the tensor-core backward against a rounding-faithful model of its own arithmetic (tests/tc_bwd_model.py),
and the rotation gradient of the saved-activation form against fp64.

The training tests hold the saved-activation tcgen05 backward (csrc/ahv_score_bwd_tc.cu) to 1e-3 of fp64 and to 2e-3
of the fp32 contractions; a conversion that rounds the wrong way moves a gradient by 5e-5 to 9e-4 of its maximum and
hides in that slack.  The model reproduces every fp16 and unorm16 conversion and the fp32 arithmetic between them,
leaving out only the tensor core's accumulation order and the order of the sums across items, CTAs and atomics, so
every gradient is held to tc_bwd_model.GATE per element and in L2 (which a coherent bias cannot pass), in the atomic
and the deterministic form, over the shapes, rotations, magnitudes and upstream gradients where the kernel's scales
and paths change.

The rotation gradient of the saved-activation form (ahv_score_backward_ex with the kept h1, fp32 contractions) is held
to fp64 autograd of the function the forward ran, with R as a leaf: directly and through verification_scores."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import tc_bwd_model as BM  # noqa: E402  (tests/tc_bwd_model.py)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)

# grad_R of the saved-activation fp32 form against fp64 autograd of the function that ran, relative to its maximum;
# measured on a B200 (profiles/r17_tc_bwd_model_residual.json)
GATE_R = 2e-5


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


_CASES = {}


@pytest.fixture(scope="module")
def case(ahv, golden, request):
    """A case's inputs, the training forward's h1 and pair_inv from the GPU, and the model's gradients given them."""
    name = request.param
    if name not in _CASES:
        _CASES.clear()
        c = BM.make_case(name, golden)
        args = [_t(c[k]) for k in ("vs", "tgt", "R", "W1", "W2", "b2")]
        _, h1, pinv = ahv.ops.score_train(*args)
        c.update(name=name, args=args, gs_t=_t(c["gs"]), h1=h1, pinv=pinv,
                 model=BM.case_model(c, h1.cpu().numpy(), pinv.cpu().numpy()))
        _CASES[name] = c
    return _CASES[name]


@pytest.mark.parametrize("case", BM.CASES, indirect=True)
@pytest.mark.parametrize("form", ["atomic", "deterministic"])
def test_tc_backward_against_the_model(ahv, case, form):
    """Every gradient of score_backward(..., h1, pair_inv, MATH_TC) within tc_bwd_model.GATE of the model, per element
    and in L2, relative to that gradient's maximum and norm; everything finite."""
    got = ahv.ops.score_backward(*case["args"], case["gs_t"], case["h1"], case["pinv"], ahv.MATH_TC,
                                 deterministic=form == "deterministic")
    for name, g in zip(BM.GRADS, got):
        g = g.cpu().numpy()
        assert np.isfinite(g).all(), (case["name"], form, name)
        r = BM.residual(g, case["model"][name])
        at = np.unravel_index(r["at"], g.shape)
        assert r["elem"] <= BM.GATE[name]["elem"] and r["l2"] <= BM.GATE[name]["l2"], \
            (case["name"], form, name, r, "worst at", tuple(int(i) for i in at))


def test_zero_conv2_agrees_with_fp64(ahv, golden):
    """W2 = 0, b2 = 0: |H2| = 0 below the clamp at every position, dH2 = (g/64) T / 1e-12.  The kernel, the model and
    fp64 agree (1e-3 of each maximum: fp16 operands) and stay finite."""
    c = BM.make_case("zero_conv2", golden)
    args = [_t(c[k]) for k in ("vs", "tgt", "R", "W1", "W2", "b2")]
    _, h1, pinv = ahv.ops.score_train(*args)
    exact = BM.case_model(c, h1.cpu().numpy(), pinv.cpu().numpy(), rounding=False)
    model = BM.case_model(c, h1.cpu().numpy(), pinv.cpu().numpy())
    got = ahv.ops.score_backward(*args, _t(c["gs"]), h1, pinv, ahv.MATH_TC)
    for name, g in zip(BM.GRADS, got):
        g = g.cpu().numpy()
        assert np.isfinite(g).all() and np.isfinite(model[name]).all(), name
        assert BM.residual(g, exact[name])["elem"] <= 1e-3, (name, BM.residual(g, exact[name]))
        assert BM.residual(model[name], exact[name])["elem"] <= 1e-3, name
    assert np.abs(exact["W2"]).max() > 1e6                            # the clamp's 1/1e-12 did reach dW2


def test_verification_scores_saved_tc_vol_src_grad_against_the_model(ahv, golden):
    """verification_scores(save_activations=True) on the golden case: vol_src enters only through the scored branch,
    so its .grad is the kernel's dV - held to the model at the same gates, given the h1 and pair_inv of a separate
    score_train call on the same inputs (the wrapper must pass the kernel the same ones)."""
    c = BM.make_case("golden", golden)
    vt = _t(golden["shared_n3000_b3"]["vol_tgt"][:3])
    W1, W2, b2, R = _t(c["W1"]), _t(c["W2"]), _t(c["b2"]), _t(c["R"])
    tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
    _, h1, pinv = ahv.ops.score_train(_t(c["vs"]), tgt, R, W1, W2, b2)
    vs = _t(c["vs"]).requires_grad_(True)
    s = ahv.training.verification_scores(vs, vt, R, W1, W2, b2, math=ahv.MATH_TC, save_activations=True)
    (s * _t(c["gs"])).sum().backward()
    model = BM.tc_backward(c["vs"], tgt.cpu().numpy(), c["R"], c["W1"], c["W2"], c["b2"], c["gs"], h1.cpu().numpy(),
                           pinv.cpu().numpy())
    r = BM.residual(vs.grad.cpu().numpy(), model["vol_src"])
    assert r["elem"] <= BM.GATE["vol_src"]["elem"] and r["l2"] <= BM.GATE["vol_src"]["l2"], r


# ---- the rotation gradient of the saved-activation form --------------------------------------------------------------
@pytest.mark.parametrize("name", list(BM.R_CASES))
@pytest.mark.parametrize("form", ["atomic", "deterministic"])
def test_saved_fp32_grad_R_against_fp64(ahv, golden, name, form):
    """score_backward(..., h1, pair_inv, MATH_FP32, want_grad_R=True): grad_R within GATE_R of fp64 autograd of the
    function that ran (R a leaf; the gradient reaches R through conv1's pre-activation under the kept mask), the other
    five gradients within 2e-5."""
    c = BM.r_case(golden, name)
    W1, W2, b2 = _t(c["W1"]), _t(c["W2"]), _t(c["b2"])
    tgt = ahv.ops.forward_3d2d(_t(c["vt"]), W1, W2, b2)
    args = (_t(c["vs"]), tgt, _t(c["R"]), W1, W2, b2)
    _, h1, pinv = ahv.ops.score_train(*args)
    got = ahv.ops.score_backward(*args, _t(c["gs"]), h1, pinv, ahv.MATH_FP32, want_grad_R=True,
                                 deterministic=form == "deterministic")
    ref = BM.fp64_autograd(c["vs"], tgt.cpu().numpy(), c["R"], c["W1"], c["W2"], c["b2"], c["gs"], h1.cpu().numpy(),
                           pinv.cpu().numpy(), want_R=True)
    for gname, a, r in zip(BM.GRADS + ("R",), got, ref):
        err = BM.residual(a.cpu().numpy(), r)["elem"]
        assert err <= (GATE_R if gname == "R" else 2e-5), (name, form, gname, err)


@pytest.mark.parametrize("name", list(BM.R_CASES))
def test_verification_scores_saved_R_grad_against_fp64(ahv, golden, name):
    """R.grad of verification_scores(save_activations=True) within GATE_R of fp64 autograd of the function that ran."""
    c = BM.r_case(golden, name)
    W1, W2, b2 = _t(c["W1"]), _t(c["W2"]), _t(c["b2"])
    vt = _t(c["vt"])
    tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
    _, h1, pinv = ahv.ops.score_train(_t(c["vs"]), tgt, _t(c["R"]), W1, W2, b2)
    R = _t(c["R"]).requires_grad_(True)
    s = ahv.training.verification_scores(_t(c["vs"]), vt, R, W1, W2, b2, math=ahv.MATH_TC, save_activations=True)
    (s * _t(c["gs"])).sum().backward()
    ref = BM.fp64_autograd(c["vs"], tgt.cpu().numpy(), c["R"], c["W1"], c["W2"], c["b2"], c["gs"], h1.cpu().numpy(),
                           pinv.cpu().numpy(), want_R=True)[5]
    err = BM.residual(R.grad.cpu().numpy(), ref)["elem"]
    assert err <= GATE_R, (name, err)
