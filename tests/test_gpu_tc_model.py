"""GPU (B200): the tensor-core scorer against a rounding-faithful model of its own arithmetic (tests/tc_model.py).

The parity tests hold AHV_MATH_TC to 1e-3 of fp64, eight times the error its fp16 operands cause; a conversion that
rounds the wrong way or a gather that sums its taps in another order moves the scores by about 1e-4 and hides in that
slack.  The model reproduces every fp16 and fp32 rounding of the forward except the tensor core's fp32 accumulation
order, so the scores are held to tc_model.GATE (3e-5) per element, in the three modes that run the kernel:
fp32 volumes under AHV_MATH_TC (fp32 gather), AHV_MATH_TC_F16GATHER, and bf16 volumes (16-bit gather).  The training
forward's kept activations are compared bit for bit, and the selections against the model's ranking."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import tc_model as M  # noqa: E402  (tests/tc_model.py)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _relerr(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-6)))


def _math(ahv, mode):
    return ahv.MATH_TC_F16GATHER if mode == "f16gather" else ahv.MATH_TC


def _vol(case, mode):
    v = torch.from_numpy(case["vs"]).to(DEV)
    return v.bfloat16() if mode == "bf16" else v


def _head(case):
    return [torch.from_numpy(case[k]).to(DEV) for k in ("W1", "W2", "b2")]


_CASES = {}


@pytest.fixture(scope="module")
def case(golden, request):
    name = request.param
    if name not in _CASES:
        _CASES.clear()
        _CASES[name] = dict(M.make_case(name, golden), name=name)
    return _CASES[name]


def _selection_ok(model, idx, gate):
    """The kernel's j-th pick scores, under the model, within 2 gates of the model's j-th best: the picks agree with
    the model's ranking wherever the model separates neighbours by more than twice the gate."""
    ranked = -np.sort(-model, axis=1)
    picked = np.take_along_axis(model, idx, axis=1)
    bad = np.abs(picked - ranked[:, : idx.shape[1]]) > 2 * gate * np.abs(ranked[:, : idx.shape[1]])
    return not bad.any(), np.argwhere(bad)[:4].tolist()


@pytest.mark.parametrize("case", M.CASES, indirect=True)
@pytest.mark.parametrize("mode", list(M.MODES))
def test_scores_against_the_model(ahv, case, mode):
    """Every score within the gate of the model; the top-4 of ahv_score in the model's order."""
    N = case["R"].shape[-3]
    k = min(4, N)
    s, _, idx = ahv.ops.score(_vol(case, mode), torch.from_numpy(case["tgt"]).to(DEV), torch.from_numpy(case["R"]).to(DEV),
                              *_head(case), k=k, math=_math(ahv, mode))
    s = s.cpu().numpy().astype(np.float64)
    model = M.case_scores(case, mode)
    err = _relerr(s, model)
    where = np.unravel_index(np.argmax(np.abs(s - model) / np.maximum(np.abs(model), 1e-6)), s.shape)
    assert err <= M.gate(mode, case["name"]), (mode, err, "at (pair, hypothesis)", tuple(int(i) for i in where))
    ok, bad = _selection_ok(model, idx.cpu().numpy(), M.gate(mode, case["name"]))
    assert ok, (mode, "top-4 off the model's ranking at (pair, rank)", bad)


@pytest.mark.parametrize("case", ["golden", "ragged_5x1000_per_pair", "pairs_150x5", "outlier_1e6", "student_t"],
                         indirect=True)
@pytest.mark.parametrize("mode", list(M.MODES))
def test_verify_top1_against_the_model(ahv, case, mode):
    """ahv_verify at k = 1 (for fp32 volumes under AHV_MATH_TC the screened arg-max): the winner is the model's, or
    within twice the gate of it."""
    _, _, idx, _ = ahv.ops.verify(_vol(case, mode), torch.from_numpy(case["vt"]).to(DEV), torch.from_numpy(case["R"]).to(DEV),
                                  *_head(case), k=1, math=_math(ahv, mode))
    ok, bad = _selection_ok(M.case_scores(case, mode), idx.cpu().numpy(), M.gate(mode, case["name"]))
    assert ok, (mode, bad)


# conv1's kept activations: the tensor core's fp32 sum of 384 products against the model's exact one, rounded to fp16
H1_MATCH = 0.995


@pytest.mark.parametrize("case", ["golden", "ragged_2x33_per_pair", "pairs_33x17", "R_x0.35", "outlier_1e6", "student_t",
                                  "W1_x2^12"], indirect=True)
def test_training_forward_against_the_model(ahv, case):
    """ahv_score_train: pair_inv bit-identical; at least 99.5 % of h1 bit-identical, and every other element within one
    fp16 ulp of the model plus 2^-20 sum |W1h| |A| (what an fp32 accumulation can explain).  A failure names the
    item, position and channel, so a wrong K slice or tap shows where it is."""
    R = case["R"] if case["R"].shape[-3] <= 1000 else case["R"][:1000]
    s, h1, pinv = ahv.ops.score_train(torch.from_numpy(case["vs"]).to(DEV), torch.from_numpy(case["tgt"]).to(DEV),
                                      torch.from_numpy(np.ascontiguousarray(R)).to(DEV), *_head(case))
    model, mh1, mpinv, bound = M.tc_forward(case["vs"], case["tgt"], R, case["W1"], case["W2"], case["b2"], gather="f32",
                                            want_h1=True)
    assert np.array_equal(pinv.cpu().numpy(), mpinv), (pinv.cpu().numpy()[:4], mpinv[:4])
    assert _relerr(s.cpu().numpy().astype(np.float64), model) <= M.GATE["tc"]
    got = h1.cpu().numpy()
    same = got.view(np.uint16) == mh1.view(np.uint16)
    frac = float(same.mean())
    diff = np.abs(got.astype(np.float64) - mh1.astype(np.float64))
    allowed = np.spacing(np.abs(mh1)).astype(np.float64) + 2.0 ** -20 * bound
    far = np.argwhere(diff > allowed)
    assert len(far) == 0, ("h1 off beyond fp32 accumulation at (item, position, channel)", far[:8].tolist(),
                           got[tuple(far[0])], mh1[tuple(far[0])])
    assert frac >= H1_MATCH, (frac, "mismatches at (item, position, channel)", np.argwhere(~same)[:8].tolist())
