"""GPU (B200): the tensor-core paths across head-weight magnitudes.

The fp16 operands of the tensor-core kernels carry W1 and W2 normalised by powers of two (csrc/ahv_tc_common.cuh
pack_weights, and the tcgen05 backward's set-up): W * 2^-e, whose largest row L1 norm lies in [4, 8) for W1 and in
[1, 2) for W2, undone with the pair scale before b2.  Trained checkpoints do not keep the scale of a default initialisation, and the score
has two exact scale symmetries along which weight decay lets them drift freely:

  S1  (W1 c, W2, b2 c)   ReLU is positively homogeneous and F.normalize removes the common factor;
  S2  (W1, W2 c, b2 c).

With c a power of two every operation of every kernel is then exact, so the scores (and the training forward's kept
activations) must be bit-identical to c = 1, and the gradients must move by exact powers of two.  Without the
normalisation, weights below 6.1e-5 went fp16-subnormal, weights above 65504 became inf, and W1's norm ate into the
volume's headroom.  The second half compares with fp64 `oracle.score_torch` at magnitudes that are not powers of two,
at weights beyond fp16's range, at trained-like weight draws, and with outlier volumes under scaled W1."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)

# the suite's score gates, relative: fp32 volumes under the tensor-core modes / the fp32 kernel; bf16 volumes against
# the scores of the bf16-rounded volume
GATE_TC, GATE_FP32, GATE_BF16 = 1e-3, 2e-5, 2e-3
# largest outlier-to-bulk ratio of each mode (include/ahv_b200.h, profiles/r06_dynamic_range.json)
MAX_RATIO = {"fp32": 3e5, "tc": 1e8, "f16gather": 1e8, "bf16": 1e8}


def _modes(ahv):
    return {"fp32": ahv.MATH_FP32, "tc": ahv.MATH_TC, "f16gather": ahv.MATH_TC_F16GATHER}


def _golden_weights(golden):
    return [torch.from_numpy(golden["weights"][k]).float() for k in ("W1", "W2", "b2")]


def _scaled(W, which, c):
    """(W1, W2, b2) with `which` multiplied by c: 'W1', 'W2', 'b2' alone, or the symmetries 'S1' / 'S2'."""
    W1, W2, b2 = W
    if which == "W1":
        return W1 * c, W2, b2
    if which == "W2":
        return W1, W2 * c, b2
    if which == "b2":
        return W1, W2, b2 * c
    if which == "S1":
        return W1 * c, W2, b2 * c
    if which == "S2":
        return W1, W2 * c, b2 * c
    raise ValueError(which)


def _to(W):
    return [t.to(DEV) for t in W]


def _volumes(B, seed):
    gen = torch.Generator().manual_seed(seed)
    vs = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    vt = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    return vs, vt


def _rotations(ahv, B, N, per_pair, seed):
    if per_pair:
        return ahv.so3.sample_rotations(B * N, seed=seed, device=DEV).reshape(B, N, 3, 3).contiguous()
    return ahv.so3.sample_rotations(N, seed=seed, device=DEV)


def _boundary_pairs(B, N):
    """Pairs whose items straddle the per-CTA item ranges of the scoring kernel, plus the first and the last pair."""
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    total = B * N
    grid = min((total + 1) // 2, sms)
    pairs = {0, B - 1}
    for c in (total * i // grid for i in range(1, grid)):
        pairs.update({(c - 1) // N, c // N})
    return sorted(pairs)


def _sample(pairs, n):
    idx = np.unique(np.linspace(0, len(pairs) - 1, n).round().astype(np.int64))
    return [pairs[i] for i in idx]


def _relerr(a, b):
    return float(((a.double() - b.double()).abs() / b.double().abs().clamp_min(1e-6)).max())


def _fp64(oracle, W, vs, vt, R, pairs):
    sel = torch.tensor(pairs)
    Rp = R.cpu()[sel] if R.dim() == 4 else R.cpu()
    return oracle.score_torch(vs[sel].double(), vt[sel].double(), Rp.double(), *(t.double() for t in W)).double()


# ---- exact symmetries ---------------------------------------------------------------------------------------------
# B*N = 300 items: about two per CTA on 148 SMs, so every CTA packs the weights itself; N >= 4 for the k = 4 selection
SYM_B, SYM_N = 75, 4
EXPONENTS = [-16, -8, -3, 3, 8, 16]


@pytest.fixture(scope="module")
def sym_inputs(ahv):
    vs, vt = _volumes(SYM_B, seed=11)
    R = {pp: _rotations(ahv, SYM_B, SYM_N, pp, seed=23 + pp) for pp in (False, True)}
    return vs.to(DEV), vt.to(DEV), R


def _all_consumers(ahv, W, vs, vt, R):
    """Every output of ahv_score (three math modes, fp32 / bf16 volumes, shared / per-pair R) and of ahv_verify
    (k = 1 and 4) for weights W."""
    out = {}
    for pp, Rx in R.items():
        for voldt, v in (("f32", vs), ("bf16", vs.bfloat16())):
            for mode, m in _modes(ahv).items():
                tgt = ahv.ops.forward_3d2d(vt, *W)
                out[pp, voldt, mode, "score"] = ahv.ops.score(v, tgt, Rx, *W, k=1, math=m)
                for k in (1, 4):
                    out[pp, voldt, mode, "verify", k] = ahv.ops.verify(v, vt, Rx, *W, k=k, math=m, return_scores=True)
    return out


@pytest.mark.parametrize("sym", ["S1", "S2"])
@pytest.mark.parametrize("a", EXPONENTS)
def test_scores_are_invariant_under_the_scale_symmetries(ahv, golden, sym_inputs, sym, a):
    """Scores, the fused arg-max, the k = 4 selection and the gathered rotations under S1 / S2 with c = 2^a are
    bit-identical to c = 1, in every math mode, for fp32 and bf16 volumes and shared and per-pair rotations."""
    vs, vt, R = sym_inputs
    W = _golden_weights(golden)
    ref = _all_consumers(ahv, _to(W), vs, vt, R)
    got = _all_consumers(ahv, _to(_scaled(W, sym, 2.0 ** a)), vs, vt, R)
    for key, r in ref.items():
        g = got[key]
        assert torch.isfinite(r[0]).all(), key
        for i, (x, y) in enumerate(zip(g, r)):
            if y is not None:
                assert torch.equal(x, y), (sym, a, key, i, float((x.double() - y.double()).abs().max()))


@pytest.mark.parametrize("sym", ["S1", "S2"])
@pytest.mark.parametrize("a", EXPONENTS)
def test_training_forward_under_the_scale_symmetries(ahv, golden, sym_inputs, sym, a):
    """ahv_score_train: scores and the kept conv1 activations are bit-identical; pair_inv, the factor that turns the
    kept activations into conv1's output, moves by exactly 2^a under S1 and not at all under S2."""
    vs, vt, R = sym_inputs
    W = _golden_weights(golden)
    for Rx in R.values():
        W0 = _to(W)
        s0, h0, p0 = ahv.ops.score_train(vs, ahv.ops.forward_3d2d(vt, *W0), Rx, *W0)
        Wc = _to(_scaled(W, sym, 2.0 ** a))
        s1, h1, p1 = ahv.ops.score_train(vs, ahv.ops.forward_3d2d(vt, *Wc), Rx, *Wc)
        assert torch.equal(s1, s0) and torch.equal(h1, h0), (sym, a)
        assert torch.equal(p1, p0 * (2.0 ** a if sym == "S1" else 1.0)), (sym, a, p0[:4], p1[:4])


def _backward(ahv, W, vs, vt, R, gs, math_):
    tgt = ahv.ops.forward_3d2d(vt, *W)
    _, h1, pinv = ahv.ops.score_train(vs, tgt, R, *W)
    return ahv.ops.score_backward(vs, tgt, R, *W, gs, h1, pinv, math_)


@pytest.mark.parametrize("sym", ["S1", "S2"])
@pytest.mark.parametrize("a", EXPONENTS)
@pytest.mark.parametrize("BN", [(1, 1), (40, 3)])
def test_saved_activation_gradients_under_the_scale_symmetries(ahv, golden, sym, a, BN):
    """Both contraction forms of the saved-activation backward.  S1: grad_vol, grad_tgt, grad_W2 unchanged, grad_W1 and
    grad_b2 times 2^-a.  S2: grad_vol, grad_tgt, grad_W1 unchanged, grad_W2 and grad_b2 times 2^-a.  One item (one CTA,
    one atomic add per output element) is exact but for grad_vol, whose adjoint sums in the order of shared-memory
    integer atomics (2e-6 of its maximum); many items are held to 1e-5 (float-atomic order across CTAs)."""
    B, N = BN
    vs, vt = (t.to(DEV) for t in _volumes(B, seed=5 + B))
    R = _rotations(ahv, B, N, True, seed=9 + B)
    gs = torch.randn(B, N, generator=torch.Generator().manual_seed(3)).to(DEV)
    W = _golden_weights(golden)
    c = 2.0 ** a
    moves = {"S1": (1.0, 1.0, 1.0 / c, 1.0, 1.0 / c), "S2": (1.0, 1.0, 1.0, 1.0 / c, 1.0 / c)}[sym]
    for math_ in (ahv.MATH_FP32, ahv.MATH_TC):
        ref = _backward(ahv, _to(W), vs, vt, R, gs, math_)
        got = _backward(ahv, _to(_scaled(W, sym, c)), vs, vt, R, gs, math_)
        for name, g, r, f in zip(("vol_src", "tgt_feat", "W1", "W2", "b2"), got, ref, moves):
            expect = r * f
            if B * N == 1 and name != "vol_src":
                assert torch.equal(g, expect), (sym, a, math_, name, float((g - expect).abs().max()))
            else:
                tol = 2e-6 if B * N == 1 else 1e-5
                err = float((g.double() - expect.double()).abs().max()) / float(expect.abs().max())
                assert err <= tol, (sym, a, math_, name, err)


# ---- fp64 gates across magnitudes ---------------------------------------------------------------------------------
GATE_B, GATE_N = 150, 3


@pytest.fixture(scope="module")
def gate_inputs(ahv):
    vs, vt = _volumes(GATE_B, seed=31)
    R = _rotations(ahv, GATE_B, GATE_N, True, seed=37)
    return vs, vt, R


def _check_against_fp64(ahv, oracle, W, vs, vt, R, what, modes=("fp32", "tc", "f16gather"), bf16=True):
    """Every mode scores the whole batch on the GPU; 64 items (32 pairs, CTA boundaries included) against fp64."""
    B, N = vs.shape[0], (R.shape[1] if R.dim() == 4 else R.shape[0])
    sample = _sample(_boundary_pairs(B, N), max(1, 64 // N))
    ref = _fp64(oracle, W, vs, vt, R, sample)
    Wd = _to(W)
    vs_d, vt_d = vs.to(DEV), vt.to(DEV)
    for mode in modes:
        s = ahv.HypothesisVerifier(*Wd, math=_modes(ahv)[mode]).score(vs_d, vt_d, R, k=1).scores
        assert torch.isfinite(s).all(), (what, mode)
        err = _relerr(s.cpu()[sample], ref)
        assert err <= (GATE_FP32 if mode == "fp32" else GATE_TC), (what, mode, err)
    if bf16:
        v16 = vs.bfloat16()
        ref16 = _fp64(oracle, W, v16, vt, R, sample)
        s = ahv.HypothesisVerifier(*Wd, math=ahv.MATH_TC).score(v16.to(DEV), vt_d, R, k=1).scores
        assert torch.isfinite(s).all(), (what, "bf16")
        err = _relerr(s.cpu()[sample], ref16)
        assert err <= GATE_BF16, (what, "bf16 vs rounded", err)


@pytest.mark.parametrize("which", ["W1", "W2", "b2", "S1", "S2"])
@pytest.mark.parametrize("k", [-16, -12, -8, -4, 4, 8, 12, 16])
def test_magnitudes_against_fp64(ahv, golden, oracle, gate_inputs, which, k):
    """c = 2^k * 1.37 (not a power of two, so no exactness can mask an error) on W1, W2 or b2 alone, and along S1, S2."""
    vs, vt, R = gate_inputs
    W = _scaled(_golden_weights(golden), which, 2.0 ** k * 1.37)
    _check_against_fp64(ahv, oracle, W, vs, vt, R, (which, k))


@pytest.mark.parametrize("which,k", [("W1", 21), ("W2", 19)])
def test_weights_beyond_the_fp16_range(ahv, golden, oracle, gate_inputs, which, k):
    """Entries above fp16's largest finite value (65504): the scores are finite and meet the gates."""
    vs, vt, R = gate_inputs
    W = _scaled(_golden_weights(golden), which, 2.0 ** k)
    assert float(W[0 if which == "W1" else 1].abs().max()) > 65504
    _check_against_fp64(ahv, oracle, W, vs, vt, R, (which, k))


def _trained_like(golden, kind, seed):
    W1, W2, b2 = _golden_weights(golden)
    gen = torch.Generator().manual_seed(seed)
    if kind == "row_scales":        # log-uniform row scales over 2^0 .. 2^6
        W1 = W1 * torch.pow(2.0, torch.rand(32, 1, generator=gen) * 6)
    elif kind == "student_t":       # heavy-tailed entries (df = 3), about 10 % exact zeros
        def draw(shape, scale):
            z = torch.randn(*shape, generator=gen)
            chi2 = sum(torch.randn(*shape, generator=gen) ** 2 for _ in range(3))
            t = z / torch.sqrt(chi2 / 3)
            return torch.where(torch.rand(*shape, generator=gen) < 0.1, torch.zeros(()), t * scale)
        W1, W2 = draw((32, 384), 1 / math.sqrt(384)), draw((32, 32), 1 / math.sqrt(32))
    elif kind == "zero_rows":       # two dead conv1 channels
        W1 = W1.clone()
        W1[[5, 22]] = 0.0
    else:
        raise ValueError(kind)
    return W1.contiguous(), W2.contiguous(), b2


@pytest.mark.parametrize("kind", ["row_scales", "student_t", "zero_rows"])
def test_trained_like_weights_against_fp64(ahv, golden, oracle, gate_inputs, kind):
    vs, vt, R = gate_inputs
    _check_against_fp64(ahv, oracle, _trained_like(golden, kind, seed=77), vs, vt, R, kind)


def _outlier_volumes(B, r, seed):
    """scripts/dynamic_range.py's pairs: standard-normal bulk, outliers +r/3 and -r (one on a corner voxel)."""
    gen = torch.Generator().manual_seed(seed)
    vs, vt = torch.randn(B, 16, 8, 8, 8, generator=gen), torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    pos = torch.randperm(16 * 512, generator=gen)[: 2 * B].reshape(B, 2)
    pos[0, 1] = 0
    flat = vs.view(B, -1)
    flat[torch.arange(B), pos[:, 0]] = r / 3
    flat[torch.arange(B), pos[:, 1]] = -r
    return vs, vt


@pytest.mark.parametrize("k", [4, 8])
@pytest.mark.parametrize("ratio", [1e2, 1e4, 3e5, 1e6, 3e7, 1e8])
def test_outlier_volumes_under_scaled_W1(ahv, golden, oracle, k, ratio):
    """The volume's headroom no longer depends on W1: at W1 * 2^k each mode meets its gate up to its header bound."""
    B, N = 4, 600
    vs, vt = _outlier_volumes(B, ratio, seed=5)
    R = ahv.so3.sample_rotations(N, seed=17, device=DEV)
    W = _scaled(_golden_weights(golden), "W1", 2.0 ** k)
    pairs = list(range(B))
    ref = _fp64(oracle, W, vs, vt, R, pairs)
    Wd = _to(W)
    for mode, m in _modes(ahv).items():
        if ratio <= MAX_RATIO[mode]:
            s = ahv.HypothesisVerifier(*Wd, math=m).score(vs.to(DEV), vt.to(DEV), R, k=1).scores.cpu()
            err = _relerr(s, ref)
            assert err <= (GATE_FP32 if mode == "fp32" else GATE_TC), (mode, k, ratio, err)
    if ratio <= MAX_RATIO["bf16"]:
        v16 = vs.bfloat16()
        ref16 = _fp64(oracle, W, v16, vt, R, pairs)
        s = ahv.HypothesisVerifier(*Wd, math=ahv.MATH_TC).score(v16.to(DEV), vt.to(DEV), R, k=1).scores.cpu()
        err = _relerr(s, ref16)
        assert err <= GATE_BF16, ("bf16 vs rounded", k, ratio, err)


# ---- backward against fp64 ----------------------------------------------------------------------------------------
def _outlier_batch(B, seed):
    """Order-one bulk plus one outlier voxel of +-2^k_b per pair (k_b in 3..19), as tests/test_gpu_pair_scale.py."""
    gen = torch.Generator().manual_seed(seed)
    vs = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    vt = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    pos = torch.randint(0, 16 * 512, (B,), generator=gen)
    sign = torch.where(torch.rand(B, generator=gen) < 0.5, -1.0, 1.0)
    vs.view(B, -1)[torch.arange(B), pos] = sign * torch.pow(2.0, torch.tensor([3.0 + (5 * b) % 17 for b in range(B)]))
    return vs, vt


@pytest.mark.parametrize("case", [("S1", 8, False), ("S1", -8, False), ("S2", -8, False), ("W1", 8, True)])
def test_saved_activation_backward_against_fp64(ahv, golden, oracle, case):
    """Both contraction forms of the saved-activation backward against fp64 autograd of the function the training
    forward evaluated (conv1's output takes the value it kept, h1 * pair_inv, and the ReLU mask of that value): 2e-5
    of each gradient's maximum for the fp32 form, 1e-3 for the tcgen05 form."""
    which, a, outliers = case
    B, N = 40, 3
    vs, vt = _outlier_batch(B, seed=99) if outliers else _volumes(B, seed=98)
    vs, vt = vs.to(DEV), vt.to(DEV)
    W1, W2, b2 = _to(_scaled(_golden_weights(golden), which, 2.0 ** a))
    R = _rotations(ahv, B, N, True, seed=41)
    tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
    gs = torch.randn(B, N, generator=torch.Generator().manual_seed(5)).to(DEV)
    scores, h1, pinv = ahv.ops.score_train(vs, tgt, R, W1, W2, b2)

    leaves = [t.double().requires_grad_(True) for t in (vs, tgt, W1, W2, b2)]
    v64, t64, w1, w2, bb = leaves
    kept_all = h1.reshape(B, N, 64, 32).double() * pinv.double()[:, None, None, None]
    ref_scores = []
    for b in range(B):
        rot = oracle.rotate_volume_torch(v64[b][None].expand(N, -1, -1, -1, -1), R[b].double())
        tri = torch.cat([rot.permute(0, 1, 4, 2, 3).reshape(N, 128, 8, 8), rot.permute(0, 1, 3, 2, 4).reshape(N, 128, 8, 8),
                         rot.reshape(N, 128, 8, 8)], dim=1)
        pre = F.conv2d(tri, w1.reshape(32, 384, 1, 1))
        kept = kept_all[b].permute(0, 2, 1).reshape(N, 32, 8, 8)
        mask = (kept > 0).double()
        hid = pre * mask + (kept - pre * mask).detach()      # value = what the forward kept, gradient = through its mask
        f = F.normalize(F.conv2d(hid, w2.reshape(32, 32, 1, 1), bb), p=2, dim=1).flatten(2)
        ref_scores.append((f * t64[b][None]).sum(dim=1).mean(dim=-1))
    ref_scores = torch.stack(ref_scores)
    assert float((ref_scores.detach().float() - scores).abs().max()) <= 1e-3        # the kept H1 reproduces the scores
    ref = torch.autograd.grad(ref_scores, leaves, grad_outputs=gs.double())
    for math_, tol in ((ahv.MATH_FP32, 2e-5), (ahv.MATH_TC, 1e-3)):
        got = ahv.ops.score_backward(vs, tgt, R, W1, W2, b2, gs, h1, pinv, math_)
        for name, g, r in zip(("vol_src", "tgt_feat", "W1", "W2", "b2"), got, ref):
            err = float((g.double() - r.reshape(g.shape)).abs().max()) / float(r.abs().max())
            assert err <= tol, (case, "tcgen05" if math_ == ahv.MATH_TC else "fp32", name, err)
