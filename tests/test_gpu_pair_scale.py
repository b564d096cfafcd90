"""GPU (B200): the per-pair power-of-two scale of the tensor-core paths, and the dynamic range of their fp16 operands.

The tensor-core kernels do not score the raw volume: stage_pair_volume (csrc/ahv_tc_common.cuh) multiplies each pair's
volume by its own power of two, chosen from max|V| and the largest L1 row norm of the normalised W1, so that the fp16
operands cannot overflow.  The gather warps hand 1/scale to the epilogue through an 8-entry ring indexed by pair; the epilogue undoes
the scale before it adds b2, and the training forward writes it out for the tcgen05 backward.  The gather runs several
tiles ahead of the epilogue, and with N = 1 or 2 every tile starts a new pair.

Batches here give every pair one outlier voxel of +-2^k_b over an order-one bulk: the outlier sets the pair's scale,
the bulk keeps the features comparable to b2 (so a scale applied to the wrong pair moves the scores by per cent rather
than cancelling in F.normalize), and k_b has period 17 - coprime to 8 - so pairs b, b+-1 and b+8 (the same ring slot)
all get different scales.  References: the AHV_MATH_FP32 kernel (an independent code path with no scaling) for every
pair, fp64 `oracle.score_torch` for a sample that includes the pairs on CTA boundaries.

The second half bounds the outlier-to-bulk ratio each mode handles (the numbers quoted in include/ahv_b200.h)."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)

# score gates, relative: fp32 volumes under the tensor-core modes / the fp32 kernel; bf16 volumes against the scores of
# the bf16-rounded volume (fp16 interpolation adds ~1e-4 on top of the tensor-core operands)
GATE_TC, GATE_FP32, GATE_BF16 = 1e-3, 2e-5, 2e-3


def _weights(golden):
    return [torch.from_numpy(golden["weights"][k]).to(DEV) for k in ("W1", "W2", "b2")]


def _modes(ahv):
    return {"fp32": ahv.MATH_FP32, "tc": ahv.MATH_TC, "f16gather": ahv.MATH_TC_F16GATHER}


def _gate(mode, voldt):
    return GATE_FP32 if mode == "fp32" else (GATE_TC if voldt == "f32" else GATE_BF16)


def _relerr(a, b):
    return float(((a.double() - b.double()).abs() / b.double().abs().clamp_min(1e-6)).max())


def _exponents(B):
    """k_b in [3, 19] with period 17: k_{b+1} - k_b = 5 and k_{b+8} - k_b = 6 (mod 17) are never 0."""
    return [3 + (5 * b) % 17 for b in range(B)]


def _mixed_batch(B, seed):
    """Order-one bulk, one outlier voxel of +-2^k_b in pair b (exact in bf16 too, so both volume types share max|V|)."""
    gen = torch.Generator().manual_seed(seed)
    vs = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    vt = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    pos = torch.randint(0, 16 * 512, (B,), generator=gen)
    sign = torch.where(torch.rand(B, generator=gen) < 0.5, -1.0, 1.0)
    vs.view(B, -1)[torch.arange(B), pos] = sign * torch.pow(2.0, torch.tensor(_exponents(B), dtype=torch.float32))
    return vs, vt


def _rotations(ahv, B, N, per_pair, seed):
    if per_pair:
        return ahv.so3.sample_rotations(B * N, seed=seed, device=DEV).reshape(B, N, 3, 3).contiguous()
    return ahv.so3.sample_rotations(N, seed=seed, device=DEV)


def _boundary_pairs(B, N):
    """Pairs whose items straddle the contiguous per-CTA item ranges of the scoring kernel (one CTA per SM, at most
    one per two-hypothesis tile), plus the first and the last pair."""
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    total = B * N
    grid = min((total + 1) // 2, sms)
    cuts = [total * i // grid for i in range(1, grid)]
    pairs = {0, B - 1}
    for c in cuts:
        pairs.update({(c - 1) // N, c // N})
    return sorted(pairs)


def _sample(pairs, n):
    idx = np.unique(np.linspace(0, len(pairs) - 1, n).round().astype(np.int64))
    return [pairs[i] for i in idx]


def _fp64_scores(oracle, golden, vs, vt, R, pairs):
    """oracle.score_torch in float64 on the CPU for `pairs` (bf16 volumes: on the bf16-rounded values)."""
    W1, W2, b2 = (torch.from_numpy(golden["weights"][k]).double() for k in ("W1", "W2", "b2"))
    sel = torch.tensor(pairs)
    Rp = R.cpu()[sel] if R.dim() == 4 else R.cpu()
    return oracle.score_torch(vs.cpu()[sel].double(), vt.cpu()[sel].double(), Rp.double(), W1, W2, b2).double()


@pytest.mark.parametrize("B,N", [(3, 1), (4, 2), (6, 7), (151, 1), (75, 2), (333, 3), (160, 7), (1201, 2), (2400, 1)])
@pytest.mark.parametrize("per_pair", [False, True])
@pytest.mark.parametrize("voldt", ["f32", "bf16"])
def test_mixed_scales_every_mode(ahv, golden, oracle, B, N, per_pair, voldt):
    """Neighbouring pairs with different scales, from a few items up to 2400 pairs of one hypothesis (each CTA crosses
    about 16 pairs, so the ring wraps): every pair against the fp32 kernel, a sample against fp64, bit-exact
    invariance of a pair's scores under batch composition, and the selections against the scores."""
    vs, vt = _mixed_batch(B, seed=1000 * B + N)
    if voldt == "bf16":
        vs = vs.bfloat16()
    R = _rotations(ahv, B, N, per_pair, seed=B + 7 * N)
    vs_d, vt_d = vs.to(DEV), vt.to(DEV)
    W = _weights(golden)
    boundary = _boundary_pairs(B, N)
    sample = _sample(boundary, 10)
    ref64 = _fp64_scores(oracle, golden, vs, vt, R, sample)
    exact = ahv.HypothesisVerifier(*W, math=ahv.MATH_FP32).score(vs_d, vt_d, R, k=1).scores
    shift = 3 if B > 3 else 1                                              # not a multiple of the ring's 8 slots
    for mode, math in _modes(ahv).items():
        v = ahv.HypothesisVerifier(*W, math=math)
        gate = _gate(mode, voldt)
        r = v.score(vs_d, vt_d, R, k=1, return_scores=True)
        s = r.scores
        assert torch.isfinite(s).all(), mode
        if mode != "fp32":
            err = _relerr(s, exact)
            assert err <= gate, (mode, "vs MATH_FP32", err)
        err = _relerr(s.cpu()[sample], ref64)
        assert err <= gate, (mode, "vs fp64", sample, err)
        # the fused arg-max, with and without the score matrix, and the k = 4 selection agree with the scores
        assert torch.equal(r.topk_idx[:, 0], s.argmax(1)) and torch.equal(r.topk_val[:, 0], s.max(1).values), mode
        noscore = v.score(vs_d, vt_d, R, k=1, return_scores=False)
        assert torch.equal(noscore.topk_idx, r.topk_idx) and torch.equal(noscore.topk_val, r.topk_val), mode
        assert torch.equal(noscore.R_best, r.R_best), mode
        k4 = v.score(vs_d, vt_d, R, k=4, return_scores=True)
        assert torch.equal(k4.scores, s), mode
        val, idx = oracle.select_np(s.cpu().numpy(), 4)
        assert np.array_equal(k4.topk_idx.cpu().numpy(), idx) and np.array_equal(k4.topk_val.cpu().numpy(), val), mode
        # batch composition: the scale and every operation are per item, so a pair's scores are bit-identical when the
        # batch is rolled (its neighbours and its ring slot change) and when it is scored alone
        Rr = R.roll(shift, 0) if per_pair else R
        rolled = v.score(vs_d.roll(shift, 0), vt_d.roll(shift, 0), Rr, k=1, return_scores=True)
        assert torch.equal(rolled.scores.roll(-shift, 0), s), mode
        assert torch.equal(rolled.topk_idx.roll(-shift, 0), r.topk_idx), mode
        for b in sample:
            alone = v.score(vs_d[b : b + 1], vt_d[b : b + 1], R[b : b + 1] if per_pair else R, k=1, return_scores=True)
            assert torch.equal(alone.scores[0], s[b]), (mode, b)


def _w1_normaliser(W1):
    """2^e1, e1 = floor(log2 of W1's largest row L1 norm) - 2: the tensor-core kernels pack W1 * 2^-e1, whose largest
    row L1 norm lies in [4, 8)."""
    return 2.0 ** (math.floor(math.log2(float(W1.double().abs().sum(1).max()))) - 2)


def _scale_bound(W1):
    """stage_pair_volume's target for max|V| * scale: 32768 / (largest L1 row norm of the normalised W1, in [4, 8)),
    capped at 8192 - so in (4096, 8192] whatever W1's magnitude."""
    l1max = float(W1.double().abs().sum(1).max()) / _w1_normaliser(W1)
    assert 4.0 <= l1max < 8.0
    return min(8192.0, 32768.0 / l1max)


@pytest.mark.parametrize("w1_exp", [0, -12, 12])
@pytest.mark.parametrize("B,N,per_pair", [(300, 1, False), (97, 2, True), (40, 3, True), (160, 7, False)])
def test_training_forward_keeps_each_pairs_scale_at_every_weight_magnitude(ahv, golden, B, N, per_pair, w1_exp):
    """ahv_score_train's pair_inv is 2^e1 / scale with the exact power of two of the scale rule for that pair's own
    max|V| (2^e1: W1's normaliser), for the golden W1 and for W1 scaled by 1.37 * 2^-12 and 1.37 * 2^12 (the rule, and
    so max|V| * scale, does not depend on W1's magnitude); pair_inv, the kept conv1 activations and the scores do not
    depend on the rest of the batch, and the scores are those of the inference kernel."""
    W1, W2, b2 = _weights(golden)
    if w1_exp:
        W1 = W1 * (1.37 * 2.0 ** w1_exp)
    vs, vt = (t.to(DEV) for t in _mixed_batch(B, seed=7 * B + N))
    R = _rotations(ahv, B, N, per_pair, seed=3 * B + N)
    tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
    scores, h1, pinv = ahv.ops.score_train(vs, tgt, R, W1, W2, b2)
    mant, _ = torch.frexp(pinv)
    assert bool((mant == 0.5).all()), pinv[mant != 0.5]
    bound = _scale_bound(W1)
    ratio = vs.abs().flatten(1).max(1).values.double() * _w1_normaliser(W1) / pinv.double()   # max|V| * scale, exact
    assert bool(((ratio > bound / 2) & (ratio <= bound)).all()), (bound, ratio[(ratio <= bound / 2) | (ratio > bound)])
    # neighbouring pairs (and pairs 8 apart) really do differ in scale, or this test could not see a mix-up
    assert bool((pinv[1:] != pinv[:-1]).all()) and bool((pinv[8:] != pinv[:-8]).all())
    infer = ahv.ops.score(vs, tgt, R, W1, W2, b2, k=0, math=ahv.MATH_TC)[0]
    assert torch.equal(scores, infer)
    h1 = h1.reshape(B, N, 64, 32)
    for b in _sample(_boundary_pairs(B, N), 12):
        s1, h1b, pb = ahv.ops.score_train(vs[b : b + 1], tgt[b : b + 1], R[b : b + 1] if per_pair else R, W1, W2, b2)
        assert torch.equal(pb[0], pinv[b]) and torch.equal(s1[0], scores[b]), b
        assert torch.equal(h1b.reshape(N, 64, 32), h1[b]), b


@pytest.mark.parametrize("per_pair", [False, True])
def test_saved_activation_backward_on_mixed_scales(ahv, golden, oracle, per_pair):
    """Both contraction forms of the saved-activation backward against fp64 autograd of the function the training
    forward evaluated (conv1's output takes the value it kept, h1 * 1/scale, and the ReLU mask of that value), on many
    pairs of few hypotheses whose scales all differ from their neighbours'.  fp32 contractions: 2e-5 of each gradient's
    maximum; tcgen05 contractions (fp16 operands): 1e-3."""
    B, N = 40, 3
    W1, W2, b2 = _weights(golden)
    vs, vt = (t.to(DEV) for t in _mixed_batch(B, seed=99 + per_pair))
    R = _rotations(ahv, B, N, per_pair, seed=41 + per_pair)
    tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
    gs = torch.randn(B, N, generator=torch.Generator().manual_seed(5)).to(DEV)
    scores, h1, pinv = ahv.ops.score_train(vs, tgt, R, W1, W2, b2)

    leaves = [t.double().requires_grad_(True) for t in (vs, tgt, W1, W2, b2)]
    v64, t64, w1, w2, bb = leaves
    kept_all = h1.reshape(B, N, 64, 32).double() * pinv.double()[:, None, None, None]
    ref_scores = []
    for b in range(B):
        Rb = (R[b] if per_pair else R).double()
        rot = oracle.rotate_volume_torch(v64[b][None].expand(N, -1, -1, -1, -1), Rb)
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
    for math, tol in ((ahv.MATH_FP32, 2e-5), (ahv.MATH_TC, 1e-3)):
        got = ahv.ops.score_backward(vs, tgt, R, W1, W2, b2, gs, h1, pinv, math)
        for name, a, r in zip(("vol_src", "tgt_feat", "W1", "W2", "b2"), got, ref):
            err = float((a.double() - r.reshape(a.shape)).abs().max()) / float(r.abs().max())
            assert err <= tol, (per_pair, "tcgen05" if math == ahv.MATH_TC else "fp32", name, err)


# ---- dynamic range of the fp16 operands --------------------------------------------------------------------------
# Outlier-to-bulk ratio r = the largest |outlier| over the bulk's standard deviation.  Each pair of a standard-normal
# bulk carries two outliers, +r/3 and -r (r = 3e4: the 1e4 and -3e4 of a trained checkpoint's heavy tail), one of
# them on a corner voxel.  With the golden head the pair scale maps r into (2^11.6, 2^12.6], so the bulk nears fp16's
# smallest normal, 2^-14, around r = 3e7.  scripts/dynamic_range.py sweeps r up to 1e9 on the same inputs; the largest
# r at which each mode met its gate there is MAX_RATIO (include/ahv_b200.h quotes it), and every mode is tested up to it.
RATIOS = [1e2, 1e3, 1e4, 3e4, 1e5, 3e5, 1e6, 1e7, 3e7, 1e8]
MAX_RATIO = {"fp32": 3e5, "tc": 1e8, "f16gather": 1e8, "bf16": 1e8}


def _outlier_volumes(B, r, seed):
    gen = torch.Generator().manual_seed(seed)
    vs, vt = torch.randn(B, 16, 8, 8, 8, generator=gen), torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    pos = torch.randperm(16 * 512, generator=gen)[: 2 * B].reshape(B, 2)
    pos[0, 1] = 0
    flat = vs.view(B, -1)
    flat[torch.arange(B), pos[:, 0]] = r / 3
    flat[torch.arange(B), pos[:, 1]] = -r
    return vs, vt


@pytest.mark.parametrize("ratio", RATIOS)
def test_dynamic_range_of_the_fp16_operands(ahv, golden, oracle, ratio):
    """fp32 volumes under AHV_MATH_TC (fp32 gather, fp16 conv operands) and AHV_MATH_TC_F16GATHER (fp16-staged volume,
    HFMA2 interpolation) against fp64 at 1e-3; bf16 volumes (always fp16-staged) at 2e-3 against fp64 on the
    bf16-rounded volume and at 1e-2 against the unrounded one; AHV_MATH_FP32 at 2e-5 as far as fp32 arithmetic holds it
    (the reference's own fp32 ATen path drifts past 2e-5 from about r = 1e6 as well)."""
    B, N = 4, 600
    vs, vt = _outlier_volumes(B, ratio, seed=5)
    R = ahv.so3.sample_rotations(N, seed=17, device=DEV)
    pairs = list(range(B))
    ref = _fp64_scores(oracle, golden, vs, vt, R, pairs)
    ref16 = _fp64_scores(oracle, golden, vs.bfloat16(), vt, R, pairs)
    W = _weights(golden)
    vt_d = vt.to(DEV)
    for mode, math, gate in (("tc", ahv.MATH_TC, GATE_TC), ("f16gather", ahv.MATH_TC_F16GATHER, GATE_TC),
                             ("fp32", ahv.MATH_FP32, GATE_FP32)):
        if ratio <= MAX_RATIO[mode]:
            r = ahv.HypothesisVerifier(*W, math=math).score(vs.to(DEV), vt_d, R, k=1, return_scores=True)
            err = _relerr(r.scores.cpu(), ref)
            assert err <= gate, (mode, "f32", ratio, err)
    if ratio <= MAX_RATIO["bf16"]:
        r = ahv.HypothesisVerifier(*W, math=ahv.MATH_TC).score(vs.bfloat16().to(DEV), vt_d, R, k=1, return_scores=True)
        s = r.scores.cpu()
        assert _relerr(s, ref16) <= GATE_BF16, ("bf16 vs rounded", ratio, _relerr(s, ref16))
        assert _relerr(s, ref) <= 1e-2, ("bf16 vs unrounded", ratio, _relerr(s, ref))
