"""GPU (B200): parity with the oracle at the STATED size of every BASELINE.json config (SURVEY.md §8d).

The oracle (`oracle.score_c`, the C restatement pinned to the reference-generated goldens) scores about
3-6e4 hypothesis-pairs per second on the host, so whole 50 000-hypothesis pairs are checked where the config
is defined by them (configs 2, 3, 4) and evenly spread samples elsewhere.  Tolerances are BASELINE.json's:
scores <= 1e-3 relative with fp32 volumes, <= 1e-2 with bf16 volumes; indices bit-exact; top-1 identical or
an equal-score tie within the score tolerance."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _weights(golden):
    w = golden["weights"]
    return w["W1"], w["W2"], w["b2"]


def _verifier(ahv, golden, math=None):
    W1, W2, b2 = (torch.from_numpy(a).to(DEV) for a in _weights(golden))
    return ahv.HypothesisVerifier(W1, W2, b2, math=math)


def _volumes(B, seed):
    gen = torch.Generator().manual_seed(seed)
    return (torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.12 - 0.18, torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.12 - 0.18)


def _relerr(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-6)))


def _top1_or_tie(ref_scores, idx_gpu, tol):
    """idx_gpu [P]: identical to the oracle's arg-max, or the oracle scores it within the tolerance of its best."""
    best = ref_scores.max(1)
    picked = ref_scores[np.arange(ref_scores.shape[0]), idx_gpu]
    return bool(np.all((idx_gpu == ref_scores.argmax(1)) | (np.abs(picked - best) <= 2 * tol * np.abs(best))))


def _topk_or_tie(ref_scores, idx_gpu, tol):
    """idx_gpu [P,k] (distinct): every selected hypothesis is scored by the oracle no lower than the oracle's own
    k-th best minus the tolerance, and every oracle score above the k-th best plus the tolerance is selected."""
    k = idx_gpu.shape[1]
    for p in range(ref_scores.shape[0]):
        s = ref_scores[p]
        kth = np.sort(s)[-k]
        band = 2 * tol * abs(kth)
        if len(set(idx_gpu[p].tolist())) != k or np.any(s[idx_gpu[p]] < kth - band):
            return False
        must = np.nonzero(s > kth + band)[0]
        if not set(must.tolist()) <= set(idx_gpu[p].tolist()):
            return False
    return True


def test_config2_full_pairs_vs_oracle(ahv, golden, oracle):
    """configs[1]: CO3D, 32 pairs x the full 50 000-hypothesis set, fp32 volumes, one GPU.  Three WHOLE pairs
    (150 000 hypothesis-pairs) against the oracle, the fused arg-max against the oracle's on those pairs; the same for
    the opt-in AHV_MATH_TC_F16GATHER mode (fp16-staged volume), which is held to the same gate."""
    B, N = 32, 50000
    vs, vt = _volumes(B, 0)
    torch.manual_seed(0)
    R = ahv.so3.random_rotations(N, device=DEV)
    pairs = [0, 13, 31]
    ref = oracle.score_c(vs[pairs].numpy(), vt[pairs].numpy(), R.cpu().numpy(), *_weights(golden))
    for math in (ahv.MATH_TC, ahv.MATH_TC_F16GATHER):
        v = _verifier(ahv, golden, math)
        r = v.score(vs.to(DEV), vt.to(DEV), R, k=1, return_scores=True)
        fused = v.score(vs.to(DEV), vt.to(DEV), R, k=1, return_scores=False)    # the 2-launch step bench.py times
        assert torch.equal(fused.topk_idx, r.topk_idx) and torch.equal(fused.topk_val, r.topk_val)
        assert torch.equal(fused.R_best[:, 0], R[fused.topk_idx[:, 0]])
        got = r.scores[pairs].cpu().numpy()
        assert _relerr(got, ref) <= 1e-3, (math, _relerr(got, ref))
        assert _top1_or_tie(ref, fused.topk_idx[pairs, 0].cpu().numpy(), 1e-3), math


def test_config3_bf16_128_pairs_vs_oracle(ahv, golden, oracle):
    """configs[2]: Objaverse, 128 pairs, bf16 volumes, 50 000 hypotheses (sharded over 8 GPUs in the config; the
    per-GPU arithmetic is the same at any shard size - tests/test_gpu_dist.py checks the sharding).  One whole
    pair + 2 048 evenly spread hypotheses of three more pairs against the oracle on the same bf16 inputs."""
    B, N = 128, 50000
    vs, vt = _volumes(B, 1)
    vs_bf = vs.bfloat16()
    R = ahv.so3.sample_rotations(N, seed=11, device=DEV)
    v = _verifier(ahv, golden)
    r = v.score(vs_bf.to(DEV), vt.to(DEV), R, k=1, return_scores=True)
    Rn = R.cpu().numpy()
    full = oracle.score_c(vs_bf[5:6].float().numpy(), vt[5:6].numpy(), Rn, *_weights(golden))
    assert _relerr(r.scores[5:6].cpu().numpy(), full) <= 1e-2
    assert _top1_or_tie(full, r.topk_idx[5:6, 0].cpu().numpy(), 1e-2)
    pairs, pick = [0, 63, 127], np.linspace(0, N - 1, 2048).astype(np.int64)
    ref = oracle.score_c(vs_bf[pairs].float().numpy(), vt[pairs].numpy(), Rn[pick], *_weights(golden))
    got = r.scores[pairs][:, torch.from_numpy(pick).to(DEV)].cpu().numpy()
    assert _relerr(got, ref) <= 1e-2
    assert torch.equal(r.topk_idx[:, 0], r.scores.argmax(1)) or torch.equal(r.topk_val[:, 0], r.scores.max(1).values)


def test_config4_grid_topk_refine_vs_oracle(ahv, golden, oracle):
    """configs[3]: LINEMOD, dense SO(3) grid (50 000 rotations) + top-k refinement.  The reference has neither;
    parity = the reference scorer (oracle) on the same rotation sets: the grid pass's top-32 against
    `topk` of the oracle's scores (ties within tolerance), the refinement pass's scores and winner against the
    oracle on the identical candidate set."""
    B, N, k, m = 2, 50000, 32, 64
    vs, vt = _volumes(B, 2)
    R = ahv.so3.grid_rotations(N, device=DEV)
    assert np.array_equal(R.cpu().numpy(), oracle.grid_rotations_c(N))          # bit-exact hypothesis set
    v = _verifier(ahv, golden)
    R_ref, val, first, cand = v.refine(vs.to(DEV), vt.to(DEV), R, k=k, m=m, max_angle_deg=4.0, seed=5)
    ref1 = oracle.score_c(vs.numpy(), vt.numpy(), R.cpu().numpy(), *_weights(golden))
    assert _topk_or_tie(ref1, first.topk_idx.cpu().numpy(), 1e-3)
    picked = np.take_along_axis(ref1, first.topk_idx.cpu().numpy(), 1)
    assert _relerr(first.topk_val.cpu().numpy(), picked) <= 1e-3
    assert torch.equal(first.R_best, R[first.topk_idx])
    # candidate set: generator against its restatement, then the scorer on exactly the GPU's candidates
    assert cand.shape == (B, k * m, 3, 3)
    want = oracle.perturb_rotations_np(first.R_best.cpu().numpy(), m, 4.0, seed=5).reshape(B, k * m, 3, 3)
    np.testing.assert_allclose(cand.cpu().numpy(), want, atol=2e-6, rtol=0)
    assert torch.equal(cand.reshape(B, k, m, 3, 3)[:, :, 0], first.R_best)      # index 0 = the centre itself
    ref2 = oracle.score_c(vs.numpy(), vt.numpy(), cand.cpu().numpy(), *_weights(golden))     # per-pair sets
    second = v.score(vs.to(DEV), vt.to(DEV), cand, k=1, return_scores=True)
    assert _relerr(second.scores.cpu().numpy(), ref2) <= 1e-3
    assert _top1_or_tie(ref2, second.topk_idx[:, 0].cpu().numpy(), 1e-3)
    assert torch.equal(second.R_best[:, 0], R_ref) and torch.equal(second.topk_val[:, 0], val)
    assert torch.all(val >= first.topk_val[:, 0])                               # the centre is a candidate


def test_config5_sweep_corners_vs_oracle(ahv, golden, oracle):
    """configs[4]: the sweep's corners.  N = 1e6 hypotheses x 1 pair: 4 096 evenly spread hypotheses and the
    winner against the oracle; 256 pairs x 1 000 hypotheses: eight whole pairs."""
    v = _verifier(ahv, golden)
    vs, vt = _volumes(1, 3)
    N = 1_000_000
    R = ahv.so3.sample_rotations(N, seed=2, device=DEV)
    r = v.score(vs.to(DEV), vt.to(DEV), R, k=4, return_scores=True)
    pick = np.unique(np.concatenate([np.linspace(0, N - 1, 4096).astype(np.int64), r.topk_idx[0].cpu().numpy()]))
    ref = oracle.score_c(vs.numpy(), vt.numpy(), R[torch.from_numpy(pick).to(DEV)].cpu().numpy(), *_weights(golden))
    assert _relerr(r.scores[:, torch.from_numpy(pick).to(DEV)].cpu().numpy(), ref) <= 1e-3
    tv, ti = torch.topk(r.scores, 4, dim=1)
    assert torch.equal(tv, r.topk_val)
    assert torch.equal(r.topk_idx[:, 0], r.scores.argmax(1)) or torch.equal(r.topk_val[:, 0], r.scores.max(1).values)
    fused = v.score(vs.to(DEV), vt.to(DEV), R, k=1, return_scores=False)
    assert torch.equal(fused.topk_idx[:, 0], r.topk_idx[:, 0]) and torch.equal(fused.topk_val[:, 0], r.topk_val[:, 0])
    B, N = 256, 1000
    vs, vt = _volumes(B, 4)
    R = ahv.so3.sample_rotations(N, seed=9, device=DEV)
    r = v.score(vs.to(DEV), vt.to(DEV), R, k=1, return_scores=True)
    pairs = [0, 37, 74, 111, 148, 185, 222, 255]
    ref = oracle.score_c(vs[pairs].numpy(), vt[pairs].numpy(), R.cpu().numpy(), *_weights(golden))
    assert _relerr(r.scores[pairs].cpu().numpy(), ref) <= 1e-3
    assert _top1_or_tie(ref, r.topk_idx[pairs, 0].cpu().numpy(), 1e-3)
    rb = v.score(vs.bfloat16().to(DEV), vt.to(DEV), R, k=1, return_scores=True)
    refb = oracle.score_c(vs.bfloat16()[pairs].float().numpy(), vt[pairs].numpy(), R.cpu().numpy(), *_weights(golden))
    assert _relerr(rb.scores[pairs].cpu().numpy(), refb) <= 1e-2


@pytest.mark.parametrize("outlier", [1e4, -3e4, 1e-4])
def test_outlier_voxel_in_an_order_one_volume(ahv, golden, oracle, outlier):
    """The tensor-core path pre-scales each pair's volume by a power of two chosen from max|V| so that fp16 conv
    operands cannot overflow.  A single outlier voxel (as a trained checkpoint's heavy tail may produce) shrinks
    that scale for the whole volume; the scores must stay within the fp32 gate."""
    B, N = 3, 1000
    vs, vt = _volumes(B, 5)
    vs[0, 3, 2, 5, 1] = outlier
    vs[1, 15, 7, 7, 7] = -outlier
    vs[2, 0, 0, 0, 0] = outlier
    R = ahv.so3.sample_rotations(N, seed=4, device=DEV)
    ref = oracle.score_c(vs.numpy(), vt.numpy(), R.cpu().numpy(), *_weights(golden))
    r = _verifier(ahv, golden).score(vs.to(DEV), vt.to(DEV), R, k=1, return_scores=True)
    assert _relerr(r.scores.cpu().numpy(), ref) <= 1e-3
    assert _top1_or_tie(ref, r.topk_idx[:, 0].cpu().numpy(), 1e-3)
    r32 = _verifier(ahv, golden, ahv.MATH_FP32).score(vs.to(DEV), vt.to(DEV), R, k=1, return_scores=True)
    assert _relerr(r32.scores.cpu().numpy(), ref) <= 2e-5


def test_generators_vs_restatements(ahv, oracle):
    """The native Philox sampler and the refinement-set generator against their numpy restatements (integer part
    exact; transcendental functions to rounding)."""
    R = ahv.so3.sample_rotations(4096, seed=3, first_index=1000, device=DEV).cpu().numpy()
    np.testing.assert_allclose(R, oracle.sample_rotations_np(4096, 3, 1000), atol=2e-6, rtol=0)
    c = torch.from_numpy(oracle.sample_rotations_np(6, 1)).to(DEV)
    P = ahv.so3.perturb_rotations(c, 33, 7.5, seed=8)
    np.testing.assert_allclose(P.cpu().numpy(), oracle.perturb_rotations_np(c.cpu().numpy(), 33, 7.5, 8), atol=2e-6, rtol=0)
    assert torch.equal(P[:, 0], c)
    rel = P @ c[:, None].transpose(-1, -2)
    ang = torch.rad2deg(torch.arccos(((rel.diagonal(dim1=-2, dim2=-1).sum(-1) - 1) / 2).clamp(-1, 1)))
    assert float(ang.max()) <= 7.5 + 1e-2


def test_graphed_refiner_equals_eager(ahv, golden):
    """The two-pass selection is one C call with nothing on the host in between: it captures into a CUDA graph."""
    B, N, k, m = 3, 5000, 16, 32
    vs, vt = _volumes(B, 7)
    R = ahv.so3.grid_rotations(N, device=DEV)
    v = _verifier(ahv, golden)
    gr = ahv.GraphedRefiner(v, B, N, k=k, m=m, max_angle_deg=3.0, seed=9, device=DEV)
    for flip in (False, True):
        a, b = (vs.flip(0), vt.flip(0)) if flip else (vs, vt)
        Rb, val = gr(a.to(DEV), b.to(DEV), R)
        R_ref, val_ref, first, cand = v.refine(a.to(DEV), b.to(DEV), R, k=k, m=m, max_angle_deg=3.0, seed=9)
        assert torch.equal(Rb, R_ref) and torch.equal(val, val_ref)
        assert torch.equal(gr.first.topk_idx, first.topk_idx) and torch.equal(gr.candidates, cand)


def test_round2_entry_edge_cases(ahv, golden):
    """Degenerate sizes of the round-2 entries: refinement with k = m = 1 is plain arg-max selection, a zero cone keeps
    every candidate on its centre, InfoNCE with no positive gives the reference's +inf loss with finite gradients, and
    empty batches are no-ops."""
    B, N = 2, 777
    vs, vt = _volumes(B, 11)
    R = ahv.so3.sample_rotations(N, seed=5, device=DEV)
    v = _verifier(ahv, golden)
    Rb, val, first, cand = v.refine(vs.to(DEV), vt.to(DEV), R, k=1, m=1, max_angle_deg=5.0)
    plain = v.score(vs.to(DEV), vt.to(DEV), R, k=1, return_scores=False)
    assert torch.equal(Rb, plain.R_best[:, 0]) and torch.equal(val, plain.topk_val[:, 0]) and torch.equal(cand[:, 0], Rb)
    P = ahv.so3.perturb_rotations(R[:5], 9, 0.0, seed=1)
    assert torch.allclose(P, R[:5, None].expand(-1, 9, -1, -1), atol=1e-6) and torch.equal(P[:, 0], R[:5])
    # InfoNCE: no hypothesis within the threshold of the ground truth (modules/model.py:58-61 gives -log(0) = inf)
    s = torch.rand(B, N, device=DEV)
    gt = ahv.so3.sample_rotations(B, seed=99, device=DEV)
    loss, grad = ahv.ops.infonce(s, R, gt, acc_thr_deg=1e-3)
    assert bool(torch.isinf(loss).all()) and bool(torch.isfinite(grad).all())
    e = torch.exp(s / 0.1)
    assert torch.allclose(grad, e / 0.1 / e.sum(-1, keepdim=True), rtol=1e-4)
    # empty batches
    assert ahv.ops.resblock3d(torch.zeros(0, 32, 8, 8, 8, device=DEV), torch.zeros(16, 32, 3, 3, 3, device=DEV),
                              torch.zeros(16, 16, 3, 3, 3, device=DEV), torch.zeros(16, 32, 1, 1, 1, device=DEV)).shape == (0, 16, 8, 8, 8)
    assert ahv.so3.perturb_rotations(R[:0], 4, 3.0).shape == (0, 4, 3, 3)
    with pytest.raises(ValueError):
        v.refine(vs.to(DEV), vt.to(DEV), R, k=8, m=0)
