"""GPU (B200): parity of the CUDA path, called through the C ABI, against the
oracle and the committed golden vectors of the reference.

Tolerances (BASELINE.json north_star): scores within 1e-3 relative in the fp32
configuration (AHV_MATH_TC, fp16 = TF32-equivalent operands on tcgen05) and
1e-2 with bf16 volumes; AHV_MATH_FP32 is held to 2e-5.  Hypothesis indices are
bit-exact; top-1 must agree or be an equal-score tie within the tolerance."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = {"fp32": 2e-5, "tc": 1e-3}


def _dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _maths(ahv):
    return [("fp32", ahv.MATH_FP32), ("tc", ahv.MATH_TC)]


def _weights(golden, dev):
    w = golden["weights"]
    return [torch.from_numpy(w[k]).to(dev) for k in ("W1", "W2", "b2")]


def _relerr(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-6)))


def _top1_ok(scores_gpu, ref_scores, idx_gpu, tol):
    ref_best = ref_scores.max(1)
    picked = ref_scores[np.arange(ref_scores.shape[0]), idx_gpu]
    # identical index, or an equal-score tie within the score tolerance
    return np.all((idx_gpu == ref_scores.argmax(1)) | (np.abs(picked - ref_best) <= 2 * tol * np.abs(ref_best)))


def test_library_loaded_and_device_is_sm100(ahv):
    dev = _dev()
    assert torch.cuda.get_device_capability(dev)[0] == 10
    assert ahv._lib.lib().ahv_version() == 200


def test_so3_from_normals_bit_exact(ahv, golden, oracle):
    dev = _dev()
    normals = golden["shared_n3000_b3"]["normals"]
    R = ahv.ops.rotations_from_normals(torch.from_numpy(normals).to(dev)).cpu().numpy()
    assert np.array_equal(R, oracle.rotations_from_normals_np(normals))     # bit-exact vs IEEE restatement
    np.testing.assert_allclose(R, golden["shared_n3000_b3"]["R"], atol=3e-7, rtol=0)


def test_random_rotations_reproduces_cpu_generator(ahv, oracle):
    dev = _dev()
    torch.manual_seed(7)
    R = ahv.so3.random_rotations(1000, device=dev).cpu().numpy()
    torch.manual_seed(7)
    ref = oracle.rotations_from_normals_np(torch.randn(1000, 4).numpy())
    assert np.array_equal(R, ref)


def test_native_sampler_properties(ahv):
    dev = _dev()
    R = ahv.so3.sample_rotations(20000, seed=3, device=dev)
    eye = R @ R.transpose(1, 2)
    assert torch.allclose(eye, torch.eye(3, device=dev).expand_as(eye), atol=3e-6)
    assert torch.allclose(torch.linalg.det(R), torch.ones(20000, device=dev), atol=1e-5)
    # shardable: a slice generated on its own equals the slice of the whole
    part = ahv.so3.sample_rotations(500, seed=3, first_index=700, device=dev)
    assert torch.equal(part, R[700:1200])
    # Haar: mean rotation angle is pi/2 + 2/pi = 126.5 degrees
    ang = torch.rad2deg(torch.arccos(((R.diagonal(dim1=1, dim2=2).sum(-1) - 1) / 2).clamp(-1, 1)))
    assert abs(ang.mean().item() - 126.5) < 1.5


def test_so3_grid_bit_exact_and_shardable(ahv, oracle):
    dev = _dev()
    R = ahv.so3.grid_rotations(50000, device=dev)
    assert np.array_equal(R.cpu().numpy(), oracle.grid_rotations_c(50000))
    part = ahv.so3.grid_rotations(50000, first_index=43750, count=6250, device=dev)   # rank 7 of 8
    assert torch.equal(part, R[43750:])


def test_rotate_volume_vs_reference(ahv, golden):
    dev = _dev()
    p, g = golden["primitives"], golden["shared_n3000_b3"]
    vol = torch.from_numpy(g["vol_src"]).to(dev)
    out = ahv.ops.rotate_volume(vol[0], torch.from_numpy(p["R"]).to(dev)).cpu().numpy()
    np.testing.assert_allclose(out, p["rotated"], atol=2e-5, rtol=0)
    out = ahv.refcompat.rotate_volume(vol[1][None].expand(8, -1, -1, -1, -1), torch.from_numpy(p["special_R"]).to(dev))
    np.testing.assert_allclose(out.cpu().numpy(), p["special_rotated"], atol=2e-5, rtol=0)
    # per-rotation volumes (modules/model.py:137)
    Rb = torch.from_numpy(p["R"][:3]).to(dev)
    per = ahv.ops.rotate_volume(vol, Rb).cpu().numpy()
    for b in range(3):
        one = ahv.ops.rotate_volume(vol[b], Rb[b : b + 1]).cpu().numpy()
        assert np.array_equal(per[b], one[0])


def test_forward_3d2d_vs_reference(ahv, golden):
    dev = _dev()
    p = golden["primitives"]
    W1, W2, b2 = _weights(golden, dev)
    f = ahv.ops.forward_3d2d(torch.from_numpy(p["rotated"]).to(dev), W1, W2, b2).cpu().numpy()
    np.testing.assert_allclose(f, p["feat"], atol=2e-6, rtol=0)
    g = golden["shared_n3000_b3"]
    t = ahv.ops.forward_3d2d(torch.from_numpy(g["vol_tgt"]).to(dev), W1, W2, b2).cpu().numpy()
    np.testing.assert_allclose(t, g["tgt_feat"], atol=2e-6, rtol=0)


@pytest.mark.parametrize("mode", ["fp32", "tc"])
def test_scores_golden_shared_rotations(ahv, golden, mode):
    """Config 1 shape: N=3000 (config.yaml:10) on 3 pairs vs the reference's own output."""
    dev = _dev()
    g = golden["shared_n3000_b3"]
    v = ahv.HypothesisVerifier(*_weights(golden, dev), math=dict(_maths(ahv))[mode])
    r = v.score(torch.from_numpy(g["vol_src"]).to(dev), torch.from_numpy(g["vol_tgt"]).to(dev),
                torch.from_numpy(g["R"]).to(dev), k=1)
    s = r.scores.cpu().numpy()
    assert _relerr(s, g["scores"]) <= TOL[mode], _relerr(s, g["scores"])
    idx = r.topk_idx[:, 0].cpu().numpy()
    assert _top1_ok(s, g["scores"], idx, TOL[mode])
    if mode == "fp32":
        assert np.array_equal(idx, g["best_idx"])
    # selection is exactly torch.max of the GPU's own scores (first maximal index)
    assert np.array_equal(idx, s.argmax(1))
    np.testing.assert_array_equal(r.topk_val[:, 0].cpu().numpy(), s.max(1))
    np.testing.assert_array_equal(r.R_best[:, 0].cpu().numpy(), g["R"][idx])


@pytest.mark.parametrize("mode", ["fp32", "tc"])
def test_scores_per_pair_rotations_and_gt_hypothesis(ahv, golden, mode):
    """modules/model.py:53-56 and :137-143: R [B,N,3,3], including N=1."""
    dev = _dev()
    g, pp = golden["shared_n3000_b3"], golden["per_pair"]
    v = ahv.HypothesisVerifier(*_weights(golden, dev), math=dict(_maths(ahv))[mode])
    vs, vt = torch.from_numpy(g["vol_src"]).to(dev), torch.from_numpy(g["vol_tgt"]).to(dev)
    r = v.score(vs, vt, torch.from_numpy(pp["R"]).to(dev), k=1)
    assert _relerr(r.scores.cpu().numpy(), pp["scores"]) <= TOL[mode]
    r1 = v.score(vs, vt, torch.from_numpy(pp["R"][:, :1]).contiguous().to(dev), k=1)
    assert _relerr(r1.scores.cpu().numpy(), pp["scores_gt"]) <= TOL[mode]
    assert r1.topk_idx.cpu().numpy().tolist() == [[0], [0], [0]]


@pytest.mark.parametrize("mode", ["fp32", "tc"])
def test_special_rotations_exact_ties_and_zero_volume(ahv, golden, mode):
    dev = _dev()
    g, p, pp = golden["shared_n3000_b3"], golden["primitives"], golden["per_pair"]
    v = ahv.HypothesisVerifier(*_weights(golden, dev), math=dict(_maths(ahv))[mode])
    vs, vt = torch.from_numpy(g["vol_src"]).to(dev), torch.from_numpy(g["vol_tgt"]).to(dev)
    r = v.score(vs, vt, torch.from_numpy(p["special_R"]).to(dev), k=8)
    s = r.scores.cpu().numpy()
    assert _relerr(s, p["special_scores"]) <= TOL[mode]
    # duplicated hypotheses give bit-identical scores; the lower index comes first
    assert np.array_equal(s[:, 4], s[:, 5]) and np.array_equal(s[:, 0], s[:, 6])
    idx = r.topk_idx.cpu().numpy()
    for b in range(3):
        order = sorted(range(8), key=lambda i: (-float(s[b, i]), i))
        assert idx[b].tolist() == order
    # all-zero source volume: every hypothesis scores the same, argmax = index 0
    z = torch.zeros(1, 16, 8, 8, 8, device=dev)
    rz = v.score(z, vt[:1], torch.from_numpy(g["R"][:16]).to(dev), k=1)
    assert _relerr(rz.scores.cpu().numpy(), pp["zero_scores"]) <= TOL[mode]
    assert int(rz.topk_idx[0, 0]) == 0


@pytest.mark.parametrize("mode", ["fp32", "tc"])
@pytest.mark.parametrize("B,N", [(1, 1), (1, 7), (2, 33), (3, 512), (5, 1000)])
def test_scores_vs_c_oracle_ragged_sizes(ahv, golden, oracle, mode, B, N):
    dev = _dev()
    w = golden["weights"]
    rng = np.random.default_rng(100 * B + N)
    vs = rng.normal(-0.2, 1.2, (B, 16, 8, 8, 8)).astype(np.float32)
    vt = rng.normal(-0.2, 1.2, (B, 16, 8, 8, 8)).astype(np.float32)
    R = oracle.rotations_from_normals_np(rng.normal(size=(N, 4)).astype(np.float32))
    ref = oracle.score_c(vs, vt, R, w["W1"], w["W2"], w["b2"])
    v = ahv.HypothesisVerifier(*_weights(golden, dev), math=dict(_maths(ahv))[mode])
    k = min(4, N)
    r = v.score(torch.from_numpy(vs).to(dev), torch.from_numpy(vt).to(dev), torch.from_numpy(R).to(dev), k=k)
    s = r.scores.cpu().numpy()
    assert _relerr(s, ref) <= TOL[mode], _relerr(s, ref)
    val, idx = oracle.select_np(s, k)
    assert np.array_equal(r.topk_idx.cpu().numpy(), idx)
    assert _top1_ok(s, ref, r.topk_idx[:, 0].cpu().numpy(), TOL[mode])


def test_bf16_volumes_within_1e2(ahv, golden):
    """Config 3 arithmetic: bf16 source volumes."""
    dev = _dev()
    g = golden["shared_n3000_b3"]
    for name, math in _maths(ahv):
        v = ahv.HypothesisVerifier(*_weights(golden, dev), math=math)
        r = v.score(torch.from_numpy(g["vol_src"]).to(dev).bfloat16(), torch.from_numpy(g["vol_tgt"]).to(dev),
                    torch.from_numpy(g["R"][:1000]).to(dev), k=1)
        assert _relerr(r.scores.cpu().numpy(), g["scores"][:, :1000]) <= 1e-2


def test_full_size_properties(ahv, golden, oracle):
    """Config 2 size (B=32, N=50000): size-independent properties + a sampled
    oracle check (the oracle cannot score 1.6M hypothesis-pairs in seconds)."""
    dev = _dev()
    w = golden["weights"]
    B, N = 32, 50000
    gen = torch.Generator().manual_seed(0)
    vs = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    vt = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    torch.manual_seed(0)
    R = ahv.so3.random_rotations(N, device=dev)
    v = ahv.HypothesisVerifier(*_weights(golden, dev))
    r = v.score(vs.to(dev), vt.to(dev), R, k=32)
    s = r.scores
    assert s.shape == (B, N) and torch.isfinite(s).all()
    assert float(s.abs().max()) <= 1.0 + 1e-5                      # mean of cosines
    # top-k: sorted, consistent with the scores, equal to an independent selection
    assert torch.all(r.topk_val[:, :-1] >= r.topk_val[:, 1:])
    assert torch.equal(torch.gather(s, 1, r.topk_idx), r.topk_val)
    tv, ti = torch.topk(s, 32, dim=1)
    assert torch.equal(tv, r.topk_val)
    assert torch.equal(r.topk_idx[:, 0], s.argmax(1)) or torch.equal(r.topk_val[:, 0], s.max(1).values)
    # permutation equivariance over hypotheses and pairs
    perm = torch.randperm(N, generator=gen).to(dev)
    rp = v.score(vs.to(dev), vt.to(dev), R[perm].contiguous(), k=1)
    assert torch.equal(rp.scores, s[:, perm])
    r_rev = v.score(vs.flip(0).to(dev), vt.flip(0).to(dev), R, k=1)
    assert torch.equal(r_rev.scores, s.flip(0))
    # sampled oracle check: 4 pairs x 64 hypotheses spread over the set
    pick_b = [0, 9, 20, 31]
    pick_n = np.linspace(0, N - 1, 64).astype(np.int64)
    Rn = R[torch.from_numpy(pick_n).to(dev)].cpu().numpy()
    ref = oracle.score_c(vs[pick_b].numpy(), vt[pick_b].numpy(), Rn, w["W1"], w["W2"], w["b2"])
    got = s[pick_b][:, torch.from_numpy(pick_n).to(dev)].cpu().numpy()
    assert _relerr(got, ref) <= TOL["tc"]


def test_topk_merge_matches_unsharded(ahv, golden):
    dev = _dev()
    g = golden["shared_n3000_b3"]
    s = torch.from_numpy(g["scores"]).to(dev)
    full_v, full_i = ahv.ops.topk(s, 8)
    parts_v, parts_i = [], []
    for lo, hi in [ahv.dist.shard_bounds(3000, r, 4) for r in range(4)]:
        v, i = ahv.ops.topk(s[:, lo:hi].contiguous(), 8, idx_offset=lo)
        parts_v.append(v)
        parts_i.append(i)
    mv, mi = ahv.ops.topk_merge(torch.stack(parts_v), torch.stack(parts_i))
    assert torch.equal(mv, full_v) and torch.equal(mi, full_i)
    # ties across shards resolve to the lowest global index
    t = torch.zeros(1, 64, device=dev)
    v0, i0 = ahv.ops.topk(t[:, :32].contiguous(), 4, 0)
    v1, i1 = ahv.ops.topk(t[:, 32:].contiguous(), 4, 32)
    _, mi = ahv.ops.topk_merge(torch.stack([v1, v0]), torch.stack([i1, i0]))
    assert mi.tolist() == [[0, 1, 2, 3]]


def test_predict_host_round_trip(ahv, golden):
    g, w = golden["shared_n3000_b3"], golden["weights"]
    T = torch.from_numpy
    scores, val, idx, Rb = ahv.ops.predict_host(T(g["vol_src"]), T(g["vol_tgt"]), T(g["R"]), T(w["W1"]), T(w["W2"]),
                                                T(w["b2"]), k=1, return_scores=True)
    assert _relerr(scores.numpy(), g["scores"]) <= TOL["tc"]
    assert np.array_equal(idx[:, 0].numpy(), scores.numpy().argmax(1))
    assert np.array_equal(Rb[:, 0].numpy(), g["R"][idx[:, 0].numpy()])


def test_refcompat_idiom(ahv, golden):
    """A test_co3d.py:137-146 style call site keeps working."""
    dev = _dev()
    g, w = golden["shared_n3000_b3"], golden["weights"]

    class Head(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.feature_embedding_2d = torch.nn.Sequential(
                torch.nn.Conv2d(384, 32, 1, bias=False), torch.nn.ReLU(inplace=True), torch.nn.Conv2d(32, 32, 1))

    fa = Head().to(dev)
    fa.feature_embedding_2d[0].weight.data.copy_(torch.from_numpy(w["W1"]).reshape(32, 384, 1, 1))
    fa.feature_embedding_2d[2].weight.data.copy_(torch.from_numpy(w["W2"]).reshape(32, 32, 1, 1))
    fa.feature_embedding_2d[2].bias.data.copy_(torch.from_numpy(w["b2"]))
    vs, vt = torch.from_numpy(g["vol_src"]).to(dev), torch.from_numpy(g["vol_tgt"]).to(dev)
    R = torch.from_numpy(g["R"][:200]).to(dev)
    # unfused, reference-shaped (every intermediate materialised)
    rot = [ahv.refcompat.rotate_volume(v[None].expand(200, -1, -1, -1, -1), R) for v in vs]
    rot = torch.stack(rot).reshape(-1, 16, 8, 8, 8)
    f = ahv.refcompat.forward_3d2d(fa, rot).reshape(3, 200, -1, 64)
    t = ahv.refcompat.forward_3d2d(fa, vt)
    sim = (f * t[:, None]).sum(dim=2).mean(dim=-1)
    # like the reference's eval loop (no torch.no_grad() around it, test_co3d.py:126-152) this records a graph,
    # because the head's parameters require a gradient; under no_grad the same calls are single kernels
    assert sim.requires_grad
    with torch.no_grad():
        f0 = ahv.refcompat.forward_3d2d(fa, rot.detach())
    assert not f0.requires_grad and torch.allclose(f0.reshape(3, 200, -1, 64), f.detach(), atol=2e-6)
    sim = sim.detach()
    assert _relerr(sim.cpu().numpy(), g["scores"][:, :200]) <= 2e-5
    # fused
    s, idx, Rbest = ahv.refcompat.verify(fa, vs, vt, R)
    assert _relerr(s.cpu().numpy(), g["scores"][:, :200]) <= TOL["tc"]
    assert torch.equal(Rbest, R[idx])


@pytest.mark.parametrize("B,N", [(1, 1), (1, 3000), (3, 37), (32, 999)])
def test_fused_verify_argmax_equals_generic_path(ahv, golden, B, N):
    """ahv_verify with k=1 (arg-max and winner decode folded into the scoring kernel, 2 launches) must agree bit for
    bit with scores + separate top-k, including ties and the odd-tail tile."""
    dev = _dev()
    w = golden["weights"]
    gen = torch.Generator().manual_seed(B * 1000 + N)
    vs = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2).to(dev)
    vt = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2).to(dev)
    R = ahv.so3.sample_rotations(N, seed=N, device=dev)
    if N > 10:
        R[N // 2] = R[3]                       # exact tie: the lower index must win
    v = ahv.HypothesisVerifier(*_weights(golden, dev))
    fused = v.score(vs, vt, R, k=1, return_scores=True)
    fused_noscores = v.score(vs, vt, R, k=1, return_scores=False)
    tgt = v.target_features(vt)
    generic = v.score(vs, vt, R, k=1, return_scores=True, tgt_feat=tgt)
    assert torch.equal(fused.scores, generic.scores)
    assert torch.equal(fused.topk_idx, generic.topk_idx) and torch.equal(fused.topk_val, generic.topk_val)
    assert torch.equal(fused_noscores.topk_idx, generic.topk_idx) and torch.equal(fused_noscores.R_best, generic.R_best)
    assert torch.equal(fused.topk_idx[:, 0], fused.scores.argmax(1))
    assert torch.equal(fused.R_best[:, 0], R[fused.topk_idx[:, 0]])
    # per-pair rotations and idx_offset
    Rp = torch.stack([ahv.so3.sample_rotations(N, seed=b, device=dev) for b in range(B)])
    fp = v.score(vs, vt, Rp, k=1, return_scores=True, idx_offset=1000)
    gp = v.score(vs, vt, Rp, k=1, return_scores=True, tgt_feat=tgt, idx_offset=1000)
    assert torch.equal(fp.scores, gp.scores) and torch.equal(fp.topk_idx, gp.topk_idx)
    assert torch.equal(fp.topk_idx[:, 0] - 1000, fp.scores.argmax(1))
    assert torch.equal(fp.R_best[:, 0], Rp[torch.arange(B), fp.topk_idx[:, 0] - 1000])


def test_bf16_staged_gather_matches_oracle_on_rounded_volume(ahv, golden, oracle):
    """bf16 volumes take the 16-bit staged gather (x-pair lines).  Against the oracle evaluated on
    the SAME bf16-rounded volume the only error left is the fp16 conv operands: 1e-3 gate."""
    dev = _dev()
    g, w = golden["shared_n3000_b3"], golden["weights"]
    vs16 = torch.from_numpy(g["vol_src"]).bfloat16()
    R = g["R"][:700]
    ref = oracle.score_c(vs16.float().numpy(), g["vol_tgt"], R, w["W1"], w["W2"], w["b2"])
    for name, math in _maths(ahv):
        v = ahv.HypothesisVerifier(*_weights(golden, dev), math=math)
        r = v.score(vs16.to(dev), torch.from_numpy(g["vol_tgt"]).to(dev), torch.from_numpy(R).to(dev), k=1)
        assert _relerr(r.scores.cpu().numpy(), ref) <= TOL[name], (name, _relerr(r.scores.cpu().numpy(), ref))
        assert _top1_ok(r.scores.cpu().numpy(), ref, r.topk_idx[:, 0].cpu().numpy(), TOL[name])
    # per-pair rotations, odd counts and a volume with large magnitude (exercises the power-of-two scale)
    big = (vs16.float() * 3000.0).bfloat16()
    Rp = np.stack([R[:33], R[100:133], R[200:233]])
    refp = oracle.score_c(big.float().numpy(), g["vol_tgt"], Rp, w["W1"], w["W2"], w["b2"])
    v = ahv.HypothesisVerifier(*_weights(golden, dev))
    rp = v.score(big.to(dev), torch.from_numpy(g["vol_tgt"]).to(dev), torch.from_numpy(Rp).to(dev), k=1)
    assert _relerr(rp.scores.cpu().numpy(), refp) <= TOL["tc"]


def test_scale_invariance_of_tc_path(ahv, golden, oracle):
    """fp32 volumes with tiny / huge magnitudes: the per-pair power-of-two pre-scale keeps the fp16
    conv operands in range (without it 1e-4-sized volumes would go subnormal, 1e4-sized overflow)."""
    dev = _dev()
    g, w = golden["shared_n3000_b3"], golden["weights"]
    R = g["R"][:300]
    for factor in (1e-5, 1.0, 3e4):
        vs = (g["vol_src"] * factor).astype(np.float32)
        ref = oracle.score_c(vs, g["vol_tgt"], R, w["W1"], w["W2"], w["b2"])
        v = ahv.HypothesisVerifier(*_weights(golden, dev))
        r = v.score(torch.from_numpy(vs).to(dev), torch.from_numpy(g["vol_tgt"]).to(dev), torch.from_numpy(R).to(dev), k=1)
        assert _relerr(r.scores.cpu().numpy(), ref) <= TOL["tc"], factor


def test_f16_gather_fast_mode_within_fp32_gate(ahv, golden):
    """Opt-in AHV_MATH_TC_F16GATHER on fp32 volumes: fp16-staged volume + packed HFMA2 interpolation
    still meets the fp32 configuration's 1e-3 gate against the reference's own scores."""
    dev = _dev()
    g = golden["shared_n3000_b3"]
    v = ahv.HypothesisVerifier(*_weights(golden, dev), math=ahv.MATH_TC_F16GATHER)
    r = v.score(torch.from_numpy(g["vol_src"]).to(dev), torch.from_numpy(g["vol_tgt"]).to(dev),
                torch.from_numpy(g["R"]).to(dev), k=1, return_scores=True)
    s = r.scores.cpu().numpy()
    err = _relerr(s, g["scores"])
    assert err <= 1e-3, err
    assert _top1_ok(s, g["scores"], r.topk_idx[:, 0].cpu().numpy(), 1e-3)
    assert np.array_equal(r.topk_idx[:, 0].cpu().numpy(), s.argmax(1))


def test_non_finite_inputs_do_not_hang_or_fault(ahv, golden):
    """NaN / Inf in rotations or volumes must neither hang the pipeline nor read out of bounds:
    coordinates are clamped with NaN-dropping min/max and the scale ignores non-finite maxima."""
    dev = _dev()
    g = golden["shared_n3000_b3"]
    vs, vt = torch.from_numpy(g["vol_src"]).to(dev), torch.from_numpy(g["vol_tgt"]).to(dev)
    R = torch.from_numpy(g["R"][:65]).to(dev).clone()
    R[3] = float("nan")
    R[7, 0, 0] = float("inf")
    R[9] = 1e30
    for math in (ahv.MATH_TC, ahv.MATH_FP32, ahv.MATH_TC_F16GATHER):
        v = ahv.HypothesisVerifier(*_weights(golden, dev), math=math)
        r = v.score(vs, vt, R, k=1, return_scores=True)
        torch.cuda.synchronize()
        ok = torch.ones(65, dtype=torch.bool, device=dev)
        ok[[3, 7, 9]] = False
        assert torch.isfinite(r.scores[:, ok]).all()
        clean = v.score(vs, vt, R[ok].contiguous(), k=1, return_scores=True)
        assert torch.equal(r.scores[:, ok], clean.scores)          # bad hypotheses do not disturb the others
        assert ((r.topk_idx >= 0) & (r.topk_idx < 65)).all()
    bad = vs.clone()
    bad[1, 3, 2, 2, 2] = float("inf")
    r = ahv.HypothesisVerifier(*_weights(golden, dev)).score(bad, vt, R[:8].contiguous(), k=1, return_scores=True)
    torch.cuda.synchronize()
    assert torch.isfinite(r.scores[0]).all() and torch.isfinite(r.scores[2]).all()


@pytest.mark.parametrize("B,N", [(64, 3), (200, 1), (7, 2), (150, 5), (33, 17), (2, 149), (3, 296), (4097, 2), (5000, 3)])
@pytest.mark.parametrize("voldt", ["f32", "bf16"])
def test_many_pairs_tiny_hypothesis_sets(ahv, golden, B, N, voldt):
    """Every CTA range crosses pair boundaries and most tiles are odd tails: stresses volume
    re-staging, the per-pair arg-max flush and the two-hypothesis tiling.  The fp32 CUDA-core
    kernel (independent code path) is the on-device reference.  Past 4096 pairs the fused call, the
    k > 1 chain and caller-computed target features must still agree bit for bit."""
    dev = _dev()
    gen = torch.Generator().manual_seed(B * 131 + N)
    vs = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2).to(dev)
    vt = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2).to(dev)
    if voldt == "bf16":
        vs = vs.bfloat16()
    for per_pair in (False, True):
        R = ahv.so3.sample_rotations(B * N if per_pair else N, seed=N + B, device=dev)
        R = R.reshape(B, N, 3, 3).contiguous() if per_pair else R
        ref = ahv.HypothesisVerifier(*_weights(golden, dev), math=ahv.MATH_FP32).score(vs, vt, R, k=1, return_scores=True)
        got = ahv.HypothesisVerifier(*_weights(golden, dev), math=ahv.MATH_TC).score(vs, vt, R, k=1, return_scores=True)
        tol = 1e-3 if voldt == "f32" else 2e-3      # bf16 volumes: fp16 interpolation adds ~1e-4 on top
        rel = ((got.scores - ref.scores).abs() / ref.scores.abs().clamp_min(1e-6)).max().item()
        assert rel <= tol, (per_pair, rel)
        assert torch.equal(got.topk_idx[:, 0], got.scores.argmax(1))
        assert torch.equal(got.topk_val[:, 0], got.scores.max(1).values)
        noscore = ahv.HypothesisVerifier(*_weights(golden, dev)).score(vs, vt, R, k=1, return_scores=False)
        assert torch.equal(noscore.topk_idx, got.topk_idx) and torch.equal(noscore.R_best, got.R_best)
        k2 = min(3, N)
        multi = ahv.HypothesisVerifier(*_weights(golden, dev)).score(vs, vt, R, k=k2, return_scores=True)
        assert torch.equal(multi.scores, got.scores)
        tv, _ = torch.topk(got.scores, k2, dim=1)
        assert torch.equal(multi.topk_val, tv)
        v = ahv.HypothesisVerifier(*_weights(golden, dev))
        given = v.score(vs, vt, R, k=1, return_scores=True, tgt_feat=v.target_features(vt))
        assert torch.equal(given.scores, got.scores) and torch.equal(given.topk_idx, got.topk_idx)


def test_graphed_verifier_matches_eager(ahv, golden):
    dev = _dev()
    g = golden["shared_n3000_b3"]
    T = lambda a: torch.from_numpy(a).to(dev)
    v = ahv.HypothesisVerifier(*_weights(golden, dev))
    eager = v.score(T(g["vol_src"]), T(g["vol_tgt"]), T(g["R"]), k=1, return_scores=False)
    gv = ahv.GraphedVerifier(v, 3, 3000, k=1, device=dev)
    out = gv(T(g["vol_src"]), T(g["vol_tgt"]), T(g["R"]))
    torch.cuda.synchronize()
    assert torch.equal(out.topk_idx, eager.topk_idx) and torch.equal(out.topk_val, eager.topk_val)
    assert torch.equal(out.R_best, eager.R_best)
    # replay with new inputs
    out2 = gv(T(g["vol_src"]).flip(0), T(g["vol_tgt"]).flip(0))
    torch.cuda.synchronize()
    assert torch.equal(out2.topk_idx, eager.topk_idx.flip(0))


def test_predict_host_topk_and_per_pair(ahv, golden):
    g, w = golden["shared_n3000_b3"], golden["weights"]
    T = torch.from_numpy
    Rp = T(np.stack([g["R"][:100], g["R"][100:200], g["R"][200:300]]))
    scores, val, idx, Rb = ahv.ops.predict_host(T(g["vol_src"]), T(g["vol_tgt"]), Rp, T(w["W1"]), T(w["W2"]), T(w["b2"]),
                                                k=5, return_scores=True)
    tv, ti = torch.topk(scores, 5, dim=1)
    assert torch.equal(val, tv)
    assert torch.equal(Rb, torch.gather(Rp, 1, idx[..., None, None].expand(-1, -1, 3, 3)))
    assert _relerr(scores[0].numpy(), g["scores"][0, :100]) <= 1e-3


def test_bitwise_determinism_and_soak(ahv, golden):
    """The pipeline has no data-dependent scheduling in its arithmetic: repeated runs are bit-identical.
    Then a soak over random (pairs, hypotheses, volume dtype, rotation layout) shapes vs the fp32 path."""
    dev = _dev()
    gen = torch.Generator().manual_seed(77)
    B, N = 32, 20000
    vs = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2).to(dev)
    vt = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2).to(dev)
    R = ahv.so3.sample_rotations(N, seed=5, device=dev)
    v = ahv.HypothesisVerifier(*_weights(golden, dev))
    first = v.score(vs, vt, R, k=1, return_scores=True)
    for _ in range(5):
        again = v.score(vs, vt, R, k=1, return_scores=True)
        assert torch.equal(again.scores, first.scores) and torch.equal(again.topk_idx, first.topk_idx)
    b16 = v.score(vs.bfloat16(), vt, R, k=1, return_scores=True)
    assert torch.equal(v.score(vs.bfloat16(), vt, R, k=1, return_scores=True).scores, b16.scores)
    rng = np.random.default_rng(2024)
    ref_v = ahv.HypothesisVerifier(*_weights(golden, dev), math=ahv.MATH_FP32)
    for it in range(24):
        b, n = int(rng.integers(1, 33)), int(rng.integers(1, 700))
        per_pair = bool(rng.integers(0, 2))
        src = vs[:b].bfloat16() if rng.integers(0, 2) else vs[:b]
        Rr = ahv.so3.sample_rotations(b * n if per_pair else n, seed=it, device=dev)
        Rr = Rr.reshape(b, n, 3, 3).contiguous() if per_pair else Rr
        got = v.score(src, vt[:b], Rr, k=1, return_scores=True)
        ref = ref_v.score(src, vt[:b], Rr, k=1, return_scores=True)
        rel = ((got.scores - ref.scores).abs() / ref.scores.abs().clamp_min(1e-6)).max().item()
        assert rel <= 2e-3, (it, b, n, per_pair, src.dtype, rel)
        assert torch.equal(got.topk_idx[:, 0], got.scores.argmax(1))


def test_concurrent_streams_and_threads(ahv, golden):
    """SURVEY.md §8b: the library is re-entrant and stream-ordered.  Four Python threads, each on its own CUDA
    stream with its own inputs, run fused verification steps concurrently (programmatically dependent
    launches, last-CTA winner decode and per-call workspaces all interleave on the device); every result must
    equal the serial one bit for bit."""
    import threading

    dev = _dev()
    w = _weights(golden, dev)
    gen = torch.Generator().manual_seed(77)
    jobs = []
    for i, (B, N) in enumerate([(1, 3000), (5, 777), (32, 500), (2, 4001)]):
        vs = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2).to(dev)
        vt = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2).to(dev)
        R = ahv.so3.sample_rotations(N, seed=100 + i, device=dev)
        jobs.append((vs, vt, R))
    serial = [ahv.HypothesisVerifier(*w).score(vs, vt, R, k=1, return_scores=True) for vs, vt, R in jobs]
    torch.cuda.synchronize()
    results, errors = [None] * len(jobs), []

    def worker(i):
        try:
            st = torch.cuda.Stream(device=dev)
            st.wait_stream(torch.cuda.current_stream(dev))
            v = ahv.HypothesisVerifier(*w)
            with torch.cuda.stream(st):
                for _ in range(10):
                    r = v.score(*jobs[i], k=1, return_scores=True)
                    r2 = v.score(*jobs[i], k=1, return_scores=False)
            st.synchronize()
            results[i] = (r, r2)
        except Exception as e:  # pragma: no cover
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(len(jobs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for (r, r2), ref in zip(results, serial):
        assert torch.equal(r.scores, ref.scores)
        assert torch.equal(r.topk_idx, ref.topk_idx) and torch.equal(r.topk_val, ref.topk_val)
        assert torch.equal(r2.topk_idx, ref.topk_idx) and torch.equal(r2.R_best, ref.R_best)


def test_misaligned_slices_are_accepted(ahv, golden):
    """A hypothesis shard R[lo:hi] starts at lo*36 bytes, which is 16-byte aligned only for lo % 4 == 0; the
    binding must hand the C ABI an aligned copy instead of failing with AHV_EINVAL (8-GPU shards of 50 000)."""
    dev = _dev()
    g = golden["shared_n3000_b3"]
    T = lambda a: torch.from_numpy(a).to(dev)
    v = ahv.HypothesisVerifier(*_weights(golden, dev))
    R = T(g["R"])
    full = v.score(T(g["vol_src"]), T(g["vol_tgt"]), R, k=1, return_scores=True)
    for lo in (1, 2, 3, 6250 % 3000):
        part = v.score(T(g["vol_src"]), T(g["vol_tgt"]), R[lo:], k=1, return_scores=True, idx_offset=lo)
        assert torch.equal(part.scores, full.scores[:, lo:])
        vs_view = T(g["vol_src"])[1:]                      # volumes: 32 KB per pair, always aligned; still a view
        assert v.score(vs_view, T(g["vol_tgt"])[1:], R[lo:], k=1).topk_idx.shape == (2, 1)


def test_peer_exchange_protocol_on_one_gpu(ahv, golden):
    """The NVLink exchange of the sharded step, exercised on ONE GPU: two "ranks" live in this process, each with its
    own exchange buffer (plain device pointers - no IPC needed inside one process), its own stream and its own shard of
    the rotation set.  Rank 0's kernel publishes its winners into both buffers and spins on rank 1's flag while rank 1's
    kernel runs beside it on the other stream (only the LAST CTA of a scoring kernel waits, so the two grids need not
    be co-resident).  Covers the fused k = 1 exchange, the top-k exchange kernel, B and k changing from step to step on
    one buffer, an empty shard and the sequence counter - the multi-process version (CUDA IPC, NCCL bootstrap, graph
    replay, host entry) is tests/test_gpu_dist.py, which needs two devices."""
    import ctypes
    from types import SimpleNamespace

    dev = _dev()
    lib = ahv._lib.lib()
    g = golden["shared_n3000_b3"]
    W1, W2, b2 = _weights(golden, dev)
    v = ahv.HypothesisVerifier(W1, W2, b2)
    vs, vt, R = (torch.from_numpy(g[k]).to(dev) for k in ("vol_src", "vol_tgt", "R"))
    cap_pairs, cap_k, world = 4, 8, 2
    bufs = []
    for _ in range(world):
        p = ctypes.c_void_p()
        ahv._lib.check(lib.ahv_peer_alloc(cap_pairs, cap_k, ctypes.byref(p)), "ahv_peer_alloc")
        bufs.append(p.value)
    peers = [SimpleNamespace(rank=r, world=world, ptrs=bufs, max_pairs=cap_pairs, max_k=cap_k) for r in range(world)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(world)]
    try:
        steps = 0
        for B, N, k in ((3, 3000, 1), (1, 1000, 1), (3, 2000, 8), (2, 501, 5), (3, 1, 1), (3, 3, 4), (3, 3000, 1)):
            want = v.score(vs[:B], vt[:B], R[:N], k=k, return_scores=False)
            torch.cuda.synchronize()
            out = [None] * world
            for r in range(world):
                lo, hi = ahv.dist.shard_bounds(N, r, world)
                streams[r].wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(streams[r]):
                    out[r] = ahv.ops.verify_sharded(vs[:B], vt[:B], R[lo:hi].contiguous(), W1, W2, b2, lo, peers[r], k=k)
            for s in streams:
                s.synchronize()
            steps += 1
            kk = min(k, N)
            for r in range(world):
                val, idx, Rb = out[r]
                if bool(torch.isnan(val).any()):      # a 20 s spin that timed out: the two streams were serialised
                    pytest.skip("the two ranks' kernels were not scheduled concurrently on this device")
                assert torch.equal(idx[:, :kk], want.topk_idx) and torch.equal(val[:, :kk], want.topk_val), (B, N, k, r)
                assert torch.equal(Rb[:, :kk], want.R_best), (B, N, k, r)
                assert bool((idx[:, kk:] == -1).all())
            seq, err = ctypes.c_uint32(), ctypes.c_uint32()
            for r in range(world):
                ahv._lib.check(lib.ahv_peer_status(bufs[r], ctypes.byref(seq), ctypes.byref(err)), "ahv_peer_status")
                assert seq.value == steps and err.value == 0
        # a call larger than the capacity the buffers were allocated with is rejected before anything is launched
        with pytest.raises(ValueError):
            ahv.ops.verify_sharded(vs, vt, R[:100].contiguous(), W1, W2, b2, 0, peers[0], k=cap_k + 1)
        mp, mk = ctypes.c_int(), ctypes.c_int()
        ahv._lib.check(lib.ahv_peer_capacity(bufs[0], ctypes.byref(mp), ctypes.byref(mk)), "ahv_peer_capacity")
        assert (mp.value, mk.value) == (cap_pairs, cap_k)
    finally:
        torch.cuda.synchronize()
        for p in bufs:
            lib.ahv_peer_free(p)


def test_plain_c_host_matches_the_python_binding(ahv, golden, tmp_path):
    """examples/predict_host.c - a host with no Python and no PyTorch in it - gets the same selection through
    ahv_predict_host_ex as the ctypes binding does."""
    import os
    import subprocess

    from test_abi import _compile_c_example

    exe = _compile_c_example(tmp_path)
    g, w = golden["shared_n3000_b3"], golden["weights"]
    B, N, k = 3, 3000, 4
    base = ahv.ops.base_coords().numpy()
    inp, outp = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    with open(inp, "wb") as f:
        f.write(np.array([B, N, k], dtype=np.int32).tobytes())
        for a in (g["vol_src"], g["vol_tgt"], g["R"], w["W1"], w["W2"], w["b2"], base):
            f.write(np.ascontiguousarray(a, dtype=np.float32).tobytes())
    run = subprocess.run([exe, inp, outp], capture_output=True, text=True, timeout=120)
    assert run.returncode == 0, run.stderr
    raw = open(outp, "rb").read()
    idx = np.frombuffer(raw, dtype=np.int64, count=B * k).reshape(B, k)
    val = np.frombuffer(raw, dtype=np.float32, count=B * k, offset=B * k * 8).reshape(B, k)
    Rb = np.frombuffer(raw, dtype=np.float32, count=B * k * 9, offset=B * k * 12).reshape(B, k, 3, 3)
    T = torch.from_numpy
    _, pv, pi, pR = ahv.ops.predict_host(T(g["vol_src"]), T(g["vol_tgt"]), T(g["R"]), T(w["W1"]), T(w["W2"]), T(w["b2"]), k=k,
                                         device=_dev())
    assert np.array_equal(idx, pi.numpy()) and np.array_equal(val, pv.numpy()) and np.array_equal(Rb, pR.numpy())
    assert np.array_equal(Rb, g["R"][idx])


def test_topk_merge_keeps_64_bit_indices(ahv):
    """Shard lists whose global indices exceed 2^32 (a set sharded with large idx_offsets): the merge orders by
    (score, low 32 index bits) and reports the full 64-bit index of the winning entries."""
    dev = _dev()
    parts, B, k = 4, 3, 5
    gen = torch.Generator().manual_seed(0)
    vals = torch.rand(parts, B, k, generator=gen).sort(dim=-1, descending=True).values
    base = (1 << 33) + 12345
    idx = base + torch.arange(parts * B * k, dtype=torch.int64).reshape(parts, B, k) * 7
    idx[1, 0, 3:] = -1                                                    # empty slots are ignored
    vals[1, 0, 3:] = float("-inf")
    out_v, out_i = ahv.ops.topk_merge(vals.to(dev), idx.to(dev))
    flat_v = vals.permute(1, 0, 2).reshape(B, -1)
    flat_i = idx.permute(1, 0, 2).reshape(B, -1)
    order = torch.argsort(flat_v, dim=1, descending=True, stable=True)[:, :k]
    assert torch.equal(out_v.cpu(), torch.gather(flat_v, 1, order))
    assert torch.equal(out_i.cpu(), torch.gather(flat_i, 1, order))
    assert int(out_i.min()) > (1 << 32)
