"""GPU: the gradient-ascent kernel (ahv_gradient_ascent / HypothesisVerifier.ascend) and the one-call chain
(ahv_refine_gradient / refine_by_gradient / GraphedRefiner(method="gradient")) against the fp32 scorer and the torch-op
reference HypothesisVerifier.refine_gradient, on the synthetic known-rotation task of test_gpu_rotation_grad.py."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _hat(u):
    z = torch.zeros_like(u[..., 0])
    return torch.stack((z, -u[..., 2], u[..., 1], u[..., 2], z, -u[..., 0], -u[..., 1], u[..., 0], z), -1).reshape(*u.shape[:-1], 3, 3)


def _expm(w):
    """exp([w]x) in fp64 (Rodrigues)."""
    th = w.norm(dim=-1, keepdim=True)[..., None]
    K = _hat(w / w.norm(dim=-1, keepdim=True))
    return torch.eye(3, dtype=w.dtype) + torch.sin(th) * K + (1 - torch.cos(th)) * (K @ K)


def _task(ahv, B):
    """Target = source rotated by a hidden R_gt, so the score peaks there whatever the head weights are."""
    import bench

    W1, W2, b2, vs, _, _ = bench.synthetic_inputs(torch, B, 16)
    v = ahv.HypothesisVerifier(W1.to(DEV), W2.to(DEV), b2.to(DEV))
    vs = vs.to(DEV)
    R_gt = ahv.so3.sample_rotations(B, seed=123, device=DEV)
    return v, vs, ahv.ops.rotate_volume(vs, R_gt), R_gt


def _around(R_gt, deg, seed):
    """[B,k,3,3] rotations deg[j] degrees off R_gt about random axes."""
    B, k = R_gt.shape[0], len(deg)
    axis = torch.randn(B, k, 3, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
    ang = torch.deg2rad(torch.tensor(deg, dtype=torch.float64))[None, :, None]
    return (_expm(ang * axis / axis.norm(dim=-1, keepdim=True)) @ R_gt.cpu().double()[:, None]).float().to(DEV).contiguous()


def _geodesic_deg(Ra, Rb):
    c = ((Ra.double() * Rb.double()).sum((-1, -2)).clamp(-1, 3) - 1) / 2
    return torch.rad2deg(torch.arccos(c.clamp(-1, 1)))


def _fp32_scores(ahv, v, vs, tgt, R):
    return ahv.ops.score(vs, tgt, R.contiguous(), v.W1, v.W2, v.b2, k=0, math=ahv.MATH_FP32)[0]


def _assert_rotations(R):
    R = R.double()
    eye = torch.eye(3, dtype=torch.float64, device=R.device)
    assert float((R @ R.transpose(-1, -2) - eye).abs().max()) <= 1e-5
    assert bool((torch.linalg.det(R) > 0).all())


@pytest.mark.parametrize("B,K", [(1, 1), (7, 1), (4, 37), (149, 1), (12, 25)])
def test_scores_are_the_fp32_scorers_and_bf16_is_exact(ahv, B, K):
    """B*K = 1, 7, 148, 149, 300: CTA ranges that span pairs, and items that wrap past the SM count."""
    v, vs, vt, R_gt = _task(ahv, B)
    R0 = _around(R_gt, [1.0 + 3.0 * (j % 7) for j in range(K)], seed=B * 100 + K)
    tgt = v.target_features(vt)
    R_out, s_out = ahv.ops.gradient_ascent(vs, tgt, R0, v.W1, v.W2, v.b2, steps=4, step_deg=1.0)
    assert torch.equal(s_out, _fp32_scores(ahv, v, vs, tgt, R_out))
    assert bool((s_out >= _fp32_scores(ahv, v, vs, tgt, R0)).all())
    _assert_rotations(R_out)
    vb = vs.bfloat16()
    Rb, sb = ahv.ops.gradient_ascent(vb, tgt, R0, v.W1, v.W2, v.b2, steps=4, step_deg=1.0)
    Rf, sf = ahv.ops.gradient_ascent(vb.float(), tgt, R0, v.W1, v.W2, v.b2, steps=4, step_deg=1.0)
    assert torch.equal(Rb, Rf) and torch.equal(sb, sf)
    assert torch.equal(sb, _fp32_scores(ahv, v, vb, tgt, Rb))


def test_zero_steps_return_the_start(ahv):
    v, vs, vt, R_gt = _task(ahv, 4)
    R0 = _around(R_gt, [2.0, 30.0, 90.0], seed=3)
    tgt = v.target_features(vt)
    R_out, s_out = ahv.ops.gradient_ascent(vs, tgt, R0, v.W1, v.W2, v.b2, steps=0)
    assert torch.equal(R_out, R0)
    assert torch.equal(s_out, _fp32_scores(ahv, v, vs, tgt, R0))


def _near_ties(ahv, v, vs, vt, R, steps, step_deg=1.0):
    """Restates refine_gradient's loop to find the candidates where some trial scored within 1e-6 of its current score:
    there the kernel and the torch ops may round the accept decision differently."""
    from importlib import import_module

    hat = import_module("3dahv_b200.verify")._hat
    tgt = v.target_features(vt)
    B, k = R.shape[:2]
    s = _fp32_scores(ahv, v, vs, tgt, R)
    theta = torch.full((B, k), math.radians(step_deg), device=DEV)
    eye = torch.eye(3, device=DEV)
    tie = torch.zeros(B, k, dtype=torch.bool, device=DEV)
    for _ in range(steps):
        G = ahv.ops.score_grad_R(vs, tgt, R, v.W1, v.W2, v.b2, torch.ones(B, k, device=DEV))
        M = G @ R.transpose(-1, -2)
        w = torch.stack((M[..., 2, 1] - M[..., 1, 2], M[..., 0, 2] - M[..., 2, 0], M[..., 1, 0] - M[..., 0, 1]), -1)
        K = hat(w / w.norm(dim=-1, keepdim=True).clamp_min(1e-30))
        Rt = (eye + torch.sin(theta)[..., None, None] * K + (1.0 - torch.cos(theta))[..., None, None] * (K @ K)) @ R
        Rt = 1.5 * Rt - 0.5 * Rt @ Rt.transpose(-1, -2) @ Rt
        st = _fp32_scores(ahv, v, vs, tgt, Rt)
        tie |= (st - s).abs() < 1e-6
        acc = st > s
        R = torch.where(acc[..., None, None], Rt, R).contiguous()
        s = torch.where(acc, st, s)
        theta = torch.where(acc, theta * 1.2, theta * 0.5)
    return tie


@pytest.mark.parametrize("steps", [1, 2, 3])
def test_same_algorithm_as_the_reference(ahv, steps):
    B = 8
    v, vs, vt, R_gt = _task(ahv, B)
    R0 = _around(R_gt, [1.0, 3.0, 9.0, 20.0, 60.0], seed=11)
    _, _, R_ref, s_ref = v.refine_gradient(vs, vt, R0, steps=steps)
    _, _, R_all, s_all = v.ascend(vs, vt, R0, steps=steps)
    tie = _near_ties(ahv, v, vs, vt, R0, steps)
    assert int(tie.sum()) <= B * 5 // 4, int(tie.sum())                 # the exemption stays an exception
    err = (R_all - R_ref).abs().amax((-1, -2))
    assert bool((err[~tie] <= 1e-5).all()), (err, tie)


def test_converges_on_the_synthetic_task(ahv):
    """From 3 degrees off, 20 steps: mean error < 0.05 degrees, max < 0.1 (the torch-op reference: 0.009 and 0.039)."""
    B = 8
    v, vs, vt, R_gt = _task(ahv, B)
    axis = torch.randn(B, 3, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    R0 = (_expm(math.radians(3.0) * axis / axis.norm(dim=-1, keepdim=True)) @ R_gt.cpu().double()).float().to(DEV)
    R_best, s_best, R_all, s_all = v.ascend(vs, vt, R0, steps=20, step_deg=1.0)
    assert R_best.shape == (B, 3, 3) and s_best.shape == (B,) and R_all.shape == (B, 1, 3, 3) and s_all.shape == (B, 1)
    err = _geodesic_deg(R_best, R_gt)
    assert float(err.mean()) < 0.05 and float(err.max()) < 0.1, err.tolist()
    _assert_rotations(R_all)


def test_scores_never_drop_and_the_best_is_the_first_arg_max(ahv):
    B = 4
    v, vs, vt, R_gt = _task(ahv, B)
    R0 = _around(R_gt, [1.0, 4.0, 9.0, 20.0, 60.0], seed=6)
    s0 = _fp32_scores(ahv, v, vs, v.target_features(vt), R0)
    R_best, s_best, R_all, s_all = v.ascend(vs, vt, R0, steps=20)
    assert bool((s_all >= s0).all())
    _assert_rotations(R_all)
    idx = torch.argmax(s_all, dim=1)
    rows = torch.arange(B, device=DEV)
    assert torch.equal(s_best, s_all[rows, idx]) and torch.equal(R_best, R_all[rows, idx])


def test_deterministic_and_replays_in_a_cuda_graph(ahv):
    B = 6
    v, vs, vt, R_gt = _task(ahv, B)
    R0 = _around(R_gt, [2.0, 7.0, 25.0], seed=9)
    eager = v.ascend(vs, vt, R0, steps=12)
    again = v.ascend(vs, vt, R0, steps=12)
    for a, b in zip(eager, again):
        assert torch.equal(a, b)
    static_R = R0.clone()
    stream = torch.cuda.Stream(device=DEV)
    stream.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(stream):
        v.ascend(vs, vt, static_R, steps=12)                # warm-up outside capture
    torch.cuda.current_stream(DEV).wait_stream(stream)
    torch.cuda.synchronize(DEV)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = v.ascend(vs, vt, static_R, steps=12)
    static_R.zero_()
    static_R.copy_(R0)
    graph.replay()
    torch.cuda.synchronize(DEV)
    for a, b in zip(out, eager):
        assert torch.equal(a, b)


@pytest.mark.parametrize("math_mode", ["MATH_TC", "MATH_FP32"])
def test_refine_by_gradient_chains_the_grid_pass_and_the_ascent(ahv, math_mode):
    B, N, k = 4, 5000, 4
    v, vs, vt, R_gt = _task(ahv, B)
    v.math = getattr(ahv, math_mode)
    grid = ahv.so3.grid_rotations(N, device=DEV)
    R_best, s_best, first, R_all, s_all = v.refine_by_gradient(vs, vt, grid, k=k, steps=10)
    ref = v.score(vs, vt, grid, k=k, return_scores=False)
    assert torch.equal(first.topk_val, ref.topk_val) and torch.equal(first.topk_idx, ref.topk_idx)
    assert torch.equal(first.R_best, ref.R_best)
    _, _, R_asc, s_asc = v.ascend(vs, vt, ref.R_best, steps=10)
    assert torch.equal(R_all, R_asc) and torch.equal(s_all, s_asc)
    idx = torch.argmax(s_all, dim=1)
    rows = torch.arange(B, device=DEV)
    assert torch.equal(s_best, s_all[rows, idx]) and torch.equal(R_best, R_all[rows, idx])
    assert float(_geodesic_deg(R_best, R_gt).max()) < float(_geodesic_deg(first.R_best[:, 0], R_gt).max()) + 1e-6


def test_graphed_refiner_gradient_method_replays_the_eager_chain(ahv):
    B, N, k = 3, 3000, 4
    v, vs, vt, R_gt = _task(ahv, B)
    grid = ahv.so3.grid_rotations(N, device=DEV)
    eager = v.refine_by_gradient(vs, vt, grid, k=k, steps=8, step_deg=1.5)
    g = ahv.GraphedRefiner(v, B, N, k=k, device=DEV, method="gradient", steps=8, step_deg=1.5)
    R_best, s_best = g(vs, vt, grid)
    torch.cuda.synchronize(DEV)
    assert torch.equal(R_best, eager[0]) and torch.equal(s_best, eager[1])
    assert torch.equal(g.first.topk_idx, eager[2].topk_idx)
    assert torch.equal(g.R_all, eager[3]) and torch.equal(g.score_all, eager[4])
    with pytest.raises(ValueError):
        ahv.GraphedRefiner(v, B, N, k=k, device=DEV, method="newton")
