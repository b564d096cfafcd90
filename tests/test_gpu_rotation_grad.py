"""GPU: gradients with respect to the rotation matrices - ahv_rotate_volume_grad_R, the rotation phase of
ahv_score_backward_ex, R.grad through the autograd functions and refcompat, and HypothesisVerifier.refine_gradient.
References: fp64 CPU autograd through the oracle's restatement of utils.py:113-131 and modules/modules.py:112-124 (the
reference's own ATen calls) with R as a leaf."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)


def _axis_rotation(axis, deg):
    """Rotation by `deg` about `axis` (Rodrigues, fp64, entries of 90/180-degree rotations rounded to exact 0/+-1)."""
    u = torch.tensor(axis, dtype=torch.float64)
    u = u / u.norm()
    K = torch.tensor([[0.0, -u[2], u[1]], [u[2], 0.0, -u[0]], [-u[1], u[0], 0.0]], dtype=torch.float64)
    a = math.radians(deg)
    R = torch.eye(3, dtype=torch.float64) + math.sin(a) * K + (1 - math.cos(a)) * (K @ K)
    if deg % 90 == 0:
        R = R.round()
    return R.float()


def _lattice_rotations():
    """I and 90/180 degrees about each axis: every sample lands on a voxel centre (exact integer coordinates)."""
    Rs = [torch.eye(3)]
    for axis in ((1, 0, 0), (0, 1, 0), (0, 0, 1)):
        Rs += [_axis_rotation(axis, 90), _axis_rotation(axis, 180)]
    return torch.stack(Rs)


def _outside_rotations():
    """Rotations that send samples outside [-1, 8): 45 degrees about z, 30 about a face diagonal, and a few more.  (Not
    about a body diagonal such as (1,1,1): that axis runs through voxel centres, whose samples then sit within rounding
    of an integer coordinate, where the resampling has a kink and fp32 and fp64 may take different sides of it.)"""
    return torch.stack([_axis_rotation((0, 0, 1), 45), _axis_rotation((1, 1, 0), 30), _axis_rotation((1, 0, 0), 45),
                        _axis_rotation((0, 1, 1), 60), _axis_rotation((1, -2, 0.5), 135)])


def _unnormalised_coords(R, dtype):
    theta = torch.cat([R.to(dtype), torch.zeros(R.shape[0], 3, 1, dtype=dtype)], -1)
    g = torch.nn.functional.affine_grid(theta, [R.shape[0], 16, 8, 8, 8], align_corners=False)
    return ((g + 1) * 8 - 1) / 2


def _rotate_ref(oracle, vol, R, gout, per_rotation):
    """fp64 autograd: d <rotate_volume(vol, R), gout> / dR."""
    Rl = R.double().requires_grad_(True)
    v = vol.double() if per_rotation else vol.double()[None].expand(R.shape[0], -1, -1, -1, -1)
    (oracle.rotate_volume_torch(v, Rl) * gout.double()).sum().backward()
    return Rl.grad


def _scores_ref(oracle, vs, vt, R, W1, W2, b2, gs):
    """fp64 autograd of sum(gs * scores) with respect to R (shared [N,3,3] or per pair [B,N,3,3])."""
    Rl = R.double().requires_grad_(True)
    W1, W2, b2 = W1.double(), W2.double(), b2.double()
    tgt = oracle.forward_3d2d_torch(vt.double(), W1, W2, b2)
    rows = []
    for b in range(vs.shape[0]):
        Rb = Rl[b] if R.dim() == 4 else Rl
        rot = oracle.rotate_volume_torch(vs[b].double()[None].expand(Rb.shape[0], -1, -1, -1, -1), Rb)
        rows.append((oracle.forward_3d2d_torch(rot, W1, W2, b2) * tgt[b][None]).sum(dim=1).mean(dim=-1))
    s = torch.stack(rows)
    (s * gs.double()).sum().backward()
    return s.detach(), Rl.grad


def _close(got, ref, tol, what):
    got = got.detach().cpu().double()
    scale = float(ref.abs().max())
    err = float((got - ref).abs().max())
    assert err <= tol * scale, (what, err, scale)


def _inputs(golden, B):
    g, w = golden["shared_n3000_b3"], golden["weights"]
    T = lambda a: torch.from_numpy(np.asarray(a))
    return T(g["vol_src"][:B]), T(g["vol_tgt"][:B]), T(w["W1"]), T(w["W2"]), T(w["b2"])


def test_lattice_rotations_sample_exact_integers():
    """The lattice cases are only a test of the floor convention if their coordinates are exact integers in both the
    fp32 the kernels use and the fp64 of the reference."""
    R = _lattice_rotations()
    for dtype in (torch.float32, torch.float64):
        u = _unnormalised_coords(R, dtype)
        assert torch.equal(u, u.round()), dtype
    # the other cases are differentiable where they sample: each coordinate is an exact integer in both precisions (an
    # axis the rotation leaves fixed) or clear of every integer, so that fp32 and fp64 agree on its floor
    for R in (_outside_rotations(), torch.cat([_lattice_rotations(), _outside_rotations()])):
        u32, u64 = _unnormalised_coords(R, torch.float32).double(), _unnormalised_coords(R, torch.float64)
        exact = (u32 == u32.round()) & (u64 == u64.round()) & (u32 == u64)
        assert ((u64 - u64.round()).abs() > 1e-4)[~exact].all()
    u = _unnormalised_coords(_outside_rotations(), torch.float64)
    assert ((u < -1) | (u >= 8)).any(dim=(1, 2, 3, 4)).all()


@pytest.mark.parametrize("case", ["random", "lattice", "outside"])
@pytest.mark.parametrize("per_rotation", [False, True])
def test_rotate_volume_grad_R_matches_autograd(ahv, oracle, case, per_rotation):
    gen = torch.Generator().manual_seed(1)
    if case == "random":
        R = ahv.so3.sample_rotations(40, seed=17, device=DEV).cpu()
    else:
        R = _lattice_rotations() if case == "lattice" else _outside_rotations()
    n = R.shape[0]
    vol = torch.randn(*((n,) if per_rotation else ()), 16, 8, 8, 8, generator=gen)
    gout = torch.randn(n, 16, 8, 8, 8, generator=gen)
    ref = _rotate_ref(oracle, vol, R, gout, per_rotation)
    got = ahv.ops.rotate_volume_grad_R(vol.to(DEV), gout.to(DEV), R.to(DEV), per_rotation)
    _close(got, ref, 2e-4, (case, per_rotation))


def _R_set(ahv, B, N, per_pair, seed):
    """Random rotations with the lattice and out-of-range cases mixed in."""
    special = torch.cat([_lattice_rotations(), _outside_rotations()])
    R = ahv.so3.sample_rotations(B * N if per_pair else N, seed=seed, device=DEV).cpu()
    R = R.reshape(B, N, 3, 3).clone() if per_pair else R.clone()
    flat = R.reshape(-1, 3, 3)
    step = max(1, flat.shape[0] // special.shape[0])
    flat[::step][: special.shape[0]] = special[: flat[::step].shape[0]]
    return R


# The backward kernels add per-CTA partial sums into the outputs with float atomics, in whatever order the CTAs finish:
# at the sizes below ahv_score_backward differs from ITSELF from run to run by up to 1.5e-6 of a gradient's maximum
# (measured on a B200: b2 1.5e-6, W2 9e-7, W1 7e-7 with shared R over 3 x 300 items).  Multi-CTA calls are therefore
# compared at 1e-5 of the maximum; a call with ONE item runs one CTA, each output element receives one atomic add onto
# zero, and there the entries are compared bit for bit (test_ex_entry_is_the_plain_kernel_bit_for_bit_on_one_item) -
# except grad_vol, whose adjoint sums each input voxel's list of contributions in the order shared-memory integer atomics
# ranked them, which varies from run to run inside one CTA too (exact only where every list has one nonzero term).
_ATOMIC_ORDER = 1e-5


def _agree(a, b, what, tol=_ATOMIC_ORDER):
    assert float((a - b).abs().max()) <= tol * float(b.abs().max()), what


@pytest.mark.parametrize("per_pair", [False, True])
def test_score_backward_ex_grad_R_matches_autograd(ahv, golden, oracle, per_pair):
    """Shared R over B=3 pairs (N=300: item ranges cross CTA boundaries, the reference is summed over pairs) and per-pair
    R; lattice and out-of-range rotations included.  The other five gradients agree with ahv_score_backward's to the
    order of float-atomic summation, and NULL outputs are honoured."""
    B, N = (3, 300) if not per_pair else (3, 60)
    vs, vt, W1, W2, b2 = _inputs(golden, B)
    R = _R_set(ahv, B, N, per_pair, seed=23)
    gs = torch.randn(B, N, generator=torch.Generator().manual_seed(7))
    _, ref = _scores_ref(oracle, vs, vt, R, W1, W2, b2, gs)
    d = [t.to(DEV) for t in (vs, vt, W1, W2, b2, R, gs)]
    tgt = ahv.ops.forward_3d2d(d[1], d[2], d[3], d[4])
    args = (d[0], tgt, d[5], d[2], d[3], d[4], d[6])
    got = ahv.ops.score_backward(*args, want_grad_R=True)
    _close(got[5], ref, 2e-4, ("grad_R", per_pair))
    plain = ahv.ops.score_backward(*args)
    for name, a, p in zip(("vol", "tgt", "W1", "W2", "b2"), got[:5], plain):
        _agree(a, p, name)
    # NULL outputs are honoured: grad_R alone, grad_R with one other, and no grad_R with some outputs missing
    _agree(ahv.ops.score_grad_R(*args), got[5], "grad_R alone")
    vs_, tg_, R_, W1_, W2_, b2_, gs_, B_, N_, pp = ahv.ops._score_backward_args(*args)
    g_tgt, g_R = torch.zeros_like(plain[1]), torch.zeros_like(got[5])
    ahv.ops._score_backward_ex(vs_, tg_, R_, W1_, W2_, b2_, gs_, None, None, (None, g_tgt, None, None, None, g_R), B_, N_, pp)
    _agree(g_tgt, plain[1], "tgt with grad_R")
    _agree(g_R, got[5], "grad_R with tgt")
    g_vol, g_w2 = torch.zeros_like(plain[0]), torch.zeros_like(plain[3])
    ahv.ops._score_backward_ex(vs_, tg_, R_, W1_, W2_, b2_, gs_, None, None, (g_vol, None, None, g_w2, None, None), B_, N_, pp)
    _agree(g_vol, plain[0], "vol without grad_R")
    _agree(g_w2, plain[3], "W2 without grad_R")


def test_ex_entry_is_the_plain_kernel_bit_for_bit_on_one_item(ahv, golden):
    """One item = one CTA = one atomic add per output element onto zero, so the order of summation is fixed: the ex
    entry's gradients are the plain entries' bit for bit (recomputing form and saved-activation fp32 form), and every
    subset of outputs returns exactly what the full call returns - grad_vol to the order of its contribution lists
    (1e-6 of its maximum, see above).  Lattice, out-of-range and random rotations."""
    def same(a, p, what):
        if what[-1] in ("vol", 0):      # grad_vol (by name or by output slot)
            _agree(a, p, what, 1e-6)
        else:
            assert torch.equal(a, p), what
    vs, vt, W1, W2, b2 = (t.to(DEV) for t in _inputs(golden, 2))
    tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
    Rs = torch.cat([_lattice_rotations(), _outside_rotations(), ahv.so3.sample_rotations(4, seed=61, device=DEV).cpu()]).to(DEV)
    gen = torch.Generator().manual_seed(10)
    for i in range(Rs.shape[0]):
        b = i % 2
        args = (vs[b:b + 1], tgt[b:b + 1], Rs[i:i + 1], W1, W2, b2, torch.randn(1, 1, generator=gen).to(DEV))
        full = ahv.ops.score_backward(*args, want_grad_R=True)
        for name, a, p in zip(("vol", "tgt", "W1", "W2", "b2"), full[:5], ahv.ops.score_backward(*args)):
            same(a, p, (i, name))
        assert torch.equal(ahv.ops.score_grad_R(*args), full[5]), i
        parts = ahv.ops._score_backward_args(*args)
        for keep in ((1, 5), (0, 3), (2, 4, 5)):
            outs = tuple(torch.zeros_like(full[k]) if k in keep else None for k in range(6))
            ahv.ops._score_backward_ex(*parts[:7], None, None, outs, *parts[7:])
            for k in keep:
                same(outs[k], full[k], (i, keep, k))
        _, h1, pinv = ahv.ops.score_train(*args[:6])
        saved = ahv.ops.score_backward(*args, h1, pinv, ahv.MATH_FP32)
        ex = ahv.ops.score_backward(*args, h1, pinv, ahv.MATH_TC, want_grad_R=True)
        for name, a, p in zip(("vol", "tgt", "W1", "W2", "b2"), ex[:5], saved):
            same(a, p, (i, "saved", name))


def test_saved_activation_form_of_the_ex_entry(ahv, golden):
    """ahv_score_backward_ex with h1_saved: the same saved values and mask as ahv_score_backward_saved's fp32 form, so
    its five gradients agree with that entry; its grad_R agrees with the recomputing form to the saved-activation
    bound (5e-2 in norm).  Many items: compared to the order of float-atomic summation (see _ATOMIC_ORDER)."""
    B, N = 2, 150
    vs, vt, W1, W2, b2 = (t.to(DEV) for t in _inputs(golden, B))
    R = ahv.so3.sample_rotations(N, seed=31, device=DEV)
    gs = torch.randn(B, N, generator=torch.Generator().manual_seed(8)).to(DEV)
    tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
    _, h1, pinv = ahv.ops.score_train(vs, tgt, R, W1, W2, b2)
    saved = ahv.ops.score_backward(vs, tgt, R, W1, W2, b2, gs, h1, pinv, ahv.MATH_FP32)
    ex = ahv.ops.score_backward(vs, tgt, R, W1, W2, b2, gs, h1, pinv, ahv.MATH_TC, want_grad_R=True)
    for name, a, p in zip(("vol", "tgt", "W1", "W2", "b2"), ex[:5], saved):
        _agree(a, p, name)
    exact = ahv.ops.score_backward(vs, tgt, R, W1, W2, b2, gs, want_grad_R=True)[5]
    assert float((ex[5] - exact).norm() / exact.norm()) <= 5e-2


@pytest.mark.parametrize("per_pair", [False, True])
def test_R_grad_through_verification_scores(ahv, golden, oracle, per_pair):
    """R.grad of training.verification_scores(math=MATH_FP32): fused form against the fp64 reference, chunked form
    against the fused form; save_activations=True against the default (tensor-core forward); R.grad stays None when R
    does not require a gradient."""
    B, N = 2, 48
    vs, vt, W1, W2, b2 = _inputs(golden, B)
    R = _R_set(ahv, B, N, per_pair, seed=41)
    gs = torch.randn(B, N, generator=torch.Generator().manual_seed(9))
    _, ref = _scores_ref(oracle, vs, vt, R, W1, W2, b2, gs)
    d = [t.to(DEV) for t in (vs, vt, W1, W2, b2)]
    grads = {}
    for name, kw in (("fused", dict(math=ahv.MATH_FP32)), ("chunked", dict(math=ahv.MATH_FP32, fused_backward=False, chunk=16)),
                     ("tc", dict(math=ahv.MATH_TC)), ("saved", dict(math=ahv.MATH_TC, save_activations=True))):
        Rl = R.to(DEV).requires_grad_(True)
        s = ahv.training.verification_scores(d[0], d[1], Rl, d[2], d[3], d[4], **kw)
        (s * gs.to(DEV)).sum().backward()
        assert Rl.grad is not None and Rl.grad.shape == R.shape, name
        grads[name] = Rl.grad.detach().cpu().double()
    _close(grads["fused"], ref, 2e-4, "fused")
    _close(grads["chunked"], grads["fused"], 2e-4, "chunked vs fused")
    assert float((grads["saved"] - grads["tc"]).norm() / grads["tc"].norm()) <= 5e-2
    # R without a gradient: nothing changes, R.grad stays None
    Rn = R.to(DEV)
    v = d[0].clone().requires_grad_(True)
    s = ahv.training.verification_scores(v, d[1], Rn, d[2], d[3], d[4], math=ahv.MATH_FP32)
    (s * gs.to(DEV)).sum().backward()
    assert Rn.grad is None and v.grad is not None


def test_refcompat_rotate_volume_differentiates_in_R(ahv, oracle):
    """Reference-style code that sets R.requires_grad_() on the drop-in rotate_volume gets R.grad (shared volume via
    expand, and one volume per rotation)."""
    gen = torch.Generator().manual_seed(3)
    R = torch.cat([ahv.so3.sample_rotations(20, seed=5, device=DEV).cpu(), _lattice_rotations(), _outside_rotations()])
    n = R.shape[0]
    gout = torch.randn(n, 16, 8, 8, 8, generator=gen)
    for per_rotation in (False, True):
        vol = torch.randn(*((n,) if per_rotation else ()), 16, 8, 8, 8, generator=gen)
        Rl = R.to(DEV).requires_grad_(True)
        v = vol.to(DEV) if per_rotation else vol.to(DEV)[None].expand(n, -1, -1, -1, -1)
        out = ahv.refcompat.rotate_volume(v, Rl)
        assert out.requires_grad
        (out * gout.to(DEV)).sum().backward()
        _close(Rl.grad, _rotate_ref(oracle, vol, R, gout, per_rotation), 2e-4, per_rotation)
    with torch.no_grad():
        assert not ahv.refcompat.rotate_volume(v, R.to(DEV).requires_grad_(True)).requires_grad


def _hat(u):
    z = torch.zeros_like(u[..., 0])
    return torch.stack((z, -u[..., 2], u[..., 1], u[..., 2], z, -u[..., 0], -u[..., 1], u[..., 0], z), -1).reshape(*u.shape[:-1], 3, 3)


def _expm(w):
    """exp([w]x) in fp64 (Rodrigues)."""
    th = w.norm(dim=-1, keepdim=True)[..., None]
    K = _hat(w / w.norm(dim=-1, keepdim=True))
    return torch.eye(3, dtype=w.dtype) + torch.sin(th) * K + (1 - torch.cos(th)) * (K @ K)


def test_grad_R_matches_a_finite_difference_of_the_fp32_scorer(ahv, golden):
    """Central difference of the AHV_MATH_FP32 score along exp(+-h [u]x) R against <G, [u]x R>, u = each item's ascent
    direction (w_i = <G, [e_i]x R>, u = w/|w|; a wrong direction or scale of G shows as a shortfall), summed over 128
    generic items.  The score is piecewise smooth (the trilinear weights at integer coordinates, the ReLU): a step h
    crosses kinks (fp64 on the same items: 1.5 % error in norm at h = 2e-4, 0.06 % at 1e-5) while fp32 rounding grows
    as 1/h; the sum over items averages both down."""
    B, N = 2, 64
    vs, vt, W1, W2, b2 = (t.to(DEV) for t in _inputs(golden, B))
    R = ahv.so3.sample_rotations(B * N, seed=51, device=DEV).reshape(B, N, 3, 3).contiguous()
    tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
    G = ahv.ops.score_grad_R(vs, tgt, R, W1, W2, b2, torch.ones(B, N, device=DEV)).cpu().double()
    R64 = R.cpu().double()
    M = G @ R64.transpose(-1, -2)
    w = torch.stack((M[..., 2, 1] - M[..., 1, 2], M[..., 0, 2] - M[..., 2, 0], M[..., 1, 0] - M[..., 0, 1]), -1)
    u = w / w.norm(dim=-1, keepdim=True)
    analytic = (G * (_hat(u) @ R64)).sum((-1, -2))
    assert torch.allclose(analytic, w.norm(dim=-1))
    h = 1e-4
    score = lambda Rc: ahv.ops.score(vs, tgt, Rc.float().to(DEV).contiguous(), W1, W2, b2, k=0, math=ahv.MATH_FP32)[0].cpu().double()
    fd = (score(_expm(h * u) @ R64) - score(_expm(-h * u) @ R64)) / (2 * h)
    assert abs(float(fd.sum() - analytic.sum())) <= 1e-2 * float(analytic.sum()), (fd, analytic)
    assert float((fd - analytic).abs().max()) <= 5e-2 * float(analytic.abs().max()), (fd, analytic)


def _synthetic_task(ahv, B, start_deg):
    import bench

    W1, W2, b2, vs, _, _ = bench.synthetic_inputs(torch, B, 16)
    v = ahv.HypothesisVerifier(W1.to(DEV), W2.to(DEV), b2.to(DEV))
    vs = vs.to(DEV)
    R_gt = ahv.so3.sample_rotations(B, seed=123, device=DEV)
    vt = ahv.ops.rotate_volume(vs, R_gt)                 # the score peaks at R_gt whatever the head weights are
    axis = torch.randn(B, 3, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    R0 = (_expm(math.radians(start_deg) * axis / axis.norm(dim=-1, keepdim=True)) @ R_gt.cpu().double()).float().to(DEV)
    return v, vs, vt, R_gt, R0


def _geodesic_deg(Ra, Rb):
    c = ((Ra.double() * Rb.double()).sum((-1, -2)).clamp(-1, 3) - 1) / 2
    return torch.rad2deg(torch.arccos(c.clamp(-1, 1)))


def test_refine_gradient_converges_on_the_synthetic_task(ahv):
    """Target = source rotated by a hidden R_gt: from 3 degrees off, 20 steps bring the mean error below 0.2 degrees,
    and no candidate ends with a lower fp32 score than it started with."""
    B = 8
    v, vs, vt, R_gt, R0 = _synthetic_task(ahv, B, 3.0)
    R_best, s_best, R_all, s_all = v.refine_gradient(vs, vt, R0, steps=20, step_deg=1.0)
    assert R_best.shape == (B, 3, 3) and s_best.shape == (B,) and R_all.shape == (B, 1, 3, 3) and s_all.shape == (B, 1)
    tgt = v.target_features(vt)
    s0 = ahv.ops.score(vs, tgt, R0[:, None].contiguous(), v.W1, v.W2, v.b2, k=0, math=ahv.MATH_FP32)[0]
    assert (s_all >= s0).all()
    err0, err = _geodesic_deg(R0, R_gt), _geodesic_deg(R_best, R_gt)
    assert float(err.mean()) < 0.2, (err0.tolist(), err.tolist())
    orth = R_best.double() @ R_best.double().transpose(-1, -2)
    assert float((orth - torch.eye(3, dtype=torch.float64, device=DEV)).abs().max()) <= 1e-5


def test_refine_gradient_top_k_scores_never_drop_and_pick_the_arg_max(ahv):
    """k candidates per pair at several distances: every final score >= its start, the best is the per-pair arg-max."""
    B, k = 4, 5
    v, vs, vt, R_gt, _ = _synthetic_task(ahv, B, 3.0)
    axis = torch.randn(B, k, 3, generator=torch.Generator().manual_seed(6), dtype=torch.float64)
    ang = torch.tensor([1.0, 4.0, 9.0, 20.0, 60.0], dtype=torch.float64)[None, :, None]
    R0 = (_expm(torch.deg2rad(ang) * axis / axis.norm(dim=-1, keepdim=True)) @ R_gt.cpu().double()[:, None]).float().to(DEV)
    tgt = v.target_features(vt)
    s0 = ahv.ops.score(vs, tgt, R0.contiguous(), v.W1, v.W2, v.b2, k=0, math=ahv.MATH_FP32)[0]
    R_best, s_best, R_all, s_all = v.refine_gradient(vs, vt, R0, steps=10)
    assert (s_all >= s0).all()
    assert torch.equal(s_best, s_all.max(dim=1).values)
    idx = torch.argmax(s_all, dim=1)
    assert torch.equal(R_best, R_all[torch.arange(B, device=DEV), idx])


def test_refine_gradient_replays_in_a_cuda_graph(ahv):
    B, k = 4, 3
    v, vs, vt, R_gt, R0 = _synthetic_task(ahv, B, 5.0)
    R0 = torch.stack([R0, R_gt, R0.transpose(-1, -2) @ R_gt @ R_gt], 1).contiguous()
    eager = v.refine_gradient(vs, vt, R0, steps=6)
    static_R = R0.clone()
    stream = torch.cuda.Stream(device=DEV)
    stream.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(stream):
        v.refine_gradient(vs, vt, static_R, steps=6)        # warm-up outside capture
    torch.cuda.current_stream(DEV).wait_stream(stream)
    torch.cuda.synchronize(DEV)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = v.refine_gradient(vs, vt, static_R, steps=6)
    static_R.zero_()
    static_R.copy_(R0)
    graph.replay()
    torch.cuda.synchronize(DEV)
    for a, b in zip(out, eager):
        assert torch.equal(a, b)
