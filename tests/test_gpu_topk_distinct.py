"""GPU: top-k of distinct rotations (ahv_topk_distinct / ops.topk_distinct) bit for bit against
distinct_oracle.select_distinct_np, its properties, and gradient refinement from distinct basins (ahv_refine_gradient_distinct)
on a volume with an exact 180-degree symmetry."""
import ctypes
import math
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import distinct_oracle  # noqa: E402  (tests/distinct_oracle.py)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
THETAS = (0.0, 0.5, 5.0, 20.0, 90.0, 180.0)
SHAPES = [(1, 1), (3, 31), (5, 33), (2, 1000), (4, 50_000), (1, 300_001)]


def _verifier(ahv, B, N, seed=0):
    import bench

    W1, W2, b2, vs, vt, normals = bench.synthetic_inputs(torch, B, max(N, 1), seed=seed)
    return ahv.HypothesisVerifier(W1.to(DEV), W2.to(DEV), b2.to(DEV)), vs.to(DEV), vt.to(DEV), normals


def _scored(ahv, B, N, per_pair):
    v, vs, vt, normals = _verifier(ahv, B, N)
    R = ahv.ops.rotations_from_normals(normals.to(DEV))
    if per_pair:
        R = ahv.so3.sample_rotations(B * N, seed=7, device=DEV).reshape(B, N, 3, 3).contiguous()
    return v.score(vs, vt, R, k=1).scores, R


def _quantised(scores, R):
    """Many ties, and every third rotation a copy of its predecessor."""
    q = (torch.round(scores * 8) / 8).contiguous()
    R = R.clone()
    n = R.shape[-3]
    src = torch.arange(0, n - 1, 3, device=R.device)
    R[..., src + 1, :, :] = R[..., src, :, :]
    return q, R.contiguous()


def _geodesic_deg(Ra, Rb):
    c = ((Ra.double() * Rb.double()).sum((-1, -2)).clamp(-1, 3) - 1) / 2
    return torch.rad2deg(torch.arccos(c.clamp(-1, 1)))


@pytest.mark.parametrize("per_pair", [False, True])
@pytest.mark.parametrize("B,N", SHAPES)
def test_oracle_parity(ahv, B, N, per_pair):
    scores, R = _scored(ahv, B, N, per_pair)
    for name, (s, Rs) in (("scorer", (scores, R)), ("quantised", _quantised(scores, R))):
        s_np, R_np = s.cpu().numpy(), Rs.cpu().numpy()
        for k in (1, 7, 32):
            for th in THETAS:
                val, idx, Rb = ahv.ops.topk_distinct(s, Rs, k, th)
                ov, oi, oR = distinct_oracle.select_distinct_np(s_np, R_np, k, th)
                assert np.array_equal(idx.cpu().numpy(), oi), (name, k, th)
                assert np.array_equal(val.cpu().numpy(), ov), (name, k, th)
                assert np.array_equal(Rb.cpu().numpy(), oR, equal_nan=True), (name, k, th)


@pytest.mark.parametrize("per_pair", [False, True])
def test_zero_and_half_turn(ahv, per_pair):
    B, N = 3, 5000
    scores, R = _scored(ahv, B, N, per_pair)
    for k in (1, 9, 32):
        val, idx, Rb = ahv.ops.topk_distinct(scores, R, k, 0.0)
        tv, ti = ahv.ops.topk(scores, k)
        assert torch.equal(val, tv) and torch.equal(idx, ti)
        assert torch.equal(Rb, ahv.ops.gather_rotations(R, ti))
        val, idx, Rb = ahv.ops.topk_distinct(scores, R, k, 180.0)
        assert torch.equal(idx[:, 0], ti[:, 0]) and torch.equal(val[:, 0], tv[:, 0])
        assert bool((idx[:, 1:] == -1).all()) and bool((val[:, 1:] == -math.inf).all()) and bool(Rb[:, 1:].isnan().all())


@pytest.mark.parametrize("th", [5.0, 20.0, 45.0])
def test_properties(ahv, th):
    B, N, k = 4, 20_000, 32
    scores, R = _scored(ahv, B, N, per_pair=True)
    val, idx, Rb = ahv.ops.topk_distinct(scores, R, k, th)
    for b in range(B):
        n = int((idx[b] >= 0).sum())
        assert n >= 1 and bool((idx[b, n:] == -1).all())
        i = idx[b, :n]
        assert bool((val[b, :n] == scores[b, i]).all())                         # strictly descending keys
        assert bool(((scores[b, i][1:] < scores[b, i][:-1]) | ((scores[b, i][1:] == scores[b, i][:-1]) & (i[1:] > i[:-1]))).all())
        d = _geodesic_deg(Rb[b, :n, None], Rb[b, None, :n])                   # winners pairwise more than th apart
        off = ~torch.eye(n, dtype=torch.bool, device=DEV)
        assert bool((d[off] > th - 1e-3).all())
        # every hypothesis ranked above the last winner is within th of a winner ranked above it
        s_last, i_last = scores[b, i[-1]], i[-1]
        above = (scores[b] > s_last) | ((scores[b] == s_last) & (torch.arange(N, device=DEV) < i_last))
        cand = torch.nonzero(above).flatten()
        dd = _geodesic_deg(R[b, cand][:, None], Rb[b, None, :n])               # [m, n]
        rank_ok = (scores[b, i][None] > scores[b, cand][:, None]) | (
            (scores[b, i][None] == scores[b, cand][:, None]) & (i[None] <= cand[:, None]))
        assert bool(((dd <= th + 1e-3) & rank_ok).any(1).all())


def test_fewer_hypotheses_than_k_repeatability_and_graph(ahv):
    scores, R = _scored(ahv, 3, 5, per_pair=False)
    val, idx, Rb = ahv.ops.topk_distinct(scores, R, 8, 1.0)
    assert bool((idx[:, 5:] == -1).all()) and bool((idx[:, :5] >= 0).all())
    scores, R = _scored(ahv, 6, 40_000, per_pair=True)
    a = ahv.ops.topk_distinct(scores, R, 32, 12.0)
    b = ahv.ops.topk_distinct(scores, R, 32, 12.0)
    assert all(torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                           y.view(torch.int32) if y.dtype == torch.float32 else y) for x, y in zip(a, b))
    s_static = scores.clone()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        ahv.ops.topk_distinct(s_static, R, 32, 12.0)
    torch.cuda.current_stream().wait_stream(stream)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ahv.ops.topk_distinct(s_static, R, 32, 12.0)
    for x in out:
        x.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out[1], a[1]) and torch.equal(out[0], a[0]) and torch.equal(out[2].nan_to_num(7.0), a[2].nan_to_num(7.0))


def test_verifier_score_with_separation(ahv):
    v, vs, vt, normals = _verifier(ahv, 2, 3000)
    R = ahv.ops.rotations_from_normals(normals.to(DEV))
    r0 = v.score(vs, vt, R, k=6)
    r = v.score(vs, vt, R, k=6, min_sep_deg=10.0)
    assert torch.equal(r.scores, r0.scores)
    val, idx, Rb = ahv.ops.topk_distinct(r0.scores, R, 6, 10.0)
    assert torch.equal(r.topk_idx, idx) and torch.equal(r.topk_val, val) and torch.equal(r.R_best, Rb)
    with pytest.raises(ValueError):
        v.score(vs, vt, R, k=6, min_sep_deg=10.0, idx_offset=3)


def _refine_distinct_c(ahv, v, vs, vt, R, k, steps, th):
    """ahv_refine_gradient_distinct called directly (ops.refine_gradient routes min_sep_deg == 0 to the plain entry)."""
    B, N = vs.shape[0], R.shape[0]
    f = dict(device=DEV, dtype=torch.float32)
    out = (torch.empty(B, k, **f), torch.empty(B, k, device=DEV, dtype=torch.int64), torch.empty(B, k, 3, 3, **f),
           torch.empty(B, k, 3, 3, **f), torch.empty(B, k, **f), torch.empty(B, **f),
           torch.empty(B, device=DEV, dtype=torch.int64), torch.empty(B, 3, 3, **f))
    lib = ahv._lib.lib()
    ws = torch.empty(int(lib.ahv_refine_gradient_workspace_bytes(B, N, k)), device=DEV, dtype=torch.uint8)
    base = ahv.ops.base_coords(DEV)
    st = lib.ahv_refine_gradient_distinct(
        vs.data_ptr(), 0, vt.data_ptr(), R.data_ptr(), 0, v.W1.data_ptr(), v.W2.data_ptr(), v.b2.data_ptr(), base.data_ptr(), k,
        steps, 1.0, th, *(t.data_ptr() for t in out), B, N, v.math, ws.data_ptr(), ws.numel(),
        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    ahv._lib.check(st, "ahv_refine_gradient_distinct")
    return out


def _same(a, b):
    if a.dtype == torch.float32:
        return torch.equal(a.view(torch.int32), b.view(torch.int32))
    return torch.equal(a, b)


@pytest.mark.parametrize("math_mode", ["tc", "fp32"])
@pytest.mark.parametrize("k", [1, 8])
def test_refinement_at_zero_separation_is_the_plain_chain(ahv, k, math_mode):
    v, vs, vt, normals = _verifier(ahv, 3, 4000)
    v.math = ahv.MATH_TC if math_mode == "tc" else ahv.MATH_FP32
    R = ahv.ops.rotations_from_normals(normals.to(DEV))
    plain = ahv.ops.refine_gradient(vs, vt, R, v.W1, v.W2, v.b2, k=k, steps=10, math=v.math)[:8]
    zero = _refine_distinct_c(ahv, v, vs, vt, R, k, 10, 0.0)
    assert all(_same(a, b) for a, b in zip(plain, zero))
    # the chain as the parent composed it: ahv_verify's top-k, then the ascent and its arg-max
    _, fv, fi, fR = ahv.ops.verify(vs, vt, R, v.W1, v.W2, v.b2, k=k, math=v.math)
    bR, bv, Ra, sa = v.ascend(vs, vt, fR, steps=10)
    for a, b in zip(plain, (fv, fi, fR, Ra, sa, bv)):
        assert _same(a, b)
    assert _same(plain[7], bR)


def test_refinement_chain_with_separation(ahv):
    v, vs, vt, normals = _verifier(ahv, 3, 4000)
    R = ahv.ops.rotations_from_normals(normals.to(DEV))
    k, th = 32, 100.0                                            # fewer than 32 rotations lie pairwise 100 degrees apart
    fv, fi, fR, Ra, sa, bv, bi, bR, _ = ahv.ops.refine_gradient(vs, vt, R, v.W1, v.W2, v.b2, k=k, steps=10, math=v.math,
                                                                min_sep_deg=th)
    scores = v.score(vs, vt, R, k=2).scores                     # k > 1: target features, then ahv_score, as in the chain
    val, idx, Rb = ahv.ops.topk_distinct(scores, R, k, th)
    assert _same(fv, val) and _same(fi, idx) and torch.equal(fR.nan_to_num(7.0), Rb.nan_to_num(7.0))
    assert bool((fi == -1).any())
    empty = fi < 0
    assert bool(Ra[empty].isnan().all()) and bool((sa[empty] == -math.inf).all())
    for b in range(3):
        n = int((~empty[b]).sum())
        R1, s1 = ahv.ops.gradient_ascent(vs[b:b + 1], v.target_features(vt[b:b + 1]), fR[b:b + 1, :n].contiguous(),
                                         v.W1, v.W2, v.b2, steps=10)
        assert _same(Ra[b:b + 1, :n], R1) and _same(sa[b:b + 1, :n], s1)
        j = int(torch.argmax(s1[0]))
        assert int(bi[b]) == j and _same(bv[b], s1[0, j]) and _same(bR[b], R1[0, j])
    g = ahv.GraphedRefiner(v, 3, 4000, k=k, method="gradient", steps=10, min_sep_deg=th)
    Rg, sg = g(vs, vt, R)
    torch.cuda.synchronize()
    assert _same(Rg, bR) and _same(sg, bv)
    with pytest.raises(ValueError):
        ahv.GraphedRefiner(v, 3, 4000, k=k, method="perturb", min_sep_deg=th)


def _hat(u):
    z = torch.zeros_like(u[..., 0])
    return torch.stack((z, -u[..., 2], u[..., 1], u[..., 2], z, -u[..., 0], -u[..., 1], u[..., 0], z), -1).reshape(*u.shape[:-1], 3, 3)


def _expm(w):
    th = w.norm(dim=-1, keepdim=True)[..., None]
    K = _hat(w / w.norm(dim=-1, keepdim=True))
    return torch.eye(3, dtype=w.dtype) + torch.sin(th) * K + (1 - torch.cos(th)) * (K @ K)


def _around(R0, deg, gen):
    """[m,3,3] rotations deg[j] degrees off R0 [3,3] about random axes (fp64 on the host)."""
    axis = torch.randn(len(deg), 3, generator=gen, dtype=torch.float64)
    ang = torch.tensor(deg, dtype=torch.float64)[:, None] * math.pi / 180
    return _expm(ang * axis / axis.norm(dim=-1, keepdim=True)) @ R0.cpu().double()


def symmetric_task(ahv, B, eps=0.1, seed=0):
    """Source V_sym + eps*A with V_sym = (V + V flipped along H and W) / 2, target = the source rotated by R_gt.  The flip
    is the lattice permutation of S = diag(-1, -1, 1), so S R_gt scores almost as high as R_gt (the false mode)."""
    import bench

    W1, W2, b2, V, A, _ = bench.synthetic_inputs(torch, B, 1, seed=seed)
    V_sym = 0.5 * (V + V.flip(3, 4))
    src = (V_sym + eps * A).to(DEV).contiguous()
    R_gt = ahv.so3.sample_rotations(B, seed=321 + seed, device=DEV)
    tgt = ahv.ops.rotate_volume(src, R_gt)
    v = ahv.HypothesisVerifier(W1.to(DEV), W2.to(DEV), b2.to(DEV))
    return v, src, tgt, R_gt


def symmetric_set(R_gt, gen, n_false=31, false_deg=2.0, true_deg=8.0):
    """n_false rotations within false_deg of S R_gt, then one true_deg from R_gt; [B, n_false + 1, 3, 3]."""
    S = torch.diag(torch.tensor([-1.0, -1.0, 1.0], dtype=torch.float64))
    out = []
    for b in range(R_gt.shape[0]):
        Rg = R_gt[b].cpu().double()
        fal = _around(S @ Rg, list(np.linspace(0.3, false_deg, n_false)), gen)
        tru = _around(Rg, [true_deg], gen)
        out.append(torch.cat((fal, tru)))
    return torch.stack(out).float().to(DEV).contiguous()


def test_distinct_basins_recover_the_true_mode_of_a_symmetric_volume(ahv):
    v, src, tgt, R_gt = symmetric_task(ahv, 1)
    R = symmetric_set(R_gt, torch.Generator().manual_seed(5))[0]
    S = torch.diag(torch.tensor([-1.0, -1.0, 1.0], device=DEV))
    # preconditions: plain top-8 lies entirely at the false mode, and so does the plain refinement from it
    r = v.score(src, tgt, R, k=8)
    assert bool((_geodesic_deg(r.R_best[0], (S @ R_gt[0])[None]) < 3.0).all())
    bR0, bv0, _, _, _ = v.refine_by_gradient(src, tgt, R, k=8, steps=40)
    assert float(_geodesic_deg(bR0[0], S @ R_gt[0])) < 1.0
    # distinct basins: the second start lies at the true mode, and its ascent wins
    bR, bv, first, _, _ = v.refine_by_gradient(src, tgt, R, k=2, steps=40, min_sep_deg=30.0)
    assert int(first.topk_idx[0, 1]) == 31
    assert float(_geodesic_deg(bR[0], R_gt[0])) < 0.1
    assert float(bv[0]) > float(bv0[0])
