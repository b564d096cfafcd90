"""GPU: posterior mass of the selected rotations (ahv_posterior_mass / ops.posterior_mass) against
posterior_oracle.posterior_mass_np, its assignment at the boundary, its value rules and determinism, agreement with
ops.infonce, and HypothesisVerifier.posterior / Estimator.predict_distribution end to end."""
import math
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import posterior_oracle  # noqa: E402  (tests/posterior_oracle.py)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _verifier(ahv, B, seed=0):
    import bench

    W1, W2, b2, vs, vt, normals = bench.synthetic_inputs(torch, B, 16, seed=seed)
    return ahv.HypothesisVerifier(W1.to(DEV), W2.to(DEV), b2.to(DEV)), vs.to(DEV), vt.to(DEV)


def _scored(ahv, B, N, per_pair, seed=0):
    v, vs, vt = _verifier(ahv, B, seed)
    if per_pair:
        R = ahv.so3.sample_rotations(B * N, seed=7 + seed, device=DEV).reshape(B, N, 3, 3).contiguous()
    else:
        R = ahv.so3.sample_rotations(N, seed=3 + seed, device=DEV)
    scores = ahv.ops.score(vs, v.target_features(vt), R, v.W1, v.W2, v.b2, k=0)[0]
    return scores, R


def _bits(t):
    return t.contiguous().view(torch.int32)


def _check_oracle(ahv, scores, R, centers, radius, T=0.1):
    log_z, mass = ahv.ops.posterior_mass(scores, R, centers, radius, T)
    o_lz, o_m = posterior_oracle.posterior_mass_np(scores.cpu().numpy(), R.cpu().numpy(),
                                                  None if centers is None else centers.cpu().numpy(), radius, T)
    assert np.allclose(log_z.cpu().numpy(), o_lz, rtol=1e-6, atol=0, equal_nan=True), (radius, T)
    assert np.allclose(mass.cpu().numpy(), o_m, rtol=0, atol=1e-6, equal_nan=True), (radius, T)
    return log_z, mass


@pytest.mark.parametrize("per_pair", [False, True])
@pytest.mark.parametrize("B,N", [(1, 1), (3, 2049), (2, 5000), (4, 50_000)])
def test_oracle_parity(ahv, B, N, per_pair):
    scores, R = _scored(ahv, B, N, per_pair)
    _check_oracle(ahv, scores, R, None, 15.0)                                          # k = 0: log_z alone
    for k in (1, 8, 32):
        for th in (0.0, 15.0, 40.0):
            if th > 0:
                _, _, Rb = ahv.ops.topk_distinct(scores, R, k, th)                   # winners, NaN empty slots
                _check_oracle(ahv, scores, R, Rb, th)
            else:
                _, idx = ahv.ops.topk(scores, min(k, N))
                Rb = ahv.ops.gather_rotations(R, idx)
                _check_oracle(ahv, scores, R, Rb, 20.0, T=0.05)


def _lattice():
    """The 24 rotations of the cube (entries 0 and +-1): traces between them are exact integers."""
    out = []
    for perm in ((0, 1, 2), (0, 2, 1), (1, 0, 2), (1, 2, 0), (2, 0, 1), (2, 1, 0)):
        for signs in ((1, 1, 1), (1, -1, -1), (-1, 1, -1), (-1, -1, 1), (-1, 1, 1), (1, -1, 1), (1, 1, -1), (-1, -1, -1)):
            M = np.zeros((3, 3), dtype=np.float32)
            for i in range(3):
                M[i, perm[i]] = signs[i]
            if round(np.linalg.det(M)) == 1:
                out.append(M)
    return np.stack(out)


def test_lattice_rotations_exactly_at_the_radius(ahv):
    L = _lattice()
    assert L.shape == (24, 3, 3)
    R = torch.from_numpy(L).to(DEV)
    gen = torch.Generator().manual_seed(0)
    scores = (torch.rand(3, 24, generator=gen) * 0.5).to(DEV)
    eye = torch.eye(3, device=DEV).expand(3, 1, 3, 3).contiguous()
    trace = np.einsum("nij,ij->n", L, np.eye(3, dtype=np.float32))
    s64 = scores.double().cpu().numpy()
    # c = fp32(1 + 2 cos(theta)): exactly 1.0 at 90 degrees, so the 90-degree rotations (trace 1) are inside; 1.0035 at
    # 89.9; 4.4e-16 at 120, so the 120-degree rotations (trace 0) fall just outside; -inf at 180
    for radius, inside in ((90.0, trace >= 1), (89.9, trace >= 3), (120.0, trace >= 1), (180.0, trace >= -1)):
        log_z, mass = _check_oracle(ahv, scores, R, eye, radius)
        for b in range(3):
            e = np.exp((s64[b] - s64[b].max()) / np.float64(np.float32(0.1)))
            assert abs(float(mass[b, 0]) - e[inside].sum() / e.sum()) < 1e-6, (radius, b)
    # centres = the distinct winners at theta = 90: every non-empty slot holds at least its own winner
    for th in (90.0, 89.9, 120.0):
        val, idx, Rb = ahv.ops.topk_distinct(scores, R, 8, th)
        log_z, mass = _check_oracle(ahv, scores, R, Rb, th)
        own = torch.exp(val.double() / np.float32(0.1) - log_z.double()[:, None])
        filled = idx >= 0
        assert bool((mass[filled].double() >= own[filled] * (1 - 1e-6)).all()) and bool((mass[~filled] == 0).all()), th


@pytest.mark.parametrize("per_pair", [False, True])
def test_distinct_winners_hold_what_they_suppressed(ahv, per_pair):
    """Centres = ahv_topk_distinct's winners and radius = min_sep_deg: every hypothesis ranked at or above the last
    winner was a winner or suppressed by one, so the slots hold at least all of that mass."""
    B, N = 3, 20_000
    scores, R = _scored(ahv, B, N, per_pair)
    for k, th in ((4, 10.0), (32, 25.0)):
        val, idx, Rb = ahv.ops.topk_distinct(scores, R, k, th)
        log_z, mass = _check_oracle(ahv, scores, R, Rb, th)
        for b in range(B):
            n = int((idx[b] >= 0).sum())
            s_last, i_last = scores[b, idx[b, n - 1]], idx[b, n - 1]
            above = (scores[b] > s_last) | ((scores[b] == s_last) & (torch.arange(N, device=DEV) <= i_last))
            p_above = torch.exp(scores[b, above].double() / np.float32(0.1) - log_z[b].double()).sum()
            assert float(mass[b].double().sum()) >= float(p_above) * (1 - 1e-6), (k, th, b)
            assert float(mass[b].sum()) <= 1 + 1e-6


def test_value_rules(ahv):
    scores, R = _scored(ahv, 4, 3000, per_pair=False)
    _, _, Rb = ahv.ops.topk_distinct(scores, R, 4, 20.0)
    Rb = Rb.clone()
    Rb[:, 2:] = float("nan")                                                           # empty slots
    s = scores.clone()
    s[1, ::3] = -math.inf                                                              # -inf scores contribute nothing
    s[2, 17] = math.nan                                                                # this pair alone turns NaN
    s[3, 5] = math.inf                                                                 # so does this one
    log_z, mass = _check_oracle(ahv, s, R, Rb, 20.0)
    assert bool((mass[:2, 2:] == 0).all()) and bool(torch.isfinite(log_z[:2]).all())
    assert bool(torch.isnan(log_z[2:]).all()) and bool(torch.isnan(mass[2:]).all())
    keep = torch.arange(3000, device=DEV) % 3 != 0
    lz1, m1 = ahv.ops.posterior_mass(s[1:2, keep].contiguous(), R[keep].contiguous(), Rb[1:2], 20.0)
    assert abs(float(lz1[0]) - float(log_z[1])) <= 1e-6 * abs(float(lz1[0])) and torch.allclose(m1, mass[1:2], atol=1e-6)
    for b in (0, 1):                                                                   # the other pairs are untouched
        lz, m = ahv.ops.posterior_mass(s[b:b + 1], R, Rb[b:b + 1], 20.0)
        assert torch.equal(_bits(lz), _bits(log_z[b:b + 1])) and torch.equal(_bits(m), _bits(mass[b:b + 1]))
    s[0] = -math.inf                                                                   # every score -inf
    log_z, mass = ahv.ops.posterior_mass(s[:1], R, Rb[:1], 20.0)
    assert float(log_z[0]) == -math.inf and bool(torch.isnan(mass).all())


@pytest.mark.parametrize("per_pair", [False, True])
def test_determinism_and_pair_alone(ahv, per_pair):
    B, N, k = 6, 30_001, 32
    scores, R = _scored(ahv, B, N, per_pair, seed=1)
    _, _, Rb = ahv.ops.topk_distinct(scores, R, k, 12.0)
    a = ahv.ops.posterior_mass(scores, R, Rb, 12.0)
    b = ahv.ops.posterior_mass(scores, R, Rb, 12.0)
    assert all(torch.equal(_bits(x), _bits(y)) for x, y in zip(a, b))
    for p in (0, 3, 5):
        Rp = R[p:p + 1].contiguous() if per_pair else R
        lz, m = ahv.ops.posterior_mass(scores[p:p + 1].contiguous(), Rp, Rb[p:p + 1].contiguous(), 12.0)
        assert torch.equal(_bits(lz), _bits(a[0][p:p + 1])) and torch.equal(_bits(m), _bits(a[1][p:p + 1])), p
        sub = slice(max(p - 1, 0), p + 1)                                              # inside a smaller batch too
        Rs = R[sub].contiguous() if per_pair else R
        lz, m = ahv.ops.posterior_mass(scores[sub].contiguous(), Rs, Rb[sub].contiguous(), 12.0)
        assert torch.equal(_bits(lz[-1:]), _bits(a[0][p:p + 1])) and torch.equal(_bits(m[-1:]), _bits(a[1][p:p + 1])), p


def test_cuda_graph_replay_with_changing_shapes(ahv):
    cases = [(3, 5000, 8), (1, 70_000, 32), (5, 2048, 0), (2, 1, 1)]
    graphs = []
    for B, N, k in cases:
        scores, R = _scored(ahv, B, N, per_pair=False, seed=B)
        Rb = ahv.ops.topk_distinct(scores, R, k, 15.0)[2] if k else None
        want = ahv.ops.posterior_mass(scores, R, Rb, 15.0)
        ws = torch.empty(ahv.ops.posterior_mass_workspace_bytes(B, N, k), device=DEV, dtype=torch.uint8)
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(stream):
            ahv.ops.posterior_mass(scores, R, Rb, 15.0, workspace=ws)
        torch.cuda.current_stream().wait_stream(stream)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = ahv.ops.posterior_mass(scores, R, Rb, 15.0, workspace=ws)
        graphs.append((g, out, want, (scores, R, Rb, ws)))                           # the graph reads these buffers
    for _ in range(2):
        for g, out, _, _ in reversed(graphs):
            for x in out:
                x.fill_(7.0)
            g.replay()
        torch.cuda.synchronize()
        for _, out, want, _ in graphs:
            assert all(torch.equal(_bits(x), _bits(y)) for x, y in zip(out, want))


def _away_from(R, G, thr_deg, margin_deg=0.5):
    """R [B,N,3,3] with every rotation within margin of the geodesic radius thr around G [B,3,3] replaced by G."""
    c = ((R.double() * G.double()[:, None]).sum((-1, -2)).clamp(-1, 3) - 1) / 2
    d = torch.rad2deg(torch.arccos(c.clamp(-1, 1)))
    band = (d - thr_deg).abs() < margin_deg
    return torch.where(band[..., None, None], G[:, None].expand_as(R), R).contiguous()


def test_single_gt_centre_agrees_with_infonce(ahv):
    B, N, thr = 8, 20_000, 15.0
    G = ahv.so3.sample_rotations(B, seed=11, device=DEV)
    near = ahv.ops.perturb_rotations(G, 200, 25.0, seed=2)                         # [B,200,3,3] around the GT
    R = torch.cat([near, ahv.so3.sample_rotations(B * (N - 200), seed=12, device=DEV).reshape(B, N - 200, 3, 3)], 1)
    R = _away_from(R, G, thr)
    gen = torch.Generator().manual_seed(1)
    s = (torch.randn(B, N, generator=gen) * 0.2).to(DEV)
    s[:, :200] += torch.linspace(0.0, 0.6, B, device=DEV)[:, None]                 # from diffuse to confident pairs
    loss, _ = ahv.ops.infonce(s, R, G, thr, 0.1, want_grad=False)
    _, mass = ahv.ops.posterior_mass(s, R, G[:, None].contiguous(), thr, 0.1)
    assert torch.allclose(-torch.log(mass[:, 0].double()), loss.double(), rtol=1e-5, atol=1e-6)


def test_verifier_posterior_end_to_end(ahv):
    B, N = 3, 6000
    v, vs, vt = _verifier(ahv, B, seed=2)
    R = ahv.so3.sample_rotations(N, seed=5, device=DEV)
    Rq = ahv.so3.sample_rotations(B * 2, seed=6, device=DEV).reshape(B, 2, 3, 3).contiguous()
    tf = v.target_features(vt)
    scores = ahv.ops.score(vs, tf, R, v.W1, v.W2, v.b2, k=0)[0]
    s_q = ahv.ops.score(vs, tf, Rq, v.W1, v.W2, v.b2, k=0)[0]
    for k, sep, radius in ((1, 0.0, 15.0), (8, 20.0, None), (4, 10.0, 30.0)):
        p = v.posterior(vs, vt, R, k=k, min_sep_deg=sep, radius_deg=radius, R_query=Rq)
        if sep > 0:
            val, idx, Rb = ahv.ops.topk_distinct(scores, R, k, sep)
        else:
            val, idx = ahv.ops.topk(scores, k)
            Rb = ahv.ops.gather_rotations(R, idx)
        assert torch.equal(p.topk_val, val) and torch.equal(p.topk_idx, idx) and torch.equal(_bits(p.R_best), _bits(Rb))
        log_z, mass = _check_oracle(ahv, scores, R, Rb, sep if radius is None else radius)
        assert torch.equal(_bits(p.mass), _bits(mass)) and torch.equal(_bits(p.log_z), _bits(log_z))
        o_lz, _ = posterior_oracle.posterior_mass_np(scores.cpu().numpy(), R.cpu().numpy(), None, 15.0)
        want = s_q.double().cpu().numpy() / np.float64(0.1) - o_lz.astype(np.float64)[:, None] + math.log(N)
        assert p.log_density.shape == (B, 2) and np.allclose(p.log_density.cpu().numpy(), want, rtol=1e-5, atol=1e-5)
    assert v.posterior(vs, vt, R, k=2, radius_deg=10.0).log_density is None
    with pytest.raises(ValueError):
        v.posterior(vs, vt, R, k=2)                                                    # radius needed when min_sep is 0


def test_estimator_predict_distribution(ahv):
    from modules.model import Estimator

    class _TinyBackbone(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.proj = torch.nn.Conv2d(3, 768, 1)

        def forward(self, img):
            return self.proj(torch.nn.functional.adaptive_avg_pool2d(img, 8))

    torch.manual_seed(0)
    cfg = {"DATA": {"NUM_ROTA": 3000, "BG": False, "SIZE_THR": 10, "ACC_THR": 15}}
    model = Estimator(cfg, feature_extractor=_TinyBackbone()).to(DEV).eval()
    gen = torch.Generator().manual_seed(3)
    vs, vt = (torch.randn(2, 2, 16, 8, 8, 8, generator=gen) * 0.1).to(DEV).unbind(0)
    R = ahv.so3.sample_rotations(3000, seed=9, device=DEV)
    gt = ahv.so3.sample_rotations(2, seed=10, device=DEV)
    post, R_out = model.predict_distribution(vs, vt, sampled_R=R, k=4, min_sep_deg=20.0, gt_R=gt)
    assert R_out is R
    want = model.verifier().posterior(vs, vt, R, k=4, min_sep_deg=20.0, radius_deg=15.0, temperature=0.1,
                                      R_query=gt[:, None].contiguous())
    for name in ("topk_val", "topk_idx", "R_best", "mass", "log_z", "log_density"):
        a, b = getattr(post, name), getattr(want, name)
        assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a,
                           b.view(torch.int32) if b.dtype == torch.float32 else b), name
    assert post.log_density.shape == (2, 1)
    post1, _ = model.predict_distribution(vs, vt, sampled_R=R)
    assert post1.mass.shape == (2, 1) and post1.log_density is None
