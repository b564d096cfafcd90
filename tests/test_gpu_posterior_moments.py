"""GPU: first moment of the posterior over each slot (ahv_posterior_moments / ops.posterior_moments) against
moments_oracle.posterior_moments_np, its value rules, bit invariance and graph replay, and the moments=True paths of
HypothesisVerifier.posterior and Estimator.predict_distribution."""
import math
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import moments_oracle  # noqa: E402  (tests/moments_oracle.py)
from test_gpu_posterior import _bits, _scored, _verifier  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _check_oracle(ahv, scores, R, centers, radius, T=0.1):
    """Every output against the oracle; log_z and mass bit-equal to ops.posterior_mass.  Returns the outputs."""
    out = ahv.ops.posterior_moments(scores, R, centers, radius, T)
    log_z, mass, mean_R, mean_cos, moment = out
    lz_m, mass_m = ahv.ops.posterior_mass(scores, R, centers, radius, T)
    assert torch.equal(_bits(log_z), _bits(lz_m)) and torch.equal(_bits(mass), _bits(mass_m)), (radius, T)
    _, _, o_R, o_cos, o_mom, gap = moments_oracle.posterior_moments_np(scores.cpu().numpy(), R.cpu().numpy(),
                                                                     centers.cpu().numpy(), radius, T)
    g_R, g_cos, g_mom = (x.double().cpu().numpy() for x in (mean_R, mean_cos, moment))
    assert np.array_equal(np.isnan(g_cos), np.isnan(o_cos)), (radius, T)
    assert np.array_equal(np.isnan(g_mom), np.isnan(o_mom)) and np.array_equal(np.isnan(g_R), np.isnan(o_R))
    assert np.allclose(g_cos, o_cos, rtol=0, atol=1e-6, equal_nan=True), (radius, T)
    assert np.allclose(g_mom, o_mom, rtol=0, atol=1e-6, equal_nan=True), (radius, T)
    sharp = gap >= 1e-3                                                          # mean_R unique and well conditioned
    assert np.allclose(g_R[sharp], o_R[sharp], rtol=0, atol=2e-6), (radius, T)
    fin = ~np.isnan(g_cos)
    Rf = g_R[fin]
    assert np.abs(np.einsum("nji,njk->nik", Rf, Rf) - np.eye(3)).max(initial=0) <= 1e-6
    assert np.abs(np.linalg.det(Rf) - 1).max(initial=0) <= 1e-6 and (np.abs(g_cos[fin]) <= 1).all()
    return out


@pytest.mark.parametrize("per_pair", [False, True])
@pytest.mark.parametrize("B,N", [(1, 1), (2, 2047), (2, 2048), (3, 2049), (2, 50_000), (1, 1_000_000)])
def test_oracle_parity(ahv, B, N, per_pair):
    if per_pair and N == 1_000_000:
        pytest.skip("one pair: the shared set is the per-pair set")
    scores, R = _scored(ahv, B, N, per_pair)
    for k in (1, 8, 32):
        _, _, Rb = ahv.ops.topk_distinct(scores, R, k, 15.0)                  # winners, NaN empty slots
        _check_oracle(ahv, scores, R, Rb, 15.0)
        C = ahv.so3.sample_rotations(B * k, seed=40 + k, device=DEV).reshape(B, k, 3, 3).contiguous()
        _check_oracle(ahv, scores, R, C, 25.0, T=0.05)                           # arbitrary centres


def test_bit_invariance(ahv):
    N, k = 30_001, 8
    scores, R = _scored(ahv, 37, N, per_pair=False, seed=1)
    _, _, Rb = ahv.ops.topk_distinct(scores, R, k, 12.0)
    full = ahv.ops.posterior_moments(scores, R, Rb, 12.0)
    again = ahv.ops.posterior_moments(scores, R, Rb, 12.0)
    assert all(torch.equal(_bits(x), _bits(y)) for x, y in zip(full, again))
    p = 20
    alone = ahv.ops.posterior_moments(scores[p:p + 1].contiguous(), R, Rb[p:p + 1].contiguous(), 12.0)
    moved = ahv.ops.posterior_moments(scores[[p, 3]].contiguous(), R, Rb[[p, 3]].contiguous(), 12.0)  # first of two
    Rpp = R.expand(2, N, 3, 3).contiguous()                                       # the shared set copied per pair
    per_pair = ahv.ops.posterior_moments(scores[[3, p]].contiguous(), Rpp, Rb[[3, p]].contiguous(), 12.0)
    for i, x in enumerate(full):
        want = _bits(x[p:p + 1])
        assert torch.equal(_bits(alone[i]), want) and torch.equal(_bits(moved[i][:1]), want), i
        assert torch.equal(_bits(per_pair[i][1:]), want) and torch.equal(_bits(per_pair[i][:1]), _bits(x[3:4])), i


def test_value_rules(ahv):
    scores, R = _scored(ahv, 5, 3000, per_pair=False)
    _, idx, Rb = ahv.ops.topk_distinct(scores, R, 4, 20.0)
    Rb = Rb.clone()
    Rb[0, 2] = float("nan")                                                        # an empty slot in pair 0 only
    s = scores.clone()
    s[1, ::3] = -math.inf                                                          # -inf scores contribute nothing
    s[2, 17] = math.nan                                                            # a NaN pair
    s[3] = -math.inf                                                               # every score -inf
    log_z, mass, mean_R, mean_cos, moment = _check_oracle(ahv, s, R, Rb, 20.0)
    assert bool(torch.isnan(moment[0, 2]).all()) and bool(torch.isnan(mean_R[0, 2]).all()) and bool(torch.isnan(mean_cos[0, 2]))
    assert bool(torch.isfinite(mean_cos[0, [0, 1, 3]]).all())
    for x in (log_z[2:3], mass[2], mean_R[2], mean_cos[2], moment[2], mass[3], mean_R[3], mean_cos[3], moment[3]):
        assert bool(torch.isnan(x).all())
    assert float(log_z[3]) == -math.inf
    # T = 1e-3: slot 1's scores all more than 0.75 below the maximum underflow in double; slot 0 holds the maximum
    s = scores[4:5].clone()
    slot = torch.from_numpy(moments_oracle.slots_np(R.cpu().numpy(), Rb[4].cpu().numpy(), 20.0)).to(DEV)
    assert bool((slot == 0).any()) and bool((slot == 1).any())
    s[0, slot == 1] = s.max() - 0.8
    log_z, mass, mean_R, mean_cos, moment = _check_oracle(ahv, s, R, Rb[4:5], 20.0, T=1e-3)
    assert float(mass[0, 1]) == 0 and bool(torch.isnan(moment[0, 1]).all()) and bool(torch.isnan(mean_cos[0, 1]))
    assert bool(torch.isfinite(mean_cos[0, 0])) and bool(torch.isfinite(mean_R[0, 0]).all())


def test_cuda_graph_replay(ahv):
    cases = [(3, 5000, 8), (1, 70_000, 32), (2, 1, 1)]
    graphs = []
    for B, N, k in cases:
        scores, R = _scored(ahv, B, N, per_pair=False, seed=B)
        Rb = ahv.ops.topk_distinct(scores, R, k, 15.0)[2]
        want = ahv.ops.posterior_moments(scores, R, Rb, 15.0)
        ws = torch.empty(ahv.ops.posterior_moments_workspace_bytes(B, N, k), device=DEV, dtype=torch.uint8)
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(stream):
            ahv.ops.posterior_moments(scores, R, Rb, 15.0, workspace=ws)
        torch.cuda.current_stream().wait_stream(stream)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = ahv.ops.posterior_moments(scores, R, Rb, 15.0, workspace=ws)
        graphs.append((g, out, want, (scores, R, Rb, ws)))                       # the graph reads these buffers
    for _ in range(2):
        for g, out, _, _ in reversed(graphs):
            for x in out:
                x.fill_(7.0)
            g.replay()
        torch.cuda.synchronize()
        for _, out, want, _ in graphs:
            assert all(torch.equal(_bits(x), _bits(y)) for x, y in zip(out, want))


def test_verifier_posterior_moments(ahv):
    B, N = 3, 6000
    v, vs, vt = _verifier(ahv, B, seed=2)
    R = ahv.so3.sample_rotations(N, seed=5, device=DEV)
    Rq = ahv.so3.sample_rotations(B, seed=6, device=DEV)[:, None].contiguous()
    for k, sep, radius in ((1, 0.0, 15.0), (8, 20.0, None)):
        a = v.posterior(vs, vt, R, k=k, min_sep_deg=sep, radius_deg=radius, R_query=Rq)
        b = v.posterior(vs, vt, R, k=k, min_sep_deg=sep, radius_deg=radius, R_query=Rq, moments=True)
        assert a.mean_R is None and a.mean_cos is None and a.moment is None and a.spread_deg is None
        for name in ("topk_val", "topk_idx", "R_best", "mass", "log_z", "log_density"):
            x, y = getattr(a, name), getattr(b, name)
            assert torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                               y.view(torch.int32) if y.dtype == torch.float32 else y), name
        want = ahv.ops.posterior_moments(v.score(vs, vt, R, k=1).scores, R, b.R_best, sep if radius is None else radius)
        for x, y in zip((b.mean_R, b.mean_cos, b.moment), want[2:]):
            assert torch.equal(_bits(x), _bits(y))
        assert b.mean_R.shape == (B, k, 3, 3) and b.moment.shape == (B, k, 3, 3) and b.spread_deg.shape == (B, k)
        fin = torch.isfinite(b.mean_cos)
        assert bool(fin[:, 0].all())
        assert torch.allclose(b.spread_deg[fin], torch.rad2deg(torch.arccos(b.mean_cos[fin].clamp(-1, 1))))


def test_estimator_predict_distribution_moments(ahv):
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
    post, _ = model.predict_distribution(vs, vt, sampled_R=R, k=4, min_sep_deg=20.0, moments=True)
    plain, _ = model.predict_distribution(vs, vt, sampled_R=R, k=4, min_sep_deg=20.0)
    assert torch.equal(_bits(post.mass), _bits(plain.mass)) and torch.equal(_bits(post.log_z), _bits(plain.log_z))
    assert post.mean_R.shape == (2, 4, 3, 3) and post.spread_deg.shape == (2, 4) and plain.mean_R is None
    assert bool(torch.isfinite(post.mean_cos[:, 0]).all())
