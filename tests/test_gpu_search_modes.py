"""GPU: ahv_search_modes (coarse-to-fine search that keeps k distinct modes) against the same chain composed from the public
ops and modes_oracle's selection steps, its slot and ordering invariants, graph replay, HypothesisVerifier.search, and the
near-symmetric and config 4 tasks."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import modes_oracle as mo  # noqa: E402  (tests/modes_oracle.py)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
ahv = importlib.import_module("3dahv_b200")
ops = ahv.ops
DEV = torch.device("cuda", 0)
BASE, THETA = 2, 30.0


def _inputs(B, seed=0):
    import bench

    W1, W2, b2, vs, vt, _ = bench.synthetic_inputs(torch, B, 1, seed=seed)
    return [t.to(DEV) for t in (W1, W2, b2, vs, vt)]


def compose(vs, vt, W1, W2, b2, base_level, levels, k, w, theta, math):
    """The search restated with the public ops (hopf_grid, score with k = 0, topk_distinct, hopf_children) and
    modes_oracle's selection steps.  Returns (first_val, first_idx, first_R, val, idx, R) and the base-level slots."""
    B = vs.shape[0]
    tf = ops.forward_3d2d(vt, W1, W2, b2)
    G = ops.hopf_grid(base_level, device=DEV)
    S0 = ops.score(vs, tf, G, W1, W2, b2, k=0, math=math)[0]
    fv, fi, fR = ops.topk_distinct(S0, G, k, theta)

    def children(lev, gen):
        ci, cR = ops.hopf_children(base_level + lev, torch.from_numpy(gen).to(DEV))
        return ci.reshape(B, -1).cpu().numpy(), cR.reshape(B, -1, 3, 3).cpu().numpy()

    def score(R):
        return ops.score(vs, tf, torch.from_numpy(R).to(DEV), W1, W2, b2, k=0, math=math)[0].cpu().numpy()

    npy = [t.cpu().numpy() for t in (fv, fi, fR)]
    val, idx, R = mo.search_modes_np(S0.cpu().numpy(), G.cpu().numpy(), *npy, theta, w, levels, children, score)
    slot = mo.slots_np(G.cpu().numpy(), npy[1], npy[2], theta)
    return (fv, fi, fR, *(torch.from_numpy(np.ascontiguousarray(a)).to(DEV) for a in (val, idx, R))), slot


NAMES = ("first_val", "first_idx", "first_R", "val", "idx", "R")


@pytest.mark.parametrize("levels", (0, 3))
@pytest.mark.parametrize("B,k,w", ((1, 1, 4), (5, 8, 4), (32, 8, 1), (5, 32, 8), (32, 32, 4), (1, 8, 8)))
@pytest.mark.parametrize("math", (ahv.MATH_TC, ahv.MATH_FP32))
@pytest.mark.parametrize("dtype", (torch.float32, torch.bfloat16))
def test_search_modes_equals_the_composed_ops_bit_for_bit(dtype, math, B, k, w, levels):
    W1, W2, b2, vs, vt = _inputs(B, seed=B + k + w)
    vs = vs.to(dtype)
    got = ops.search_modes(vs, vt, W1, W2, b2, base_level=BASE, levels=levels, k=k, beam=w, min_sep_deg=THETA, math=math)[:6]
    ref, _ = compose(vs, vt, W1, W2, b2, BASE, levels, k, w, THETA, math)
    for name, a, b in zip(NAMES, got, ref):
        assert torch.equal(a.nan_to_num(7.0), b.nan_to_num(7.0)), name                # empty modes: NaN in both
    if levels == 0:
        for a, b in zip(got[:3], got[3:]):
            assert torch.equal(a.nan_to_num(7.0), b.nan_to_num(7.0))


@pytest.mark.parametrize("math", (ahv.MATH_TC, ahv.MATH_FP32))
def test_first_is_topk_distinct_of_the_base_scores(math):
    B, k = 6, 8
    W1, W2, b2, vs, vt = _inputs(B, seed=21)
    fv, fi, fR = ops.search_modes(vs, vt, W1, W2, b2, base_level=BASE, levels=2, k=k, min_sep_deg=THETA, math=math)[:3]
    G = ops.hopf_grid(BASE, device=DEV)
    S0 = ops.score(vs, ops.forward_3d2d(vt, W1, W2, b2), G, W1, W2, b2, k=0, math=math)[0]
    for a, b in zip((fv, fi, fR), ops.topk_distinct(S0, G, k, THETA)):
        assert torch.equal(a.nan_to_num(7.0), b.nan_to_num(7.0))


@pytest.mark.parametrize("levels", (1, 4))
def test_every_mode_descends_from_its_own_slot(levels):
    B, k, w = 8, 8, 4
    W1, W2, b2, vs, vt = _inputs(B, seed=13)
    _, fi, _, val, idx, R, _ = ops.search_modes(vs, vt, W1, W2, b2, base_level=BASE, levels=levels, k=k, beam=w,
                                                min_sep_deg=THETA)
    _, slot = compose(vs, vt, W1, W2, b2, BASE, 0, k, w, THETA, ahv.MATH_TC)
    G = ops.hopf_grid(BASE + levels, device=DEV)
    fi, idx, val = fi.cpu().numpy(), idx.cpu().numpy(), val.cpu()
    for b in range(B):
        n = int((fi[b] >= 0).sum())
        assert (idx[b, :n] >= 0).all() and (idx[b, n:] == -1).all() and torch.isneginf(val[b, n:]).all()
        origin = slot[b, idx[b, :n] // 8 ** levels]                                    # the base cell each mode came from
        assert sorted(origin.tolist()) == list(range(n))                              # one mode per non-empty slot
        assert torch.equal(R[b, :n], G[torch.from_numpy(idx[b, :n]).to(DEV)]) and torch.isnan(R[b, n:]).all()
        assert (val[b, : n - 1] >= val[b, 1:n]).all()


def test_min_sep_180_keeps_one_mode_and_empty_slots_last():
    B, k = 4, 8
    W1, W2, b2, vs, vt = _inputs(B, seed=17)
    fv, fi, fR, val, idx, R, _ = ops.search_modes(vs, vt, W1, W2, b2, base_level=BASE, levels=3, k=k, min_sep_deg=180.0)
    assert (fi[:, 0] >= 0).all() and (fi[:, 1:] == -1).all() and torch.isnan(fR[:, 1:]).all()
    assert (idx[:, 0] >= 0).all() and (idx[:, 1:] == -1).all()
    assert torch.isfinite(val[:, 0]).all() and torch.isneginf(val[:, 1:]).all()
    assert torch.isfinite(R[:, 0]).all() and torch.isnan(R[:, 1:]).all()
    # one slot holding every cell: with k = 1 (the same candidate sets) the beam of 4 is the plain search's top-4
    one = ops.search_modes(vs, vt, W1, W2, b2, base_level=BASE, levels=3, k=1, beam=4, min_sep_deg=180.0)
    plain = ops.search_hierarchical(vs, vt, W1, W2, b2, base_level=BASE, levels=3, k=4)
    assert torch.equal(one[4][:, 0], plain[4][:, 0]) and torch.equal(one[3][:, 0], plain[3][:, 0])


def test_repeated_calls_and_graph_replay_are_bit_identical():
    B, k, w = 5, 8, 4
    W1, W2, b2, vs, vt = _inputs(B, seed=3)
    run = lambda out=None, ws=None: ops.search_modes(vs, vt, W1, W2, b2, base_level=BASE, levels=4, k=k, beam=w,
                                                     min_sep_deg=THETA, out=out, workspace=ws)
    same = lambda xs, ys: all(torch.equal(x.nan_to_num(7.0), y.nan_to_num(7.0)) for x, y in zip(xs, ys))
    a = [t.clone() for t in run()[:6]]
    b = run()
    assert same(a, b[:6])
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        res = run(b[:6], b[6])
    torch.cuda.current_stream().wait_stream(stream)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run(res[:6], res[6])
    for t in res[:6]:
        t.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert same(a, res[:6])
    # new inputs through the same graph equal an eager call on them
    _, _, _, vs2, vt2 = _inputs(B, seed=4)
    vs.copy_(vs2)
    vt.copy_(vt2)
    graph.replay()
    eager = ops.search_modes(vs2, vt2, W1, W2, b2, base_level=BASE, levels=4, k=k, beam=w, min_sep_deg=THETA)
    torch.cuda.synchronize()
    assert same(eager[:6], res[:6])


def test_verifier_search_keeps_todays_call_and_rejects_a_misplaced_beam():
    W1, W2, b2, vs, vt = _inputs(3, seed=5)
    v = ahv.HypothesisVerifier(W1, W2, b2)
    Rb, sb, first, final = v.search(vs, vt, base_level=BASE, levels=3, k=8, min_sep_deg=0.0)
    ref = ops.search_hierarchical(vs, vt, W1, W2, b2, base_level=BASE, levels=3, k=8)
    for a, b in zip((first.topk_val, first.topk_idx, first.R_best, final.topk_val, final.topk_idx, final.R_best), ref[:6]):
        assert torch.equal(a, b)
    assert torch.equal(Rb, ref[5][:, 0]) and torch.equal(sb, ref[3][:, 0])
    Rm, sm, first_m, final_m = v.search(vs.bfloat16(), vt, base_level=BASE, levels=3, k=8, min_sep_deg=THETA, beam=2)
    ref = ops.search_modes(vs.bfloat16(), vt, W1, W2, b2, base_level=BASE, levels=3, k=8, beam=2, min_sep_deg=THETA)
    got = (first_m.topk_val, first_m.topk_idx, first_m.R_best, final_m.topk_val, final_m.topk_idx, final_m.R_best)
    assert all(torch.equal(a.nan_to_num(7.0), b.nan_to_num(7.0)) for a, b in zip(got, ref[:6]))
    assert torch.equal(Rm, ref[5][:, 0]) and torch.equal(sm, ref[3][:, 0])
    with pytest.raises(ValueError):
        v.search(vs, vt, beam=2)
    with pytest.raises(ValueError):
        v.search(vs, vt, min_sep_deg=-1.0)


def _geodesic_deg(Ra, Rb):
    c = ((Ra.double() * Rb.double()).sum((-1, -2)) - 1) / 2
    return torch.rad2deg(torch.arccos(c.clamp(-1, 1)))


def _symmetric_task(eps=0.1):
    """scripts/hierarchical_search.py's near-symmetric task: 64 pairs whose source is nearly its own 180-degree turn."""
    import bench

    W1, W2, b2, V, A, _ = bench.synthetic_inputs(torch, 64, 1)
    src = (0.5 * (V + V.flip(3, 4)) + eps * A).to(DEV).contiguous()
    R_gt = ahv.so3.sample_rotations(64, seed=321, device=DEV)
    return (W1.to(DEV), W2.to(DEV), b2.to(DEV)), src, ops.rotate_volume(src, R_gt), R_gt


@pytest.mark.parametrize("math", (ahv.MATH_TC, ahv.MATH_FP32))
def test_modes_find_the_true_mode_of_every_near_symmetric_pair(math):
    head, vs, vt, R_gt = _symmetric_task()
    v = ahv.HypothesisVerifier(*head, math=math)
    Rp, _, _, _ = v.search(vs, vt, base_level=2, levels=4, k=32)
    assert float(_geodesic_deg(Rp, R_gt).max()) > 90.0                              # the plain search loses the basin
    _, _, _, final = v.search(vs, vt, base_level=2, levels=4, k=8, min_sep_deg=30.0, beam=4)
    live = final.topk_idx >= 0
    e = _geodesic_deg(final.R_best, R_gt[:, None]).masked_fill(~live, 360.0).min(1).values   # the best of the modes
    R0 = torch.where(live[..., None, None], final.R_best, final.R_best[:, :1]).contiguous()
    Ra, _, _, _ = v.ascend(vs, vt, R0, steps=20)                                     # ascend from every mode
    # The bounds come from the measured run (profiles/r18_search_modes.jsonl, B200), identical under both math modes: the
    # plain search's top-1 misses by up to 179.6 deg; the nearest mode lies at most 5.24 deg from R_gt (its beam of 4 ends
    # on a coarser cell of the right basin than base level 3 reaches), and ascending from every mode ends within 0.035 deg.
    assert float(e.max()) < 6.0, e
    assert float(_geodesic_deg(Ra, R_gt).max()) < 0.05


@pytest.mark.parametrize("beam,bound", ((8, 0.75), (4, 1.5)))
@pytest.mark.parametrize("math", (ahv.MATH_TC, ahv.MATH_FP32))
def test_config4_known_rotation_task(math, beam, bound):
    """Config 4's task as scripts/config4_distinct.py builds it: 8 pairs, the target is the source rotated by R_gt."""
    import bench

    W1, W2, b2, vs, _, _ = bench.synthetic_inputs(torch, 8, 16)
    v = ahv.HypothesisVerifier(W1.to(DEV), W2.to(DEV), b2.to(DEV), math=math)
    vs = vs.to(DEV)
    R_gt = ahv.so3.sample_rotations(8, seed=123, device=DEV)
    Rb, _, _, _ = v.search(vs, ops.rotate_volume(vs, R_gt), base_level=2, levels=4, k=8, min_sep_deg=30.0, beam=beam)
    # test_gpu_hierarchical_search.py holds the plain search at (2, 4, 8) to 0.75 deg on this task.  Measured
    # (profiles/r18_search_modes.jsonl, B200, both math modes): a beam of 8 keeps it (largest error 0.60 deg); the default
    # beam of 4 does not (1.21 deg on one pair of 8), so it is held to 1.5 deg.
    assert float(_geodesic_deg(Rb, R_gt).max()) < bound
