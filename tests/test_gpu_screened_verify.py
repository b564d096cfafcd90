"""GPU (B200): the screened arg-max of ahv_verify (fp32 volumes, MATH_TC, k = 1, no scores returned; csrc/ahv_score_tc.cu
launch_verify_tc_screened) returns what the single fp32-gather pass returns, bit for bit.

The single pass is the same call with the scores returned (the screened form never serves it).  Cases: the bench
workload; per-pair rotation sets with an index offset; duplicated rotations (equal scores: ties go to the lowest
index); a zero source volume (every hypothesis ties: every pair overflows its contender list and falls back to the
exact pass, which picks index 0); an outlier volume of ratio 1e9 (beyond the 16-bit gather's range: the guard trips);
a call below the size threshold (single pass); and the set sharded over two GPUs through the peer exchange."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda", 0)


def _bench_inputs(B, N):
    sys.path.insert(0, ROOT)
    import bench

    return bench.synthetic_inputs(torch, B, N)


def _verify(ahv, W, vs, vt, R, idx_offset=0):
    """(screened result, single-pass result, screen stats) of one call shape."""
    B, N = vs.shape[0], R.shape[-3]
    ws = torch.empty(ahv.ops.workspace_bytes(B, N, 1), dtype=torch.uint8, device=DEV)
    args = (vs.to(DEV), vt.to(DEV), R.to(DEV), *(t.to(DEV) for t in W))
    _, val, idx, Rb = ahv.ops.verify(*args, k=1, idx_offset=idx_offset, math=ahv.MATH_TC, workspace=ws)
    stats = ahv.ops.verify_screen_stats(ws, B, N)
    scores, sval, sidx, sRb = ahv.ops.verify(*args, k=1, idx_offset=idx_offset, math=ahv.MATH_TC, return_scores=True)
    torch.cuda.synchronize()
    return (val, idx, Rb), (sval, sidx, sRb), stats, scores


def _assert_equal(got, want):
    for g, w in zip(got, want):
        assert torch.equal(g, w)


def _golden_weights(golden):
    return [torch.from_numpy(golden["weights"][k]) for k in ("W1", "W2", "b2")]


def test_bench_workload(ahv):
    W1, W2, b2, vs, vt, normals = _bench_inputs(32, 50000)
    R = ahv.ops.rotations_from_normals(normals.to(DEV))
    got, want, stats, scores = _verify(ahv, (W1, W2, b2), vs, vt, R)
    assert stats is not None
    flagged, count, err = stats
    _assert_equal(got, want)
    assert torch.equal(want[1][:, 0], scores.argmax(dim=1))
    assert bool((count >= 1).all()) and bool((count <= 224).all())
    assert flagged == 0 and float(err.max()) <= 0.5e-3


def test_per_pair_rotations_and_index_offset(ahv, golden):
    B, N = 8, 40000
    gen = torch.Generator().manual_seed(11)
    vs = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    vt = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    R = ahv.so3.sample_rotations(B * N, seed=3, device=DEV).reshape(B, N, 3, 3).contiguous()
    got, want, stats, _ = _verify(ahv, _golden_weights(golden), vs, vt, R, idx_offset=12345)
    assert stats is not None and stats[0] == 0
    _assert_equal(got, want)


def test_duplicated_rotations_tie_to_lowest_index(ahv, golden):
    B, N = 8, 40000
    gen = torch.Generator().manual_seed(12)
    vs = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    vt = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    R0 = ahv.so3.sample_rotations(N // 4, seed=4, device=DEV)
    R = R0.repeat(4, 1, 1).contiguous()                          # rotation n == n + N/4 == n + N/2 == ...
    got, want, stats, scores = _verify(ahv, _golden_weights(golden), vs, vt, R)
    assert stats is not None
    _assert_equal(got, want)
    assert bool((got[1] < N // 4).all())
    assert torch.equal(scores[:, : N // 4], scores[:, N // 4: N // 2])


def test_zero_source_volume_falls_back_to_index_zero(ahv, golden):
    B, N = 8, 40000
    gen = torch.Generator().manual_seed(13)
    vs = torch.zeros(B, 16, 8, 8, 8)
    vt = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    R = ahv.so3.sample_rotations(N, seed=5, device=DEV)
    got, want, stats, _ = _verify(ahv, _golden_weights(golden), vs, vt, R, idx_offset=7)
    assert stats is not None
    flagged, count, _ = stats
    assert flagged == B and bool((count == N).all())           # every hypothesis ties: overflow, then the exact pass
    _assert_equal(got, want)
    assert bool((got[1] == 7).all())


def test_outlier_volume_beyond_the_16bit_range_trips_the_guard(ahv, golden):
    B, N, r = 8, 40000, 1e9
    gen = torch.Generator().manual_seed(14)
    vs, vt = torch.randn(B, 16, 8, 8, 8, generator=gen), torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    pos = torch.randperm(16 * 512, generator=gen)[: 2 * B].reshape(B, 2)
    flat = vs.view(B, -1)
    flat[torch.arange(B), pos[:, 0]] = r / 3
    flat[torch.arange(B), pos[:, 1]] = -r
    R = ahv.so3.sample_rotations(N, seed=6, device=DEV)
    got, want, stats, _ = _verify(ahv, _golden_weights(golden), vs, vt, R)
    assert stats is not None and stats[0] >= 1
    _assert_equal(got, want)


def test_small_call_stays_on_the_single_pass(ahv, golden):
    assert ahv.ops.verify_screen_stats(None, 1, 3000) is None
    assert ahv.ops.verify_screen_stats(None, 32, 20000) is None   # the lists would not fit the workspace
    g = golden["shared_n3000_b3"]
    T = torch.from_numpy
    got, want, stats, _ = _verify(ahv, _golden_weights(golden), T(g["vol_src"]), T(g["vol_tgt"]), T(g["R"]))
    assert stats is None
    _assert_equal(got, want)


def _worker(rank, world, port, out_q):
    sys.path.insert(0, ROOT)
    import importlib

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    ahv = importlib.import_module("3dahv_b200")
    W1, W2, b2, vs, vt, normals = _bench_inputs(16, 2 * 40000)
    T = lambda t: t.to(dev)
    v = ahv.HypothesisVerifier(T(W1), T(W2), T(b2))
    R = ahv.ops.rotations_from_normals(T(normals))
    lo, hi = ahv.dist.shard_bounds(R.shape[0], rank, world)
    peer = ahv.dist.PeerExchange(16, dev, max_k=1)
    ws = torch.empty(ahv.ops.workspace_bytes(16, hi - lo, 1), dtype=torch.uint8, device=dev)
    got = ahv.ops.verify_sharded(T(vs), T(vt), R[lo:hi].contiguous(), v.W1, v.W2, v.b2, lo, peer, k=1, workspace=ws)
    stats = ahv.ops.verify_screen_stats(ws, 16, hi - lo)
    single = v.score(T(vs), T(vt), R, k=1, return_scores=True)
    torch.cuda.synchronize()
    out_q.put((rank, [t.cpu() for t in got], [t.cpu() for t in (single.topk_val, single.topk_idx, single.R_best)],
               stats is not None))
    dist.barrier()
    peer.close()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_peer_form():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, 29641, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = dict((r, rest) for r, *rest in (q.get(timeout=600) for _ in range(world)))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank in range(world):
        got, want, was_screened = res[rank]
        assert was_screened
        for g, w in zip(got, want):
            assert torch.equal(g, w)
