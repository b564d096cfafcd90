"""GPU: gradient refinement and distinct top-k over a hypothesis set sharded across ranks, exchanged through peer memory.

Every output of `ops.refine_gradient_sharded` (and of `ShardedVerifier.refine_by_gradient`, `.scores()` and the
distinct `.score()`), on every rank, is bit for bit the one-GPU result over the whole set.  On one GPU, two or four
"ranks" live in this process, each with its own exchange buffer (plain device pointers), stream and verifier, as in
test_gpu_parity.py::test_peer_exchange_protocol_on_one_gpu; with two or more GPUs a spawned-process test adds CUDA IPC,
the NCCL composition and CUDA-graph replay."""
import ctypes
import math
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAP_PAIRS, CAP_K, CAP_HYPS = 4, 32, 3000


def _bits(t):
    """int32 view of a float tensor (NaN slots compare too), the tensor itself otherwise."""
    t = t.detach().contiguous()
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _assert_same(got, want, what):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape, (what, i, g.shape, w.shape)
        assert torch.equal(_bits(g), _bits(w)), (what, i)


class _Ranks:
    """`world` in-process ranks on one GPU: exchange buffers with a score region, one stream each."""

    def __init__(self, ahv, world, dev):
        self.ahv, self.world, self.dev = ahv, world, dev
        self.lib = ahv._lib.lib()
        self.bufs = []
        for _ in range(world):
            p = ctypes.c_void_p()
            ahv._lib.check(self.lib.ahv_peer_alloc_ex(CAP_PAIRS, CAP_K, CAP_HYPS, ctypes.byref(p)), "ahv_peer_alloc_ex")
            self.bufs.append(p.value)
        self.peers = [SimpleNamespace(rank=r, world=world, ptrs=self.bufs, max_pairs=CAP_PAIRS, max_k=CAP_K, max_hyps=CAP_HYPS)
                      for r in range(world)]
        self.streams = [torch.cuda.Stream(device=dev) for _ in range(world)]
        self.exchanges = 0

    def run(self, fn, exchanges):
        """fn(rank, peer) on every rank's stream, all enqueued before any is waited for."""
        torch.cuda.synchronize()
        out = [None] * self.world
        for r in range(self.world):
            self.streams[r].wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(self.streams[r]):
                out[r] = fn(r, self.peers[r])
        for s in self.streams:
            s.synchronize()
        self.exchanges += exchanges
        return out

    def check_status(self):
        seq, err = ctypes.c_uint32(), ctypes.c_uint32()
        for r in range(self.world):
            self.ahv._lib.check(self.lib.ahv_peer_status(self.bufs[r], ctypes.byref(seq), ctypes.byref(err)), "ahv_peer_status")
            if err.value != 0:   # a 20 s spin that timed out: the ranks' kernels were not scheduled concurrently
                pytest.skip("the ranks' kernels were not scheduled concurrently on this device")
            assert seq.value == self.exchanges, (r, seq.value, self.exchanges)

    def close(self):
        torch.cuda.synchronize()
        for p in self.bufs:
            self.lib.ahv_peer_free(p)


def _setup(ahv, golden):
    dev = torch.device("cuda", 0)
    g, w = golden["shared_n3000_b3"], golden["weights"]
    T = lambda a: torch.from_numpy(a).to(dev)
    return dev, T(g["vol_src"]), T(g["vol_tgt"]), T(g["R"]), [T(w[k]) for k in ("W1", "W2", "b2")]


def test_sharded_gradient_refinement_equals_one_gpu(ahv, golden):
    dev, vs, vt, R, (W1, W2, b2) = _setup(ahv, golden)
    ops = ahv.ops
    TC, FP32 = ahv.MATH_TC, ahv.MATH_FP32
    Rp = torch.stack([R[b * 900:(b + 1) * 900] for b in range(3)]).contiguous()        # per-pair sets [3,900,3,3]
    Rc = ops.perturb_rotations(R[5:6], 20, 5.0, seed=1).reshape(20, 3, 3).contiguous()  # 20 rotations within 5 deg
    # (world, B, set, k, min_sep_deg, bf16, math); B, k and N change from call to call on the same buffers
    cases = [
        (2, 3, R, 8, 0.0, False, TC), (2, 3, R, 8, 15.0, False, TC), (2, 3, R, 1, 0.0, False, TC),
        (2, 3, R, 32, 30.0, False, TC), (2, 3, Rp, 8, 15.0, False, TC), (2, 3, Rp, 3, 0.0, False, TC),
        (2, 3, R, 8, 30.0, True, TC), (2, 2, R[:1000], 3, 15.0, False, FP32), (2, 3, R[:1000], 32, 0.0, False, FP32),
        (2, 1, Rc, 8, 30.0, False, TC),                           # one winner, seven empty slots
        (4, 3, R[:2999], 3, 15.0, False, TC), (4, 3, R[:2999], 8, 0.0, True, TC),   # N not divisible by world
        (4, 3, R[:7], 3, 0.0, False, TC), (4, 3, R[:7], 3, 30.0, False, TC),        # N < world * k
        (4, 1, R[:5], 1, 30.0, False, TC), (4, 1, R[:5], 1, 0.0, False, FP32),      # k < world: ranks without items
        (4, 2, Rc, 8, 30.0, False, FP32), (4, 3, R, 32, 15.0, False, TC),
    ]
    for world in (2, 4):
        ranks = _Ranks(ahv, world, dev)
        try:
            for cw, B, Rs, k, sep, bf16, math_mode in cases:
                if cw != world:
                    continue
                src = vs[:B].bfloat16() if bf16 else vs[:B]
                RB = Rs[:B] if Rs.dim() == 4 else Rs
                want = ops.refine_gradient(src, vt[:B], RB, W1, W2, b2, k=k, steps=12, step_deg=1.0, math=math_mode,
                                           min_sep_deg=sep)[:8]
                got = ranks.run(lambda r, p: ops.refine_gradient_sharded(src, vt[:B], RB, W1, W2, b2, p, k=k, steps=12,
                                                                         step_deg=1.0, math=math_mode, min_sep_deg=sep)[:8],
                                exchanges=2)
                ranks.check_status()
                what = (world, B, tuple(RB.shape), k, sep, bf16, math_mode)
                for r in range(world):
                    _assert_same(got[r], want, (what, r))
                if Rs is Rc:
                    assert bool((want[1][:, 1:] == -1).all()) and bool(torch.isnan(want[3][:, 1:]).all())
                    assert bool(torch.isneginf(want[4][:, 1:]).all())
        finally:
            ranks.close()


def test_sharded_verifier_scores_and_distinct_score_equal_one_gpu(ahv, golden):
    dev, vs, vt, R, (W1, W2, b2) = _setup(ahv, golden)
    world = 2
    ranks = _Ranks(ahv, world, dev)
    try:
        vers = [ahv.HypothesisVerifier(W1, W2, b2) for _ in range(world)]       # one workspace per rank
        one = ahv.HypothesisVerifier(W1, W2, b2)
        svs = []
        for r in range(world):
            sv = ahv.dist.ShardedVerifier(vers[r], peer=ranks.peers[r])
            sv.rank, sv.world = r, world
            svs.append(sv)
        for N in (3000, 2999, 3):
            want = one.score(vs, vt, R[:N], k=1, return_scores=True).scores
            got = ranks.run(lambda r, p: svs[r].scores(vs, vt, R[:N]), exchanges=1)
            ranks.check_status()
            for r in range(world):
                assert torch.equal(_bits(got[r]), _bits(want)), (N, r)
            # the exchange on its own, on ahv_score(k = 0) slices
            tf = one.target_features(vt)

            def part(r, p, N=N):
                lo, hi = ahv.dist.shard_bounds(N, r, world)
                sl = ahv.ops.score(vs, tf, R[lo:hi], W1, W2, b2, k=0)[0] if hi > lo else torch.zeros(3, 0, device=dev)
                return ahv.ops.scores_exchange(sl, N, p)

            want0 = ahv.ops.score(vs, tf, R[:N], W1, W2, b2, k=0)[0]
            got = ranks.run(part, exchanges=1)
            ranks.check_status()
            for r in range(world):
                assert torch.equal(_bits(got[r]), _bits(want0)), (N, r)
        for k, sep in ((8, 15.0), (32, 30.0), (3, 0.0)):
            w = one.score(vs, vt, R, k=k, min_sep_deg=sep) if sep > 0 else one.score(vs, vt, R, k=k, return_scores=False)
            got = ranks.run(lambda r, p: svs[r].score(vs, vt, R, k=k, min_sep_deg=sep), exchanges=1)
            ranks.check_status()
            for r in range(world):
                _assert_same(got[r], (w.topk_val, w.topk_idx, w.R_best), (k, sep, r))
        for sep in (0.0, 15.0):                                       # the wrapper returns refine_by_gradient's tuple
            bR, bv, first, Ra, sa = one.refine_by_gradient(vs, vt, R, k=8, steps=10, min_sep_deg=sep)
            got = ranks.run(lambda r, p: svs[r].refine_by_gradient(vs, vt, R, k=8, steps=10, min_sep_deg=sep), exchanges=2)
            ranks.check_status()
            for r in range(world):
                gR, gv, gf, gRa, gsa = got[r]
                _assert_same((gR, gv, gf.topk_val, gf.topk_idx, gf.R_best, gRa, gsa),
                             (bR, bv, first.topk_val, first.topk_idx, first.R_best, Ra, sa), (sep, r))
    finally:
        ranks.close()


def test_distinct_selection_is_not_a_merge_of_shard_lists(ahv, golden):
    """x (best) on rank 1; a (second) within theta of x and c (third) within theta of a but farther than theta from x,
    both on rank 0.  Global greedy suppression keeps x and c; NMS on each shard keeps a and drops c on rank 0, and a
    merge of the shard lists can then only give x (a is suppressed by x): c is lost."""
    dev, vs, vt, R, (W1, W2, b2) = _setup(ahv, golden)
    ops = ahv.ops
    one = ahv.HypothesisVerifier(W1, W2, b2)
    theta = 15.0
    tf = one.target_features(vt[:1])
    s0 = ops.score(vs[:1], tf, R, W1, W2, b2, k=0)[0][0]
    x = R[int(torch.argmax(s0))]
    # candidates along geodesics from x: a at 8 deg, c at 20 deg on the same axis (d(a,c) = 12 < theta < d(x,c))
    gen = torch.Generator().manual_seed(0)
    axes = torch.nn.functional.normalize(torch.randn(256, 3, generator=gen), dim=1).to(dev)

    def rot(axis, deg):
        K = torch.zeros(axis.shape[0], 3, 3, device=dev)
        K[:, 0, 1], K[:, 0, 2], K[:, 1, 2] = -axis[:, 2], axis[:, 1], -axis[:, 0]
        K = K - K.transpose(1, 2)
        t = math.radians(deg)
        return (torch.eye(3, device=dev) + math.sin(t) * K + (1 - math.cos(t)) * K @ K) @ x

    A, C = rot(axes, 8.0), rot(axes, 20.0)
    sx = ops.score(vs[:1], tf, x[None].contiguous(), W1, W2, b2, k=0)[0][0, 0]
    sa = ops.score(vs[:1], tf, A.contiguous(), W1, W2, b2, k=0)[0][0]
    sc = ops.score(vs[:1], tf, C.contiguous(), W1, W2, b2, k=0)[0][0]
    ok = torch.nonzero((sx > sa) & (sa > sc)).flatten()
    assert ok.numel() > 0, "no geodesic with decreasing scores found"
    i = int(ok[0])
    Rs = torch.stack([A[i], C[i], x]).contiguous()          # N = 3 over 2 ranks: rank 0 holds a, c; rank 1 holds x
    k = 3
    want = ops.refine_gradient(vs[:1], vt[:1], Rs, W1, W2, b2, k=k, steps=5, min_sep_deg=theta)[:8]
    assert want[1][0].tolist() == [2, 1, -1]                  # x, then c
    shard0 = ops.topk_distinct(ops.score(vs[:1], tf, Rs[:2], W1, W2, b2, k=0)[0], Rs[:2], 2, theta)[1][0].tolist()
    assert shard0 == [0, -1]                                  # rank 0 alone keeps a and suppresses c
    ranks = _Ranks(ahv, 2, dev)
    try:
        got = ranks.run(lambda r, p: ops.refine_gradient_sharded(vs[:1], vt[:1], Rs, W1, W2, b2, p, k=k, steps=5,
                                                                 min_sep_deg=theta)[:8], exchanges=2)
        ranks.check_status()
        for r in range(2):
            _assert_same(got[r], want, r)
    finally:
        ranks.close()


def _worker(rank, world, port, out_q):
    sys.path.insert(0, ROOT)
    import importlib

    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    ahv = importlib.import_module("3dahv_b200")
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "shared_n3000_b3.npz")))
    w = dict(np.load(os.path.join(ROOT, "tests", "golden", "weights.npz")))
    T = lambda a: torch.from_numpy(a).to(dev)
    cpu = lambda ts: tuple(t.cpu() for t in ts)
    W1, W2, b2 = T(w["W1"]), T(w["W2"]), T(w["b2"])
    vs, vt, R = T(g["vol_src"]), T(g["vol_tgt"]), T(g["R"])
    one = ahv.HypothesisVerifier(W1, W2, b2)
    peer = ahv.dist.PeerExchange(4, dev, max_k=32, max_hyps=3000)
    sv_peer = ahv.dist.ShardedVerifier(ahv.HypothesisVerifier(W1, W2, b2), peer=peer)
    sv_nccl = ahv.dist.ShardedVerifier(ahv.HypothesisVerifier(W1, W2, b2))
    flat = lambda o: (o[0], o[1], o[2].topk_val, o[2].topk_idx, o[2].R_best, o[3], o[4])
    out, steps = {}, 0
    for k, sep in ((8, 0.0), (8, 15.0), (32, 30.0), (1, 0.0)):
        out[("one", k, sep)] = cpu(flat(one.refine_by_gradient(vs, vt, R, k=k, steps=10, min_sep_deg=sep)))
        out[("peer", k, sep)] = cpu(flat(sv_peer.refine_by_gradient(vs, vt, R, k=k, steps=10, min_sep_deg=sep)))
        out[("nccl", k, sep)] = cpu(flat(sv_nccl.refine_by_gradient(vs, vt, R, k=k, steps=10, min_sep_deg=sep)))
        steps += 2
    out["scores"] = (sv_peer.scores(vs, vt, R).cpu(), sv_nccl.scores(vs, vt, R).cpu(),
                     one.score(vs, vt, R, k=1, return_scores=True).scores.cpu())
    steps += 1
    # CUDA-graph capture and replay of the one-call chain
    res = None
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(stream):
        res = ahv.ops.refine_gradient_sharded(vs, vt, R, W1, W2, b2, peer, k=8, steps=10, min_sep_deg=15.0)
        steps += 2
    torch.cuda.current_stream(dev).wait_stream(stream)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ahv.ops.refine_gradient_sharded(vs, vt, R, W1, W2, b2, peer, k=8, steps=10, min_sep_deg=15.0, out=res[:8],
                                        workspace=res[8])
    want = ahv.ops.refine_gradient(vs, vt, R, W1, W2, b2, k=8, steps=10, min_sep_deg=15.0)[:8]
    out["graph"] = []
    for _ in range(3):
        for t in res[:8]:
            t.zero_()
        graph.replay()
        torch.cuda.synchronize(dev)
        out["graph"].append((cpu(res[:8]), cpu(want)))
        steps += 2
    out["seq"] = (peer.check(), steps)
    out_q.put((rank, out))
    dist.barrier()
    peer.close()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_gradient_refinement_across_gpus():
    import torch.multiprocessing as mp

    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, 29631, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=900) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank in range(world):
        o = res[rank]
        for key in [k for k in o if isinstance(k, tuple) and k[0] == "one"]:
            _assert_same(o[("peer",) + key[1:]], o[key], ("peer", rank, key))
            _assert_same(o[("nccl",) + key[1:]], o[key], ("nccl", rank, key))
        _assert_same(o["scores"][:2], (o["scores"][2], o["scores"][2]), ("scores", rank))
        for got, want in o["graph"]:
            _assert_same(got, want, ("graph", rank))
        assert o["seq"][0] == o["seq"][1]
