#!/usr/bin/env python
"""Benchmark of the 3DAHV hypothesis-and-verification hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Metric (BASELINE.json): rotation hypotheses scored per second x pairs.
Workload at any N: BASELINE config 2 per GPU — CO3D shape, B=32 pairs, 50 000
hypotheses (test_co3d.py:212), fp32 volumes, one shared rotation set.  With N>1
each rank scores its own 50 000-hypothesis shard of an N x 50 000 set for all 32
pairs (weak scaling); the scoring kernels exchange and merge the per-rank winners
over NVLink peer memory inside the timed step (`--collective nccl`: NCCL
all-gather + merge kernel).  After the timed loop the exchanged winners are
checked against an unsharded recompute on rank 0 (`sharded_parity`), and a
`strong` sub-record reports BASELINE config 3 (128 pairs, bf16 volumes, ONE
50 000 set sharded over the ranks) and the B=1 x 50 000 step latency, so the
driver's per-N files carry the strong-scaling curve as well.

A step = target features (forward_3d2d on the 32 target volumes) + fused
score kernel + top-k (+ all-gather/merge) + gather of the winning rotations.
`value` is timed with CUDA events on resident inputs, L2 flushed between
steps; `e2e` goes through the host-buffer C-ABI entry (ahv_predict_host_ex; at
N>1 the sharded form, exchange included) with H2D/D2H inside the timed region.  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PAIRS, HYPS, TOPK = 32, 50000, 1
METRIC, UNIT = "rotation hypotheses scored/sec (x pairs)", "hyp*pairs/s"
GATHER_BYTES_PER_HYP = 512 * 8 * 16 * 4      # SURVEY.md §8d: 262 144 B of smem gather per hypothesis (fp32)
FLOP_PER_HYP = 1_843_200                     # SURVEY.md §8d
HBM_BYTES_PER_HYP = 40                       # 36 B rotation in + 4 B score out
DUMP_LIMIT_BYTES = 64_000_000                # --dump-outputs writes at most this much


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "bf16_tflops": d.get("bf16_tflops", 1590.0),
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", 1400.0),
                "sm_max_mhz": d.get("sm_max_mhz", 1965.0), "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0,
            "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the score kernel, per launch, from the committed
    `ncu --set full` capture of this same workload (profiles/); None if the summary is absent."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_score_tc_summary.csv")))
    if not files:
        return None
    rd = wr = None
    for row in csv.reader(l for l in open(files[-1]) if not l.startswith("#")):
        if len(row) >= 4 and row[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(row[1], 1.0)
            v = float(row[-1]) * scale
            rd, wr = (v, wr) if row[0].endswith("read.sum") else (rd, v)
    return None if rd is None or wr is None else rd + wr


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6), ("sw_power_cap", 7)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_inputs(torch, pairs, hyps, seed=0):
    """Random-init head of the named architecture (Conv2d 384->32 no bias, ReLU,
    Conv2d 32->32; PyTorch default init, modules/modules.py:66-70), Gaussian
    volumes with the statistics forward_2d3d produces, restated random_rotations
    from torch's CPU generator (SURVEY.md §8d)."""
    torch.manual_seed(seed)
    head = torch.nn.Sequential(torch.nn.Conv2d(384, 32, 1, bias=False), torch.nn.ReLU(), torch.nn.Conv2d(32, 32, 1))
    W1 = head[0].weight.detach().reshape(32, 384).clone()
    W2 = head[2].weight.detach().reshape(32, 32).clone()
    b2 = head[2].bias.detach().clone()
    vol_src = torch.randn(pairs, 16, 8, 8, 8) * 1.12 - 0.18
    vol_tgt = torch.randn(pairs, 16, 8, 8, 8) * 1.12 - 0.18
    normals = torch.randn(hyps, 4)
    return W1, W2, b2, vol_src, vol_tgt, normals


def cpu_reference_rate(torch, sample_pairs, sample_hyps, steps=1, warmup=0):
    """The reference's PyTorch CPU path (restated in oracle/ahv_oracle.py with the
    same ATen calls) on all host threads, on a bounded sample of the workload.  Also returns what the last step
    computed, named as the product arm's outputs, plus the scores."""
    from oracle import ahv_oracle as orc

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    W1, W2, b2, vs, vt, normals = synthetic_inputs(torch, sample_pairs, sample_hyps)
    R = orc.rotations_from_normals_torch(normals)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        s = orc.score_torch(vs, vt, R, W1, W2, b2)
        best = torch.max(s, dim=1)
        R_best = R[best.indices]
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    per_step = sum(times) / len(times)
    last = {"topk_val": best.values[:, None].float(), "topk_idx": best.indices[:, None].double(),
            "R_best": R_best[:, None].float(), "scores": s.float()}
    return {"value": sample_pairs * sample_hyps / per_step, "unit": UNIT, "cores": cores, "kind": "port",
            "threads": torch.get_num_threads(),
            "sample": f"{sample_pairs} pairs x {sample_hyps} hypotheses of the config-2 workload, "
                      f"oracle.score_torch (F.affine_grid/F.grid_sample/conv1x1/normalize, the reference's ATen calls), "
                      f"{per_step:.2f} s per pass"}, per_step, last


def run_reference(args):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sp, sh = 2, 10000
    base, per_step, last = cpu_reference_rate(torch, sp, sh, steps=max(1, args.steps), warmup=min(args.warmup, 1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": per_step * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # same workload as the product arm; each timed step scores a bounded sample of it on the host cores
            "config": {"workload": (f"CO3D config 2 (BASELINE.json configs[1]): B={PAIRS} pairs x N={HYPS} hypotheses per GPU, "
                                    f"fp32 volumes, shared rotation set, top-1; N>1 = weak scaling over hypothesis shards "
                                    f"+ in-kernel NVLink exchange of the winners"), "pairs": PAIRS, "hypotheses_per_gpu": HYPS,
                       "math": "reference ATen calls on the host CPU", "sample_per_step": f"{sp} pairs x {sh} hypotheses"},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def _events(torch, n):
    return [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]


def dump_outputs(out_dir, tensors, limit_bytes=DUMP_LIMIT_BYTES):
    """Write each tensor as out_dir/<name>.npy, so that two builds run with the same arguments (hence the same seeded
    inputs) can be compared output for output.  The tensors share their leading (pair) axis; when together they
    exceed `limit_bytes`, a fixed seeded sample of pairs is written instead and its pair numbers go to rows.npy."""
    import numpy as np

    arrays = {name: t.cpu().numpy() for name, t in tensors.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > limit_bytes:
        pairs = next(iter(arrays.values())).shape[0]
        keep = max(1, (limit_bytes - 4096) * pairs // (total + 8 * pairs))    # 8 B for each row number, 4 KiB for headers
        rows = np.sort(np.random.default_rng(0).choice(pairs, keep, replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def gpu_eager_rate(torch, dev, sample_pairs, sample_hyps):
    """Informational (SURVEY.md TL;DR bar ii): the reference's own ATen calls (oracle.score_torch: F.affine_grid /
    F.grid_sample / conv1x1 / normalize, then torch.max) executed eagerly ON THE B200, on a bounded sample."""
    from oracle import ahv_oracle as orc

    W1, W2, b2, vs, vt, normals = synthetic_inputs(torch, sample_pairs, sample_hyps)
    R = orc.rotations_from_normals_torch(normals).to(dev)
    W1, W2, b2, vs, vt = (t.to(dev) for t in (W1, W2, b2, vs, vt))

    def once():
        s = orc.score_torch(vs, vt, R, W1, W2, b2)
        best = torch.max(s, dim=1)
        return R[best.indices]

    once()
    torch.cuda.synchronize()
    a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        once()
    b_.record()
    torch.cuda.synchronize()
    per = a.elapsed_time(b_) * 1e-3 / 3
    return {"value": sample_pairs * sample_hyps / per, "unit": UNIT,
            "what": "the reference's ATen calls (oracle.score_torch) run eagerly on this GPU, cuDNN/cuBLAS defaults",
            "sample": f"{sample_pairs} pairs x {sample_hyps} hypotheses, {per * 1e3:.1f} ms per pass"}


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the 3DAHV hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    ahv = importlib.import_module("3dahv_b200")
    lib = ahv._lib.lib()
    math = {"tc": ahv.MATH_TC, "fp32": ahv.MATH_FP32}[args.math]
    steps, warmup = args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)    # > 126 MB L2
    peer = None
    if world > 1 and args.collective == "peer":
        try:
            peer = ahv.dist.PeerExchange(max(128, args.pairs), dev, max_k=1)
        except RuntimeError as e:   # raised on every rank together: fall back to NCCL all-gather + merge
            if rank == 0:
                print(f"[bench] {e}", file=sys.stderr)

    def timed(step_fn, n_steps, n_warm):
        """W untimed steps, then K steps each bracketed by CUDA events on the launching stream with the L2 flushed
        (untimed) in between; barrier + synchronize on both sides.  Returns the MAX over ranks of the summed step
        times and what the last timed step returned."""
        out = None
        for _ in range(n_warm):
            out = step_fn()
        barrier()
        ev = _events(torch, n_steps)
        for a, b_ in ev:
            flush.zero_()
            a.record()
            out = step_fn()
            b_.record()
        barrier()
        return max_over_ranks(sum(a.elapsed_time(b_) for a, b_ in ev))[0], out

    def make_step(verifier, vs, vt, R, B, N, shard_lo, k=1):
        ws = verifier._workspace(B, N, k, dev)
        if world == 1:   # ahv_verify: target-feature prologue + fused score/arg-max/selection = 2 launches
            def step():
                r = verifier.score(vs, vt, R, k=k, return_scores=False, idx_offset=0, gather=True)
                return r.topk_val, r.topk_idx, r.R_best
            return step, 2
        if peer is not None and math != ahv.MATH_FP32:
            # the scoring kernels exchange and merge their winners over NVLink peer memory: still 2 launches
            def step():
                return ahv.ops.verify_sharded(vs, vt, R, verifier.W1, verifier.W2, verifier.b2, shard_lo, peer, k=k, math=math,
                                              workspace=ws)
            return step, 2

        def step():
            r = verifier.score(vs, vt, R, k=k, return_scores=False, idx_offset=shard_lo, gather=False)
            vals, idxs = ahv.dist.all_gather_topk(r.topk_val, r.topk_idx)
            val, idx = ahv.ops.topk_merge(vals, idxs)
            own = (idx >= shard_lo) & (idx < shard_lo + N)
            Rb = ahv.ops.gather_rotations(R, torch.where(own, idx, torch.full_like(idx, shard_lo)), shard_lo)
            Rb = Rb * own[..., None, None]           # the owner contributes the rotation, everyone else exact zeros
            dist.all_reduce(Rb)
            return val, idx, Rb
        return step, 4                     # + merge + winner gather (NCCL and torch kernels not counted)

    # ------------------------------------------------------------------ headline: config 2, weak scaling ----
    B, N, k = args.pairs, args.hyps, TOPK
    if args.config == 3:   # explicit --config 3: the strong-scaling workload as the headline line
        B = 128 if args.pairs == PAIRS else args.pairs
        lo, hi = ahv.dist.shard_bounds(args.hyps, rank, world)
        N, shard_lo = hi - lo, lo
        W1, W2, b2, vs_h, vt_h, normals_all = synthetic_inputs(torch, B, args.hyps)
        vs_h = vs_h.bfloat16()
    else:
        W1, W2, b2, vs_h, vt_h, normals_all = synthetic_inputs(torch, B, N * world)
        shard_lo = rank * N            # this rank's shard of the N*world rotation set
    strong_headline = args.config == 3
    normals_h = normals_all[shard_lo:shard_lo + N].contiguous()
    verifier = ahv.HypothesisVerifier(W1.to(dev), W2.to(dev), b2.to(dev), math=math)
    vs, vt = vs_h.to(dev), vt_h.to(dev)
    R = ahv.ops.rotations_from_normals(normals_h.to(dev))
    step, launches_per_step = make_step(verifier, vs, vt, R, B, N, shard_lo)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms, last = timed(step, steps, warmup)
    n_launch = launches_per_step * steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"topk_val": last[0].float(), "topk_idx": last[1].double(), "R_best": last[2].float()})

    # ------------------------------------------------ sharded parity: the exchange's winners vs an unsharded recompute
    sharded_parity = None
    if world > 1:
        val, idx, Rb = step()
        val, idx, Rb = val.reshape(B, -1)[:, 0], idx.reshape(B, -1)[:, 0], Rb.reshape(B, -1, 3, 3)[:, 0]
        packed = torch.cat([val.view(torch.int32).long(), idx, Rb.reshape(B, 9).contiguous().view(torch.int32).long().flatten()])
        every = [torch.empty_like(packed) for _ in range(world)]
        dist.all_gather(every, packed)            # outside the timed region
        ranks_identical = all(torch.equal(every[0], e) for e in every)
        ok = None
        if rank == 0:   # the WHOLE set on one GPU, no sharding, no exchange: ahv_verify on all world*N hypotheses
            R_full = ahv.ops.rotations_from_normals(normals_all.to(dev))
            full = verifier.score(vs, vt, R_full, k=1, return_scores=False, idx_offset=0, gather=True)
            ok = (torch.equal(full.topk_val[:, 0], val) and torch.equal(full.topk_idx[:, 0], idx)
                  and torch.equal(full.R_best[:, 0], Rb) and torch.equal(Rb, R_full[idx]))
            del R_full
        sharded_parity = {"ok": bool(ok) and ranks_identical if rank == 0 else None, "pairs_checked": B,
                          "hypotheses_unsharded": int(normals_all.shape[0]), "ranks_bit_identical": ranks_identical,
                          "checked": "(score, global index, rotation) of the in-kernel NVLink exchange == ahv_verify over the "
                                     "unsharded set on rank 0, bit for bit, all pairs"}
        if peer is not None:
            peer.check()
        barrier()

    # ------------------------------------------------ dominant kernel alone: score kernel, no selection (k=0)
    tgt = verifier.target_features(vt)
    ws = torch.empty(max(ahv.ops.workspace_bytes(B, N, 1), 16), dtype=torch.uint8, device=dev)
    kev = _events(torch, steps)
    for a, b_ in kev:
        flush.zero_()
        a.record()
        ahv.ops.score(vs, tgt, R, verifier.W1, verifier.W2, verifier.b2, k=0, math=math, return_scores=False, workspace=ws)
        b_.record()
    torch.cuda.synchronize()
    kernel_ms = max_over_ranks(sum(a.elapsed_time(b_) for a, b_ in kev) / steps)[0]
    clocks = sampler.stop() if rank == 0 else None

    # ------------------------------------------------ e2e: HOST buffers through the C ABI, copies inside the timed region
    # (N > 1: every rank passes its host slice of the rotation set; the kernels exchange the winners; the result is
    # the selection over the whole set on every rank's host)
    session = ahv.ops.HostSession(dev)
    vs_p, vt_p = vs_h.pin_memory(), vt_h.pin_memory()
    R_p = R.cpu().pin_memory()
    e2e_peer = peer if (world > 1 and peer is not None and math != ahv.MATH_FP32) else None

    def e2e_step():
        if world > 1 and e2e_peer is None:   # NCCL fallback: host entry on the shard, then all-gather + merge on the device
            _, v_h, i_h, _ = ahv.ops.predict_host(vs_p, vt_p, R_p, W1, W2, b2, k=k, math=math, device=dev, session=session,
                                                  idx_offset=shard_lo)
            vals, idxs = ahv.dist.all_gather_topk(v_h.to(dev), i_h.to(dev))
            v2, i2 = ahv.ops.topk_merge(vals, idxs)
            return v2.cpu(), i2.cpu()
        return ahv.ops.predict_host(vs_p, vt_p, R_p, W1, W2, b2, k=k, math=math, device=dev, session=session,
                                    idx_offset=shard_lo, peer=e2e_peer)

    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_out = e2e_step()
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)[0]
    session.close()
    h2d = vs_p.numel() * vs_p.element_size() + vt_p.numel() * 4 + R_p.numel() * 4 + (32 * 384 + 32 * 32 + 32 + 8) * 4
    d2h = B * k * (4 + 8 + 36)

    # ------------------------------------------------ strong scaling (every N, N = 1 included so the driver's SCALE
    # file holds the curve): config 3 = 128 pairs, bf16 volumes, ONE 50 000-hypothesis set sharded over the ranks;
    # and the B = 1 x 50 000 step latency (p50 of 100 CUDA-graph replays in lockstep), exchange inside the kernel
    strong = None
    if not strong_headline and not args.no_strong:
        try:
            sB, sN = 128, HYPS
            slo, shi = ahv.dist.shard_bounds(sN, rank, world)
            sW1, sW2, sb2, svs_h, svt_h, snorm = synthetic_inputs(torch, sB, sN, seed=3)
            sver = ahv.HypothesisVerifier(sW1.to(dev), sW2.to(dev), sb2.to(dev), math=math)
            svs, svt = svs_h.bfloat16().to(dev), svt_h.to(dev)
            sR = ahv.ops.rotations_from_normals(snorm[slo:shi].contiguous().to(dev))
            sstep, _ = make_step(sver, svs, svt, sR, sB, shi - slo, slo)
            c3_ms = timed(sstep, steps, warmup)[0] / steps
            strong = {"config3": {"workload": f"BASELINE configs[2]: B={sB} pairs, bf16 volumes, ONE set of {sN} hypotheses sharded "
                                              f"over {world} GPU(s), top-1, exchange inside the scoring kernel",
                                  "ms_per_step": c3_ms, "value": sB * sN / (c3_ms * 1e-3), "unit": UNIT, "scaling": "strong"}}
            if world > 1:   # check this workload's sharded result as well
                val3, idx3, _ = sstep()
                if rank == 0:
                    R3 = ahv.ops.rotations_from_normals(snorm.to(dev))
                    f3 = sver.score(svs, svt, R3, k=1, return_scores=False)
                    strong["config3"]["sharded_parity"] = bool(torch.equal(f3.topk_idx, idx3.reshape(sB, -1)[:, :1])
                                                               and torch.equal(f3.topk_val, val3.reshape(sB, -1)[:, :1]))
                barrier()
            gpeer = peer if (world > 1 and peer is not None and math != ahv.MATH_FP32) else None
            if world == 1 or gpeer is not None:
                gv = ahv.GraphedVerifier(sver, 1, shi - slo, k=1, device=dev, peer=gpeer, idx_offset=slo)
                gv(svs[:1].float(), svt[:1], sR)
                for _ in range(10):
                    gv()
                barrier()
                lev = _events(torch, 100)
                for a, b_ in lev:
                    a.record(); gv(); b_.record()
                barrier()
                p50 = statistics.median(a.elapsed_time(b_) for a, b_ in lev) * 1e3
                strong["b1_n50000_latency"] = {"p50_us": max_over_ranks(p50)[0], "calls": 100,
                                               "what": f"B=1 pair, {sN} hypotheses sharded over {world} GPU(s), whole step "
                                                       f"(target features + scoring + selection + exchange) as one CUDA-graph "
                                                       f"replay, max over ranks of the per-rank median"}
        except Exception as e:  # noqa: BLE001   informational: must never cost the run its JSON line
            strong = {"error": repr(e)}
            if world > 1:
                raise   # ranks out of lockstep cannot continue safely

    # ------------------------------------------------ informational sections on rank 0 (no exchange below this line)
    other, latency, eager, training = {}, {}, None, {}
    smem_peak_gbs = None
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    if rank == 0:
        def _rate(src, m):
            for _ in range(2):
                ahv.ops.score(src, tgt, R, verifier.W1, verifier.W2, verifier.b2, k=0, math=m, return_scores=False, workspace=ws)
            a2, b2_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a2.record()
            for _ in range(3):
                ahv.ops.score(src, tgt, R, verifier.W1, verifier.W2, verifier.b2, k=0, math=m, return_scores=False, workspace=ws)
            b2_.record()
            torch.cuda.synchronize()
            return B * N * 3 / (a2.elapsed_time(b2_) * 1e-3)
        if not strong_headline:
            try:   # other arithmetic modes on the same workload (the headline stays fp32 volumes + AHV_MATH_TC)
                other["bf16_volumes_tc"] = _rate(vs.bfloat16(), ahv.MATH_TC)
                other["fp32_volumes_tc_f16gather"] = _rate(vs, ahv.MATH_TC_F16GATHER)
            except Exception as e:  # noqa: BLE001
                other["error"] = repr(e)

        # training variant (SURVEY.md §8f-3): scores + InfoNCE forward/backward on the reference's training shape
        # (12 pairs x 9 000 per-pair hypotheses, ground truth first), p50 of 7 steps after 2 warm-ups, three backward forms
        if not strong_headline and world == 1 and not args.no_train:
            try:
                Bt, Nt = 12, 9000
                tW1, tW2, tb2, tvs, tvt, _ = synthetic_inputs(torch, Bt, 16)
                leaves = [x.to(dev).requires_grad_(True) for x in (tvs, tvt, tW1, tW2, tb2)]
                gt_t = ahv.so3.sample_rotations(Bt, 1, 0, dev)
                Rs_t = torch.cat([gt_t[:, None], ahv.so3.sample_rotations(Bt * (Nt - 1), 2, 0, dev).reshape(Bt, Nt - 1, 3, 3)], 1).contiguous()
                for name, kw in (("exact_fp32_backward", {}), ("saved_h1_fp32_backward", {"save_activations": True, "tc_backward": False}),
                                 ("saved_h1_tcgen05_backward", {"save_activations": True})):
                    ms = []
                    for i in range(9):
                        for x in leaves:
                            x.grad = None
                        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        ea.record()
                        sc = ahv.training.verification_scores(leaves[0], leaves[1], Rs_t, *leaves[2:], **kw)
                        ahv.training.infonce_loss(sc, Rs_t, gt_t, acc_thr_deg=15.0).mean().backward()
                        eb.record()
                        torch.cuda.synchronize()
                        if i >= 2:
                            ms.append(ea.elapsed_time(eb))
                    training[name] = {"ms_per_step_p50": sorted(ms)[len(ms) // 2]}
                training["shape"] = f"{Bt} pairs x {Nt} per-pair hypotheses; scores + InfoNCE + gradients to volumes and head weights"
                del leaves, Rs_t, sc
            except Exception as e:  # noqa: BLE001
                training["error"] = repr(e)

        # measured shared-memory read peak (no such figure in MEASURED_PEAKS.json)
        import ctypes
        nbytes = ctypes.c_ulonglong(0)
        out = torch.zeros(2 * sms, device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        lib.ahv_diag_smem_read(out.data_ptr(), 2 * sms, 200, ctypes.byref(nbytes), st)
        torch.cuda.synchronize()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        lib.ahv_diag_smem_read(out.data_ptr(), 2 * sms, 4000, ctypes.byref(nbytes), st)
        b_.record()
        torch.cuda.synchronize()
        smem_peak_gbs = nbytes.value / (a.elapsed_time(b_) * 1e-3) / 1e9

        # p50 per-pair latency, B=1 on ONE GPU (SURVEY.md §8d): CUDA-graph replay of the whole step, CUDA events
        if not strong_headline:
            for n_lat in (3000, 50000):
                try:
                    gv = ahv.GraphedVerifier(verifier, 1, n_lat, k=1, device=dev)
                    R_lat = R[:n_lat] if N >= n_lat else ahv.so3.sample_rotations(n_lat, 1, 0, dev)
                    gv(vs[:1].float(), vt[:1], R_lat)
                    for _ in range(10):
                        gv()
                    lev = _events(torch, 100)
                    for a, b_ in lev:
                        a.record(); gv(); b_.record()
                    torch.cuda.synchronize()
                    latency[f"N={n_lat}"] = {"p50_us": statistics.median(a.elapsed_time(b_) for a, b_ in lev) * 1e3, "calls": 100}
                except Exception as e:  # noqa: BLE001
                    latency[f"N={n_lat}"] = {"error": repr(e)}
            try:   # the same replay in the opt-in 16-bit-gather mode
                vfast = ahv.HypothesisVerifier(verifier.W1, verifier.W2, verifier.b2, math=ahv.MATH_TC_F16GATHER)
                gv = ahv.GraphedVerifier(vfast, 1, 3000, k=1, device=dev)
                gv(vs[:1].float(), vt[:1], R[:3000] if N >= 3000 else ahv.so3.sample_rotations(3000, 1, 0, dev))
                for _ in range(10):
                    gv()
                lev = _events(torch, 100)
                for a, b_ in lev:
                    a.record(); gv(); b_.record()
                torch.cuda.synchronize()
                latency["N=3000, AHV_MATH_TC_F16GATHER"] = {"p50_us": statistics.median(a.elapsed_time(b_) for a, b_ in lev) * 1e3, "calls": 100}
            except Exception as e:  # noqa: BLE001
                latency["extra_error"] = repr(e)
        if world == 1 and not args.no_cpu:
            try:
                eager = gpu_eager_rate(torch, dev, 2, 10000)
            except Exception as e:  # noqa: BLE001
                eager = {"error": repr(e)}

    if rank == 0:
        peaks = load_peaks()
        units_per_step = B * args.hyps if strong_headline else B * N * world
        value = units_per_step * steps / (total_ms * 1e-3)
        hyp_per_s_kernel = B * N / (kernel_ms * 1e-3)              # one GPU's kernel
        gather_bytes = GATHER_BYTES_PER_HYP // 2 if strong_headline else GATHER_BYTES_PER_HYP   # 16-bit staged volume: 256 B per voxel sample
        gather_gbs = hyp_per_s_kernel * gather_bytes / 1e9
        nominal_smem = sms * 128 * peaks["sm_max_mhz"] * 1e6 / 1e9
        collective = ("none (1 GPU)" if world == 1 else "peer memory, fused into the scoring kernel" if e2e_peer is not None
                      else "NCCL all-gather + merge kernel")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": total_ms / steps, "higher_is_better": True,
            "scaling": "strong" if strong_headline else "weak", "vs_baseline": None, "dtype": "bf16 volumes" if strong_headline else "f32",
            "data": "synthetic",
            "dtype_detail": "fp32 volumes, trilinear gather / normalise / correlate in fp32; the two 1x1 convs use fp16 "
                            "operands (10-bit mantissa, TF32-equivalent) with fp32 accumulation on tcgen05; scores within "
                            "1.3e-4 relative of the reference's fp32 CPU path (gate 1e-3)",
            "config": {"workload": (f"Objaverse config 3 (BASELINE.json configs[2]): B={B} pairs, bf16 volumes, one set of "
                                    f"{args.hyps} hypotheses sharded over {world} GPU(s)") if strong_headline else
                                   (f"CO3D config 2 (BASELINE.json configs[1]): B={B} pairs x N={N} hypotheses per GPU, "
                                    f"fp32 volumes, shared rotation set, top-{k}; N>1 = weak scaling over hypothesis shards "
                                    f"+ in-kernel NVLink exchange of the winners"), "pairs": B, "hypotheses_per_gpu": N, "math": args.math,
                       "collective": collective,
                       "l2": "flushed between timed steps (256 MiB memset, untimed)"},
            "voxel_samples_per_s": value * 512,
            "clocks": clocks,
            "latency_p50_per_pair": latency,
            "other_modes_hyp_pairs_per_s": other,
            "training_step": training,
            "e2e": {"value": units_per_step * steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h,
                    "api": ("ahv_predict_host_ex (C ABI, pinned host buffers, caller-owned session)" +
                            ("; every rank passes its host slice, the kernels exchange the winners over NVLink, every rank's "
                             "host receives the selection over the whole set" if e2e_peer is not None else
                             "; per-shard selection merged by NCCL all-gather + merge kernel" if world > 1 else ""))},
            "gpu_launches": n_launch,
            "roofline": {
                "bound": "smem", "kernel": "score (fused rotate+head+correlate)", "achieved": gather_gbs,
                "peak": smem_peak_gbs, "unit": "GB/s", "frac": gather_gbs / smem_peak_gbs,
                "peak_source": "measured in this run (ahv_diag_smem_read, conflict-free LDS.128)",
                "nominal_peak": nominal_smem, "kernel_ms": kernel_ms, "traffic": ncu_traffic(), "traffic_note": "DRAM bytes per launch from the committed ncu --set full capture (profiles/); algorithmic HBM bytes per launch = %d" % (HBM_BYTES_PER_HYP * B * N),
                "algorithmic_bytes_per_unit": gather_bytes,
                "alt": {
                    "hbm": {"achieved": hyp_per_s_kernel * HBM_BYTES_PER_HYP / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": hyp_per_s_kernel * HBM_BYTES_PER_HYP / 1e9 / peaks["hbm_gbs"]},
                    "tensor": {"achieved": hyp_per_s_kernel * FLOP_PER_HYP / 1e12, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                               "frac": hyp_per_s_kernel * FLOP_PER_HYP / 1e12 / peaks["bf16_tflops"]},
                    "peaks": peaks["source"]},
            },
        }
        if sharded_parity is not None:
            line["sharded_parity"] = sharded_parity["ok"]
            line["sharded_parity_detail"] = sharded_parity
        if strong is not None:
            line["strong"] = strong
        if eager is not None:
            line["gpu_eager_baseline"] = eager
        if world == 1 and not args.no_cpu:
            base, _, _ = cpu_reference_rate(torch, 2, 10000)
            line["cpu_baseline"] = base
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        if peer is not None:
            peer.close()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--collective", choices=["peer", "nccl"], default="peer",
                    help="N>1: winners exchanged by the scoring kernels through NVLink peer memory (default) or "
                         "NCCL all-gather + merge kernel")
    ap.add_argument("--math", choices=["tc", "fp32"], default=os.environ.get("AHV_BENCH_MATH", "tc"))
    ap.add_argument("--pairs", type=int, default=PAIRS)
    ap.add_argument("--hyps", type=int, default=HYPS)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline and gpu_eager_baseline legs")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling sub-record (config 3, B=1 latency)")
    ap.add_argument("--no-train", action="store_true", help="skip the training_step sub-record (profiling runs: keeps the launch list to the path)")
    ap.add_argument("--config", type=int, choices=[2, 3], default=2,
                    help="2 (default): BASELINE configs[1], weak scaling; 3: configs[2], bf16 volumes, hypothesis set sharded (strong)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (topk_val, topk_idx, R_best; the reference arm also "
                         "its scores) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
