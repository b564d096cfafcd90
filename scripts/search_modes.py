"""Coarse-to-fine search that keeps k distinct modes (ops.search_modes / ahv_search_modes) against the plain search and
the dense 50 000-point grid.  Writes one JSONL file (default profiles/r18_search_modes.jsonl); the card's name and power
limit are read in the same run.  Four kinds of rows:
  time:       search_modes at (2, 4, k, w, 30 deg) for k in {4, 8, 16} and w in {1, 2, 4, 8}, alternated with the plain
              search at (2, 4, 32) and (3, 4, 32) and verify(k = 1) on the 50 000-point grid, for B in {1, 8, 32}; every
              call captured in a CUDA graph and timed with CUDA events around single replays, three rounds of 10 replays
              per call taken in turn (median of the 30, after 5 warm-up replays);
  kernels:    torch.profiler's CUDA time per kernel of one eager search_modes call at (2, 4, 8, 4, 30 deg), B in {1, 8, 32};
  accuracy:   config 4's known-rotation task (8 pairs) and the near-symmetric task (64 pairs), both built as in
              scripts/hierarchical_search.py, under AHV_MATH_TC and AHV_MATH_FP32: geodesic error to R_gt (mean / max) of the
              top-1, of the best of the modes, and of the best score after `ascend` from every non-empty mode;
  robustness: on 256 random synthetic pairs under AHV_MATH_FP32, the fraction where the top-1 score is >= the 50 000-grid
              top-1's, and the number of final mode pairs closer than min_sep / 2.
    python scripts/search_modes.py [out.jsonl]"""
import importlib, json, os, statistics, subprocess, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
ahv = importlib.import_module("3dahv_b200")
ops = ahv.ops
dev = torch.device("cuda", 0)
out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r18_search_modes.jsonl")
N_GRID, STEPS, THETA = 50_000, 20, 30.0
MODES = [(k, w) for k in (4, 8, 16) for w in (1, 2, 4, 8)]
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
rows = []


def emit(row):
    row = {"gpu": gpu, **row}
    rows.append(row)
    print(json.dumps(row), flush=True)


def geodesic_deg(Ra, Rb):
    c = ((Ra.double() * Rb.double()).sum((-1, -2)) - 1) / 2
    return torch.rad2deg(torch.arccos(c.clamp(-1, 1)))


def capture(fn):
    s = torch.cuda.Stream(device=dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        fn()
        fn()
    torch.cuda.current_stream(dev).wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    for _ in range(5):
        g.replay()
    return g


def timed(graphs, rounds=3, per=10):
    """Median single-replay time of each graph, the graphs taken in turn `rounds` times, `per` replays each."""
    times = {name: [] for name in graphs}
    for _ in range(rounds):
        for name, g in graphs.items():
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(per)]
            for a, b in ev:
                a.record(); g.replay(); b.record()
            torch.cuda.synchronize()
            times[name] += [a.elapsed_time(b) for a, b in ev]
    return {name: statistics.median(t) for name, t in times.items()}


grid = ahv.so3.grid_rotations(N_GRID, device=dev)

# ---- time ------------------------------------------------------------------------------------------------------------
for B in (1, 8, 32):
    W1, W2, b2, vs, vt, _ = [t.to(dev) for t in bench.synthetic_inputs(torch, B, 1)]
    graphs, meta = {}, {}
    for k, w in MODES:
        res = ops.search_modes(vs, vt, W1, W2, b2, base_level=2, levels=4, k=k, beam=w, min_sep_deg=THETA)
        graphs[("modes", k, w)] = capture(lambda res=res, k=k, w=w: ops.search_modes(
            vs, vt, W1, W2, b2, base_level=2, levels=4, k=k, beam=w, min_sep_deg=THETA, out=res[:6], workspace=res[6]))
        meta[("modes", k, w)] = {"what": "search_modes", "base_level": 2, "levels": 4, "k": k, "beam": w, "min_sep_deg": THETA,
                                 "hypotheses_per_pair": 72 * 8 ** 2 + 4 * 8 * k * w}
    for base in (2, 3):
        res = ops.search_hierarchical(vs, vt, W1, W2, b2, base_level=base, levels=4, k=32)
        graphs[("plain", base)] = capture(lambda res=res, base=base: ops.search_hierarchical(
            vs, vt, W1, W2, b2, base_level=base, levels=4, k=32, out=res[:6], workspace=res[6]))
        meta[("plain", base)] = {"what": "search", "base_level": base, "levels": 4, "k": 32,
                                 "hypotheses_per_pair": 72 * 8 ** base + 4 * 8 * 32}
    ws = torch.empty(ops.workspace_bytes(B, N_GRID, 1), device=dev, dtype=torch.uint8)
    graphs["grid"] = capture(lambda: ops.verify(vs, vt, grid, W1, W2, b2, k=1, workspace=ws))
    meta["grid"] = {"what": "verify_k1_grid50k", "hypotheses_per_pair": N_GRID}
    ms = timed(graphs)
    for name, t in ms.items():
        emit({"kind": "time", "B": B, **meta[name], "ms": t, "ratio_to_search_2_4_32": t / ms[("plain", 2)]})
    del graphs

# ---- kernels ---------------------------------------------------------------------------------------------------------
from torch.profiler import ProfilerActivity, profile

for B in (1, 8, 32):
    W1, W2, b2, vs, vt, _ = [t.to(dev) for t in bench.synthetic_inputs(torch, B, 1)]
    res = ops.search_modes(vs, vt, W1, W2, b2, base_level=2, levels=4, k=8, beam=4, min_sep_deg=THETA)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            ops.search_modes(vs, vt, W1, W2, b2, base_level=2, levels=4, k=8, beam=4, min_sep_deg=THETA, out=res[:6],
                             workspace=res[6])
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        if e.self_device_time_total > 0:   # kernels and copies (host-side ops carry no device time of their own)
            per[e.key] = {"calls_per_search": e.count / 10, "us_per_search": e.self_device_time_total / 10}
    emit({"kind": "kernels", "B": B, "what": "search_modes", "k": 8, "beam": 4, "min_sep_deg": THETA, "kernels": per})


# ---- accuracy --------------------------------------------------------------------------------------------------------
def config4_task():
    W1, W2, b2, vs, _, _ = bench.synthetic_inputs(torch, 8, 16)
    vs = vs.to(dev)
    R_gt = ahv.so3.sample_rotations(8, seed=123, device=dev)
    return (W1.to(dev), W2.to(dev), b2.to(dev)), vs, ops.rotate_volume(vs, R_gt), R_gt


def symmetric_task(eps=0.1):
    W1, W2, b2, V, A, _ = bench.synthetic_inputs(torch, 64, 1)
    src = (0.5 * (V + V.flip(3, 4)) + eps * A).to(dev).contiguous()
    R_gt = ahv.so3.sample_rotations(64, seed=321, device=dev)
    return (W1.to(dev), W2.to(dev), b2.to(dev)), src, ops.rotate_volume(src, R_gt), R_gt


stat = lambda e: {"mean_deg": float(e.mean()), "max_deg": float(e.max())}


def ascend_modes(v, vs, vt, final):
    """`ascend` from every non-empty mode (an empty one starts at the pair's top-1 instead); the best score's rotation."""
    R0 = torch.where((final.topk_idx >= 0)[..., None, None], final.R_best, final.R_best[:, :1]).contiguous()
    Ra, _, _, _ = v.ascend(vs, vt, R0, steps=STEPS)
    return Ra


for task, (head, vs, vt, R_gt) in (("config4", config4_task()), ("near_symmetric", symmetric_task())):
    for math_name, math in (("tc", ahv.MATH_TC), ("fp32", ahv.MATH_FP32)):
        v = ahv.HypothesisVerifier(*head, math=math)
        for base in (2, 3):
            Rb, _, _, final = v.search(vs, vt, base_level=base, levels=4, k=32)
            emit({"kind": "accuracy", "task": task, "math": math_name, "what": "search", "base_level": base, "levels": 4,
                  "k": 32, "pairs": vs.shape[0], "top1": stat(geodesic_deg(Rb, R_gt)),
                  "best_of_k": stat(geodesic_deg(final.R_best, R_gt[:, None]).min(1).values),
                  "ascend_all": stat(geodesic_deg(ascend_modes(v, vs, vt, final), R_gt))})
        for k, w in MODES:
            Rb, _, first, final = v.search(vs, vt, base_level=2, levels=4, k=k, min_sep_deg=THETA, beam=w)
            e_modes = geodesic_deg(final.R_best, R_gt[:, None]).nan_to_num(360.0).min(1).values
            emit({"kind": "accuracy", "task": task, "math": math_name, "what": "search_modes", "base_level": 2, "levels": 4,
                  "k": k, "beam": w, "min_sep_deg": THETA, "pairs": vs.shape[0], "top1": stat(geodesic_deg(Rb, R_gt)),
                  "best_of_modes": stat(e_modes), "ascend_all": stat(geodesic_deg(ascend_modes(v, vs, vt, final), R_gt)),
                  "modes_per_pair_mean": float((final.topk_idx >= 0).double().sum(1).mean()),
                  "pairs_best_of_modes_within_2deg": int((e_modes <= 2.0).sum())})

# ---- robustness: basin misses and close modes on random pairs --------------------------------------------------------
W1, W2, b2, vs, vt, _ = [t.to(dev) for t in bench.synthetic_inputs(torch, 256, 1, seed=1)]
v = ahv.HypothesisVerifier(W1, W2, b2, math=ahv.MATH_FP32)
g1 = v.score(vs, vt, grid, k=1, return_scores=False).topk_val[:, 0]
_, sp, _, _ = v.search(vs, vt, base_level=2, levels=4, k=32)
emit({"kind": "robustness", "pairs": 256, "math": "fp32", "what": "search", "base_level": 2, "levels": 4, "k": 32,
      "fraction_top1_ge_grid50k": float((sp >= g1).double().mean())})
for k, w in MODES:
    _, sb, _, final = v.search(vs, vt, base_level=2, levels=4, k=k, min_sep_deg=THETA, beam=w)
    live = final.topk_idx >= 0
    d = geodesic_deg(final.R_best[:, :, None], final.R_best[:, None])
    close = (d < THETA / 2) & live[:, :, None] & live[:, None] & torch.ones(k, k, dtype=torch.bool, device=dev).triu(1)
    emit({"kind": "robustness", "pairs": 256, "math": "fp32", "what": "search_modes", "base_level": 2, "levels": 4, "k": k,
          "beam": w, "min_sep_deg": THETA, "fraction_top1_ge_grid50k": float((sb >= g1).double().mean()),
          "close_mode_pairs": int(close.sum()), "pairs_with_close_modes": int(close.any(2).any(1).sum()),
          "modes_per_pair_mean": float(live.double().sum(1).mean())})

os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    for r in rows:
        f.write(json.dumps(r) + "\n")
