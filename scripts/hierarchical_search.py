"""Coarse-to-fine search on the nested Hopf grid (HypothesisVerifier.search / ahv_search_hierarchical) against the dense
50 000-point super-Fibonacci grid.  Writes one JSONL file (default profiles/r14_hierarchical_search.jsonl); the card's name
and power limit are read in the same run.  Four kinds of rows:
  time:       search at (base_level, levels, k) in {2,3} x {3,4,5} x {1,8,32}, verify(k = 1) on the 50 000-point grid and
              refine_by_gradient (k = 8 and 32, 20 steps) on it, for B in {1, 8, 32}; every call captured in a CUDA graph
              and timed with CUDA events around single replays (median of 30 after 5 warm-up replays);
  accuracy:   config 4's known-rotation task (8 pairs) and the near-symmetric task (64 pairs), both built as in
              scripts/config4_distinct.py, under AHV_MATH_TC and AHV_MATH_FP32: mean / max geodesic error to R_gt of the
              search, of the search followed by `ascend` from final.R_best, and of the 50 000-grid top-1;
  ties:       per level of the default search under AHV_MATH_TC, the fp32 score gap between the best and second-best
              candidate, and the pairs where it is below 1e-4 (the tensor-core path's error);
  robustness: on 256 random synthetic pairs, the fraction where the search's fp32 top-1 score is >= the 50 000-grid's.
    python scripts/hierarchical_search.py [out.jsonl]"""
import importlib, json, os, statistics, subprocess, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
ahv = importlib.import_module("3dahv_b200")
ops = ahv.ops
dev = torch.device("cuda", 0)
out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r14_hierarchical_search.jsonl")
N_GRID, STEPS = 50_000, 20
CONFIGS = [(b, l, k) for b in (2, 3) for l in (3, 4, 5) for k in (1, 8, 32)]
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


def graph_ms(fn, n=30):
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
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for a, b in ev:
        a.record(); g.replay(); b.record()
    torch.cuda.synchronize()
    return statistics.median(a.elapsed_time(b) for a, b in ev)


grid = ahv.so3.grid_rotations(N_GRID, device=dev)

# ---- time ------------------------------------------------------------------------------------------------------------
for B in (1, 8, 32):
    W1, W2, b2, vs, vt, _ = [t.to(dev) for t in bench.synthetic_inputs(torch, B, 1)]
    v = ahv.HypothesisVerifier(W1, W2, b2)
    for base, levels, k in CONFIGS:
        res = ops.search_hierarchical(vs, vt, W1, W2, b2, base_level=base, levels=levels, k=k)
        ms = graph_ms(lambda: ops.search_hierarchical(vs, vt, W1, W2, b2, base_level=base, levels=levels, k=k, out=res[:6],
                                                      workspace=res[6]))
        emit({"kind": "time", "what": "search", "B": B, "base_level": base, "levels": levels, "k": k,
              "hypotheses_per_pair": 72 * 8 ** base + levels * 8 * k, "ms": ms})
    ws = torch.empty(ops.workspace_bytes(B, N_GRID, 1), device=dev, dtype=torch.uint8)
    emit({"kind": "time", "what": "verify_k1_grid50k", "B": B, "hypotheses_per_pair": N_GRID,
          "ms": graph_ms(lambda: ops.verify(vs, vt, grid, W1, W2, b2, k=1, workspace=ws))})
    for k in (8, 32):
        res = ops.refine_gradient(vs, vt, grid, W1, W2, b2, k=k, steps=STEPS)
        emit({"kind": "time", "what": f"refine_by_gradient_k{k}_grid50k", "B": B, "k": k, "steps": STEPS,
              "ms": graph_ms(lambda: ops.refine_gradient(vs, vt, grid, W1, W2, b2, k=k, steps=STEPS, out=res[:8],
                                                         workspace=res[8]))})


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
for task, (head, vs, vt, R_gt) in (("config4", config4_task()), ("near_symmetric", symmetric_task())):
    for math_name, math in (("tc", ahv.MATH_TC), ("fp32", ahv.MATH_FP32)):
        v = ahv.HypothesisVerifier(*head, math=math)
        g1 = v.score(vs, vt, grid, k=1, return_scores=False)
        e_grid = geodesic_deg(g1.R_best[:, 0], R_gt)
        Rg, _, _, _, _ = v.refine_by_gradient(vs, vt, grid, k=8, steps=STEPS)
        emit({"kind": "accuracy", "task": task, "math": math_name, "what": "grid50k_top1", "pairs": vs.shape[0],
              **stat(e_grid), "refine_by_gradient_k8": stat(geodesic_deg(Rg, R_gt))})
        for base, levels, k in CONFIGS:
            Rb, sb, first, final = v.search(vs, vt, base_level=base, levels=levels, k=k)
            Ra, sa, _, _ = v.ascend(vs, vt, final.R_best, steps=STEPS)
            e = geodesic_deg(Rb, R_gt)
            emit({"kind": "accuracy", "task": task, "math": math_name, "what": "search", "base_level": base, "levels": levels,
                  "k": k, "pairs": vs.shape[0], "search": stat(e), "search_then_ascend": stat(geodesic_deg(Ra, R_gt)),
                  "base_level_top1": stat(geodesic_deg(first.R_best[:, 0], R_gt)), "grid50k_top1": stat(e_grid),
                  "pairs_search_better_than_grid": int((e < e_grid).sum())})

# ---- ties at fine levels under the tensor-core path ------------------------------------------------------------------
head, vs, vt, R_gt = config4_task()
W1, W2, b2 = head
tf = ops.forward_3d2d(vt, W1, W2, b2)
B, k, base, levels = vs.shape[0], 8, 2, 4
G = ops.hopf_grid(base, device=dev)
_, _, idx = ops.score(vs, tf, G, W1, W2, b2, k=k, math=ahv.MATH_TC, return_scores=False)
par = idx.sort(1).values
for l in range(levels):
    ci, cR = ops.hopf_children(base + l, par)
    cR = cR.reshape(B, 8 * k, 3, 3)
    s32 = ops.score(vs, tf, cR, W1, W2, b2, k=0, math=ahv.MATH_FP32)[0]
    stc, _, li = ops.score(vs, tf, cR, W1, W2, b2, k=k, math=ahv.MATH_TC)
    top2 = s32.topk(2, dim=1).values
    gap = top2[:, 0] - top2[:, 1]
    emit({"kind": "ties", "task": "config4", "level": base + l + 1, "cell_deg": float(torch.rad2deg(torch.tensor(
              (torch.pi ** 2 / (72 * 8 ** (base + l + 1))) ** (1 / 3)))),
          "fp32_top2_gap_median": float(gap.median()), "fp32_top2_gap_min": float(gap.min()),
          "pairs_gap_below_1e-4": int((gap < 1e-4).sum()), "tc_minus_fp32_max_abs": float((stc - s32).abs().max()),
          "pairs_tc_top1_differs_from_fp32_top1": int((stc.argmax(1) != s32.argmax(1)).sum()), "pairs": B})
    par = ci.reshape(B, 8 * k).gather(1, li).sort(1).values

# ---- robustness: basin misses on random pairs ------------------------------------------------------------------------
W1, W2, b2, vs, vt, _ = [t.to(dev) for t in bench.synthetic_inputs(torch, 256, 1, seed=1)]
v = ahv.HypothesisVerifier(W1, W2, b2, math=ahv.MATH_FP32)
g1 = v.score(vs, vt, grid, k=1, return_scores=False).topk_val[:, 0]
for base, levels, k in CONFIGS:
    _, sb, _, _ = v.search(vs, vt, base_level=base, levels=levels, k=k)
    emit({"kind": "robustness", "pairs": 256, "math": "fp32", "base_level": base, "levels": levels, "k": k,
          "fraction_search_ge_grid50k": float((sb >= g1).double().mean()), "search_score_mean": float(sb.mean()),
          "grid50k_score_mean": float(g1.mean())})

os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    for r in rows:
        f.write(json.dumps(r) + "\n")
