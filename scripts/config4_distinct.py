"""Top-k of distinct rotations (ahv_topk_distinct) and gradient refinement from distinct basins (refine_by_gradient with
min_sep_deg > 0).  Three parts, all in one run; the card's name and power limit are read in the same run:
  selection: ahv_topk_distinct against ahv_topk, k = 32, (B, N) in AHV_SEL_SHAPES, theta in {10, 30} (CUDA events, median);
  accuracy:  refine_by_gradient, theta in {0, 15, 30} x k in {4, 8, 32}, on config 4's known-rotation task (as
             config4_gradient.py) and on a near-symmetric task built as in tests/test_gpu_topk_distinct.py (source
             V_sym + eps A with V_sym invariant under the 180-degree rotation S = diag(-1,-1,1); a 50 000-point grid);
  spread:    the largest geodesic angle from the top-1 to the other k - 1 of plain top-k on both tasks.
Prints one JSON line.   AHV_B (8), AHV_N (50000), AHV_SYM_B (64), AHV_STEPS (20)."""
import importlib, json, os, statistics, subprocess, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
ahv = importlib.import_module("3dahv_b200")
dev = torch.device("cuda", 0)
B, N = int(os.environ.get("AHV_B", "8")), int(os.environ.get("AHV_N", "50000"))
B_sym, steps = int(os.environ.get("AHV_SYM_B", "64")), int(os.environ.get("AHV_STEPS", "20"))
sel_shapes = [(1, 50_000), (8, 50_000), (32, 50_000), (128, 50_000), (1, 1_000_000)]


def geodesic_deg(Ra, Rb):
    c = ((Ra.double() * Rb.double()).sum((-1, -2)) - 1) / 2
    return torch.rad2deg(torch.arccos(c.clamp(-1, 1)))


def timed(fn, n=20):
    for _ in range(3):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return statistics.median(a.elapsed_time(b) for a, b in ev)


# ---- selection cost ------------------------------------------------------------------------------------------------
selection = []
for Bs, Ns in sel_shapes:
    W1, W2, b2, vs, vt, normals = bench.synthetic_inputs(torch, Bs, 16)
    v = ahv.HypothesisVerifier(W1.to(dev), W2.to(dev), b2.to(dev))
    R = ahv.so3.grid_rotations(Ns, device=dev)
    scores = v.score(vs.to(dev), vt.to(dev), R, k=2).scores
    row = {"B": Bs, "N": Ns, "k": 32, "ms_topk": timed(lambda: ahv.ops.topk(scores, 32))}
    for th in (10.0, 30.0):
        row[f"ms_topk_distinct_{th:g}"] = timed(lambda: ahv.ops.topk_distinct(scores, R, 32, th))
        row[f"winners_mean_{th:g}"] = float((ahv.ops.topk_distinct(scores, R, 32, th)[1] >= 0).sum(1).float().mean())
    selection.append(row)


# ---- accuracy ------------------------------------------------------------------------------------------------------
def config4_task():
    W1, W2, b2, vs, _, _ = bench.synthetic_inputs(torch, B, 16)
    v = ahv.HypothesisVerifier(W1.to(dev), W2.to(dev), b2.to(dev))
    vs = vs.to(dev)
    R_gt = ahv.so3.sample_rotations(B, seed=123, device=dev)
    return v, vs, ahv.ops.rotate_volume(vs, R_gt), R_gt


def symmetric_task(eps=0.1):
    W1, W2, b2, V, A, _ = bench.synthetic_inputs(torch, B_sym, 1)
    src = (0.5 * (V + V.flip(3, 4)) + eps * A).to(dev).contiguous()
    R_gt = ahv.so3.sample_rotations(B_sym, seed=321, device=dev)
    v = ahv.HypothesisVerifier(W1.to(dev), W2.to(dev), b2.to(dev))
    return v, src, ahv.ops.rotate_volume(src, R_gt), R_gt


grid = ahv.so3.grid_rotations(N, device=dev)
tasks = {}
for name, (v, vs, vt, R_gt) in (("config4", config4_task()), ("near_symmetric", symmetric_task())):
    rows, spread = [], {}
    for k in (4, 8, 32):
        top = v.score(vs, vt, grid, k=k, return_scores=False)
        sp = geodesic_deg(top.R_best[:, 1:], top.R_best[:, :1]).max(1).values
        spread[k] = {"mean_deg": float(sp.mean()), "max_deg": float(sp.max()), "min_deg": float(sp.min())}
        for th in (0.0, 15.0, 30.0):
            Rb, sb, first, _, _ = v.refine_by_gradient(vs, vt, grid, k=k, steps=steps, min_sep_deg=th)
            e = geodesic_deg(Rb, R_gt)
            rows.append({"k": k, "min_sep_deg": th, "err_deg_mean": float(e.mean()), "err_deg_max": float(e.max()),
                         "acc5": float((e < 5).double().mean()), "acc15": float((e < 15).double().mean()),
                         "acc30": float((e < 30).double().mean()), "score_mean": float(sb.mean()),
                         "starts_mean": float((first.topk_idx >= 0).sum(1).float().mean()),
                         "ms_refine_by_gradient": timed(lambda: v.refine_by_gradient(vs, vt, grid, k=k, steps=steps,
                                                                                     min_sep_deg=th), n=10)})
    tasks[name] = {"pairs": vs.shape[0], "runs": rows, "plain_topk_spread_from_top1": spread}

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
print(json.dumps({"what": "top-k of distinct rotations (greedy geodesic NMS on SO(3)): selection cost against plain top-k, "
                          "and grid + distinct top-k + gradient ascent (refine_by_gradient min_sep_deg) accuracy",
                  "gpu": gpu, "torch": torch.__version__, "grid_hypotheses": N, "gradient_steps": steps,
                  "selection": selection, "accuracy": tasks}))
