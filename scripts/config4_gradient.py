"""BASELINE config 4 with gradient refinement: dense SO(3) grid -> top-k -> `HypothesisVerifier.refine_gradient` (torch
ops) and its one-kernel form `ascend`, and the whole chain in one C call (`refine_by_gradient`), against the
random-perturbation refinement pass (`refine`), on the synthetic known-rotation task of config4_linemod.py (the target
volume is the source rotated by a hidden rotation, so the score peaks there whatever the random-init head).
For k in AHV_KS (1,4,32): geodesic error (mean, max) and time per pair batch of each method, all timed in one run; the
card's name and power limit are read in the same run.  Prints one JSON line.   AHV_B (8), AHV_N (50000), AHV_M (64), AHV_STEPS (20)."""
import importlib, json, os, statistics, subprocess, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
ahv = importlib.import_module("3dahv_b200")
dev = torch.device("cuda", 0)
B, N = int(os.environ.get("AHV_B", "8")), int(os.environ.get("AHV_N", "50000"))
m, steps = int(os.environ.get("AHV_M", "64")), int(os.environ.get("AHV_STEPS", "20"))
ks = [int(x) for x in os.environ.get("AHV_KS", "1,4,32").split(",")]
W1, W2, b2, vs, _, _ = bench.synthetic_inputs(torch, B, 16)
v = ahv.HypothesisVerifier(W1.to(dev), W2.to(dev), b2.to(dev))
vs = vs.to(dev)
R_gt = ahv.so3.sample_rotations(B, seed=123, device=dev)
vt = ahv.ops.rotate_volume(vs, R_gt)
grid = ahv.so3.grid_rotations(N, device=dev)


def geodesic_deg(Ra, Rb):
    c = ((Ra.double() * Rb.double()).sum((-1, -2)) - 1) / 2
    return torch.rad2deg(torch.arccos(c.clamp(-1, 1)))


def stats(e):
    return {"mean": float(e.mean()), "max": float(e.max())}


def timed(fn, n=10):
    for _ in range(2):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return statistics.median(a.elapsed_time(b) for a, b in ev)


def grid_then_gradient(k):
    first = v.score(vs, vt, grid, k=k, return_scores=False)
    return first, v.refine_gradient(vs, vt, first.R_best, steps=steps, step_deg=1.0)


rows = []
for k in ks:
    first, (Rg, sg, _, _) = grid_then_gradient(k)
    Rr, sr, _, _ = v.refine(vs, vt, grid, k=k, m=m, max_angle_deg=6.0)
    Ra, sa, _, _ = v.ascend(vs, vt, first.R_best, steps=steps, step_deg=1.0)
    Rc, sc, _, _, _ = v.refine_by_gradient(vs, vt, grid, k=k, steps=steps, step_deg=1.0)
    rows.append({"k": k,
                 "grid_top1_err_deg": stats(geodesic_deg(first.R_best[:, 0], R_gt)),
                 "gradient_err_deg": stats(geodesic_deg(Rg, R_gt)), "gradient_score_mean": float(sg.mean()),
                 "perturbation_err_deg": stats(geodesic_deg(Rr, R_gt)), "perturbation_score_mean": float(sr.mean()),
                 "ms_grid_plus_gradient": timed(lambda: grid_then_gradient(k)),
                 "ms_gradient_only": timed(lambda: v.refine_gradient(vs, vt, first.R_best, steps=steps, step_deg=1.0)),
                 "ms_grid_plus_perturbation": timed(lambda: v.refine(vs, vt, grid, k=k, m=m, max_angle_deg=6.0)),
                 "ascend_err_deg": stats(geodesic_deg(Ra, R_gt)), "ascend_score_mean": float(sa.mean()),
                 "refine_by_gradient_err_deg": stats(geodesic_deg(Rc, R_gt)), "refine_by_gradient_score_mean": float(sc.mean()),
                 "ms_ascend_only": timed(lambda: v.ascend(vs, vt, first.R_best, steps=steps, step_deg=1.0)),
                 "ms_refine_by_gradient": timed(lambda: v.refine_by_gradient(vs, vt, grid, k=k, steps=steps, step_deg=1.0))})
    rows[-1]["ascend_speedup_over_refine_gradient"] = rows[-1]["ms_gradient_only"] / rows[-1]["ms_ascend_only"]
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
print(json.dumps({"what": "config 4: dense SO(3) grid + top-k, then gradient refinement (refine_gradient: torch ops; ascend: "
                          "one kernel; refine_by_gradient: grid + top-k + ascent in one C call) or perturbation refinement "
                          "(refine), synthetic task with a known rotation",
                  "gpu": gpu, "torch": torch.__version__, "pairs": B, "grid_hypotheses": N, "gradient_steps": steps,
                  "perturbations_per_candidate": m, "perturbation_max_angle_deg": 6.0, "runs": rows}))
