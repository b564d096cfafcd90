"""The screened arg-max of ahv_verify on the bench workload (config 2: 32 pairs x 50 000 hypotheses, fp32 volumes,
MATH_TC, top-1, no scores): the whole call against the single fp32-gather pass (the same call returning its scores,
which the screened form never serves) by CUDA events, L2 flushed between calls; the kernels of one screened call under
torch.profiler (16-bit screening pass, selection, list gather, fp32 re-scoring of the lists, guard, exact pass over the
flagged pairs, in launch order); contender counts per pair and the largest realised |fp32 - 16-bit| score difference
on each pair's list over tau.  The card's name and power limit are read in the same run.  Prints one JSON line
(also written to $AHV_OUT when set).   AHV_B (32), AHV_N (50000), AHV_STEPS (20)."""
import importlib, json, os, subprocess, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
ahv = importlib.import_module("3dahv_b200")
dev = torch.device("cuda", 0)
B, N, STEPS = int(os.environ.get("AHV_B", "32")), int(os.environ.get("AHV_N", "50000")), int(os.environ.get("AHV_STEPS", "20"))
TAU = 2e-3  # kScreenTau (csrc/ahv_common.cuh)

W1, W2, b2, vs, vt, normals = bench.synthetic_inputs(torch, B, N)
W1, W2, b2, vs, vt = (t.to(dev) for t in (W1, W2, b2, vs, vt))
R = ahv.ops.rotations_from_normals(normals.to(dev))
ws = torch.empty(ahv.ops.workspace_bytes(B, N, 1), dtype=torch.uint8, device=dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def screened():
    return ahv.ops.verify(vs, vt, R, W1, W2, b2, k=1, math=ahv.MATH_TC, workspace=ws)


def single():
    return ahv.ops.verify(vs, vt, R, W1, W2, b2, k=1, math=ahv.MATH_TC, return_scores=True, workspace=ws)


def timed(fn):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(STEPS):
        flush.zero_()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b_.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b_))
    ts.sort()
    return {"median_ms": ts[len(ts) // 2], "min_ms": ts[0], "max_ms": ts[-1]}


t_single = timed(single)
t_screened = timed(screened)
t_single2 = timed(single)
_, val, idx, Rb = screened()
stats = ahv.ops.verify_screen_stats(ws, B, N)
_, sval, sidx, sRb = single()
same = bool(torch.equal(val, sval) and torch.equal(idx, sidx) and torch.equal(Rb, sRb))

from torch.profiler import ProfilerActivity, profile
screened()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    screened()
    torch.cuda.synchronize()
kernels = [(e.name, e.device_time_total / 1e3) for e in prof.events() if e.device_type.name == "CUDA"]

try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as e:  # noqa: BLE001
    card = f"unavailable ({e})"
line = {"card": card, "B": B, "N": N, "steps": STEPS, "single_pass": [t_single, t_single2], "screened": t_screened,
        "speedup_median": 0.5 * (t_single["median_ms"] + t_single2["median_ms"]) / t_screened["median_ms"],
        "bit_identical": same, "kernels_ms_in_launch_order": [[n[:60], round(t, 4)] for n, t in kernels]}
if stats is not None:
    flagged, count, err = stats
    line.update({"flagged_pairs": flagged, "contenders_per_pair": count.tolist(),
                 "realised_err_over_tau": [round(float(e) / TAU, 4) for e in err]})
dst = os.environ.get("AHV_OUT")
if dst:
    with open(dst, "w") as f:
        json.dump(line, f)
print(json.dumps(line))
