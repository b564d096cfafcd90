"""First moment of the posterior over each slot (ahv_posterior_moments).  Two parts in one run; the card's name and power
limit are read in the same run:
  timing:         ahv_posterior_moments alternated with ahv_posterior_mass, call for call, at the sizes of
                  posterior_time.py: B x N in {1, 8, 32, 128} x 5e4 and 1 x 1e6 (a super-Fibonacci grid), k in {1, 8, 32},
                  the distinct winners at theta = 15 degrees as centres and radius 15; CUDA events, median of 20 after 3
                  warm-up calls of each.  `ms_*`: replays of a CUDA graph of 20 back-to-back calls, divided by 20 (the
                  kernels' time; at these sizes an eager call waits on the Python wrapper's launches).  `ms_*_eager`:
                  the ops.* calls themselves, as posterior_time.py timed them.  Every input fits in L2 and is read from
                  there.  Each row also records that the moments call's log_z and mass equal the mass call's bit for bit.
  demonstration:  HypothesisVerifier.posterior(moments=True) on config 4's known-rotation task (as posterior_time.py:
                  8 pairs) with k = 1 and radius 15 degrees, on super-Fibonacci grids of 5 000 and 50 000 rotations and
                  at T in {0.1, 0.03, 0.01}: the geodesic error of the top-1 and of slot 0's mean_R, spread_deg, and the
                  Spearman rank correlation of spread and mean_R error over the pairs.  The verification head is the
                  synthetic one of bench.py (random weights, not trained): the numbers show what the call reports, not
                  a calibration.
Writes one JSON line per row to AHV_OUT (profiles/r13_posterior_moments.jsonl).   AHV_B (8)."""
import importlib, json, os, statistics, subprocess, sys, torch
from scipy.stats import spearmanr
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
ahv = importlib.import_module("3dahv_b200")
dev = torch.device("cuda", 0)
B = int(os.environ.get("AHV_B", "8"))
out_path = os.environ.get("AHV_OUT", os.path.join(ROOT, "profiles", "r13_posterior_moments.jsonl"))
sizes = [(1, 50_000), (8, 50_000), (32, 50_000), (128, 50_000), (1, 1_000_000)]
THETA = 15.0


def geodesic_deg(Ra, Rb):
    c = ((Ra.double() * Rb.double()).sum((-1, -2)) - 1) / 2
    return torch.rad2deg(torch.arccos(c.clamp(-1, 1)))


def alternated(fa, fb, n=20):
    """Median ms of fa and of fb, timed call for call in alternation after 3 warm-up calls of each."""
    for _ in range(3):
        fa(); fb()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(n)]
    for e in ev:
        e[0].record(); fa(); e[1].record()
        e[2].record(); fb(); e[3].record()
    torch.cuda.synchronize()
    return statistics.median(e[0].elapsed_time(e[1]) for e in ev), statistics.median(e[2].elapsed_time(e[3]) for e in ev)


def graphed(fn, reps=20):
    """A CUDA graph of `reps` back-to-back calls of fn: its replay times the kernels, not the Python wrapper."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    return lambda: g.replay(), g


def bits(t):
    return t.contiguous().view(torch.int32)


rows = []
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
rows.append({"what": "first moment of the posterior over each slot (ahv_posterior_moments): time against ahv_posterior_mass, "
                     "and mean rotation / spread on config 4's task", "gpu": gpu, "torch": torch.__version__})
print(json.dumps(rows[-1]), flush=True)

# ---- timing --------------------------------------------------------------------------------------------------------
for Bs, Ns in sizes:
    W1, W2, b2, vs, vt, _ = bench.synthetic_inputs(torch, Bs, 16)
    v = ahv.HypothesisVerifier(W1.to(dev), W2.to(dev), b2.to(dev))
    R = ahv.so3.grid_rotations(Ns, device=dev)
    scores = ahv.ops.score(vs.to(dev), v.target_features(vt.to(dev)), R, v.W1, v.W2, v.b2, k=0)[0]
    for k in (1, 8, 32):
        _, idx, Rb = ahv.ops.topk_distinct(scores, R, k, THETA)
        ws_mass = torch.empty(ahv.ops.posterior_mass_workspace_bytes(Bs, Ns, k), device=dev, dtype=torch.uint8)
        ws_mom = torch.empty(ahv.ops.posterior_moments_workspace_bytes(Bs, Ns, k), device=dev, dtype=torch.uint8)
        lz, mass = ahv.ops.posterior_mass(scores, R, Rb, THETA, workspace=ws_mass)
        lz2, mass2, mean_R, mean_cos, _ = ahv.ops.posterior_moments(scores, R, Rb, THETA, workspace=ws_mom)
        call_mass = lambda: ahv.ops.posterior_mass(scores, R, Rb, THETA, workspace=ws_mass)
        call_mom = lambda: ahv.ops.posterior_moments(scores, R, Rb, THETA, workspace=ws_mom)
        eager_mass, eager_mom = alternated(call_mass, call_mom)
        (rep_mass, g1), (rep_mom, g2) = graphed(call_mass), graphed(call_mom)
        ms_mass, ms_mom = (x / 20 for x in alternated(rep_mass, rep_mom))
        target = 1.25 if k == 1 else (2.0 if k == 32 else None)
        spread = torch.rad2deg(torch.arccos(mean_cos[:, 0].clamp(-1, 1)))
        row = {"part": "timing", "B": Bs, "N": Ns, "k": k, "theta_deg": THETA, "ms_posterior_mass": ms_mass,
               "ms_posterior_moments": ms_mom, "ratio": ms_mom / ms_mass, "ms_posterior_mass_eager": eager_mass,
               "ms_posterior_moments_eager": eager_mom, "ratio_eager": eager_mom / eager_mass, "target_ratio": target,
               "target_met": None if target is None else ms_mom / ms_mass <= target,
               "log_z_mass_bit_equal": bool(torch.equal(bits(lz), bits(lz2)) and torch.equal(bits(mass), bits(mass2))),
               "slot0_spread_deg_mean": float(spread.mean()),
               "slot0_mean_R_to_winner_deg_mean": float(geodesic_deg(mean_R[:, 0], Rb[:, 0]).mean())}
        rows.append(row)
        print(json.dumps(row), flush=True)

# ---- demonstration -------------------------------------------------------------------------------------------------
W1, W2, b2, vs, _, _ = bench.synthetic_inputs(torch, B, 16)
v = ahv.HypothesisVerifier(W1.to(dev), W2.to(dev), b2.to(dev))
vs = vs.to(dev)
R_gt = ahv.so3.sample_rotations(B, seed=123, device=dev)
vt = ahv.ops.rotate_volume(vs, R_gt)
for N_grid in (5000, 50_000):
    grid = ahv.so3.grid_rotations(N_grid, device=dev)
    for T in (0.1, 0.03, 0.01):
        p = v.posterior(vs, vt, grid, k=1, radius_deg=15.0, temperature=T, moments=True)
        err_top1 = geodesic_deg(p.R_best[:, 0], R_gt)
        err_mean = geodesic_deg(p.mean_R[:, 0], R_gt)
        spread = p.spread_deg[:, 0]
        rho = spearmanr(spread.cpu().numpy(), err_mean.cpu().numpy()).statistic
        row = {"part": "demo_config4", "pairs": B, "grid": N_grid, "k": 1, "radius_deg": 15.0, "temperature": T,
               "err_top1_deg": [round(float(x), 3) for x in err_top1], "err_mean_R_deg": [round(float(x), 3) for x in err_mean],
               "spread_deg": [round(float(x), 3) for x in spread], "mass_top1": [round(float(x), 4) for x in p.mass[:, 0]],
               "err_top1_deg_mean": float(err_top1.mean()), "err_mean_R_deg_mean": float(err_mean.mean()),
               "spread_deg_mean": float(spread.mean()), "spearman_spread_vs_err_mean_R": float(rho)}
        rows.append(row)
        print(json.dumps(row), flush=True)

os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    for r in rows:
        f.write(json.dumps(r) + "\n")
print("wrote", out_path)
