"""Posterior mass of the selected rotations (ahv_posterior_mass).  Three parts in one run; the card's name and power limit
are read in the same run:
  timing:         ahv_posterior_mass with the distinct winners (theta = 15 degrees) as centres, next to ahv_topk_distinct
                  and ahv_score(k = 0) at the same sizes: B x N in {1, 8, 32, 128} x 5e4 and 1 x 1e6 (a super-Fibonacci
                  grid), k in {1, 8, 32}; CUDA events, median of 20 calls after 3 warm-up calls.  Every input of the
                  posterior call fits in L2 (at most 26 MB of scores plus 36 MB of rotations) and is read from there.
                  `pass_fraction`: the share of the hypotheses that some slot holds (the rest test all k centres).
  demonstration:  HypothesisVerifier.posterior on config 4's known-rotation task (as config4_gradient.py) with k = 1 and
                  radius 15 degrees (ACC_THR), and on the near-symmetric task of config4_distinct.py (source V_sym + 0.1 A,
                  V_sym invariant under the half-turn S = diag(-1,-1,1)) with the distinct top-2 at theta = 30: the masses
                  of the mode near R_gt and of the flip mode near S R_gt.  The verification head is the synthetic one of
                  bench.py (random weights, not trained), so the masses show what the call reports, not a calibration.
Writes one JSON line per row to AHV_OUT (profiles/r10_posterior.jsonl).   AHV_N (50000), AHV_B (8), AHV_SYM_B (64)."""
import importlib, json, math, os, statistics, subprocess, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
ahv = importlib.import_module("3dahv_b200")
dev = torch.device("cuda", 0)
N_grid, B, B_sym = int(os.environ.get("AHV_N", "50000")), int(os.environ.get("AHV_B", "8")), int(os.environ.get("AHV_SYM_B", "64"))
out_path = os.environ.get("AHV_OUT", os.path.join(ROOT, "profiles", "r10_posterior.jsonl"))
sizes = [(1, 50_000), (8, 50_000), (32, 50_000), (128, 50_000), (1, 1_000_000)]
THETA = 15.0


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


def pass_fraction(R, centers, theta):
    """Share of the hypotheses whose fp32 trace against some centre reaches c (what ahv_posterior_mass assigns)."""
    c = (1.0 + 2.0 * math.cos(theta * math.pi / 180.0))
    c = torch.tensor(c, dtype=torch.float32).item()
    hit = torch.zeros(centers.shape[0], R.shape[0], dtype=torch.bool, device=dev)
    for j in range(centers.shape[1]):
        t = R.reshape(-1, 9)[None] * centers[:, j].reshape(-1, 1, 9)
        tr = t[..., 0]
        for e in range(1, 9):
            tr = tr + t[..., e]
        hit |= tr >= c
    return float(hit.float().mean())


rows = []
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
rows.append({"what": "posterior mass of the selected rotations (ahv_posterior_mass): time against ahv_topk_distinct and "
                     "ahv_score(k = 0), and HypothesisVerifier.posterior on two tasks", "gpu": gpu, "torch": torch.__version__})

# ---- timing --------------------------------------------------------------------------------------------------------
for Bs, Ns in sizes:
    W1, W2, b2, vs, vt, _ = bench.synthetic_inputs(torch, Bs, 16)
    v = ahv.HypothesisVerifier(W1.to(dev), W2.to(dev), b2.to(dev))
    vs, vt = vs.to(dev), vt.to(dev)
    R = ahv.so3.grid_rotations(Ns, device=dev)
    tf = v.target_features(vt)
    ws_score = torch.empty(ahv.ops.workspace_bytes(Bs, Ns, 1), device=dev, dtype=torch.uint8)
    scores = ahv.ops.score(vs, tf, R, v.W1, v.W2, v.b2, k=0, workspace=ws_score)[0]
    ms_score = timed(lambda: ahv.ops.score(vs, tf, R, v.W1, v.W2, v.b2, k=0, workspace=ws_score))
    for k in (1, 8, 32):
        _, idx, Rb = ahv.ops.topk_distinct(scores, R, k, THETA)
        ws = torch.empty(ahv.ops.posterior_mass_workspace_bytes(Bs, Ns, k), device=dev, dtype=torch.uint8)
        log_z, mass = ahv.ops.posterior_mass(scores, R, Rb, THETA, workspace=ws)
        row = {"part": "timing", "B": Bs, "N": Ns, "k": k, "theta_deg": THETA,
               "ms_posterior_mass": timed(lambda: ahv.ops.posterior_mass(scores, R, Rb, THETA, workspace=ws)),
               "ms_topk_distinct": timed(lambda: ahv.ops.topk_distinct(scores, R, k, THETA)),
               "ms_score_k0": ms_score,
               "winners_mean": float((idx >= 0).sum(1).float().mean()),
               "mass_sum_mean": float(mass.sum(1).mean()), "mass_top1_mean": float(mass[:, 0].mean())}
        if Bs * Ns <= 32 * 50_000:
            row["pass_fraction"] = pass_fraction(R, Rb, THETA)
        rows.append(row)
        print(json.dumps(row), flush=True)


# ---- demonstration -------------------------------------------------------------------------------------------------
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


grid = ahv.so3.grid_rotations(N_grid, device=dev)
v, vs, vt, R_gt = config4_task()
p = v.posterior(vs, vt, grid, k=1, radius_deg=15.0, R_query=R_gt[:, None].contiguous())
err = geodesic_deg(p.R_best[:, 0], R_gt)
rows.append({"part": "demo_config4", "pairs": B, "grid": N_grid, "k": 1, "radius_deg": 15.0, "temperature": 0.1,
             "err_deg": [round(float(x), 3) for x in err], "mass_top1": [float(x) for x in p.mass[:, 0]],
             "log_z": [float(x) for x in p.log_z], "gt_log_density": [float(x) for x in p.log_density[:, 0]],
             "gt_log_density_pi2": [float(x) - 2 * math.log(math.pi) for x in p.log_density[:, 0]]})
print(json.dumps(rows[-1]), flush=True)

v, vs, vt, R_gt = symmetric_task()
S = torch.diag(torch.tensor([-1.0, -1.0, 1.0], device=dev))
p = v.posterior(vs, vt, grid, k=2, min_sep_deg=30.0, R_query=torch.stack([R_gt, S @ R_gt], 1).contiguous())
d_true = geodesic_deg(p.R_best, R_gt[:, None])                                   # [B,2]
d_flip = geodesic_deg(p.R_best, (S @ R_gt)[:, None])
near_true, near_flip = d_true < 15, d_flip < 15
both = near_true.any(1) & near_flip.any(1)
m_true = (p.mass * near_true).sum(1)
m_flip = (p.mass * near_flip).sum(1)
rows.append({"part": "demo_near_symmetric", "pairs": B_sym, "grid": N_grid, "k": 2, "min_sep_deg": 30.0, "radius_deg": 30.0,
             "temperature": 0.1, "pairs_with_both_modes_selected": int(both.sum()),
             "top1_is_true_mode": int(near_true[:, 0].sum()), "top1_is_flip_mode": int(near_flip[:, 0].sum()),
             "mass_true_mode_mean": float(m_true[both].mean()) if bool(both.any()) else None,
             "mass_flip_mode_mean": float(m_flip[both].mean()) if bool(both.any()) else None,
             "mass_both_modes_mean": float((m_true + m_flip)[both].mean()) if bool(both.any()) else None,
             "mass_true_mode": [round(float(x), 4) for x in m_true[:8]], "mass_flip_mode": [round(float(x), 4) for x in m_flip[:8]],
             "log_density_gt_minus_flip_mean": float((p.log_density[:, 0] - p.log_density[:, 1]).mean())})
print(json.dumps(rows[-1]), flush=True)

os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    for r in rows:
        f.write(json.dumps(r) + "\n")
print("wrote", out_path)
