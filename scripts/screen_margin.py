"""How far the 16-bit gather's scores (AHV_MATH_TC_F16GATHER) stray from the fp32 gather's (AHV_MATH_TC) on fp32
volumes: the measurement behind the screening margin tau of ahv_verify's screened arg-max (csrc/ahv_api.cu).

Cases: the bench workload (config 2: 32 pairs x 50 000 hypotheses, `bench.synthetic_inputs`, seed 0); outlier
volumes (order-one bulk, outliers +r/3 and -r, r = 1e2 .. 1e9, as tests/test_gpu_weight_range.py) under W1 * 2^k;
the mixed per-pair scales of tests/test_gpu_pair_scale.py; the golden head with W1, W2, b2 or the symmetries S1/S2
scaled by 1.37 * 2^k, one W1 row times 2^k, and the trained-like weight draws.  Per case: the largest
|s16 - s32| in score units; for the bench workload also per pair the top-1/top-2 gap and, for candidate tau, how many
hypotheses lie within 2 tau of the screened maximum and whether the fp32 winner is among them.  The card's name and
power limit are read in the same run.  Prints one JSON line per case; with $AHV_OUT set, writes the whole record there."""
import importlib, json, math, os, subprocess, sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
ahv = importlib.import_module("3dahv_b200")
dev = torch.device("cuda", 0)
TAUS = [1e-4, 2e-4, 5e-4, 1e-3, 2e-3, 5e-3, 1e-2]


def scores(W, vs, vt, R, math_mode):
    v = ahv.HypothesisVerifier(*(t.to(dev) for t in W), math=math_mode)
    return v.score(vs.to(dev), vt.to(dev), R.to(dev), k=1).scores.double()


def deviation(W, vs, vt, R):
    s32 = scores(W, vs, vt, R, ahv.MATH_TC)
    s16 = scores(W, vs, vt, R, ahv.MATH_TC_F16GATHER)
    d = (s16 - s32).abs()
    return s32, s16, float(d.max()), float(d.quantile(0.999)) if d.numel() <= 1 << 24 else None


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception as e:  # noqa: BLE001
        return f"unavailable ({e})"


out = {"card": card(), "cases": []}

# ---- the bench workload ----
W1, W2, b2, vs, vt, normals = bench.synthetic_inputs(torch, 32, 50000)
R = ahv.ops.rotations_from_normals(normals.to(dev))
s32, s16, dmax, dq = deviation((W1, W2, b2), vs, vt, R)
top2 = s32.topk(2, dim=1).values
m16 = s16.max(dim=1).values
win = s32.argmax(dim=1)
per_tau = {}
for tau in TAUS:
    cand = (s16 >= (m16 - 2 * tau)[:, None])
    kept = bool(cand[torch.arange(32, device=dev), win].all())
    cnt = cand.sum(1).cpu().tolist()
    per_tau[f"{tau:g}"] = {"contenders_max": max(cnt), "contenders_median": float(np.median(cnt)), "winner_kept": kept}
bench_row = {"case": "bench config 2 (32 x 50000)", "max_abs_dev": dmax, "p999_abs_dev": dq,
             "per_pair_max_abs_dev": (s16 - s32).abs().max(1).values.cpu().tolist(),
             "gap12": (top2[:, 0] - top2[:, 1]).cpu().tolist(), "score_max": float(s32.max()), "score_std": float(s32.std()),
             "per_tau": per_tau}
out["cases"].append(bench_row)
print(json.dumps({k: bench_row[k] for k in ("case", "max_abs_dev", "p999_abs_dev", "per_tau")}), flush=True)

# ---- outlier volumes ----
g = dict(np.load(os.path.join(ROOT, "tests", "golden", "weights.npz")))
W0 = [torch.from_numpy(g[k]).float() for k in ("W1", "W2", "b2")]


def outlier_volumes(B, r, seed):
    gen = torch.Generator().manual_seed(seed)
    vs, vt = torch.randn(B, 16, 8, 8, 8, generator=gen), torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    pos = torch.randperm(16 * 512, generator=gen)[: 2 * B].reshape(B, 2)
    pos[0, 1] = 0
    flat = vs.view(B, -1)
    flat[torch.arange(B), pos[:, 0]] = r / 3
    flat[torch.arange(B), pos[:, 1]] = -r
    return vs, vt


def mixed_batch(B, seed):
    gen = torch.Generator().manual_seed(seed)
    vs = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    vt = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    pos = torch.randint(0, 16 * 512, (B,), generator=gen)
    sign = torch.where(torch.rand(B, generator=gen) < 0.5, -1.0, 1.0)
    vs.view(B, -1)[torch.arange(B), pos] = sign * torch.pow(2.0, torch.tensor([3.0 + (5 * b) % 17 for b in range(B)]))
    return vs, vt


Rs = ahv.so3.sample_rotations(3000, seed=17, device=dev)


def record(name, W, vs, vt, R=Rs):
    _, _, dmax, dq = deviation(W, vs, vt, R)
    out["cases"].append({"case": name, "max_abs_dev": dmax, "p999_abs_dev": dq})
    print(json.dumps(out["cases"][-1]), flush=True)


for k in (0, 4, 8):
    for r in (1e2, 1e4, 1e6, 1e7, 3e7, 1e8, 3e8, 1e9):
        vs_o, vt_o = outlier_volumes(4, r, seed=5)
        record(f"outlier r={r:g} W1*2^{k}", (W0[0] * 2.0 ** k, W0[1], W0[2]), vs_o, vt_o)
vs_m, vt_m = mixed_batch(16, seed=3)
record("mixed per-pair scales (2^3 .. 2^19 outliers)", W0, vs_m, vt_m)

gen = torch.Generator().manual_seed(5)
vs_w = torch.randn(4, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
vt_w = torch.randn(4, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
for which in ("W1", "W2", "b2", "S1", "S2"):
    for k in (-24, -12, -4, 0, 4, 12, 24):
        c = 1.37 * 2.0 ** k
        W1s, W2s, b2s = W0
        W = {"W1": (W1s * c, W2s, b2s), "W2": (W1s, W2s * c, b2s), "b2": (W1s, W2s, b2s * c),
             "S1": (W1s * c, W2s, b2s * c), "S2": (W1s, W2s * c, b2s * c)}[which]
        record(f"{which} * 1.37*2^{k}", W, vs_w, vt_w)
for k in (0, 6, 12):
    W1r = W0[0].clone()
    W1r[7] *= 2.0 ** k
    record(f"W1 row 7 * 2^{k}", (W1r, W0[1], W0[2]), vs_w, vt_w)
gen = torch.Generator().manual_seed(77)
W1t = W0[0] * torch.pow(2.0, torch.rand(32, 1, generator=gen) * 6)
record("trained-like row_scales", (W1t.contiguous(), W0[1], W0[2]), vs_w, vt_w)
W1z = W0[0].clone()
W1z[[5, 22]] = 0.0
record("trained-like zero_rows", (W1z, W0[1], W0[2]), vs_w, vt_w)

dst = os.environ.get("AHV_OUT")
if dst:
    with open(dst, "w") as f:
        json.dump(out, f, indent=1)
print("card:", out["card"])
