"""Weight range of the tensor-core paths: the golden head with W1, W2 or b2 scaled by c = 1.37 * 2^k (k = -24 .. 24),
alone and along the two exact symmetries of the score (S1: W1 and b2; S2: W2 and b2), entries beyond fp16's range
(W1 * 2^21, W2 * 2^19), and the spread between W1's rows (one row times 2^k, k = 0 .. 12, the limit that fp16 H1 sets).
Order-one volumes, scored under every math mode and volume type against fp64 `oracle.score_torch`; per case the worst
relative score error against each gate: fp32 volumes against the volume itself (1e-3 for AHV_MATH_TC and
AHV_MATH_TC_F16GATHER, 2e-5 for AHV_MATH_FP32), bf16 volumes against the bf16-rounded volume (2e-3).  The card's name
and power limit are read in the same run.  Prints one JSON line.   AHV_B (4), AHV_N (300)."""
import importlib, json, os, subprocess, sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ahv_oracle as orc
ahv = importlib.import_module("3dahv_b200")
dev = torch.device("cuda", 0)
B, N = int(os.environ.get("AHV_B", "4")), int(os.environ.get("AHV_N", "300"))
w = dict(np.load(os.path.join(ROOT, "tests", "golden", "weights.npz")))
W0 = [torch.from_numpy(w[k]) for k in ("W1", "W2", "b2")]
MODES = (("tc", ahv.MATH_TC), ("f16gather", ahv.MATH_TC_F16GATHER), ("fp32", ahv.MATH_FP32))


def scaled(which, c):
    W1, W2, b2 = W0
    return {"W1": (W1 * c, W2, b2), "W2": (W1, W2 * c, b2), "b2": (W1, W2, b2 * c),
            "S1": (W1 * c, W2, b2 * c), "S2": (W1, W2 * c, b2 * c)}[which]


def row_spread(k):
    W1 = W0[0].clone()
    W1[7] *= 2.0 ** k
    return W1, W0[1], W0[2]


def relerr(a, b):
    return float(((a.double() - b).abs() / b.abs().clamp_min(1e-6)).max())


gen = torch.Generator().manual_seed(5)
vs = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
vt = torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
vs16 = vs.bfloat16()
R = ahv.so3.sample_rotations(N, seed=17, device=dev)


def measure(W):
    Wd = [t.double() for t in W]
    ref = orc.score_torch(vs.double(), vt.double(), R.cpu().double(), *Wd).double()
    ref16 = orc.score_torch(vs16.double(), vt.double(), R.cpu().double(), *Wd).double()
    row = {}
    for name, math in MODES:
        v = ahv.HypothesisVerifier(*(t.to(dev) for t in W), math=math)
        s = v.score(vs.to(dev), vt.to(dev), R, k=1).scores.cpu()
        s16 = v.score(vs16.to(dev), vt.to(dev), R, k=1).scores.cpu()
        row[name] = {"f32_vs_fp64": relerr(s, ref), "bf16_vs_rounded": relerr(s16, ref16)}
    return row


rows = []
for which in ("W1", "W2", "b2", "S1", "S2"):
    for k in range(-24, 25, 4):
        row = {"scaled": which, "factor": 1.37 * 2.0 ** k, **measure(scaled(which, 1.37 * 2.0 ** k))}
        rows.append(row)
        print(json.dumps(row), file=sys.stderr)
for which, k in (("W1", 21), ("W2", 19)):
    row = {"scaled": which, "factor": 2.0 ** k, **measure(scaled(which, 2.0 ** k))}
    rows.append(row)
    print(json.dumps(row), file=sys.stderr)
for k in range(0, 13, 2):
    row = {"scaled": "one W1 row", "factor": 2.0 ** k, **measure(row_spread(k))}
    rows.append(row)
    print(json.dumps(row), file=sys.stderr)
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
print(json.dumps({"what": "worst relative score error against fp64 oracle.score_torch, golden head with scaled weights, "
                          "order-one volumes", "gpu": gpu, "torch": torch.__version__, "pairs": B, "hypotheses": N,
                  "gates": {"f32_vs_fp64": {"tc": 1e-3, "f16gather": 1e-3, "fp32": 2e-5}, "bf16_vs_rounded": 2e-3},
                  "rows": rows}))
