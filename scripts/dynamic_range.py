"""Dynamic range of the per-pair power-of-two scale of the tensor-core paths: pairs with an order-one bulk (standard
normal) and two outlier voxels, +r/3 and -r, scored under every math mode and volume type against fp64
`oracle.score_torch`, for r = 1e2 .. 1e9.  Per (mode, volume type, r) the worst relative score error against each gate:
fp32 volumes against the volume itself (1e-3 for AHV_MATH_TC and AHV_MATH_TC_F16GATHER, 2e-5 for AHV_MATH_FP32); bf16
volumes against the bf16-rounded volume (2e-3) and against the unrounded one (1e-2).  The card's name and power limit
are read in the same run.  Prints one JSON line.   AHV_B (4), AHV_N (1000)."""
import importlib, json, os, subprocess, sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ahv_oracle as orc
ahv = importlib.import_module("3dahv_b200")
dev = torch.device("cuda", 0)
B, N = int(os.environ.get("AHV_B", "4")), int(os.environ.get("AHV_N", "1000"))
RATIOS = [1e2, 1e3, 1e4, 3e4, 1e5, 3e5, 1e6, 3e6, 1e7, 3e7, 1e8, 1e9]
w = dict(np.load(os.path.join(ROOT, "tests", "golden", "weights.npz")))
W = [torch.from_numpy(w[k]) for k in ("W1", "W2", "b2")]


def outlier_volumes(B, r, seed):
    gen = torch.Generator().manual_seed(seed)
    vs, vt = torch.randn(B, 16, 8, 8, 8, generator=gen), torch.randn(B, 16, 8, 8, 8, generator=gen) * 1.1 - 0.2
    pos = torch.randperm(16 * 512, generator=gen)[: 2 * B].reshape(B, 2)
    pos[0, 1] = 0                                                        # one outlier on a corner of the volume
    flat = vs.view(B, -1)
    flat[torch.arange(B), pos[:, 0]] = r / 3
    flat[torch.arange(B), pos[:, 1]] = -r
    return vs, vt


def relerr(a, b):
    return float(((a.double() - b).abs() / b.abs().clamp_min(1e-6)).max())


R = ahv.so3.sample_rotations(N, seed=17, device=dev)
rows = []
for r in RATIOS:
    vs, vt = outlier_volumes(B, r, seed=5)
    ref = orc.score_torch(vs.double(), vt.double(), R.cpu().double(), *(t.double() for t in W)).double()
    vs16 = vs.bfloat16()
    ref16 = orc.score_torch(vs16.double(), vt.double(), R.cpu().double(), *(t.double() for t in W)).double()
    row = {"ratio": r}
    for name, math in (("tc", ahv.MATH_TC), ("f16gather", ahv.MATH_TC_F16GATHER), ("fp32", ahv.MATH_FP32)):
        v = ahv.HypothesisVerifier(*(t.to(dev) for t in W), math=math)
        s = v.score(vs.to(dev), vt.to(dev), R, k=1).scores.cpu()
        s16 = v.score(vs16.to(dev), vt.to(dev), R, k=1).scores.cpu()
        row[name] = {"f32_vs_fp64": relerr(s, ref), "bf16_vs_rounded": relerr(s16, ref16), "bf16_vs_unrounded": relerr(s16, ref)}
    rows.append(row)
    print(json.dumps(row), file=sys.stderr)
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
print(json.dumps({"what": "worst relative score error against fp64 oracle.score_torch, order-one bulk + outliers +r/3 and -r",
                  "gpu": gpu, "torch": torch.__version__, "pairs": B, "hypotheses": N,
                  "gates": {"f32_vs_fp64": {"tc": 1e-3, "f16gather": 1e-3, "fp32": 2e-5}, "bf16_vs_rounded": 2e-3,
                            "bf16_vs_unrounded": 1e-2},
                  "rows": rows}))
