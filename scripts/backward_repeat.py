"""Repeatability of the fused backward, atomic (default) against deterministic (ahv_score_backward_det): three
identical calls per form and shape, and how many output elements differ in their bits from the first call; then the
kernel times of one call per form at 12 x 9000 under torch.profiler.  Prints JSON lines."""
import importlib, json, os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
ahv = importlib.import_module("3dahv_b200")
dev = torch.device("cuda", 0)
w = dict(np.load(os.path.join(ROOT, "tests", "golden", "weights.npz")))
out = []
def inputs(B, N, per_pair, seed=0):
    gen = torch.Generator().manual_seed(seed)
    vs = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 0.5).to(dev)
    vt = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 0.5).to(dev)
    W1, W2, b2 = (torch.from_numpy(w[k]).to(dev) for k in ("W1", "W2", "b2"))
    R = ahv.so3.sample_rotations(B * N if per_pair else N, seed=seed + 11, device=dev)
    R = (R.reshape(B, N, 3, 3) if per_pair else R).contiguous()
    tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
    gs = torch.randn(B, N, generator=gen).to(dev)
    return vs, tgt, R, W1, W2, b2, gs
names = ("vol", "tgt", "W1", "W2", "b2", "R")
for B, N, pp in ((1, 1, False), (3, 50, False), (12, 9000, True), (12, 9000, False)):
    a = inputs(B, N, pp)
    _, h1, pi = ahv.ops.score_train(*a[:6])
    for form in ("recompute", "saved_tc", "recompute_R"):
        if form == "recompute_R" and B * N > 100000 and pp: continue
        for det in (False, True):
            def run():
                if form == "recompute": return ahv.ops.score_backward(*a, deterministic=det)
                if form == "recompute_R": return ahv.ops.score_backward(*a, want_grad_R=True, deterministic=det)
                return ahv.ops.score_backward(*a, h1, pi, ahv.MATH_TC, deterministic=det)
            r = [run() for _ in range(3)]
            diff = {}
            for i, n in enumerate(names[:len(r[0])]):
                d = max(float((r[0][i] - r[k][i]).abs().max()) for k in (1, 2))
                nbits = sum(int((r[0][i].view(torch.int32) != r[k][i].view(torch.int32)).sum()) for k in (1, 2))
                diff[n] = [nbits, d / max(float(r[0][i].abs().max()), 1e-30)]
            out.append({"B": B, "N": N, "per_pair": pp, "form": form, "deterministic": det, "differing_elements_and_rel_max": diff})
            print(json.dumps(out[-1]), flush=True)
# kernel times of one call per form at 12 x 9000 (profiler run of its own)
a = inputs(12, 9000, True)
_, h1, pi = ahv.ops.score_train(*a[:6])
from torch.profiler import profile, ProfilerActivity
for form in ("recompute", "saved_tc"):
    for det in (False, True):
        f = (lambda: ahv.ops.score_backward(*a, deterministic=det)) if form == "recompute" else (lambda: ahv.ops.score_backward(*a, h1, pi, ahv.MATH_TC, deterministic=det))
        f(); torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3): f()
            torch.cuda.synchronize()
        ks = {}
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" or "kernel" in e.key or "reduce" in e.key:
                ks[e.key[:60]] = round(e.device_time_total / 3 / 1000, 3) if hasattr(e, "device_time_total") else round(e.cuda_time_total / 3 / 1000, 3)
        print(json.dumps({"form": form, "deterministic": det, "kernel_ms_per_call": ks}), flush=True)
