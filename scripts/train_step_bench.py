"""Training-step timing (SURVEY.md §8f-3): scores + InfoNCE forward/backward, per-pair rotation sets.
AHV_B (12), AHV_N (9000), AHV_CHUNK (1024), AHV_FUSED_BWD (1), AHV_SAVE (0), AHV_TC_BWD (1), AHV_DETERMINISTIC (0:
1 runs the step under torch.use_deterministic_algorithms(True), i.e. the deterministic backward, with cuBLAS's
deterministic workspace setting).  Prints one JSON line."""
import importlib, json, os, sys, time
det = os.environ.get("AHV_DETERMINISTIC", "0") != "0"
if det:   # read by cuBLAS when torch first initialises CUDA
    os.environ["CUBLAS_WORKSPACE_CONFIG"] = ":4096:8"
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
ahv = importlib.import_module("3dahv_b200")
if os.environ.get("AHV_VARIANT_LIB"):   # scripts-only: time an experiment / diagnostics build (the product reads no environment)
    ahv._lib.LIB_PATH = os.path.abspath(os.environ["AHV_VARIANT_LIB"])
torch.use_deterministic_algorithms(det)
dev = torch.device("cuda", 0)
B, N = int(os.environ.get("AHV_B", "12")), int(os.environ.get("AHV_N", "9000"))
chunk = int(os.environ.get("AHV_CHUNK", "1024"))
fused = os.environ.get("AHV_FUSED_BWD", "1") != "0"
save = os.environ.get("AHV_SAVE", "0") != "0"
tc_bwd = os.environ.get("AHV_TC_BWD", "1") != "0"
W1, W2, b2, vs, vt, _ = bench.synthetic_inputs(torch, B, 16)
W1, W2, b2 = (t.to(dev).requires_grad_(True) for t in (W1, W2, b2))
vs, vt = vs.to(dev).requires_grad_(True), vt.to(dev).requires_grad_(True)
gt = ahv.so3.sample_rotations(B, seed=1, device=dev)
Rs = torch.cat([gt[:, None], ahv.so3.sample_rotations(B * (N - 1), seed=2, device=dev).reshape(B, N - 1, 3, 3)], 1).contiguous()

def step():
    s = ahv.training.verification_scores(vs, vt, Rs, W1, W2, b2, chunk=chunk, fused_backward=fused, save_activations=save, tc_backward=tc_bwd)
    loss = ahv.training.infonce_loss(s, Rs, gt, acc_thr_deg=15.0).mean()
    loss.backward()
    return loss

for _ in range(2):
    step()
torch.cuda.synchronize()
n = 5
ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
for a, b in ev:
    a.record(); loss = step(); b.record()
torch.cuda.synchronize()
ms = sorted(a.elapsed_time(b) for a, b in ev)[n // 2]
print(json.dumps({"what": "training step: fused scores forward + InfoNCE + backward to volumes and head weights",
                  "pairs": B, "hyps_per_pair": N, "saved_activations": save and fused, "tcgen05_backward": save and fused and tc_bwd, "backward": "fused kernel (ahv_score_backward)" if fused else f"chunked recomputation (chunk {chunk})",
                  "deterministic": det,
                  "ms_per_step_p50": ms, "hyp_pairs_per_s_fwd_bwd": B * N / (ms * 1e-3), "loss": float(loss.detach())}))
