"""Every output of the fused backward, deterministic (`ahv_score_backward_det`) and atomic, on fixed seeded inputs, saved
to one .npz per library; and the comparison of two such files.  A change to the backward kernels that is meant to keep
their arithmetic keeps every deterministic array's bits; the atomic arrays are compared to 1e-5 of each maximum, since
their float atomics make them differ from run to run.

    python scripts/backward_bits.py OUT_DIR [TAG]         # writes OUT_DIR/backward_bits_TAG.npz (AHV_VARIANT_LIB: another build)
    python scripts/backward_bits.py --compare A.npz B.npz  # prints one JSON line, exit status 1 on a mismatch

Cases: B x N in (1, 1), (3, 50), (300, 3), (12, 9000) with a shared and a per-pair R, and (2, 150) with R * 0.35 (matrices
that crowd the samples: the tcgen05 form's exact path); each in the five forms of tests/test_gpu_backward_deterministic.py
(recompute, recompute_R, saved_fp32, saved_fp32_R, saved_tc), plus the plain `ahv_score_backward` entry.
"""
import importlib, json, os, sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FORMS = ("recompute", "recompute_R", "saved_fp32", "saved_fp32_R", "saved_tc")
CASES = [(1, 1, 1.0), (3, 50, 1.0), (300, 3, 1.0), (12, 9000, 1.0), (2, 150, 0.35)]
NAMES = ("vol", "tgt", "W1", "W2", "b2", "R")


def compare(a_path, b_path):
    a, b = np.load(a_path), np.load(b_path)
    bad, worst = [], 0.0
    if sorted(a.files) != sorted(b.files):
        bad.append("different keys")
    for k in sorted(set(a.files) & set(b.files)):
        x, y = a[k], b[k]
        if x.shape != y.shape:
            bad.append(k)
        elif k.startswith("atomic/"):
            err = float(np.abs(x.astype(np.float64) - y).max(initial=0.0))
            scale = float(np.abs(x).max(initial=0.0))
            worst = max(worst, err / scale if scale > 0 else err)
            if err > 1e-5 * scale:
                bad.append(k)
        elif not np.array_equal(x.view(np.uint32), y.view(np.uint32)):
            bad.append(k)
    n_det = sum(not k.startswith("atomic/") for k in a.files)
    print(json.dumps({"a": a_path, "b": b_path, "arrays": len(a.files), "bit_compared": n_det,
                      "atomic_worst_rel_err": worst, "mismatches": bad}))
    return not bad


def run(out_dir, tag):
    import torch
    sys.path.insert(0, ROOT)
    ahv = importlib.import_module("3dahv_b200")
    if os.environ.get("AHV_VARIANT_LIB"):   # scripts-only: another build of the library
        ahv._lib.LIB_PATH = os.path.abspath(os.environ["AHV_VARIANT_LIB"])
    dev = torch.device("cuda", 0)
    w = np.load(os.path.join(ROOT, "tests", "golden", "weights.npz"))
    W1, W2, b2 = (torch.from_numpy(w[k]).to(dev) for k in ("W1", "W2", "b2"))
    out = {}
    for B, N, shrink in CASES:
        for per_pair in (False, True):
            gen = torch.Generator().manual_seed(B * 100003 + N)
            vs = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 0.5).to(dev)
            vt = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 0.5).to(dev)
            R = ahv.so3.sample_rotations(B * N if per_pair else N, seed=N + 11, device=dev)
            R = ((R.reshape(B, N, 3, 3) if per_pair else R) * shrink).contiguous()
            gs = torch.randn(B, N, generator=gen).to(dev)
            tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
            _, h1, pinv = ahv.ops.score_train(vs, tgt, R, W1, W2, b2)
            case = f"{B}x{N}{'_pp' if per_pair else ''}{'_shrink' if shrink != 1.0 else ''}"
            out[f"in/{case}/pair_inv"] = pinv.cpu().numpy()
            args = (vs, tgt, R, W1, W2, b2, gs)
            for det in (True, False):
                for form in FORMS:
                    want_R = form.endswith("_R")
                    saved = (h1, pinv, ahv.MATH_TC if form == "saved_tc" else ahv.MATH_FP32) if form.startswith("saved") else ()
                    g = ahv.ops.score_backward(*args, *saved, want_grad_R=want_R, deterministic=det)
                    for name, t in zip(NAMES, g):
                        out[f"{'det' if det else 'atomic'}/{case}/{form}/{name}"] = t.cpu().numpy()
            z = lambda *s: torch.zeros(*s, device=dev)
            g = (z(B, 16, 8, 8, 8), z(B, 32, 64), z(32, 384), z(32, 32), z(32))
            ahv.ops._call("ahv_score_backward", dev, vs.data_ptr(), tgt.data_ptr(), R.data_ptr(), int(per_pair), W1.data_ptr(),
                          W2.data_ptr(), b2.data_ptr(), ahv.ops.base_coords(dev).data_ptr(), gs.data_ptr(),
                          *(t.data_ptr() for t in g), B, N)
            for name, t in zip(NAMES, g):
                out[f"atomic/{case}/plain/{name}"] = t.cpu().numpy()
    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, f"backward_bits_{tag}.npz")
    np.savez(path, **out)
    print(json.dumps({"wrote": path, "arrays": len(out), "gpu": torch.cuda.get_device_name(dev),
                      "lib": ahv._lib.LIB_PATH}))


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        sys.exit(0 if compare(sys.argv[2], sys.argv[3]) else 1)
    run(sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else "lib")
