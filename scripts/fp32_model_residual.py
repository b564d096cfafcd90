"""Residual of the fp32 CUDA-core kernels against the numpy model of their arithmetic (tests/fp32_model.py).

    python scripts/fp32_model_residual.py [OUT.json]      # default profiles/r20_fp32_model_residual.json

Per case and kernel the share of outputs bit-identical to the model and the largest distance in fp32 ulps:
AHV_MATH_FP32 scores on every case of tests/tc_model.py (fp32 and bf16 volumes, the items tests/test_gpu_fp32_model.py
compares), the target features of ahv_forward_3d2d at m = 1 .. 9000 (sampled volumes) and rotate_volume (shared and
per rotation, five kinds of matrices).  For the backward of rotate_volume, which adds with float atomics in no fixed
order, the largest ratio of its error against the exact sum of its own rounded terms to the model's bound on any order
of those additions."""
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import fp32_model as F  # noqa: E402
import kernel_arith as K  # noqa: E402
import tc_model as M  # noqa: E402  (the cases)
import test_gpu_fp32_model as G  # noqa: E402  (its inputs: rotation kinds, volumes, sizes)

f32 = np.float32


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def _cmp(got, want):
    got, want = np.asarray(got, f32), np.asarray(want, f32)
    same = got.view(np.uint32) == want.view(np.uint32)
    return {"identical": float(same.mean()), "max_ulp": int(K.ulp_distance(got, want).max()), "outputs": int(same.size)}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r20_fp32_model_residual.json")
    ahv = importlib.import_module("3dahv_b200")
    T = G._T
    golden = {k: dict(np.load(os.path.join(ROOT, "tests", "golden", k + ".npz"))) for k in ("weights", "shared_n3000_b3")}
    rec = {"gpu": _gpu(), "scores": {}, "target_features": {}, "rotate_volume": {}, "rotate_volume_backward": {}}
    t0 = time.time()
    for name in M.CASES:
        case = M.make_case(name, golden)
        head = [T(case[k]) for k in ("W1", "W2", "b2")]
        B, N = case["vs"].shape[0], case["R"].shape[-3]
        items = F.case_items(name, B, N, cap=48)
        row = {}
        for voldt in ("f32", "bf16"):
            v, vs = T(case["vs"]), case["vs"]
            if voldt == "bf16":
                v, vs = v.bfloat16(), K.bf16_round(vs)
            s = ahv.ops.score(v, T(case["tgt"]), T(case["R"]), *head, k=1, math=ahv.MATH_FP32)[0]
            model = F.score(vs, case["tgt"], case["R"], case["W1"], case["W2"], case["b2"], items=items)
            row[voldt] = _cmp(s.cpu().numpy().reshape(-1)[items], model)
        rec["scores"][name] = row
        print(name, row, flush=True)
    w = golden["weights"]
    W = [T(w[k]) for k in ("W1", "W2", "b2")]
    V = (np.random.default_rng(2024).standard_normal((9000, 16, 8, 8, 8), dtype=f32) * f32(1.1) - f32(0.2)).astype(f32)
    for m in (1, 3, 4096, 4097, 9000):
        feat = ahv.ops.forward_3d2d(T(V[:m]), *W).cpu().numpy()
        rows = np.unique(np.concatenate([[0, m - 1], np.arange(4094, 4098), np.random.default_rng(m).choice(m, min(m, 48),
                                                                                                           replace=False)]))
        rows = rows[rows < m]
        rec["target_features"][str(m)] = _cmp(feat[rows], F.target_features(V[rows], w["W1"], w["W2"], w["b2"]))
    print("target features", rec["target_features"], flush=True)
    for kind in G.KINDS:
        for n in G.NS:
            vol, R = G._vol(n), G._rotations(kind, n, seed=n + 17)
            got = ahv.ops.rotate_volume(T(vol), T(R)).cpu().numpy()
            rec["rotate_volume"][f"shared_{kind}_{n}"] = _cmp(got, F.rotate_volume(vol, R))
        for n in (1, 9, 300):
            vol, R = G._vol(n + 1, n), G._rotations(kind, n, seed=n + 29)
            got = ahv.ops.rotate_volume(T(vol), T(R)).cpu().numpy()
            rec["rotate_volume"][f"per_rotation_{kind}_{n}"] = _cmp(got, F.rotate_volume(vol, R))
    print("rotate_volume", {k: v["identical"] for k, v in rec["rotate_volume"].items()}, flush=True)
    for per_rotation in (False, True):
        for n in G.NS:
            pool = np.concatenate([G._rotations(k, n, seed=n + 53) for k in G.KINDS])
            R = np.ascontiguousarray(pool[np.random.default_rng(n).permutation(len(pool))[:n]])
            g = np.random.default_rng(n + 7).normal(size=(n, 16, 8, 8, 8)).astype(f32)
            got = ahv.ops.rotate_volume_backward(T(g), T(R), per_rotation).cpu().numpy().astype(np.float64)
            exact, cnt, bound = F.rotate_volume_adjoint(g, R, per_rotation)
            err = np.abs(got - exact)
            ratio = np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err > 0, np.inf, 0.0))
            rec["rotate_volume_backward"][f"{'per_rotation' if per_rotation else 'shared'}_{n}"] = {
                "max_error_to_bound": float(ratio.max()), "identical_to_exact_rounded": float(np.mean(got == exact.astype(f32))),
                "max_terms": int(cnt.max())}
    print("backward", rec["rotate_volume_backward"], flush=True)
    rec["largest"] = {
        "scores_max_ulp": max(r[d]["max_ulp"] for r in rec["scores"].values() for d in r),
        "target_features_max_ulp": max(r["max_ulp"] for r in rec["target_features"].values()),
        "rotate_volume_max_ulp": max(r["max_ulp"] for r in rec["rotate_volume"].values()),
        "backward_max_error_to_bound": max(r["max_error_to_bound"] for r in rec["rotate_volume_backward"].values()),
    }
    rec["seconds"] = round(time.time() - t0, 1)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec["largest"]))


if __name__ == "__main__":
    main()
