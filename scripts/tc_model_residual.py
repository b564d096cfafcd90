"""Residual of the tensor-core scorer against the rounding-faithful model of its arithmetic (tests/tc_model.py).

    python scripts/tc_model_residual.py [OUT.json]        # default profiles/r16_tc_model_residual.json

For every case of tests/test_gpu_tc_model.py and every mode that runs the kernel (fp32 volumes under AHV_MATH_TC,
AHV_MATH_TC_F16GATHER, bf16 volumes) the largest per-element relative score difference (1e-6 floor) and where it is;
for the training forward (ahv_score_train, fp32 gather) the fraction of conv1's kept fp16 activations that are
bit-identical to the model's, the largest difference in fp16 ulps, and the largest share of the fp32-accumulation
allowance 2^-20 sum |W1h| |A| a differing element uses.  The gates of the test file are set from these numbers."""
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
import tc_model as M  # noqa: E402

H1_CASES = ["golden", "ragged_2x33_per_pair", "pairs_33x17", "R_x0.35", "outlier_1e6", "student_t", "W1_x2^12"]


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r16_tc_model_residual.json")
    ahv = importlib.import_module("3dahv_b200")
    dev = torch.device("cuda", 0)
    golden = {k: dict(np.load(os.path.join(ROOT, "tests", "golden", k + ".npz"))) for k in ("weights", "shared_n3000_b3")}
    rec = {"gpu": _gpu(), "gates": M.GATE, "scores": {}, "h1": {}}
    t0 = time.time()
    for name in M.CASES:
        case = M.make_case(name, golden)
        head = [torch.from_numpy(case[k]).to(dev) for k in ("W1", "W2", "b2")]
        R = torch.from_numpy(case["R"]).to(dev)
        tgt = torch.from_numpy(case["tgt"]).to(dev)
        row = {}
        for mode in M.MODES:
            v = torch.from_numpy(case["vs"]).to(dev)
            v = v.bfloat16() if mode == "bf16" else v
            math = ahv.MATH_TC_F16GATHER if mode == "f16gather" else ahv.MATH_TC
            s = ahv.ops.score(v, tgt, R, *head, k=1, math=math)[0].cpu().numpy().astype(np.float64)
            model = M.case_scores(case, mode)
            rel = np.abs(s - model) / np.maximum(np.abs(model), 1e-6)
            at = np.unravel_index(int(np.argmax(rel)), rel.shape)
            row[mode] = {"max_rel": float(rel.max()), "mean_rel": float(rel.mean()), "at": [int(i) for i in at],
                         "items": int(rel.size)}
        rec["scores"][name] = row
        print(name, {m: f"{r['max_rel']:.2e}" for m, r in row.items()}, flush=True)
        if name in H1_CASES:
            Rn = case["R"] if case["R"].shape[-3] <= 1000 else np.ascontiguousarray(case["R"][:1000])
            s, h1, pinv = ahv.ops.score_train(torch.from_numpy(case["vs"]).to(dev), tgt, torch.from_numpy(Rn).to(dev), *head)
            model, mh1, mpinv, bound = M.tc_forward(case["vs"], case["tgt"], Rn, case["W1"], case["W2"], case["b2"],
                                                    gather="f32", want_h1=True)
            got = h1.cpu().numpy()
            same = got.view(np.uint16) == mh1.view(np.uint16)
            diff = np.abs(got.astype(np.float64) - mh1.astype(np.float64))
            ulp = np.spacing(np.abs(mh1)).astype(np.float64)
            share = np.where(same, 0.0, np.maximum(diff - ulp, 0.0) / np.maximum(2.0 ** -20 * bound, 1e-300))
            rec["h1"][name] = {
                "match": float(same.mean()), "elements": int(same.size),
                "max_ulp": float((diff / ulp).max()),
                "max_allowance_share": float(share.max()),
                "pair_inv_identical": bool(np.array_equal(pinv.cpu().numpy(), mpinv)),
                "score_max_rel": float((np.abs(s.cpu().numpy() - model) / np.maximum(np.abs(model), 1e-6)).max()),
            }
            print("  h1", rec["h1"][name], flush=True)
    rec["largest"] = {m: max(r[m]["max_rel"] for r in rec["scores"].values()) for m in M.MODES}
    rec["seconds"] = round(time.time() - t0, 1)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec["largest"]))


if __name__ == "__main__":
    main()
