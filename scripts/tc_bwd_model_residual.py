"""Residual of the tensor-core backward against the rounding-faithful model of its arithmetic (tests/tc_bwd_model.py),
and of the saved-activation form's rotation gradient against fp64.

    python scripts/tc_bwd_model_residual.py [OUT.json]        # default profiles/r17_tc_bwd_model_residual.json

For every case of tests/test_gpu_tc_bwd_model.py, both forms of score_backward(..., h1, pair_inv, MATH_TC) (atomic and
deterministic) and every gradient: the largest per-element residual relative to the gradient's maximum, the L2
residual relative to its norm, and the flat index of the worst element; the same for vol_src.grad of
verification_scores(save_activations=True) on the golden case.  For the rotation-gradient cases: grad_R of
score_backward(..., MATH_FP32, want_grad_R=True) in both forms, and R.grad of verification_scores(save_activations=True),
against fp64 autograd of the function that ran.  The card's name and power limit are read in the same run.  The gates
of the test file are set from these numbers."""
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import tc_bwd_model as BM  # noqa: E402


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r17_tc_bwd_model_residual.json")
    ahv = importlib.import_module("3dahv_b200")
    dev = torch.device("cuda", 0)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    golden = {k: dict(np.load(os.path.join(ROOT, "tests", "golden", k + ".npz"))) for k in ("weights", "shared_n3000_b3")}
    rec = {"gpu": _gpu(), "gates": BM.GATE, "cases": {}, "grad_R": {}}
    t0 = time.time()
    for name in BM.CASES:
        c = BM.make_case(name, golden)
        args = [T(c[k]) for k in ("vs", "tgt", "R", "W1", "W2", "b2")]
        _, h1, pinv = ahv.ops.score_train(*args)
        model, info = BM.case_model(c, h1.cpu().numpy(), pinv.cpu().numpy(), info=True)
        row = {"items": int(c["gs"].size), "exact_path_items": int(info["exact"].sum()),
               "largest_count": int(info["count"].max())}
        for form in ("atomic", "deterministic"):
            got = ahv.ops.score_backward(*args, T(c["gs"]), h1, pinv, ahv.MATH_TC, deterministic=form == "deterministic")
            row[form] = {g: BM.residual(a.cpu().numpy(), model[g]) for g, a in zip(BM.GRADS, got)}
        rec["cases"][name] = row
        print(name, {f: {g: f"{r['elem']:.1e}/{r['l2']:.1e}" for g, r in row[f].items()} for f in ("atomic", "deterministic")},
              flush=True)
    # vol_src.grad through the autograd wrapper on the golden case
    c = BM.make_case("golden", golden)
    vt = T(golden["shared_n3000_b3"]["vol_tgt"][:3])
    W1, W2, b2, R = T(c["W1"]), T(c["W2"]), T(c["b2"]), T(c["R"])
    tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
    _, h1, pinv = ahv.ops.score_train(T(c["vs"]), tgt, R, W1, W2, b2)
    vs = T(c["vs"]).requires_grad_(True)
    s = ahv.training.verification_scores(vs, vt, R, W1, W2, b2, math=ahv.MATH_TC, save_activations=True)
    (s * T(c["gs"])).sum().backward()
    model = BM.tc_backward(c["vs"], tgt.cpu().numpy(), c["R"], c["W1"], c["W2"], c["b2"], c["gs"], h1.cpu().numpy(),
                           pinv.cpu().numpy())
    rec["verification_scores_vol_src"] = BM.residual(vs.grad.cpu().numpy(), model["vol_src"])
    # the rotation gradient of the saved-activation form against fp64
    for name in BM.R_CASES:
        c = BM.r_case(golden, name)
        W1, W2, b2 = T(c["W1"]), T(c["W2"]), T(c["b2"])
        vt = T(c["vt"])
        tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
        args = (T(c["vs"]), tgt, T(c["R"]), W1, W2, b2)
        _, h1, pinv = ahv.ops.score_train(*args)
        ref = BM.fp64_autograd(c["vs"], tgt.cpu().numpy(), c["R"], c["W1"], c["W2"], c["b2"], c["gs"], h1.cpu().numpy(),
                               pinv.cpu().numpy(), want_R=True)
        row = {}
        for form in ("atomic", "deterministic"):
            got = ahv.ops.score_backward(*args, T(c["gs"]), h1, pinv, ahv.MATH_FP32, want_grad_R=True,
                                         deterministic=form == "deterministic")
            row[form] = {g: BM.residual(a.cpu().numpy(), r) for g, a, r in zip(BM.GRADS + ("R",), got, ref)}
        Rl = T(c["R"]).requires_grad_(True)
        s = ahv.training.verification_scores(T(c["vs"]), vt, Rl, W1, W2, b2, math=ahv.MATH_TC, save_activations=True)
        (s * T(c["gs"])).sum().backward()
        row["verification_scores_R"] = BM.residual(Rl.grad.cpu().numpy(), ref[5])
        rec["grad_R"][name] = row
        print("grad_R", name, {f: f"{row[f]['R']['elem']:.1e}" for f in ("atomic", "deterministic")},
              f"{row['verification_scores_R']['elem']:.1e}", flush=True)
    forms = [r[f] for r in rec["cases"].values() for f in ("atomic", "deterministic")]
    rec["largest"] = {g: {m: max(f[g][m] for f in forms) for m in ("elem", "l2")} for g in BM.GRADS}
    rec["largest"]["vol_src"] = {m: max(rec["largest"]["vol_src"][m], rec["verification_scores_vol_src"][m])
                                 for m in ("elem", "l2")}
    rec["largest_grad_R"] = max(max(r["atomic"]["R"]["elem"], r["deterministic"]["R"]["elem"], r["verification_scores_R"]["elem"])
                                for r in rec["grad_R"].values())
    rec["seconds"] = round(time.time() - t0, 1)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"largest": rec["largest"], "grad_R": rec["largest_grad_R"]}))


if __name__ == "__main__":
    main()
