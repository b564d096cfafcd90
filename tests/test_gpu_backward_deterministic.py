"""GPU: the deterministic form of the fused backward (ahv_score_backward_det, `ops.score_backward(deterministic=True)`,
and the training path under torch.use_deterministic_algorithms).

- Repeatability: three calls give the same bits in every form (recompute, saved activations with fp32 or tcgen05
  contractions, the subsets of NULL outputs, the rotation gradient for shared and per-pair R), over item counts below
  the SM count, not a multiple of the grid, pairs spanning many CTAs and many pairs per CTA; the tcgen05 form's exact
  path; CUDA-graph replay.
- Same function as the atomic entries: bit for bit on one-item calls except grad_vol (whose adjoint lists are summed
  in another order), 1e-5 of each gradient's maximum on large calls.
- fp64 autograd of the oracle at the gates tests/test_gpu_training.py uses for each form.
- End to end in a fresh process: Feature_Aligner.forward_2d3d -> verification_scores -> infonce_loss -> backward,
  twice, with every .grad bit-identical.
- The paths without a deterministic form raise (or warn) under the flag; without it nothing changes."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
NAMES = ("vol_src", "tgt_feat", "W1", "W2", "b2", "R")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _inputs(ahv, golden, B, N, per_pair, shrink=1.0, seed=0):
    w = golden["weights"]
    gen = torch.Generator().manual_seed(seed)
    vs = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 0.5).to(DEV)
    vt = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 0.5).to(DEV)
    W1, W2, b2 = (torch.from_numpy(w[k]).to(DEV) for k in ("W1", "W2", "b2"))
    R = ahv.so3.sample_rotations(B * N if per_pair else N, seed=seed + 11, device=DEV)
    R = (R.reshape(B, N, 3, 3) if per_pair else R) * shrink
    tgt = ahv.ops.forward_3d2d(vt, W1, W2, b2)
    gs = torch.randn(B, N, generator=gen).to(DEV)
    return vs, tgt, R.contiguous(), W1, W2, b2, gs


def _bits(t):
    return t.contiguous().view(torch.int32)


def _same_bits(a, b):
    return all((x is None and y is None) or torch.equal(_bits(x), _bits(y)) for x, y in zip(a, b))


def _run(ahv, form, args, deterministic, h1=None, pinv=None):
    """One backward in `form`: (grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2[, grad_R])."""
    vs, tgt, R, W1, W2, b2, gs = args
    if form == "recompute":
        return ahv.ops.score_backward(vs, tgt, R, W1, W2, b2, gs, deterministic=deterministic)
    if form == "recompute_R":
        return ahv.ops.score_backward(vs, tgt, R, W1, W2, b2, gs, want_grad_R=True, deterministic=deterministic)
    math = ahv.MATH_TC if form in ("saved_tc",) else ahv.MATH_FP32
    return ahv.ops.score_backward(vs, tgt, R, W1, W2, b2, gs, h1, pinv, math, want_grad_R=form == "saved_fp32_R",
                                  deterministic=deterministic)


def _raw_det(ahv, args, outs, h1=None, pinv=None, mode=None):
    """ahv_score_backward_det with some outputs NULL (the kEx subsets the Python wrapper does not expose)."""
    vs, tgt, R, W1, W2, b2, gs = args
    B = vs.shape[0]
    per_pair = R.dim() == 4
    N = R.shape[1] if per_pair else R.shape[0]
    want_R = outs[5] is not None
    ws = torch.empty(max(ahv.ops.score_backward_det_workspace_bytes(B, N, per_pair, want_R), 16), device=DEV, dtype=torch.uint8)
    ptr = lambda t: t.data_ptr() if t is not None else None
    ahv.ops._call("ahv_score_backward_det", DEV, vs.data_ptr(), tgt.data_ptr(), R.data_ptr(), int(per_pair),
                  W1.data_ptr(), W2.data_ptr(), b2.data_ptr(), ahv.ops.base_coords(DEV).data_ptr(), gs.data_ptr(),
                  ptr(h1), ptr(pinv), *(ptr(t) for t in outs), B, N, ahv.MATH_FP32 if mode is None else mode,
                  ws.data_ptr(), ws.numel())
    return outs


def _zeros_like_outputs(B, R, mask):
    shapes = ((B, 16, 8, 8, 8), (B, 32, 64), (32, 384), (32, 32), (32,), tuple(R.shape))
    return tuple(torch.zeros(*s, device=DEV) if m else None for s, m in zip(shapes, mask))


FORMS = ("recompute", "recompute_R", "saved_fp32", "saved_fp32_R", "saved_tc")
SHAPES = [(1, 1), (1, 7), (3, 50), (300, 3), (12, 9000)]


@pytest.mark.parametrize("per_pair", [False, True])
@pytest.mark.parametrize("B,N", SHAPES)
def test_three_calls_give_the_same_bits(ahv, golden, B, N, per_pair):
    args = _inputs(ahv, golden, B, N, per_pair)
    vs, tgt, R, W1, W2, b2, gs = args
    _, h1, pinv = ahv.ops.score_train(vs, tgt, R, W1, W2, b2)
    forms = FORMS if B * N < 100_000 else ("recompute", "saved_fp32", "saved_tc")   # grad_R at 12 x 9000 costs 3 more steps
    for form in forms:
        first = _run(ahv, form, args, True, h1, pinv)
        assert all(torch.isfinite(t).all() for t in first), form
        for _ in range(2):
            assert _same_bits(first, _run(ahv, form, args, True, h1, pinv)), (B, N, per_pair, form)


@pytest.mark.parametrize("B,N,per_pair", [(1, 1, False), (3, 50, False), (3, 50, True), (12, 400, False)])
def test_null_output_subsets_are_repeatable_and_equal_the_full_call(ahv, golden, B, N, per_pair):
    """The kEx instance: any subset of outputs; each output equals the full deterministic call's bit for bit (the
    phases left out do not touch the others' arithmetic)."""
    args = _inputs(ahv, golden, B, N, per_pair, seed=3)
    full = _raw_det(ahv, args, _zeros_like_outputs(B, args[2], (1, 1, 1, 1, 1, 1)))
    for mask in ((0, 0, 0, 0, 0, 1), (1, 0, 1, 0, 0, 0), (0, 1, 0, 1, 1, 0), (1, 1, 1, 1, 1, 0), (0, 0, 1, 0, 0, 1)):
        runs = [_raw_det(ahv, args, _zeros_like_outputs(B, args[2], mask)) for _ in range(3)]
        assert _same_bits(runs[0], runs[1]) and _same_bits(runs[0], runs[2]), mask
        for name, got, ref in zip(NAMES, runs[0], full):
            if got is not None:
                assert torch.equal(_bits(got), _bits(ref)), (mask, name)


def test_tensor_core_exact_path_is_repeatable(ahv, golden):
    """Matrices scaled by 0.35 crowd dozens of contributions onto an input voxel: the tcgen05 form's row lists
    overflow and its exact path (counting sort) runs."""
    for per_pair in (False, True):
        args = _inputs(ahv, golden, 2, 150, per_pair, shrink=0.35, seed=5)
        vs, tgt, R, W1, W2, b2, gs = args
        _, h1, pinv = ahv.ops.score_train(vs, tgt, R, W1, W2, b2)
        for form in ("saved_tc", "saved_fp32", "recompute"):
            first = _run(ahv, form, args, True, h1, pinv)
            for _ in range(2):
                assert _same_bits(first, _run(ahv, form, args, True, h1, pinv)), (per_pair, form)


def test_cuda_graph_replay_gives_the_eager_bits(ahv, golden):
    args = _inputs(ahv, golden, 3, 500, True, seed=7)
    vs, tgt, R, W1, W2, b2, gs = args
    _, h1, pinv = ahv.ops.score_train(vs, tgt, R, W1, W2, b2)
    ws = torch.empty(ahv.ops.score_backward_det_workspace_bytes(3, 500, True, True), device=DEV, dtype=torch.uint8)
    for form, math, want_R in (("saved_tc", ahv.MATH_TC, False), ("saved_fp32_R", ahv.MATH_FP32, True)):
        eager = ahv.ops.score_backward(vs, tgt, R, W1, W2, b2, gs, h1, pinv, math, want_grad_R=want_R, deterministic=True)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):   # warm-up on the capture stream
            ahv.ops.score_backward(vs, tgt, R, W1, W2, b2, gs, h1, pinv, math, want_grad_R=want_R, deterministic=True,
                                   workspace=ws)
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = ahv.ops.score_backward(vs, tgt, R, W1, W2, b2, gs, h1, pinv, math, want_grad_R=want_R,
                                         deterministic=True, workspace=ws)
        for _ in range(3):
            graph.replay()
            torch.cuda.synchronize()
            assert _same_bits(out, eager), form


@pytest.mark.parametrize("per_pair", [False, True])
def test_one_item_calls_equal_the_atomic_entries(ahv, golden, per_pair):
    """One item runs one CTA: every sum but grad_vol's adjoint lists runs in the atomic kernel's order."""
    args = _inputs(ahv, golden, 1, 1, per_pair, seed=13)
    vs, tgt, R, W1, W2, b2, gs = args
    _, h1, pinv = ahv.ops.score_train(vs, tgt, R, W1, W2, b2)
    for form in FORMS:
        a, d = _run(ahv, form, args, False, h1, pinv), _run(ahv, form, args, True, h1, pinv)
        for name, x, y in zip(NAMES, a, d):
            if name == "vol_src":
                err = float((x - y).abs().max()) / max(float(x.abs().max()), 1e-30)
                assert err <= 1e-6, (form, name, err)
            else:
                assert torch.equal(_bits(x), _bits(y)), (form, name)


@pytest.mark.parametrize("B,N,per_pair", [(3, 50, False), (12, 9000, True), (300, 3, False), (4, 2000, False)])
def test_large_calls_agree_with_the_atomic_entries(ahv, golden, B, N, per_pair):
    """Atomic and deterministic sums of the same partials: within the atomic-vs-atomic bound of
    test_gpu_rotation_grad.py, 1e-5 of each gradient's maximum."""
    args = _inputs(ahv, golden, B, N, per_pair, seed=17)
    vs, tgt, R, W1, W2, b2, gs = args
    _, h1, pinv = ahv.ops.score_train(vs, tgt, R, W1, W2, b2)
    forms = FORMS if B * N < 100_000 else ("recompute", "saved_fp32", "saved_tc")
    for form in forms:
        a, d = _run(ahv, form, args, False, h1, pinv), _run(ahv, form, args, True, h1, pinv)
        for name, x, y in zip(NAMES, a, d):
            err = float((x - y).abs().max()) / max(float(x.abs().max()), 1e-30)
            assert err <= 1e-5, (B, N, per_pair, form, name, err)


def _fp64_recompute(oracle, args, want_R):
    vs, tgt, R, W1, W2, b2, gs = (t.detach().cpu().double() for t in args)
    leaves = [t.clone().requires_grad_(True) for t in (vs, tgt, W1, W2, b2)] + ([R.clone().requires_grad_(True)] if want_R else [])
    v64, t64, w1, w2, bb = leaves[:5]
    R64 = leaves[5] if want_R else R
    per_pair = R.dim() == 4
    rows = []
    for b in range(vs.shape[0]):
        Rb = R64[b] if per_pair else R64
        rot = oracle.rotate_volume_torch(v64[b][None].expand(Rb.shape[0], -1, -1, -1, -1), Rb)
        f = oracle.forward_3d2d_torch(rot, w1, w2, bb)
        rows.append((f * t64[b][None]).sum(dim=1).mean(dim=-1))
    return torch.autograd.grad((torch.stack(rows) * gs).sum(), leaves)


@pytest.mark.parametrize("per_pair", [False, True])
def test_recompute_form_against_fp64_autograd(ahv, golden, oracle, per_pair):
    """The gate test_gpu_training.py holds the fused backward to: 2e-4 of each gradient's maximum; grad_R as well."""
    args = _inputs(ahv, golden, 2, 40, per_pair, seed=19)
    got = _run(ahv, "recompute_R", args, True)
    ref = _fp64_recompute(oracle, args, True)
    for name, a, r in zip(NAMES, got, ref):
        err = float((a.cpu().double() - r.reshape(a.shape)).abs().max()) / float(r.abs().max())
        assert err <= 2e-4, (per_pair, name, err)


@pytest.mark.parametrize("per_pair,shrink", [(False, 1.0), (True, 1.0), (False, 0.35)])
def test_saved_forms_against_fp64_autograd_of_the_function_that_ran(ahv, golden, oracle, per_pair, shrink):
    """As test_gpu_training.py's check of the saved-activation backward: conv1's output takes the value the forward
    kept and the ReLU mask of that value; fp32 contractions 2e-5, tcgen05 1e-3 of each gradient's maximum."""
    import torch.nn.functional as F

    args = _inputs(ahv, golden, 2, 150, per_pair, shrink=shrink, seed=23)
    vs, tgt, R, W1, W2, b2, gs = args
    B, N = 2, 150
    _, h1, pinv = ahv.ops.score_train(vs, tgt, R, W1, W2, b2)
    leaves = [t.double().requires_grad_(True) for t in (vs, tgt, W1, W2, b2)]
    v64, t64, w1, w2, bb = leaves
    rows = []
    for b in range(B):
        Rb = (R[b] if per_pair else R).double()
        rot = oracle.rotate_volume_torch(v64[b][None].expand(N, -1, -1, -1, -1), Rb)
        tri = torch.cat([rot.permute(0, 1, 4, 2, 3).reshape(N, 128, 8, 8), rot.permute(0, 1, 3, 2, 4).reshape(N, 128, 8, 8),
                         rot.reshape(N, 128, 8, 8)], dim=1)
        pre = F.conv2d(tri, w1.reshape(32, 384, 1, 1))
        kept = (h1.reshape(B, N, 64, 32)[b].double() * pinv[b].double()).permute(0, 2, 1).reshape(N, 32, 8, 8)
        mask = (kept > 0).double()
        hid = pre * mask + (kept - pre * mask).detach()
        f = F.normalize(F.conv2d(hid, w2.reshape(32, 32, 1, 1), bb), p=2, dim=1).flatten(2)
        rows.append((f * t64[b][None]).sum(dim=1).mean(dim=-1))
    ref = torch.autograd.grad(torch.stack(rows), leaves, grad_outputs=gs.double())
    for form, tol in (("saved_fp32", 2e-5), ("saved_tc", 1e-3)):
        got = _run(ahv, form, args, True, h1, pinv)
        for name, a, r in zip(NAMES, got, ref):
            err = float((a.double() - r.reshape(a.shape)).abs().max()) / float(r.abs().max())
            assert err <= tol, (per_pair, shrink, form, name, err)


E2E = textwrap.dedent(r"""
    import importlib, json, sys
    import numpy as np
    import torch
    sys.path.insert(0, sys.argv[1])
    torch.use_deterministic_algorithms(True)
    ahv = importlib.import_module("3dahv_b200")
    from modules.modules import Feature_Aligner
    dev = torch.device("cuda", 0)

    def run(save):
        torch.manual_seed(0)
        fa = Feature_Aligner(in_channel=768, mid_channel=256, out_channel=32, n_heads=4, depth=1).to(dev)
        gen = torch.Generator().manual_seed(1)
        B, N = 4, 700
        a = torch.randn(B, 768, 8, 8, generator=gen).to(dev).requires_grad_(True)
        b = torch.randn(B, 768, 8, 8, generator=gen).to(dev).requires_grad_(True)
        gt = ahv.so3.sample_rotations(B, seed=1, device=dev)
        R = torch.cat([gt[:, None], ahv.so3.sample_rotations(B * (N - 1), seed=2, device=dev).reshape(B, N - 1, 3, 3)], 1)
        vs, vt = fa.forward_2d3d(a, b, random_mask=False, mask_ratio=0.0)
        head = fa.feature_embedding_2d
        s = ahv.training.verification_scores(vs, vt, R.contiguous(), head[0].weight, head[2].weight, head[2].bias,
                                             save_activations=save)
        ahv.training.infonce_loss(s, R, gt, acc_thr_deg=15.0).mean().backward()
        grads = {n: p.grad for n, p in fa.named_parameters() if p.grad is not None}
        grads["img_feat_src"], grads["img_feat_tgt"] = a.grad, b.grad
        return grads

    out = {}
    for save in (False, True):
        g1, g2 = run(save), run(save)
        assert g1.keys() == g2.keys()
        out[str(save)] = {"n": len(g1), "differ": sorted(k for k in g1 if not torch.equal(g1[k].view(torch.int32), g2[k].view(torch.int32))),
                          "head": [k for k in g1 if k.startswith("feature_embedding_2d")]}
    print(json.dumps(out))
""")


def test_end_to_end_training_step_is_bit_reproducible_in_a_fresh_process(ahv):
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    p = subprocess.run([sys.executable, "-c", E2E, ROOT], env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-4000:]
    import json

    res = json.loads(p.stdout.strip().splitlines()[-1])
    for save, r in res.items():
        assert r["differ"] == [], (save, r["differ"])
        assert len(r["head"]) == 3 and r["n"] > 10, r   # W1, W2, b2 of the head, the aligner's parameters, both inputs


def test_paths_without_a_deterministic_form_alert_under_the_flag(ahv, golden, monkeypatch):
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")   # the head's matmuls under the flag
    args = _inputs(ahv, golden, 2, 20, False, seed=29)
    vs, tgt, R, W1, W2, b2, gs = args
    vt = torch.randn(2, 16, 8, 8, 8, device=DEV)

    def chunked():
        v = vs.clone().requires_grad_(True)
        s = ahv.training.verification_scores(v, vt, R, W1, W2, b2, chunk=8, fused_backward=False)
        s.sum().backward()

    def rotate():
        v = vs[0].clone().requires_grad_(True)
        ahv.training.rotate_volume(v, R).sum().backward()

    try:
        torch.use_deterministic_algorithms(True)
        for fn in (chunked, rotate):
            with pytest.raises(RuntimeError, match="ahv_rotate_volume_backward"):
                fn()
        torch.use_deterministic_algorithms(True, warn_only=True)
        for fn in (chunked, rotate):
            with pytest.warns(UserWarning, match="ahv_rotate_volume_backward"):
                fn()
    finally:
        torch.use_deterministic_algorithms(False)
    rotate()   # no alert without the flag
    chunked()


def test_the_flag_picks_the_atomic_or_deterministic_entry(ahv, golden, monkeypatch):
    """Without the flag the training path calls the atomic entries: ahv_score_backward_saved for saved activations on
    tcgen05, ahv_score_backward_ex for every other form; with it, the deterministic one."""
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")   # the head's matmuls under the flag
    args = _inputs(ahv, golden, 2, 30, True, seed=31)
    vs, tgt, R, W1, W2, b2, gs = args
    vt = torch.randn(2, 16, 8, 8, 8, device=DEV)
    called = []
    real = ahv.ops._call
    monkeypatch.setattr(ahv.ops, "_call", lambda name, *a: (called.append(name), real(name, *a))[1])

    def step(save, want_R):
        v = vs.clone().requires_grad_(True)
        Rl = R.clone().requires_grad_(want_R)
        s = ahv.training.verification_scores(v, vt, Rl, W1, W2, b2, save_activations=save)
        called.clear()
        (s * gs).sum().backward()
        return [c for c in called if c.startswith("ahv_score_backward")]

    expect_atomic = {(False, False): "ahv_score_backward_ex", (True, False): "ahv_score_backward_saved",
                     (False, True): "ahv_score_backward_ex", (True, True): "ahv_score_backward_ex"}
    for (save, want_R), name in expect_atomic.items():
        assert step(save, want_R) == [name], (save, want_R)
    try:
        torch.use_deterministic_algorithms(True)
        for save, want_R in expect_atomic:
            assert step(save, want_R) == ["ahv_score_backward_det"], (save, want_R)
    finally:
        torch.use_deterministic_algorithms(False)
