"""Every output of the selection chains of ahv_api.cu on fixed seeded inputs, saved to one .npz per library; and the
comparison of two such files.  A change to the host layer that is meant to keep the launch sequence keeps every bit.

    python scripts/chain_bits.py OUT_DIR [TAG]         # writes OUT_DIR/chain_bits_TAG.npz (AHV_VARIANT_LIB: another build)
    python scripts/chain_bits.py --compare A.npz B.npz  # prints one JSON line, exit status 1 on a mismatch
    python scripts/chain_bits.py --sizes A.so B.so      # every workspace-size entry of two builds over a grid of sizes
                                                        # (no device needed); one JSON line, exit status 1 on a mismatch

Entries, through their ops wrappers, for fp32 and bf16 source volumes under MATH_TC and MATH_FP32:
  ahv_verify                    k = 1 without scores (screened at 32 x 50 000 with fp32 volumes under MATH_TC), k = 1
                                with scores (the single pass), k = 4; B x N = 32 x 50 000 (config 2) and 3 x 3 000 per pair
  ahv_refine                    k = 8, m = 16
  ahv_refine_gradient(_distinct) k = 8, min_sep_deg 0 and 15
  ahv_search_hierarchical       base level 2, 3 levels, k = 8
  ahv_search_modes              base level 2, 3 levels, k = 8, beam 4, 30 degrees
  ahv_score                     k = 0 (scores only) and k = 4 with scores, on ahv_forward_3d2d's target features
  ahv_score_train               fp32 volumes (scores, h1, pair scales)
  ahv_gradient_ascent           8 starting rotations per pair, 10 steps
  ahv_verify_sharded and ahv_refine_gradient_sharded at world 1, and at world 2 as two in-process ranks on one GPU (the
  launcher of tests/test_gpu_sharded_refine.py; its buffers hold 4 pairs and 3 000 scores, so B = 4 there).  World 2
  also runs ahv_verify_sharded at k = 4 with shards shorter than k (N = 5) and with an empty shard (N = 1).
"""
import importlib, json, os, sys
from types import SimpleNamespace

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [(32, 50000, False), (3, 3000, True)]   # B, N, one rotation set per pair


def compare(a_path, b_path):
    a, b = np.load(a_path), np.load(b_path)
    bad = [] if sorted(a.files) == sorted(b.files) else ["different keys"]
    for k in sorted(set(a.files) & set(b.files)):
        x, y = a[k], b[k]
        if x.shape != y.shape or x.dtype != y.dtype or x.tobytes() != y.tobytes():
            bad.append(k)
    print(json.dumps({"a": a_path, "b": b_path, "arrays": len(a.files), "mismatches": bad}))
    return not bad


def _size_calls():
    """(entry, argtypes, argument tuples): each size entry over a grid with 0, invalid sizes and k up to 32."""
    from ctypes import c_int, c_int64
    from itertools import product
    Bs, Ns, ks = (-1, 0, 1, 3, 32, 257), (-1, 0, 1, 5, 3000, 50000, 2**31 - 1, 2**31), (-1, 0, 1, 2, 4, 8, 31, 32, 33)
    BNk = list(product(Bs, Ns, ks))
    levels = (-1, 0, 1, 2, 3, 6, 7)
    return [
        ("ahv_workspace_bytes", (c_int, c_int64, c_int), BNk),
        ("ahv_refine_workspace_bytes", (c_int, c_int64, c_int, c_int), [a + (m,) for a in BNk for m in (0, 1, 16)]),
        ("ahv_refine_gradient_workspace_bytes", (c_int, c_int64, c_int), BNk),
        ("ahv_refine_gradient_sharded_workspace_bytes", (c_int, c_int64, c_int, c_int),
         [a + (w,) for a in BNk for w in range(0, 10)]),
        ("ahv_search_hierarchical_workspace_bytes", (c_int, c_int, c_int), list(product(Bs, levels, ks))),
        ("ahv_search_modes_workspace_bytes", (c_int, c_int, c_int, c_int),
         [a + (w,) for a in product(Bs, levels, ks) for w in range(0, 10)]),
        ("ahv_posterior_mass_workspace_bytes", (c_int, c_int64, c_int), BNk),
        ("ahv_posterior_moments_workspace_bytes", (c_int, c_int64, c_int), BNk),
        ("ahv_score_backward_det_workspace_bytes", (c_int, c_int64, c_int, c_int),
         [(B, N, r, g) for B, N in product(Bs, Ns) for r in (0, 1) for g in (0, 1)]),
    ]


def sizes(a_path, b_path):
    """Every workspace size, and whether ahv_verify screens, from two builds; these entries do not touch the device."""
    import ctypes
    libs = [ctypes.CDLL(os.path.abspath(p)) for p in (a_path, b_path)]
    bad, n = [], 0
    for name, argtypes, calls in _size_calls():
        fns = [getattr(lib, name) for lib in libs]
        for f in fns:
            f.argtypes, f.restype = list(argtypes), ctypes.c_size_t
        for args in calls:
            x, y = (f(*args) for f in fns)
            n += 1
            if x != y:
                bad.append([name, args, x, y])
    for B in (0, 1, 3, 32, 257):
        for N in (0, 1, 3000, 40000, 50000, 100000, 2**20):
            flags = []
            for lib in libs:
                v = ctypes.c_int(-7)
                st = lib.ahv_verify_screen_stats(None, B, ctypes.c_int64(N), ctypes.byref(v), None, None, None)
                flags.append((st, v.value))
            n += 1
            if flags[0] != flags[1]:
                bad.append(["ahv_verify_screen_stats", (B, N), flags[0], flags[1]])
    print(json.dumps({"a": a_path, "b": b_path, "calls": n, "mismatches": bad[:20], "n_mismatches": len(bad)}))
    return not bad


def run(out_dir, tag):
    import torch
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    ahv = importlib.import_module("3dahv_b200")
    if os.environ.get("AHV_VARIANT_LIB"):   # scripts-only: another build of the library
        ahv._lib.LIB_PATH = os.path.abspath(os.environ["AHV_VARIANT_LIB"])
    from test_gpu_sharded_refine import _Ranks

    ops = ahv.ops
    dev = torch.device("cuda", 0)
    w = np.load(os.path.join(ROOT, "tests", "golden", "weights.npz"))
    head = tuple(torch.from_numpy(w[k]).to(dev) for k in ("W1", "W2", "b2"))
    out = {}

    def save(name, tensors):
        for i, t in enumerate(tensors):
            if isinstance(t, torch.Tensor):
                out[f"{name}/{i}"] = t.detach().cpu().numpy()

    def volumes(B, seed, bf16):
        gen = torch.Generator().manual_seed(seed)
        vs = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 0.5).to(dev)
        vt = (torch.randn(B, 16, 8, 8, 8, generator=gen) * 0.5).to(dev)
        return (vs.bfloat16() if bf16 else vs), vt

    modes = [(bf16, math) for bf16 in (False, True) for math in (ahv.MATH_TC, ahv.MATH_FP32)]
    for B, N, per_pair in SIZES:
        R = ahv.so3.sample_rotations(B * N if per_pair else N, seed=N + 5, device=dev)
        R = R.reshape(B, N, 3, 3) if per_pair else R
        for bf16, math in modes:
            vs, vt = volumes(B, B * 7 + N, bf16)
            case = f"{B}x{N}{'_pp' if per_pair else ''}/{'bf16' if bf16 else 'fp32'}/math{math}"
            save(f"verify_k1/{case}", ops.verify(vs, vt, R, *head, k=1, math=math))
            save(f"verify_k1_scores/{case}", ops.verify(vs, vt, R, *head, k=1, math=math, return_scores=True))
            save(f"verify_k4/{case}", ops.verify(vs, vt, R, *head, k=4, math=math))
            tf = ops.forward_3d2d(vt, *head)
            save(f"score_k0/{case}", ops.score(vs, tf, R, *head, k=0, math=math))
            save(f"score_k4/{case}", ops.score(vs, tf, R, *head, k=4, math=math))
            if not bf16 and math == ahv.MATH_TC:
                save(f"score_train/{case}", ops.score_train(vs, tf, R, *head))
            if math == ahv.MATH_TC:   # the ascent scores in fp32 whatever the math mode
                R0 = ahv.so3.sample_rotations(B * 8, seed=B + 11, device=dev).reshape(B, 8, 3, 3)
                save(f"gradient_ascent/{case}", ops.gradient_ascent(vs, tf, R0, *head, steps=10))
            save(f"refine/{case}", ops.refine(vs, vt, R, *head, k=8, m=16, max_angle_deg=4.0, seed=3, math=math)[:7])
            for sep in (0.0, 15.0):
                save(f"refine_gradient_sep{sep}/{case}",
                     ops.refine_gradient(vs, vt, R, *head, k=8, steps=10, math=math, min_sep_deg=sep)[:8])
            one = SimpleNamespace(rank=0, world=1, ptrs=[], max_pairs=32, max_k=32, max_hyps=0)
            save(f"verify_sharded_w1/{case}", ops.verify_sharded(vs, vt, R, *head, 0, one, k=4, math=math))
            for sep in (0.0, 15.0):
                save(f"refine_gradient_sharded_w1_sep{sep}/{case}",
                     ops.refine_gradient_sharded(vs, vt, R, *head, one, k=8, steps=10, math=math, min_sep_deg=sep)[:8])
    for bf16, math in modes:
        vs, vt = volumes(8, 17, bf16)
        save(f"search_hierarchical/8/{'bf16' if bf16 else 'fp32'}/math{math}",
             ops.search_hierarchical(vs, vt, *head, base_level=2, levels=3, k=8, math=math)[:6])
        save(f"search_modes/8/{'bf16' if bf16 else 'fp32'}/math{math}",
             ops.search_modes(vs, vt, *head, base_level=2, levels=3, k=8, beam=4, min_sep_deg=30.0, math=math)[:6])

    # world 2: B = 4 pairs, N = 3 000 shared hypotheses (the in-process ranks' exchange capacity)
    B, N, world = 4, 3000, 2
    R = ahv.so3.sample_rotations(N, seed=N + 5, device=dev)
    ranks = _Ranks(ahv, world, dev)
    try:
        for bf16, math in modes:
            vs, vt = volumes(B, 29, bf16)
            case = f"{B}x{N}/{'bf16' if bf16 else 'fp32'}/math{math}"
            for k in (1, 4):
                def step(r, peer, k=k):
                    lo, hi = ahv.dist.shard_bounds(N, r, world)
                    return ops.verify_sharded(vs, vt, R[lo:hi], *head, lo, peer, k=k, math=math)
                for r, res in enumerate(ranks.run(step, 1)):
                    save(f"verify_sharded_w2_k{k}/{case}/rank{r}", res)
            for sep in (0.0, 15.0):
                res = ranks.run(lambda r, peer, sep=sep: ops.refine_gradient_sharded(
                    vs, vt, R, *head, peer, k=8, steps=10, math=math, min_sep_deg=sep)[:8], 2)
                for r, rr in enumerate(res):
                    save(f"refine_gradient_sharded_w2_sep{sep}/{case}/rank{r}", rr)
            for n in (5, 1):   # shards of 3 and 2, and of 1 and 0, hypotheses at k = 4
                def short(r, peer, n=n):
                    lo, hi = ahv.dist.shard_bounds(n, r, world)
                    return ops.verify_sharded(vs, vt, R[lo:hi], *head, lo, peer, k=4, math=math)
                for r, res in enumerate(ranks.run(short, 1)):
                    save(f"verify_sharded_w2_N{n}_k4/{B}x{n}/{'bf16' if bf16 else 'fp32'}/math{math}/rank{r}", res)
    finally:
        ranks.close()
    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, f"chain_bits_{tag}.npz")
    np.savez(path, **out)
    print(json.dumps({"wrote": path, "arrays": len(out), "gpu": torch.cuda.get_device_name(dev), "lib": ahv._lib.LIB_PATH}))


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        sys.exit(0 if compare(sys.argv[2], sys.argv[3]) else 1)
    if sys.argv[1] == "--sizes":
        sys.exit(0 if sizes(sys.argv[2], sys.argv[3]) else 1)
    run(sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else "lib")
