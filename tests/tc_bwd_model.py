"""numpy model of the tensor-core backward's arithmetic (csrc/ahv_score_bwd_tc.cu, atomic and deterministic forms).

TEST INFRASTRUCTURE ONLY.  It restates, rounding for rounding, what the saved-activation backward computes from the
training forward's kept conv1 output (h1, fp16) and pair factor (pair_inv = 2^e1 / s), so that the suite can hold the
kernel to what the model leaves out - the tensor core's fp32 accumulation inside each MMA and the order of the fp32
sums across items, CTAs and atomics, which the model takes in fp64 - instead of to 1e-3 of fp64:

  fp32 gather     gather_rotated: kernel_arith.gather32 with make_tap's coordinate order fmaf(R2, z, fmaf(R1, y, R0 x))
                  (not the tensor-core scorer's) and the x-tap swap (line ^ w) & 1 (parity="w").
  A^T operand     RN16(X * s), s = 1 / (pair_inv 2^-e1).
  packing         W1h = RN16(W1 2^-e1), W2h = RN16(W2 2^-e2) with tc_model's exponents; kappa from the fp32 column
                  L1 sums of W1h (o = 0 .. 31 in order): 2^floor(log2(2 / (3 c))).
  conv2           v = fmaf(acc, pinv 2^e2, b2); |v|^2 and <v, T> by kernel_arith.head_dots; the 1e-12 clamp;
                  dH2 = (g/64) inv (T - F <F,T>), dT += (g/64) F, db2 += dH2.
  per-item scales dH2: 2^(13 - e), e = floor(log2(2 |g/64| / max(sqrt(min_p |v_p|^2), 1e-12))) (13 when that is 0);
                  dH1: 2^(13 - e), e = floor(log2 max |dH1|) (13 when 0); both clamped to [-100, 100].
  fp16 operands   dH2h = RN16(dH2 S2), dH1h = RN16(mask (dH2h W2h) 2^(e2 - ...) S), mask = kept h1 > 0.
  dX fold         view x: RN16(acc_x kappa); views y, z: RN16(fmaf(acc, kappa, dX)) in that order (double rounding).
  adjoint         make_tap's corners; row path: weight (wx wy) wz in fp32 -> unorm16 __float2uint_rn(w 65535), read
                  back as float(w16) * (unscale * fp32(1/65535)); the exact path (some input voxel collects more than 16
                  contributions, zero weights included) keeps the fp32 weight times unscale.
  outputs         dW1 = acc (invS pvol), dW2 = acc (inv_s2 pinv), dV = dX unscale-weighted, dT, db2.

The roundings, taps, gathers and head_dots are kernel_arith's.  `rounding=False` evaluates every step in fp64: the
exact gradient of the function the forward ran (its kept H1 and that value's ReLU mask).  `rz` names sites whose
conversion is made round-toward-zero instead: "AT" (the A^T operand), "W1t" (the W1^T operand), "dH2", "dH1", "dX"
(all three fold conversions), "w16" (__float2uint_rz) - the defects the gates of tests/test_gpu_tc_bwd_model.py must
see.  `fold` is the order the three views are folded in ("xyz", as the kernel).
"""
from __future__ import annotations

import numpy as np

import tc_model as M
from kernel_arith import (C, KTRI, NPOS, OCH, S, VOX, exp_bits, fma32, gather32, gather64, head_dots, lattice_rotations,
                          outside_rotations, random_rotations, random_volumes, rn16, run_chunks, rz16, sample_coords,
                          sample_coords64, tap_at, trained_like)
from oracle import ahv_oracle as oracle

LIST_CAP = 16                                                   # kListCap: contributions a row of the work list holds
f16, f32, f64 = np.float16, np.float32, np.float64
GRADS = ("vol_src", "tgt_feat", "W1", "W2", "b2")


# ---- scalar helpers -------------------------------------------------------------------------------------------------
def _pow2(e) -> np.ndarray:
    return np.ldexp(f32(1.0), np.asarray(e, np.int64)).astype(f32)


def item_scale(m) -> tuple[np.ndarray, np.ndarray]:
    """(S, 1/S) of an item whose bound is m (fp32): S = 2^(13 - e), e = floor(log2 m) clamped to [-100, 100], so that
    2^13 <= m S < 2^14; e = 13 (S = 1) when m is not positive."""
    m = np.asarray(m, f32)
    e = np.where(m > 0, np.clip(exp_bits(m), -100, 100), 13)
    return _pow2(13 - e), _pow2(e - 13)


def dh2_bound(g64, ssmin) -> np.ndarray:
    """2 |g/64| / max(sqrt(min_p |H2_p|^2), 1e-12) in fp32, the bound the dH2 scale is taken from."""
    g64, ssmin = np.asarray(g64, f32), np.asarray(ssmin, f32)
    return (f32(2.0) * np.abs(g64) / np.maximum(np.sqrt(ssmin), f32(1e-12))).astype(f32)


def kappa_of(W1h: np.ndarray, e1: int) -> tuple[f32, f32]:
    """(kappa, inv_kappa): kappa = 2^e, e = floor(log2(2 / (3 c))) clamped to [-60, 60], c the largest column L1 norm
    of W1h summed in fp32 over o = 0 .. 31; inv_kappa = 2^-e 2^e1.  (1, 2^e1) when W1h is zero."""
    col = np.zeros(KTRI, f32)
    a = np.abs(W1h.astype(f32))
    for o in range(OCH):
        col = (col + a[o]).astype(f32)
    c = f32(col.max())
    w1s = f32(np.ldexp(1.0, e1))
    if not c > 0:
        return f32(1.0), w1s
    x = f32(f32(2.0) / f32(f32(3.0) * c))
    e = int(np.clip(exp_bits(x), -60, 60))
    return f32(np.ldexp(1.0, e)), f32(f32(np.ldexp(1.0, -e)) * w1s)


def unorm16(w, rz: bool = False) -> np.ndarray:
    """__float2uint_rn(w * 65535.0f) (ties to even), or __float2uint_rz: the adjoint's 16-bit weights."""
    p = (np.asarray(w, f32) * f32(65535.0)).astype(f32)
    return (np.floor(p) if rz else np.rint(p)).astype(np.int64)


# ---- the adjoint's taps ---------------------------------------------------------------------------------------------
def corners(taps):
    """The 8 (input voxel [n,512], inside [n,512], weight (wx wy) wz [n,512]) of every output voxel, dlt = dx + 2 dy +
    4 dz as list_pass walks them; weights in the taps' precision."""
    (x0, y0, z0), (fx, fy, fz), _ = taps
    one = fx.dtype.type(1.0)
    out = []
    for dlt in range(8):
        dx, dy, dz = dlt & 1, (dlt >> 1) & 1, dlt >> 2
        x, y, z = x0 + dx, y0 + dy, z0 + dz
        inside = (x >= 0) & (x < 8) & (y >= 0) & (y < 8) & (z >= 0) & (z < 8)
        w = ((fx if dx else one - fx) * (fy if dy else one - fy)).astype(fx.dtype) * (fz if dz else one - fz)
        out.append((np.where(inside, z * 64 + y * 8 + x, 0), inside, w.astype(fx.dtype)))
    return out


def contributions(R: np.ndarray, base=None) -> np.ndarray:
    """The largest number of contributions any input voxel collects, per matrix R [n,3,3] (the work list's row holds
    LIST_CAP; above that the item takes the exact path)."""
    R = np.asarray(R, f32).reshape(-1, 9)
    cs = corners(tap_at(sample_coords(R, base)))
    n = len(R)
    cnt = np.zeros((n, VOX), np.int64)
    rows = np.repeat(np.arange(n)[:, None], VOX, 1)
    for v, inside, _ in cs:
        np.add.at(cnt, (rows[inside], v[inside]), 1)
    return cnt.max(axis=1)


def fold_views(dA: np.ndarray):
    """dA [n,64 pos,384 k] -> its three views as [n,16,8,8,8] (c, d, h, w) arrays, in the order x, y, z (the adjoint of
    oracle.triplane_np)."""
    n = dA.shape[0]
    v = dA.reshape(n, 8, 8, 3, C, 8)                           # [n, pos/8, pos%8, view, c, k%8]
    x = v[:, :, :, 0].transpose(0, 3, 1, 2, 4)                 # pos (d, h), k (c, w)
    y = v[:, :, :, 1].transpose(0, 3, 1, 4, 2)                 # pos (d, w), k (c, h)
    z = v[:, :, :, 2].transpose(0, 3, 4, 1, 2)                 # pos (h, w), k (c, d)
    return {"x": x, "y": y, "z": z}


# ---- the backward ---------------------------------------------------------------------------------------------------
def base64_coords() -> np.ndarray:
    """The base coordinates torch's affine_grid makes in fp64 (linspace(-1, 1, 8) * 7/8): what fp64 autograd samples."""
    return np.linspace(-1.0, 1.0, 8) * (7.0 / 8.0)


def tc_backward(vol_src, tgt_feat, R, W1, W2, b2, grad_scores, h1, pair_inv, *, rounding: bool = True, rz=(),
                fold: str = "xyz", base=None, base64=None, chunk: int = 96, info: bool = False):
    """Gradients (vol_src [B,16,8,8,8], tgt_feat [B,32,64], W1 [32,384], W2 [32,32], b2 [32]) in fp64 of
    sum(grad_scores * scores) as the tensor-core backward computes them from the kernel's own h1 [B*N,64,32] fp16 and
    pair_inv [B].  R [N,3,3] shared or [B,N,3,3] per pair.  info=True also returns, per item, whether the adjoint
    took the exact path and the largest contribution count of an input voxel."""
    vs = np.asarray(vol_src, f32).reshape(-1, C, S, S, S)
    tg = np.asarray(tgt_feat, f32).reshape(-1, OCH, NPOS)
    B = vs.shape[0]
    R = np.asarray(R, f32)
    per_pair = R.ndim == 4
    N = R.shape[1] if per_pair else R.shape[0]
    Rall = R.reshape(-1, 9) if per_pair else R.reshape(N, 9)
    gs = np.asarray(grad_scores, f32).reshape(-1)
    h1 = np.asarray(h1, f16).reshape(-1, NPOS, OCH)
    pinv = np.asarray(pair_inv, f32).reshape(B)
    rz = tuple(rz)
    b2v = np.asarray(b2, f32).reshape(OCH)
    if rounding:
        W1h, W2h, e1, e2 = M.packed_weights(W1, W2, ("W1h",) if "W1t" in rz else ())
        kappa, inv_kappa = kappa_of(M.packed_weights(W1, W2)[0], e1)   # from RN16 W1 whatever the operand's rounding
        W1d, W2d = W1h.astype(f64), W2h.astype(f64)
        n1, w2s = f32(np.ldexp(1.0, -e1)), f32(np.ldexp(1.0, e2))
    else:
        W1d, W2d = np.asarray(W1, f64).reshape(OCH, KTRI), np.asarray(W2, f64).reshape(OCH, OCH)
        base64 = base64_coords() if base64 is None else np.asarray(base64, f64)
    wq_unit = f32(f32(1.0) / f32(65535.0))

    def run(i0):
        items = np.arange(i0, min(i0 + chunk, B * N))
        n = len(items)
        pair = items // N
        Rc = Rall[items if per_pair else items % N]
        used, slot = np.unique(pair, return_inverse=True)
        g_item = gs[items]
        H = h1[items].astype(f64)                              # [n,64 pos,32 ch] kept value in the kernel's units
        tgp = tg[pair].transpose(0, 2, 1)                      # [n,64,32]
        out = {"vol_src": np.zeros((len(used), C, VOX)), "tgt_feat": np.zeros((len(used), NPOS, OCH)),
               "W1": np.zeros((OCH, KTRI)), "W2": np.zeros((OCH, OCH)), "b2": np.zeros(OCH)}
        if rounding:
            taps = tap_at(sample_coords(Rc, base))
            X = gather32(vs[used], Rc, base, slot)             # [n,16,512] fp32
            pv = (pinv[pair] * n1).astype(f32)                 # 1/s
            sb = (f32(1.0) / pv).astype(f32)
            Xs = (X * sb[:, None, None]).astype(f32)
            AT = (rz16(Xs) if "AT" in rz else rn16(Xs)).astype(f64)
            tri = oracle.triplane_np(AT.reshape(n, C, S, S, S)).reshape(n, KTRI, NPOS)
            acc2 = np.einsum("npi,oi->npo", H, W2d).astype(f32)
            v = fma32(acc2, (pinv[pair] * w2s).astype(f32)[:, None, None], b2v)      # [n,64,32] fp32
            ss, ft = head_dots(v, tgp)
            nraw = np.sqrt(ss)
            inv = (f32(1.0) / np.maximum(nraw, f32(1e-12))).astype(f32)[..., None]
            fdot = (ft[..., None] * inv).astype(f32)
            g64 = (g_item * f32(1.0 / 64.0)).astype(f32)[:, None, None]
            F = (v * inv).astype(f32)
            par = np.where((nraw < f32(1e-12))[..., None], tgp, fma32(-F, fdot, tgp))
            d2 = ((g64 * inv).astype(f32) * par).astype(f32)
            S2, inv_s2 = item_scale(dh2_bound(g64[:, 0, 0], ss.min(axis=1)))
            p2 = (d2 * S2[:, None, None]).astype(f32)
            dH2h = (rz16(p2) if "dH2" in rz else rn16(p2)).astype(f64)
            accH1 = np.einsum("npo,oi->npi", dH2h, W2d).astype(f32)
            dh1 = np.where(H > 0, (accH1 * (inv_s2 * w2s).astype(f32)[:, None, None]).astype(f32), f32(0.0))
            Sd, invS = item_scale(np.abs(dh1).max(axis=(1, 2)))
            p1 = (dh1 * Sd[:, None, None]).astype(f32)
            dH1h = (rz16(p1) if "dH1" in rz else rn16(p1)).astype(f64)
            accW2 = np.einsum("npo,npi->noi", dH2h, H).astype(f32)
            out["W2"] += np.einsum("noi,n->oi", accW2.astype(f64), (inv_s2 * pinv[pair]).astype(f32).astype(f64))
            accW1 = np.einsum("npo,nkp->nok", dH1h, tri).astype(f32)
            out["W1"] += np.einsum("nok,n->ok", accW1.astype(f64), (invS * pv).astype(f32).astype(f64))
            views = fold_views(np.einsum("npo,ok->npk", dH1h, W1d).astype(f32))
            dX = None
            for vname in fold:
                a = views[vname].reshape(n, C, VOX)
                p = (a * kappa).astype(f32) if dX is None else fma32(a, kappa, dX)
                dX = (rz16(p) if "dX" in rz else rn16(p)).astype(f32)
            unscale = (invS * inv_kappa).astype(f32)
            cs = corners(taps)
            cnt = np.zeros((n, VOX), np.int64)
            rows = np.repeat(np.arange(n)[:, None], VOX, 1)
            for vi, inside, _ in cs:
                np.add.at(cnt, (rows[inside], vi[inside]), 1)
            exact = cnt.max(axis=1) > LIST_CAP
            wq = (unscale * wq_unit).astype(f32)[:, None]
            wts = []
            for vi, inside, w in cs:
                row = (unorm16(w, "w16" in rz).astype(f32) * wq).astype(f32)
                ex = (w * unscale[:, None]).astype(f32)
                wts.append(np.where(exact[:, None], ex, row))
            dT = g64.astype(f64) * F.astype(f64)
            dX = dX.astype(f64)
        else:
            taps = tap_at(sample_coords64(Rc, base64))
            X = gather64(vs[used], Rc, base64, slot)
            tri = oracle.triplane_np(X.reshape(n, C, S, S, S)).reshape(n, KTRI, NPOS)
            Ht = H * pinv[pair].astype(f64)[:, None, None]
            v = np.einsum("npi,oi->npo", Ht, W2d) + b2v.astype(f64)
            nraw = np.sqrt((v * v).sum(axis=2, keepdims=True))
            inv = 1.0 / np.maximum(nraw, 1e-12)
            F = v * inv
            fdot = (F * tgp).sum(axis=2, keepdims=True)
            g64 = (g_item.astype(f64) / 64.0)[:, None, None]
            d2 = g64 * inv * np.where(nraw < 1e-12, tgp, tgp - F * fdot)
            dh1 = np.where(H > 0, np.einsum("npo,oi->npi", d2, W2d), 0.0)
            out["W2"] += np.einsum("npo,npi->oi", d2, Ht)
            out["W1"] += np.einsum("npo,nkp->ok", dh1, tri)
            views = fold_views(np.einsum("npo,ok->npk", dh1, W1d))
            dX = sum(views[c] for c in "xyz").reshape(n, C, VOX)
            cs = corners(taps)
            wts = [w for _, _, w in cs]
            exact = np.zeros(n, bool)
            cnt = np.zeros((n, VOX), np.int64)
            dT = g64 * F
        out["b2"] += d2.astype(f64).sum(axis=(0, 1))
        np.add.at(out["tgt_feat"], slot, dT)
        dV = out["vol_src"]
        for (vi, inside, _), w in zip(cs, wts):
            idx = (slot[:, None] * VOX + vi)[inside]
            for c in range(C):
                dV[:, c] += np.bincount(idx, (w.astype(f64) * dX[:, c])[inside], len(used) * VOX).reshape(len(used), VOX)
        return used, out, exact, cnt.max(axis=1)

    res = {"vol_src": np.zeros((B, C, VOX)), "tgt_feat": np.zeros((B, NPOS, OCH)), "W1": np.zeros((OCH, KTRI)),
           "W2": np.zeros((OCH, OCH)), "b2": np.zeros(OCH)}
    exact, count = np.zeros(B * N, bool), np.zeros(B * N, np.int64)
    starts = range(0, B * N, chunk)
    for i0, (used, out, ex, cn) in zip(starts, run_chunks(run, starts)):    # the chunks' sums added in chunk order
        res["vol_src"][used] += out["vol_src"]
        res["tgt_feat"][used] += out["tgt_feat"]
        for k in ("W1", "W2", "b2"):
            res[k] += out[k]
        exact[i0 : i0 + len(ex)], count[i0 : i0 + len(cn)] = ex, cn
    grads = {"vol_src": res["vol_src"].reshape(B, C, S, S, S), "tgt_feat": res["tgt_feat"].transpose(0, 2, 1).copy(),
             "W1": res["W1"], "W2": res["W2"], "b2": res["b2"]}
    if info:
        return grads, {"exact": exact, "count": count}
    return grads


# ---- comparison -----------------------------------------------------------------------------------------------------
def residual(got, ref) -> dict:
    """Per-element (largest |got - ref| / max |ref|) and L2 (|got - ref| / |ref|) residuals of one gradient, and the
    flat index of the worst element.  A zero reference asks for a zero result."""
    got, ref = np.asarray(got, f64).reshape(-1), np.asarray(ref, f64).reshape(-1)
    d = np.abs(got - ref)
    mx, nrm = float(np.abs(ref).max()), float(np.linalg.norm(ref))
    at = int(np.argmax(d))
    elem = float(d[at]) / mx if mx > 0 else (0.0 if d[at] == 0 else np.inf)
    l2 = float(np.linalg.norm(got - ref)) / nrm if nrm > 0 else (0.0 if d[at] == 0 else np.inf)
    return {"elem": elem, "l2": l2, "at": at}


# Gates of tests/test_gpu_tc_bwd_model.py, relative to each gradient's maximum (per element) and norm (L2), against
# this model.  Set from the residuals measured on a B200 at 1 000 W (profiles/r17_tc_bwd_model_residual.json, 24 cases x
# 2 forms): each is at least three times the largest residual of its gradient and metric.  Largest per element / L2:
# vol_src 2.3e-4 / 4.7e-5, tgt_feat 5.2e-7 / 2.2e-7, W1 1.9e-5 / 1.3e-5, W2 1.6e-5 / 4.6e-6, b2 1.2e-6 / 8.6e-7.  The
# vol_src residual is the fp16 rounding of dX turning the other way where the tensor core's fp32 sum of dA differs from
# the model's in its last bits (a few dX elements per item move by one fp16 ulp); it is largest where a pair has few
# items (lattice 2 x 24, 300 x 3) and the atomic and deterministic forms show the same.  On the golden case every
# round-toward-zero defect but the adjoint's weights (w16) moves some gradient by 4.0x to 24x its gate; w16 (0.4x) and
# folding the views in the order y, x, z (1.8x) move only vol_src and stay within 3x of it on the golden case
# (tests/test_oracle_tc_bwd_model.py).  Built into the kernel, the fold order still fails most cases of the GPU file,
# where pairs with few items let its per-element shift exceed the gate; truncated weights fail none.
GATE = {"vol_src": {"elem": 7.5e-4, "l2": 1.5e-4}, "tgt_feat": {"elem": 2e-6, "l2": 7e-7},
        "W1": {"elem": 6e-5, "l2": 4e-5}, "W2": {"elem": 5e-5, "l2": 1.5e-5}, "b2": {"elem": 4e-6, "l2": 3e-6}}


# ---- the cases tests/test_gpu_tc_bwd_model.py and scripts/tc_bwd_model_residual.py run -------------------------------
CASES = (["golden"]
         + ["shape_1x1", "shape_1x3", "shape_3x49_per_pair", "shape_300x3", "shape_12x400_per_pair"]
         + ["lattice", "outside", "R_x0.35", "R_mixed_x0.35"]
         + ["vol_x1e-3", "vol_x300", "outlier_4e3"]
         + ["W1_x2^12", "W1_x2^-12", "W1_x40", "W2_x0.05", "student_t", "row_scales", "zero_rows"]
         + ["g_decades", "g_x1e6", "g_x1e-8", "zero_conv2"])


def make_case(name: str, golden: dict) -> dict:
    """Inputs of one case: vs [B,16,8,8,8], tgt [B,32,64] (the target features the kernel and the model are given),
    R [N,3,3] or [B,N,3,3], W1, W2, b2, gs [B,N] (the upstream gradient)."""
    g, w = golden["shared_n3000_b3"], golden["weights"]
    W1, W2, b2 = (np.asarray(w[k], f32) for k in ("W1", "W2", "b2"))
    rng = np.random.default_rng(sum(map(ord, name)) * 7919 + len(name))
    vs, vt = g["vol_src"], g["vol_tgt"]
    B, N, per_pair = 3, 200, False
    R = None
    tgt_w = None                                              # head weights of the target side, when not the case's
    if name == "golden":
        B, N = 3, 700
        R = g["R"][:N]
    elif name.startswith("shape_"):
        B, N = map(int, name.split("_")[1].split("x"))
        per_pair = name.endswith("per_pair")
        vs, vt = random_volumes(rng, B)
    elif name == "lattice":
        B, R = 2, lattice_rotations()
    elif name == "outside":
        R = np.concatenate([outside_rotations(), random_rotations(rng, 60)])
    elif name == "R_x0.35":                                   # not rotations: every item takes the exact path
        B, N = 2, 150
        R = (random_rotations(rng, N) * f32(0.35)).astype(f32)
    elif name == "R_mixed_x0.35":                             # every fifth matrix shrunk: the path changes per item
        B, N = 2, 150
        R = random_rotations(rng, B, N)
        R[:, ::5] *= f32(0.35)
    elif name.startswith("vol_x"):
        vs = (np.asarray(vs) * f32(float(name[5:]))).astype(f32)
    elif name == "outlier_4e3":
        B, N = 2, 150
        vs = np.array(vs[:B])
        vs[1, 3, 2, 5, 1] = 4.0e3
    elif name.startswith("W1_x"):
        c = 2.0 ** int(name[6:]) if "^" in name else float(name[4:])
        W1 = (W1 * f32(c)).astype(f32)
        if c < 1:
            b2 = (b2 * f32(c)).astype(f32)
    elif name == "W2_x0.05":
        W2 = (W2 * f32(0.05)).astype(f32)
    elif name in ("student_t", "row_scales", "zero_rows"):
        W1, W2 = trained_like(W1, W2, name, seed=77)
    elif name == "zero_conv2":                                # H2 = 0 everywhere: the normalisation's clamp
        tgt_w = (W1, W2, b2)
        W2, b2 = np.zeros_like(W2), np.zeros_like(b2)
    if R is None:
        R = random_rotations(rng, B, N) if per_pair else random_rotations(rng, N)
    N = R.shape[-3]
    vs = np.ascontiguousarray(np.asarray(vs)[:B], f32)
    vt = np.ascontiguousarray(np.asarray(vt)[:B], f32)
    gs = rng.normal(size=(B, N)).astype(f32)
    if name == "g_decades":                                   # six decades per item, one item exactly zero
        gs = (gs * np.logspace(-6, 0, B * N)[rng.permutation(B * N)].reshape(B, N)).astype(f32)
        gs[0, min(1, N - 1)] = 0.0
    elif name == "g_x1e6":
        gs = (gs * f32(1e6)).astype(f32)
    elif name == "g_x1e-8":
        gs = (gs * f32(1e-8)).astype(f32)
    if name == "golden":
        tgt = g["tgt_feat"][:B]
    else:
        tgt = oracle.forward_3d2d_np(vt, *(tgt_w or (W1, W2, b2)))
    return dict(vs=vs, tgt=np.ascontiguousarray(tgt, f32), R=np.ascontiguousarray(R, f32), W1=W1, W2=W2, b2=b2,
                gs=np.ascontiguousarray(gs, f32))


def fp64_autograd(vs, tgt, R, W1, W2, b2, gs, h1, pair_inv, want_R: bool = False):
    """fp64 autograd (torch, CPU) of the function the training forward ran: conv1's output takes the VALUE it kept
    (h1 pair_inv) and the ReLU MASK of that value, the rest is utils.py:113-131 and modules/modules.py:112-124.
    Returns the gradients of sum(gs * scores) with respect to (vol_src, tgt_feat, W1, W2, b2[, R]) as numpy fp64."""
    import torch
    import torch.nn.functional as F

    T = lambda a: torch.as_tensor(np.asarray(a, f32)).double()
    leaves = [T(a).requires_grad_(True) for a in (vs, tgt, W1, W2, b2)]
    Rl = T(R).requires_grad_(want_R)
    v64, t64, w1, w2, bb = leaves
    B = v64.shape[0]
    per_pair = Rl.dim() == 4
    N = Rl.shape[1] if per_pair else Rl.shape[0]
    kept_all = torch.as_tensor(np.asarray(h1, f16)).double().reshape(B, N, NPOS, OCH)
    rows = []
    for b in range(B):
        Rb = Rl[b] if per_pair else Rl
        rot = oracle.rotate_volume_torch(v64[b][None].expand(N, -1, -1, -1, -1), Rb)
        tri = torch.cat([rot.permute(0, 1, 4, 2, 3).reshape(N, 128, 8, 8), rot.permute(0, 1, 3, 2, 4).reshape(N, 128, 8, 8),
                         rot.reshape(N, 128, 8, 8)], dim=1)
        pre = F.conv2d(tri, w1.reshape(32, 384, 1, 1))
        kept = (kept_all[b] * float(np.asarray(pair_inv, f32)[b])).permute(0, 2, 1).reshape(N, 32, 8, 8)
        mask = (kept > 0).double()
        hid = pre * mask + (kept - pre * mask).detach()       # value = what the forward kept, gradient = through its mask
        f = F.normalize(F.conv2d(hid, w2.reshape(32, 32, 1, 1), bb), p=2, dim=1).flatten(2)
        rows.append((f * t64[b][None]).sum(dim=1).mean(dim=-1))
    s = torch.stack(rows)
    wrt = leaves + ([Rl] if want_R else [])
    out = torch.autograd.grad(s, wrt, grad_outputs=T(gs).reshape(B, N))
    return [o.numpy() for o in out]


def r_set(B, N, per_pair, seed):
    """Random rotations with the 24 lattice rotations and the out-of-range ones mixed in (evenly spaced)."""
    special = np.concatenate([lattice_rotations(), outside_rotations()])
    R = random_rotations(np.random.default_rng(seed), *((B, N) if per_pair else (N,)))
    flat = R.reshape(-1, 3, 3)
    step = max(1, flat.shape[0] // len(special))
    k = len(flat[::step][: len(special)])
    flat[::step][:k] = special[:k]
    return np.ascontiguousarray(R, f32)


R_CASES = {"shared": (False, 1.0), "per_pair": (True, 1.0), "shared_x0.35": (False, 0.35)}


def r_case(golden, name):
    """B = 2 x N = 120 with an outlier voxel in the second volume and upstream gradients over six decades."""
    per_pair, shrink = R_CASES[name]
    g, w = golden["shared_n3000_b3"], golden["weights"]
    B, N = 2, 120
    vs = g["vol_src"][:B].copy()
    vs[1, 3, 2, 5, 1] = 4.0e3
    R = (r_set(B, N, per_pair, seed=31) * f32(shrink)).astype(f32)
    rng = np.random.default_rng(17)
    gs = (rng.normal(size=(B, N)) * np.logspace(-6, 0, N)[rng.permutation(N)][None]).astype(f32)
    return dict(vs=vs, vt=g["vol_tgt"][:B], R=R, W1=w["W1"], W2=w["W2"], b2=w["b2"], gs=gs)


def case_model(case: dict, h1, pair_inv, **kw):
    """The model's gradients of a case given the training forward's h1 and pair_inv."""
    return tc_backward(case["vs"], case["tgt"], case["R"], case["W1"], case["W2"], case["b2"], case["gs"], h1, pair_inv,
                       **kw)
