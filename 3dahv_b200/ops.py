"""Tensor-level wrappers over the C ABI: device pointers, current stream, checks.

PyTorch is used only for device memory and streams; all arithmetic of the hot
path happens inside lib3dahv_b200.so.
"""
from __future__ import annotations

import ctypes

import torch
import torch.nn.functional as F

from . import _lib
from ._lib import MATH_FP32, MATH_TC, MATH_TC_F16GATHER, VOL_BF16, VOL_F32

_BASE_CPU = None
_BASE_DEV = {}


def base_coords(device=None) -> torch.Tensor:
    """The 8 base coordinates F.affine_grid(align_corners=False) uses for size 8
    (ATen: linspace(-1,1,8)*7/8 — not exactly (2i+1)/8-1), taken from ATen itself
    so the kernel sees the reference's values (utils.py:126).  Cached per device
    (no host->device copy on the hot path, CUDA-graph safe)."""
    global _BASE_CPU
    if _BASE_CPU is None:
        g = F.affine_grid(torch.eye(3, 4)[None], (1, 1, 8, 8, 8), align_corners=False)
        _BASE_CPU = g[0, 0, 0, :, 0].contiguous().clone()
    if device is None:
        return _BASE_CPU
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    if device not in _BASE_DEV:
        _BASE_DEV[device] = _BASE_CPU.to(device)
    return _BASE_DEV[device]


def _call(name: str, device, *args) -> None:
    """lib3dahv_b200's `name`(*args, current stream of `device`) with `device` current; raises on a failing status."""
    with torch.cuda.device(device):
        _lib.check(getattr(_lib.lib(), name)(*args, torch.cuda.current_stream(device).cuda_stream), name)


def _dev(t: torch.Tensor, name: str, dtype=torch.float32) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: the 3DAHV hot path has no CPU fallback")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    t = t.contiguous()
    if t.data_ptr() % 16:   # the C ABI wants 16-byte aligned buffers; a slice such as R[lo:hi] need not be
        t = t.clone()
    return t


def _vol_src(vol_src):
    """A bf16 source volume stays bf16, any other must be fp32: (tensor, AHV_VOL_* code)."""
    if vol_src.dtype == torch.bfloat16:
        return _dev(vol_src, "vol_src", torch.bfloat16), VOL_BF16
    return _dev(vol_src, "vol_src"), VOL_F32


def _head(W1, W2, b2):
    """The verification head's weights as the kernels read them: W1 [32,384], W2 [32,32], b2 [32]."""
    return _dev(W1.reshape(32, 384), "W1"), _dev(W2.reshape(32, 32), "W2"), _dev(b2, "b2")


def _rotations(R, B: int):
    """R [N,3,3] shared by the B pairs or [B,N,3,3] one set per pair -> (R, per_pair, N)."""
    per_pair = R.dim() == 4
    if per_pair and R.shape[0] != B:
        raise ValueError("per-pair R must be [B,N,3,3]")
    if tuple(R.shape[-2:]) != (3, 3):
        raise ValueError("R must be [...,3,3]")
    return R, per_pair, R.shape[1] if per_pair else R.shape[0]


def _workspace(ws, need: int, device):
    """`ws` if it holds `need` bytes, else a new buffer that does: (workspace, its size in bytes)."""
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = torch.empty(max(need, 16), device=device, dtype=torch.uint8)
    return ws, ws.numel() * ws.element_size()


def rotations_from_normals(normals: torch.Tensor) -> torch.Tensor:
    """[n,4] normals (GPU) -> [n,3,3]; pytorch3d random_rotations arithmetic."""
    o = _dev(normals, "normals")
    n = o.shape[0]
    R = torch.empty(n, 3, 3, device=o.device, dtype=torch.float32)
    _call("ahv_so3_from_normals", o.device, o.data_ptr(), R.data_ptr(), n)
    return R


def sample_rotations(n: int, seed: int, first_index: int = 0, device="cuda") -> torch.Tensor:
    """Native Philox sampler: hypothesis i depends only on (seed, first_index+i)."""
    R = torch.empty(n, 3, 3, device=torch.device(device), dtype=torch.float32)
    _call("ahv_so3_sample", R.device, seed & (2**64 - 1), first_index, R.data_ptr(), n)
    return R


def grid_rotations(n_total: int, first_index: int = 0, count: int | None = None, device="cuda") -> torch.Tensor:
    """Deterministic super-Fibonacci SO(3) grid, points [first, first+count) of n_total."""
    count = n_total - first_index if count is None else count
    R = torch.empty(count, 3, 3, device=torch.device(device), dtype=torch.float32)
    _call("ahv_so3_grid", R.device, n_total, first_index, R.data_ptr(), count)
    return R


HOPF_MAX_LEVEL, HOPF_MAX_BASE_LEVEL = 16, 6


def hopf_cells(level: int) -> int:
    """Cells of level `level` of the nested Hopf grid: 72 * 8^level."""
    return 72 * 8 ** level


def hopf_grid(level: int, first_index: int = 0, count: int | None = None, device="cuda") -> torch.Tensor:
    """ahv_so3_hopf_grid: cells [first_index, first_index + count) of level `level` (0..16) of the nested, equal-volume
    Hopf x HEALPix SO(3) grid, as rotations [count,3,3] (cell i's children at level + 1 are 8i .. 8i+7)."""
    count = hopf_cells(level) - first_index if count is None else count
    R = torch.empty(count, 3, 3, device=torch.device(device), dtype=torch.float32)
    _call("ahv_so3_hopf_grid", R.device, int(level), int(first_index), R.data_ptr(), int(count))
    return R


def hopf_children(level: int, parent_idx: torch.Tensor):
    """ahv_so3_hopf_children: cells parent_idx [...] of level `level` (0..15) -> their 8 children at level + 1 in child
    order, (child_idx [...,8] int64, R [...,8,3,3]); bit for bit `hopf_grid(level + 1)` at child_idx.  A parent outside the
    level gives children -1 with NaN rotations."""
    p = _dev(parent_idx, "parent_idx", torch.int64)
    n = p.numel()
    child = torch.empty(*p.shape, 8, device=p.device, dtype=torch.int64)
    R = torch.empty(*p.shape, 8, 3, 3, device=p.device, dtype=torch.float32)
    _call("ahv_so3_hopf_children", p.device, int(level), p.data_ptr(), n, child.data_ptr(), R.data_ptr())
    return child, R


def search_hierarchical_workspace_bytes(B: int, base_level: int, k: int) -> int:
    """Bytes of scratch `search_hierarchical` needs (0 for invalid sizes); it holds the base grid, 36 B per cell."""
    return int(_lib.lib().ahv_search_hierarchical_workspace_bytes(B, base_level, k))


def search_hierarchical(vol_src, vol_tgt, W1, W2, b2, base_level: int = 2, levels: int = 4, k: int = 8, math: int = MATH_TC,
                        workspace: torch.Tensor | None = None, out=None):
    """ahv_search_hierarchical: coarse-to-fine search on the nested Hopf grid in one C call - the whole base level scored
    and cut to its top-k, then `levels` times the 8 children of each pair's k cells scored and cut to their top-k.  No
    torch ops, no host synchronisation, CUDA-graph capturable (pass `out` = the tuple a previous call returned to reuse
    its buffers).  Returns (first_val [B,k], first_idx [B,k], first_R [B,k,3,3] - the base level's top-k, indices of
    level base_level - val [B,k], idx [B,k], R [B,k,3,3] - the finest level's top-k, indices of level
    base_level + levels; slot 0 is the answer - workspace)."""
    vs, vdt = _vol_src(vol_src)
    vt = _dev(vol_tgt, "vol_tgt")
    B = vs.shape[0]
    if tuple(vs.shape[1:]) != (16, 8, 8, 8) or tuple(vt.shape) != (B, 16, 8, 8, 8):
        raise ValueError("vol_src / vol_tgt must be [B,16,8,8,8]")
    if not (1 <= k <= 32 and 0 <= base_level <= HOPF_MAX_BASE_LEVEL and levels >= 0 and base_level + levels <= HOPF_MAX_LEVEL):
        raise ValueError("1 <= k <= 32, 0 <= base_level <= 6, levels >= 0 and base_level + levels <= 16 expected")
    W1, W2, b2 = _head(W1, W2, b2)
    dev = vs.device
    if out is None:
        f = dict(device=dev, dtype=torch.float32)
        out = (torch.empty(B, k, **f), torch.empty(B, k, device=dev, dtype=torch.int64), torch.empty(B, k, 3, 3, **f),
               torch.empty(B, k, **f), torch.empty(B, k, device=dev, dtype=torch.int64), torch.empty(B, k, 3, 3, **f))
    fv, fi, fR, v, i, R = out[:6]
    workspace, ws_bytes = _workspace(workspace, search_hierarchical_workspace_bytes(B, base_level, k), dev)
    _call("ahv_search_hierarchical", dev, vs.data_ptr(), vdt, vt.data_ptr(), W1.data_ptr(), W2.data_ptr(), b2.data_ptr(),
          base_coords(dev).data_ptr(), int(base_level), int(levels), int(k), fv.data_ptr(), fi.data_ptr(), fR.data_ptr(),
          v.data_ptr(), i.data_ptr(), R.data_ptr(), B, int(math), workspace.data_ptr(), ws_bytes)
    return fv, fi, fR, v, i, R, workspace


def perturb_rotations(R_center: torch.Tensor, m: int, max_angle_deg: float, seed: int = 0) -> torch.Tensor:
    """ahv_so3_perturb: [...,3,3] centres -> [...,m,3,3] rotations within `max_angle_deg` of them (index 0 = the
    centre itself)."""
    c = _dev(R_center, "R_center")
    lead = c.shape[:-2]
    n = c.numel() // 9
    out = torch.empty(*lead, m, 3, 3, device=c.device, dtype=torch.float32)
    _call("ahv_so3_perturb", c.device, c.data_ptr(), n, m, float(max_angle_deg), seed & (2**64 - 1), out.data_ptr())
    return out


def rotate_volume(volume: torch.Tensor, R: torch.Tensor) -> torch.Tensor:
    """utils.rotate_volume (utils.py:113-131) on the GPU.  `volume` is
    [16,8,8,8] (one volume under n rotations) or [n,16,8,8,8] (one per rotation)."""
    R = _dev(R, "R")
    n = R.shape[0]
    per_rot = volume.dim() == 5
    if per_rot and volume.shape[0] != n:
        raise ValueError("volume batch must match the number of rotations")
    if tuple(volume.shape[-4:]) != (16, 8, 8, 8):
        raise ValueError("volume must be [...,16,8,8,8]")
    v = _dev(volume, "volume")
    out = torch.empty(n, 16, 8, 8, 8, device=v.device, dtype=torch.float32)
    base = base_coords(v.device)
    _call("ahv_rotate_volume", v.device, v.data_ptr(), int(per_rot), R.data_ptr(), base.data_ptr(), out.data_ptr(), n)
    return out


def rotate_volume_backward(grad_out: torch.Tensor, R: torch.Tensor, per_rotation: bool) -> torch.Tensor:
    """Adjoint of rotate_volume w.r.t. the volume: [n,16,8,8,8] -> [16,8,8,8] (shared volume, summed)
    or [n,16,8,8,8] (one volume per rotation)."""
    g, R = _dev(grad_out, "grad_out"), _dev(R, "R")
    n = R.shape[0]
    if tuple(g.shape) != (n, 16, 8, 8, 8):
        raise ValueError("grad_out must be [n,16,8,8,8]")
    out = (torch.empty(n, 16, 8, 8, 8, device=g.device, dtype=torch.float32) if per_rotation
           else torch.zeros(16, 8, 8, 8, device=g.device, dtype=torch.float32))
    base = base_coords(g.device)
    _call("ahv_rotate_volume_backward", g.device, g.data_ptr(), int(per_rotation), R.data_ptr(), base.data_ptr(), out.data_ptr(),
          n)
    return out


def rotate_volume_grad_R(vol: torch.Tensor, grad_out: torch.Tensor, R: torch.Tensor, per_rotation: bool) -> torch.Tensor:
    """Gradient of rotate_volume w.r.t. the rotations, as F.grid_sample's backward gives it through F.affine_grid:
    `vol` [16,8,8,8] (shared) or [n,16,8,8,8] (one per rotation), grad_out [n,16,8,8,8] -> grad_R [n,3,3]."""
    v, g, R = _dev(vol, "vol"), _dev(grad_out, "grad_out"), _dev(R, "R")
    n = R.shape[0]
    if tuple(R.shape) != (n, 3, 3) or tuple(g.shape) != (n, 16, 8, 8, 8):
        raise ValueError("R [n,3,3] and grad_out [n,16,8,8,8] expected")
    if tuple(v.shape) != ((n, 16, 8, 8, 8) if per_rotation else (16, 8, 8, 8)):
        raise ValueError("vol must be [n,16,8,8,8] (per rotation) or [16,8,8,8] (shared)")
    out = torch.empty(n, 3, 3, device=g.device, dtype=torch.float32)
    base = base_coords(g.device)
    _call("ahv_rotate_volume_grad_R", g.device, v.data_ptr(), int(per_rotation), R.data_ptr(), base.data_ptr(), g.data_ptr(),
          out.data_ptr(), n)
    return out


def score_train(vol_src: torch.Tensor, tgt_feat: torch.Tensor, R: torch.Tensor, W1: torch.Tensor, W2: torch.Tensor,
                b2: torch.Tensor, workspace: torch.Tensor | None = None):
    """ahv_score_train: the training forward - scores [B,N] from the tensor-core kernel, plus what the backward pass
    wants back: conv1's ReLU'd output of every item (fp16 [B*N,64,32], 4 KB per item) and per pair [B] the factor
    that turns it back into conv1's output (2^e1 / scale: the pair scale and W1's normaliser)."""
    vs, tf, R = _dev(vol_src, "vol_src"), _dev(tgt_feat, "tgt_feat"), _dev(R, "R")
    W1, W2, b2 = _head(W1, W2, b2)
    B = vs.shape[0]
    if tuple(vs.shape) != (B, 16, 8, 8, 8) or tuple(tf.shape) != (B, 32, 64):
        raise ValueError("vol_src [B,16,8,8,8], tgt_feat [B,32,64], R [N,3,3] or [B,N,3,3] expected")
    R, per_pair, N = _rotations(R, B)
    dev = vs.device
    scores = torch.empty(B, N, device=dev, dtype=torch.float32)
    h1 = torch.empty(B * N, 64, 32, device=dev, dtype=torch.float16)
    pair_inv = torch.empty(B, device=dev, dtype=torch.float32)
    workspace, ws_bytes = _workspace(workspace, workspace_bytes(B, N, 1), dev)
    _call("ahv_score_train", dev, vs.data_ptr(), tf.data_ptr(), R.data_ptr(), int(per_pair), W1.data_ptr(), W2.data_ptr(),
          b2.data_ptr(), base_coords(dev).data_ptr(), scores.data_ptr(), h1.data_ptr(), pair_inv.data_ptr(), B, N,
          workspace.data_ptr(), ws_bytes)
    return scores, h1, pair_inv


def _score_backward_ex(vs, tg, R, W1, W2, b2, gs, h1, pi, outs, B, N, per_pair):
    """ahv_score_backward_ex into `outs` = (grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2, grad_R), each a zeroed
    tensor or None."""
    ptr = lambda t: t.data_ptr() if t is not None else None
    _call("ahv_score_backward_ex", vs.device, vs.data_ptr(), tg.data_ptr(), R.data_ptr(), int(per_pair), W1.data_ptr(),
          W2.data_ptr(), b2.data_ptr(), base_coords(vs.device).data_ptr(), gs.data_ptr(), ptr(h1), ptr(pi),
          *(ptr(t) for t in outs), B, N)


def _score_backward_args(vol_src, tgt_feat, R, W1, W2, b2, grad_scores):
    vs, tg, R, gs = _dev(vol_src, "vol_src"), _dev(tgt_feat, "tgt_feat"), _dev(R, "R"), _dev(grad_scores, "grad_scores")
    W1, W2, b2 = _head(W1, W2, b2)
    B = vs.shape[0]
    R, per_pair, N = _rotations(R, B)
    if tuple(vs.shape) != (B, 16, 8, 8, 8) or tuple(tg.shape) != (B, 32, 64) or tuple(gs.shape) != (B, N):
        raise ValueError("vol_src [B,16,8,8,8], tgt_feat [B,32,64], grad_scores [B,N] expected")
    return vs, tg, R, W1, W2, b2, gs, B, N, per_pair


def score_backward(vol_src: torch.Tensor, tgt_feat: torch.Tensor, R: torch.Tensor, W1: torch.Tensor, W2: torch.Tensor,
                   b2: torch.Tensor, grad_scores: torch.Tensor, h1_saved: torch.Tensor | None = None,
                   pair_inv: torch.Tensor | None = None, math: int = MATH_TC, want_grad_R: bool = False,
                   deterministic: bool = False, workspace: torch.Tensor | None = None):
    """Fused gradient of the verification scores (modules/model.py:53-56 under autograd): returns
    (grad_vol_src [B,16,8,8,8], grad_tgt_feat [B,32,64], grad_W1 [32,384], grad_W2 [32,32], grad_b2 [32]).
    With `h1_saved` / `pair_inv` from `score_train` the kernel reads conv1's output instead of recomputing it, and
    `math` picks how it contracts dA = dH1 W1 and dW1 = dH1^T A: MATH_TC on tcgen05, MATH_FP32 in FFMA.  Without them
    it is the exact fp32 kernel whatever `math` says.
    `want_grad_R`: also the gradient w.r.t. the rotations, appended to the tuple - grad_R [N,3,3] (summed over pairs)
    or [B,N,3,3] - from `ahv_score_backward_ex`, which contracts in fp32 FFMA whatever `math` says (the tcgen05
    backward has no rotation phase; with saved activations this is the MATH_FP32 form on the same saved values).
    `deterministic`: the same kernels and routing, in the form of `ahv_score_backward_det`, which sums every gradient
    in a fixed order instead of with float atomics: bit-identical results from run to run on one device (the bits
    depend on the inputs and on min(SM count, 160)).  It needs `ahv_score_backward_det_workspace_bytes` of scratch,
    about 15 MB at B = 12 (16 MB more with a shared R's gradient at N = 9000); `workspace` re-uses a buffer of at least
    that size, else one is allocated."""
    vs, tg, R, W1, W2, b2, gs, B, N, per_pair = _score_backward_args(vol_src, tgt_feat, R, W1, W2, b2, grad_scores)
    dev = vs.device
    z = lambda *shape: torch.zeros(*shape, device=dev, dtype=torch.float32)
    g_vol, g_tgt, g_w1, g_w2, g_b2 = z(B, 16, 8, 8, 8), z(B, 32, 64), z(32, 384), z(32, 32), z(32)
    h1 = pi = None
    if h1_saved is not None:
        h1 = _dev(h1_saved, "h1_saved", torch.float16)
        pi = _dev(pair_inv, "pair_inv")
        if h1.numel() != B * N * 64 * 32 or pi.numel() != B:
            raise ValueError("h1_saved [B*N,64,32] fp16 and pair_inv [B] expected")
    if deterministic:
        g_R = z(*R.shape) if want_grad_R else None
        outs = (g_vol, g_tgt, g_w1, g_w2, g_b2, g_R)
        mode = int(math) if h1 is not None and not want_grad_R else MATH_FP32
        need = score_backward_det_workspace_bytes(B, N, per_pair, want_grad_R)
        workspace, ws_bytes = _workspace(workspace, need, dev)
        ptr = lambda t: t.data_ptr() if t is not None else None
        _call("ahv_score_backward_det", dev, vs.data_ptr(), tg.data_ptr(), R.data_ptr(), int(per_pair), W1.data_ptr(),
              W2.data_ptr(), b2.data_ptr(), base_coords(dev).data_ptr(), gs.data_ptr(), ptr(h1), ptr(pi),
              *(ptr(t) for t in outs), B, N, mode, workspace.data_ptr(), ws_bytes)
        return outs if want_grad_R else outs[:5]
    if h1 is not None and not want_grad_R and math != MATH_FP32:   # the tcgen05 kernel (the entry checks `math`)
        _call("ahv_score_backward_saved", dev, vs.data_ptr(), tg.data_ptr(), R.data_ptr(), int(per_pair), W1.data_ptr(),
              W2.data_ptr(), b2.data_ptr(), base_coords(dev).data_ptr(), gs.data_ptr(), h1.data_ptr(), pi.data_ptr(),
              g_vol.data_ptr(), g_tgt.data_ptr(), g_w1.data_ptr(), g_w2.data_ptr(), g_b2.data_ptr(), B, N, int(math))
        return g_vol, g_tgt, g_w1, g_w2, g_b2
    g_R = z(*R.shape) if want_grad_R else None
    _score_backward_ex(vs, tg, R, W1, W2, b2, gs, h1, pi, (g_vol, g_tgt, g_w1, g_w2, g_b2, g_R), B, N, per_pair)
    return (g_vol, g_tgt, g_w1, g_w2, g_b2, g_R) if want_grad_R else (g_vol, g_tgt, g_w1, g_w2, g_b2)


def score_backward_det_workspace_bytes(B: int, N: int, per_pair: bool, want_grad_R: bool) -> int:
    """Bytes of scratch `score_backward(..., deterministic=True)` needs (0 for invalid sizes)."""
    return int(_lib.lib().ahv_score_backward_det_workspace_bytes(B, N, int(per_pair), int(want_grad_R)))


def score_grad_R(vol_src: torch.Tensor, tgt_feat: torch.Tensor, R: torch.Tensor, W1: torch.Tensor, W2: torch.Tensor,
                 b2: torch.Tensor, grad_scores: torch.Tensor) -> torch.Tensor:
    """d(sum grad_scores * scores)/dR alone - `ahv_score_backward_ex` with every other output NULL, so the kernel
    skips the adjoint of the resampling and the dW1 contraction.  R [N,3,3] -> [N,3,3] (summed over pairs) or
    [B,N,3,3] -> [B,N,3,3]."""
    vs, tg, R, W1, W2, b2, gs, B, N, per_pair = _score_backward_args(vol_src, tgt_feat, R, W1, W2, b2, grad_scores)
    g_R = torch.zeros(*R.shape, device=vs.device, dtype=torch.float32)
    _score_backward_ex(vs, tg, R, W1, W2, b2, gs, None, None, (None, None, None, None, None, g_R), B, N, per_pair)
    return g_R


def infonce(scores: torch.Tensor, sampled_R: torch.Tensor, gt_delta_R: torch.Tensor, acc_thr_deg: float,
            temperature: float = 0.1, want_grad: bool = True):
    """ahv_infonce: (loss [B], d loss / d scores [B,N] or None) in one launch (modules/model.py:43-63).
    The masses of the positives and the negatives are summed apart in double, so confident pairs (loss far below
    fp32's epsilon) keep fp32 relative accuracy in the loss and in every gradient.  Domain: exp(scores/T) is fp32,
    so |scores|/T must stay below ~88; the reference overflows there too.  Scores that are means of cosines lie in
    [-1, 1] and cannot reach it at T = 0.1."""
    s, R, g = _dev(scores, "scores"), _dev(sampled_R, "sampled_R"), _dev(gt_delta_R, "gt_delta_R")
    B, N = s.shape
    per_pair = R.dim() == 4
    if (R.shape[1] if per_pair else R.shape[0]) != N or tuple(g.shape) != (B, 3, 3) or (per_pair and R.shape[0] != B):
        raise ValueError("scores [B,N], sampled_R [N,3,3] or [B,N,3,3], gt_delta_R [B,3,3] expected")
    loss = torch.empty(B, device=s.device, dtype=torch.float32)
    grad = torch.empty(B, N, device=s.device, dtype=torch.float32) if want_grad else None
    _call("ahv_infonce", s.device, s.data_ptr(), R.data_ptr(), int(per_pair), g.data_ptr(), float(acc_thr_deg),
          float(temperature), loss.data_ptr(), grad.data_ptr() if want_grad else None, B, N)
    return loss, grad


def resblock3d(x: torch.Tensor, conv1_w: torch.Tensor, conv2_w: torch.Tensor, down_w: torch.Tensor) -> torch.Tensor:
    """ResNetBlock_3D(32->16) of the lifting stage (modules/modules.py:9-47, :100-101): [m,32,8,8,8] -> [m,16,8,8,8]
    in one cluster launch (inference only)."""
    v = _dev(x, "x")
    if tuple(v.shape[1:]) != (32, 8, 8, 8):
        raise ValueError("x must be [m,32,8,8,8]")
    w1, w2, wd = _dev(conv1_w, "conv1_w"), _dev(conv2_w, "conv2_w"), _dev(down_w, "down_w")
    if tuple(w1.shape) != (16, 32, 3, 3, 3) or tuple(w2.shape) != (16, 16, 3, 3, 3) or w1.numel() * 0 + wd.numel() != 16 * 32:
        raise ValueError("weights must be conv1 [16,32,3,3,3], conv2 [16,16,3,3,3], downsample [16,32,1,1,1]")
    m = v.shape[0]
    out = torch.empty(m, 16, 8, 8, 8, device=v.device, dtype=torch.float32)
    _call("ahv_resblock3d", v.device, v.data_ptr(), w1.data_ptr(), w2.data_ptr(), wd.data_ptr(), out.data_ptr(), m)
    return out


def forward_3d2d(vol: torch.Tensor, W1: torch.Tensor, W2: torch.Tensor, b2: torch.Tensor) -> torch.Tensor:
    """Feature_Aligner.forward_3d2d (modules/modules.py:112-124): [m,16,8,8,8] -> [m,32,64]."""
    v = _dev(vol, "vol")
    if tuple(v.shape[1:]) != (16, 8, 8, 8):
        raise ValueError("vol must be [m,16,8,8,8]")
    W1, W2, b2 = _head(W1, W2, b2)
    m = v.shape[0]
    feat = torch.empty(m, 32, 64, device=v.device, dtype=torch.float32)
    _call("ahv_forward_3d2d", v.device, v.data_ptr(), W1.data_ptr(), W2.data_ptr(), b2.data_ptr(), feat.data_ptr(), m)
    return feat


def workspace_bytes(B: int, N: int, k: int) -> int:
    return int(_lib.lib().ahv_workspace_bytes(B, N, k))


def score(vol_src, tgt_feat, R, W1, W2, b2, k: int = 1, idx_offset: int = 0, math: int = MATH_TC,
          return_scores: bool = True, workspace: torch.Tensor | None = None):
    """The fused hot path (modules/model.py:186-196).

    vol_src [B,16,8,8,8] fp32|bf16, tgt_feat [B,32,64], R [N,3,3] or [B,N,3,3].
    Returns (scores [B,N] or None, topk_val [B,k], topk_idx [B,k] int64)."""
    vs, vdt = _vol_src(vol_src)
    B = vs.shape[0]
    if tuple(vs.shape[1:]) != (16, 8, 8, 8):
        raise ValueError("vol_src must be [B,16,8,8,8]")
    tf = _dev(tgt_feat, "tgt_feat")
    if tuple(tf.shape) != (B, 32, 64):
        raise ValueError("tgt_feat must be [B,32,64]")
    R, per_pair, N = _rotations(_dev(R, "R"), B)
    if k < 0 or k > 32:
        raise ValueError("k must be in [0,32]")
    W1, W2, b2 = _head(W1, W2, b2)
    dev = vs.device
    scores = torch.empty(B, N, device=dev, dtype=torch.float32) if return_scores else None
    kk = max(k, 1)
    val = torch.empty(B, kk, device=dev, dtype=torch.float32)
    idx = torch.empty(B, kk, device=dev, dtype=torch.int64)
    workspace, ws_bytes = _workspace(workspace, workspace_bytes(B, N, kk), dev)
    _call("ahv_score", dev, vs.data_ptr(), vdt, tf.data_ptr(), R.data_ptr(), int(per_pair), W1.data_ptr(), W2.data_ptr(),
          b2.data_ptr(), base_coords(dev).data_ptr(), scores.data_ptr() if scores is not None else None,
          val.data_ptr() if k > 0 else None, idx.data_ptr() if k > 0 else None, k, idx_offset, B, N, math,
          workspace.data_ptr(), ws_bytes)
    if k == 0:
        return scores, None, None
    return scores, val, idx


def verify(vol_src, vol_tgt, R, W1, W2, b2, k: int = 1, idx_offset: int = 0, math: int = MATH_TC,
           return_scores: bool = False, gather: bool = True, workspace: torch.Tensor | None = None):
    """ahv_verify: target features + fused scoring + selection + winner gather in one C call.
    Returns (scores|None, topk_val [B,k], topk_idx [B,k], R_best [B,k,3,3]|None)."""
    vs, vdt = _vol_src(vol_src)
    vt = _dev(vol_tgt, "vol_tgt")
    B = vs.shape[0]
    if tuple(vs.shape[1:]) != (16, 8, 8, 8) or tuple(vt.shape) != (B, 16, 8, 8, 8):
        raise ValueError("vol_src / vol_tgt must be [B,16,8,8,8]")
    R, per_pair, N = _rotations(_dev(R, "R"), B)
    if k < 1 or k > 32:
        raise ValueError("k must be in [1,32]")
    W1, W2, b2 = _head(W1, W2, b2)
    dev = vs.device
    scores = torch.empty(B, N, device=dev, dtype=torch.float32) if return_scores else None
    val = torch.empty(B, k, device=dev, dtype=torch.float32)
    idx = torch.empty(B, k, device=dev, dtype=torch.int64)
    Rb = torch.empty(B, k, 3, 3, device=dev, dtype=torch.float32) if gather else None
    workspace, ws_bytes = _workspace(workspace, workspace_bytes(B, N, k), dev)
    _call("ahv_verify", dev, vs.data_ptr(), vdt, vt.data_ptr(), R.data_ptr(), int(per_pair), W1.data_ptr(), W2.data_ptr(),
          b2.data_ptr(), base_coords(dev).data_ptr(), scores.data_ptr() if scores is not None else None, val.data_ptr(),
          idx.data_ptr(), Rb.data_ptr() if Rb is not None else None, k, idx_offset, B, N, math, workspace.data_ptr(), ws_bytes)
    return scores, val, idx, Rb


def verify_screen_stats(workspace: torch.Tensor | None, B: int, N: int):
    """What the last screened `verify` (k = 1, fp32 volumes, MATH_TC, no scores) over `workspace` found: None when a
    call of that shape takes the single pass, else (number of pairs that fell back to the exact pass, contenders per
    pair [B] int32, largest |fp32 - 16-bit| score difference on each pair's list [B] fp32).  Synchronises."""
    lib = _lib.lib()
    is_screened = ctypes.c_int(0)
    _lib.check(lib.ahv_verify_screen_stats(None, B, N, ctypes.byref(is_screened), None, None, None), "ahv_verify_screen_stats")
    if not is_screened.value:
        return None
    flagged = ctypes.c_int(0)
    count = (ctypes.c_int * B)()
    err = (ctypes.c_float * B)()
    _lib.check(lib.ahv_verify_screen_stats(workspace.data_ptr(), B, N, ctypes.byref(is_screened), ctypes.byref(flagged),
                                           count, err), "ahv_verify_screen_stats")
    return flagged.value, torch.tensor(list(count), dtype=torch.int32), torch.tensor(list(err), dtype=torch.float32)


def refine(vol_src, vol_tgt, R, W1, W2, b2, k: int = 32, m: int = 64, max_angle_deg: float = 5.0, seed: int = 0,
           math: int = MATH_TC, workspace: torch.Tensor | None = None, out=None):
    """ahv_refine: top-k over the set, m local candidates around each winner, arg-max over them - one C call, no
    torch ops, CUDA-graph capturable (pass `out` = the tuple a previous call returned to reuse its buffers).
    Returns (first_val [B,k], first_idx [B,k], first_R [B,k,3,3], cand [B,k*m,3,3], best_val [B], best_idx [B],
    R_best [B,3,3], workspace)."""
    vs, vdt = _vol_src(vol_src)
    vt = _dev(vol_tgt, "vol_tgt")
    B = vs.shape[0]
    R, per_pair, N = _rotations(_dev(R, "R"), B)
    if tuple(vs.shape[1:]) != (16, 8, 8, 8) or tuple(vt.shape) != (B, 16, 8, 8, 8):
        raise ValueError("vol_src / vol_tgt must be [B,16,8,8,8]")
    if not (1 <= k <= min(32, N)) or m < 1:
        raise ValueError("1 <= k <= min(32, N) and m >= 1 expected")
    W1, W2, b2 = _head(W1, W2, b2)
    dev = vs.device
    if out is None:
        f = dict(device=dev, dtype=torch.float32)
        out = (torch.empty(B, k, **f), torch.empty(B, k, device=dev, dtype=torch.int64), torch.empty(B, k, 3, 3, **f),
               torch.empty(B, k * m, 3, 3, **f), torch.empty(B, **f), torch.empty(B, device=dev, dtype=torch.int64),
               torch.empty(B, 3, 3, **f))
    fv, fi, fR, cand, bv, bi, bR = out[:7]
    workspace, ws_bytes = _workspace(workspace, int(_lib.lib().ahv_refine_workspace_bytes(B, N, k, m)), dev)
    _call("ahv_refine", dev, vs.data_ptr(), vdt, vt.data_ptr(), R.data_ptr(), int(per_pair), W1.data_ptr(), W2.data_ptr(),
          b2.data_ptr(), base_coords(dev).data_ptr(), k, m, float(max_angle_deg), seed & (2**64 - 1), fv.data_ptr(),
          fi.data_ptr(), fR.data_ptr(), cand.data_ptr(), bv.data_ptr(), bi.data_ptr(), bR.data_ptr(), B, N, math,
          workspace.data_ptr(), ws_bytes)
    return fv, fi, fR, cand, bv, bi, bR, workspace


def gradient_ascent(vol_src, tgt_feat, R_init, W1, W2, b2, steps: int = 20, step_deg: float = 1.0, out=None):
    """ahv_gradient_ascent: backtracking Riemannian gradient ascent of the AHV_MATH_FP32 score on SO(3), every step of
    every candidate in one launch.  vol_src [B,16,8,8,8] fp32|bf16, tgt_feat [B,32,64], R_init [B,K,3,3].  Returns
    (R_out [B,K,3,3], score_out [B,K]); score_out is the fp32 scorer's score of R_out, never below that of R_init.
    `out` = a previous result to write into (CUDA-graph replays)."""
    vs, vdt = _vol_src(vol_src)
    tf, R = _dev(tgt_feat, "tgt_feat"), _dev(R_init, "R_init")
    B = vs.shape[0]
    if tuple(vs.shape[1:]) != (16, 8, 8, 8) or tuple(tf.shape) != (B, 32, 64):
        raise ValueError("vol_src [B,16,8,8,8] and tgt_feat [B,32,64] expected")
    if R.dim() != 4 or R.shape[0] != B or tuple(R.shape[2:]) != (3, 3):
        raise ValueError("R_init must be [B,K,3,3]")
    W1, W2, b2 = _head(W1, W2, b2)
    K = R.shape[1]
    if out is None:
        out = (torch.empty(B, K, 3, 3, device=vs.device, dtype=torch.float32), torch.empty(B, K, device=vs.device, dtype=torch.float32))
    R_out, s_out = out
    _call("ahv_gradient_ascent", vs.device, vs.data_ptr(), vdt, tf.data_ptr(), R.data_ptr(), W1.data_ptr(), W2.data_ptr(),
          b2.data_ptr(), base_coords(vs.device).data_ptr(), int(steps), float(step_deg), R_out.data_ptr(), s_out.data_ptr(), B, K)
    return R_out, s_out


def refine_gradient(vol_src, vol_tgt, R, W1, W2, b2, k: int = 32, steps: int = 20, step_deg: float = 1.0, math: int = MATH_TC,
                    workspace: torch.Tensor | None = None, out=None, min_sep_deg: float = 0.0):
    """ahv_refine_gradient: top-k over the set, gradient ascent of the fp32 score from each winner, per-pair arg-max -
    one C call, no torch ops, CUDA-graph capturable (pass `out` = the tuple a previous call returned to reuse its buffers).
    min_sep_deg > 0 calls ahv_refine_gradient_distinct: the first pass keeps the k winners of `topk_distinct` instead, and
    its empty slots come back as first_idx -1, R_all NaN, score_all -inf.
    Returns (first_val [B,k], first_idx [B,k], first_R [B,k,3,3], R_all [B,k,3,3], score_all [B,k], best_val [B],
    best_idx [B], R_best [B,3,3], workspace)."""
    vs, vdt = _vol_src(vol_src)
    vt = _dev(vol_tgt, "vol_tgt")
    B = vs.shape[0]
    R, per_pair, N = _rotations(_dev(R, "R"), B)
    if tuple(vs.shape[1:]) != (16, 8, 8, 8) or tuple(vt.shape) != (B, 16, 8, 8, 8):
        raise ValueError("vol_src / vol_tgt must be [B,16,8,8,8]")
    if not 1 <= k <= min(32, N):
        raise ValueError("1 <= k <= min(32, N) expected")
    W1, W2, b2 = _head(W1, W2, b2)
    dev = vs.device
    if out is None:
        f = dict(device=dev, dtype=torch.float32)
        out = (torch.empty(B, k, **f), torch.empty(B, k, device=dev, dtype=torch.int64), torch.empty(B, k, 3, 3, **f),
               torch.empty(B, k, 3, 3, **f), torch.empty(B, k, **f), torch.empty(B, **f),
               torch.empty(B, device=dev, dtype=torch.int64), torch.empty(B, 3, 3, **f))
    fv, fi, fR, Ra, sa, bv, bi, bR = out[:8]
    workspace, ws_bytes = _workspace(workspace, int(_lib.lib().ahv_refine_gradient_workspace_bytes(B, N, k)), dev)
    head = (vs.data_ptr(), vdt, vt.data_ptr(), R.data_ptr(), int(per_pair), W1.data_ptr(), W2.data_ptr(), b2.data_ptr(),
            base_coords(dev).data_ptr(), k, int(steps), float(step_deg))
    tail = (fv.data_ptr(), fi.data_ptr(), fR.data_ptr(), Ra.data_ptr(), sa.data_ptr(), bv.data_ptr(), bi.data_ptr(), bR.data_ptr(),
            B, N, math, workspace.data_ptr(), ws_bytes)
    if min_sep_deg == 0:
        _call("ahv_refine_gradient", dev, *head, *tail)
    else:
        _call("ahv_refine_gradient_distinct", dev, *head, float(min_sep_deg), *tail)
    return fv, fi, fR, Ra, sa, bv, bi, bR, workspace


def _peer_array(peer):
    import ctypes

    return (ctypes.c_void_p * peer.world)(*[int(p) for p in peer.ptrs])


def verify_sharded(vol_src, vol_tgt, R, W1, W2, b2, idx_offset: int, peer, k: int = 1, math: int = MATH_TC,
                   workspace: torch.Tensor | None = None):
    """ahv_verify_sharded on this rank's slice `R` of the rotation set (global index = local + idx_offset); `peer`
    is a `dist.PeerExchange`.  The kernels exchange the per-shard winners through NVLink peer memory and merge
    them (k == 1 with tensor-core arithmetic: inside the scoring kernel; otherwise one exchange kernel after the
    shard's top-k).  Returns (topk_val [B,k], topk_idx [B,k] global, R_best [B,k,3,3]) over the whole set,
    identical on every rank.  An empty slice ([0,3,3]) is allowed."""
    vs, vdt = _vol_src(vol_src)
    vt = _dev(vol_tgt, "vol_tgt")
    R = _dev(R, "R")
    W1, W2, b2 = _head(W1, W2, b2)
    B = vs.shape[0]
    R, per_pair, N = _rotations(R, B)
    if tuple(vs.shape[1:]) != (16, 8, 8, 8) or tuple(vt.shape) != (B, 16, 8, 8, 8):
        raise ValueError("vol_src / vol_tgt must be [B,16,8,8,8]")
    if B > peer.max_pairs or k > peer.max_k:
        raise ValueError(f"exchange buffer holds {peer.max_pairs} pairs x top-{peer.max_k}; got B={B}, k={k}")
    dev = vs.device
    val = torch.empty(B, k, device=dev, dtype=torch.float32)
    idx = torch.empty(B, k, device=dev, dtype=torch.int64)
    Rb = torch.empty(B, k, 3, 3, device=dev, dtype=torch.float32)
    workspace, ws_bytes = _workspace(workspace, workspace_bytes(B, N, k), dev)
    _call("ahv_verify_sharded", dev, vs.data_ptr(), vdt, vt.data_ptr(), R.data_ptr() if N else None, int(per_pair), W1.data_ptr(),
          W2.data_ptr(), b2.data_ptr(), base_coords(dev).data_ptr(), val.data_ptr(), idx.data_ptr(), Rb.data_ptr(), k, idx_offset,
          B, N, math, workspace.data_ptr(), ws_bytes, peer.rank, peer.world, _peer_array(peer), peer.max_pairs, peer.max_k)
    return val, idx, Rb


def topk_exchange(val, idx, R, idx_offset: int, peer):
    """ahv_topk_exchange: this shard's [B,k] list (global indices, -1 = empty) -> the whole set's top-k on every
    rank, with the winning rotations.  Returns (topk_val [B,k], topk_idx [B,k], R_best [B,k,3,3])."""
    v, i, R = _dev(val, "val"), _dev(idx, "idx", torch.int64), _dev(R, "R")
    B, k = v.shape
    R, per_pair, N = _rotations(R, B)
    dev = v.device
    out_v = torch.empty(B, k, device=dev, dtype=torch.float32)
    out_i = torch.empty(B, k, device=dev, dtype=torch.int64)
    Rb = torch.empty(B, k, 3, 3, device=dev, dtype=torch.float32)
    _call("ahv_topk_exchange", dev, v.data_ptr(), i.data_ptr(), R.data_ptr() if N else None, int(per_pair), idx_offset, N, B, k,
          out_v.data_ptr(), out_i.data_ptr(), Rb.data_ptr(), peer.rank, peer.world, _peer_array(peer), peer.max_pairs, peer.max_k)
    return out_v, out_i, Rb


def scores_exchange(part, N: int, peer, out=None):
    """ahv_scores_exchange: this rank's columns part [B, hi-lo] (lo, hi = `dist.shard_bounds(N, rank, world)`) of a
    [B,N] score matrix -> the whole [B,N] on every rank, through the score region of `peer` (a `dist.PeerExchange`
    with max_hyps >= N).  `out`: a [B,N] fp32 tensor to write into (CUDA-graph replays)."""
    from .dist import shard_bounds

    p = _dev(part, "part")
    B = p.shape[0]
    lo, hi = shard_bounds(N, peer.rank, peer.world)
    if p.dim() != 2 or p.shape[1] != hi - lo:
        raise ValueError(f"part must be [B,{hi - lo}] (rank {peer.rank}'s columns [{lo},{hi}) of N={N})")
    max_hyps = getattr(peer, "max_hyps", 0)
    if B > peer.max_pairs or N > max_hyps:
        raise ValueError(f"exchange buffer holds {peer.max_pairs} pairs x {max_hyps} scores; got B={B}, N={N}")
    out = torch.empty(B, N, device=p.device, dtype=torch.float32) if out is None else out
    _call("ahv_scores_exchange", p.device, p.data_ptr() if hi > lo else None, B, N, out.data_ptr(), peer.rank, peer.world,
          _peer_array(peer), peer.max_pairs, peer.max_k, max_hyps)
    return out


def refine_gradient_sharded(vol_src, vol_tgt, R, W1, W2, b2, peer, k: int = 32, steps: int = 20, step_deg: float = 1.0,
                            math: int = MATH_TC, workspace: torch.Tensor | None = None, out=None, min_sep_deg: float = 0.0):
    """ahv_refine_gradient_sharded: `refine_gradient` over a rotation set sharded across the ranks of `peer` (a
    `dist.PeerExchange`).  Every rank passes the WHOLE set R and gets the whole-set result, bit for bit what
    `refine_gradient` returns on one GPU: the rank scores its `dist.shard_bounds` slice, the kernels exchange the
    first pass (top-k lists, or with min_sep_deg > 0 the score matrix, after which the distinct selection runs on
    every rank) and the ascended slots through NVLink peer memory.  min_sep_deg > 0 needs peer.max_hyps >= N.
    One C call, no NCCL, CUDA-graph capturable (`out` = a previous result's tuple).  Returns `refine_gradient`'s tuple."""
    vs, vdt = _vol_src(vol_src)
    vt = _dev(vol_tgt, "vol_tgt")
    B = vs.shape[0]
    R, per_pair, N = _rotations(_dev(R, "R"), B)
    if tuple(vs.shape[1:]) != (16, 8, 8, 8) or tuple(vt.shape) != (B, 16, 8, 8, 8):
        raise ValueError("vol_src / vol_tgt must be [B,16,8,8,8]")
    if not 1 <= k <= min(32, N):
        raise ValueError("1 <= k <= min(32, N) expected")
    max_hyps = getattr(peer, "max_hyps", 0)
    if peer.world > 1 and (B > peer.max_pairs or k > peer.max_k or (min_sep_deg > 0 and N > max_hyps)):
        raise ValueError(f"exchange buffer holds {peer.max_pairs} pairs x top-{peer.max_k} x {max_hyps} scores; got B={B}, k={k}, "
                         f"N={N}")
    W1, W2, b2 = _head(W1, W2, b2)
    dev = vs.device
    if out is None:
        f = dict(device=dev, dtype=torch.float32)
        out = (torch.empty(B, k, **f), torch.empty(B, k, device=dev, dtype=torch.int64), torch.empty(B, k, 3, 3, **f),
               torch.empty(B, k, 3, 3, **f), torch.empty(B, k, **f), torch.empty(B, **f),
               torch.empty(B, device=dev, dtype=torch.int64), torch.empty(B, 3, 3, **f))
    fv, fi, fR, Ra, sa, bv, bi, bR = out[:8]
    need = int(_lib.lib().ahv_refine_gradient_sharded_workspace_bytes(B, N, k, peer.world))
    workspace, ws_bytes = _workspace(workspace, need, dev)
    _call("ahv_refine_gradient_sharded", dev, vs.data_ptr(), vdt, vt.data_ptr(), R.data_ptr(), int(per_pair), W1.data_ptr(),
          W2.data_ptr(), b2.data_ptr(), base_coords(dev).data_ptr(), k, int(steps), float(step_deg), float(min_sep_deg),
          fv.data_ptr(), fi.data_ptr(), fR.data_ptr(), Ra.data_ptr(), sa.data_ptr(), bv.data_ptr(), bi.data_ptr(), bR.data_ptr(),
          B, N, math, workspace.data_ptr(), ws_bytes, peer.rank, peer.world, _peer_array(peer), peer.max_pairs, peer.max_k,
          max_hyps)
    return fv, fi, fR, Ra, sa, bv, bi, bR, workspace


def topk(scores: torch.Tensor, k: int, idx_offset: int = 0):
    """torch.max / top-k with the reference's tie rule (lowest index wins)."""
    s = _dev(scores, "scores")
    B, N = s.shape
    val = torch.empty(B, k, device=s.device, dtype=torch.float32)
    idx = torch.empty(B, k, device=s.device, dtype=torch.int64)
    ws, ws_bytes = _workspace(None, workspace_bytes(B, N, k), s.device)
    _call("ahv_topk", s.device, s.data_ptr(), B, N, k, idx_offset, val.data_ptr(), idx.data_ptr(), ws.data_ptr(), ws_bytes)
    return val, idx


def topk_distinct(scores: torch.Tensor, R: torch.Tensor, k: int, min_sep_deg: float, gather: bool = True):
    """ahv_topk_distinct: per pair, the k best hypotheses whose rotations lie pairwise more than `min_sep_deg` apart
    (greedy geodesic non-maximum suppression in `topk`'s order).  scores [B,N]; R [N,3,3] or [B,N,3,3].  Returns
    (topk_val [B,k], topk_idx [B,k], R_best [B,k,3,3] or None); slots no hypothesis fills are (-inf, -1, NaN).
    min_sep_deg = 0 gives `topk` bit for bit, 180 the top-1 alone."""
    s, R = _dev(scores, "scores"), _dev(R, "R")
    B, N = s.shape
    per_pair = R.dim() == 4
    if tuple(R.shape) != ((B, N, 3, 3) if per_pair else (N, 3, 3)):
        raise ValueError("R must be [N,3,3] or [B,N,3,3] for scores [B,N]")
    if not 1 <= k <= 32:
        raise ValueError("k must be in [1,32]")
    val = torch.empty(B, k, device=s.device, dtype=torch.float32)
    idx = torch.empty(B, k, device=s.device, dtype=torch.int64)
    Rb = torch.empty(B, k, 3, 3, device=s.device, dtype=torch.float32) if gather else None
    _call("ahv_topk_distinct", s.device, s.data_ptr(), R.data_ptr(), int(per_pair), B, N, k, float(min_sep_deg), val.data_ptr(),
          idx.data_ptr(), Rb.data_ptr() if gather else None)
    return val, idx, Rb


def posterior_mass_workspace_bytes(B: int, N: int, k: int) -> int:
    """Bytes of scratch `posterior_mass` needs (0 for invalid sizes)."""
    return int(_lib.lib().ahv_posterior_mass_workspace_bytes(B, N, k))


def _posterior_args(scores, R, centers):
    """The checks `posterior_mass` and `posterior_moments` share: (scores, R, per_pair, centers or None)."""
    s, R = _dev(scores, "scores"), _dev(R, "R")
    B, N = s.shape
    per_pair = R.dim() == 4
    if tuple(R.shape) != ((B, N, 3, 3) if per_pair else (N, 3, 3)):
        raise ValueError("R must be [N,3,3] or [B,N,3,3] for scores [B,N]")
    c = None
    if centers is not None:
        c = _dev(centers, "centers")
        if c.dim() != 4 or c.shape[0] != B or tuple(c.shape[2:]) != (3, 3):
            raise ValueError("centers must be [B,k,3,3]")
    return s, R, per_pair, c


def posterior_mass(scores: torch.Tensor, R: torch.Tensor, centers: torch.Tensor | None, radius_deg: float,
                   temperature: float = 0.1, workspace: torch.Tensor | None = None):
    """ahv_posterior_mass: the softmax p_b(n) = exp(scores[b,n]/T) / Z_b over the hypothesis set, summarised per pair.
    Returns (log_z [B] = log Z_b, mass [B,k]): mass[b,j] is the probability of the hypotheses whose lowest slot j with
    trace(R_n c_j^T) >= fp32(1 + 2 cos(radius_deg)) is j - `topk_distinct`'s trace test, so with centers = its R_best
    and radius_deg = its min_sep_deg, slot j holds its winner and the hypotheses that winner suppressed.  scores [B,N];
    R [N,3,3] or [B,N,3,3]; centers [B,k,3,3] (NaN = empty slot, mass 0) or None (k = 0: mass is [B,0]).  A pair with a
    NaN or +inf score gets NaN outputs.  Deterministic, bit-identical whatever the batch around a pair."""
    s, R, per_pair, c = _posterior_args(scores, R, centers)
    B, N = s.shape
    k = 0 if c is None else c.shape[1]
    log_z = torch.empty(B, device=s.device, dtype=torch.float32)
    mass = torch.empty(B, k, device=s.device, dtype=torch.float32)
    workspace, ws_bytes = _workspace(workspace, posterior_mass_workspace_bytes(B, N, k), s.device)
    _call("ahv_posterior_mass", s.device, s.data_ptr(), R.data_ptr(), int(per_pair), c.data_ptr() if k else None, B, N, k,
          float(radius_deg), float(temperature), log_z.data_ptr(), mass.data_ptr() if k else None, workspace.data_ptr(),
          ws_bytes)
    return log_z, mass


def posterior_moments_workspace_bytes(B: int, N: int, k: int) -> int:
    """Bytes of scratch `posterior_moments` needs (0 for invalid sizes)."""
    return int(_lib.lib().ahv_posterior_moments_workspace_bytes(B, N, k))


def posterior_moments(scores: torch.Tensor, R: torch.Tensor, centers: torch.Tensor, radius_deg: float,
                      temperature: float = 0.1, workspace: torch.Tensor | None = None):
    """ahv_posterior_moments: `posterior_mass` (the same slots, and log_z and mass bit for bit) and the first moment of
    p_b over each slot.  Returns (log_z [B], mass [B,k], mean_R [B,k,3,3], mean_cos [B,k], moment [B,k,3,3]):
    moment[b,j] = M_j, the p-weighted mean of the hypothesis matrices in slot j; mean_R[b,j] = argmax over SO(3) of
    tr(R^T M_j), a proper rotation; mean_cos[b,j] = (tr(mean_R^T M_j) - 1) / 2, the p-weighted mean of cos(angle
    between R_n and mean_R) over the slot.  centers [B,k,3,3], 1 <= k <= 32.  NaN moments, mean_R and mean_cos for a
    slot that holds no probability (an empty centre, all -inf scores, or exp((s - max)/T) underflowing in double) and
    for a pair with a NaN or +inf score.  Deterministic, bit-identical whatever the batch around a pair."""
    s, R, per_pair, c = _posterior_args(scores, R, centers)
    B, N = s.shape
    k = 0 if c is None else c.shape[1]
    if k == 0:
        raise ValueError("posterior_moments needs centers [B,k,3,3] with k >= 1")
    f32 = dict(device=s.device, dtype=torch.float32)
    log_z, mass, mean_cos = torch.empty(B, **f32), torch.empty(B, k, **f32), torch.empty(B, k, **f32)
    mean_R, moment = torch.empty(B, k, 3, 3, **f32), torch.empty(B, k, 3, 3, **f32)
    workspace, ws_bytes = _workspace(workspace, posterior_moments_workspace_bytes(B, N, k), s.device)
    _call("ahv_posterior_moments", s.device, s.data_ptr(), R.data_ptr(), int(per_pair), c.data_ptr(), B, N, k,
          float(radius_deg), float(temperature), log_z.data_ptr(), mass.data_ptr(), mean_R.data_ptr(), mean_cos.data_ptr(),
          moment.data_ptr(), workspace.data_ptr(), ws_bytes)
    return log_z, mass, mean_R, mean_cos, moment


def topk_merge(vals: torch.Tensor, idx: torch.Tensor):
    """Merge [parts,B,k] shard lists into [B,k] (same ordering rule)."""
    v, i = _dev(vals, "vals"), _dev(idx, "idx", torch.int64)
    parts, B, k = v.shape
    out_v = torch.empty(B, k, device=v.device, dtype=torch.float32)
    out_i = torch.empty(B, k, device=v.device, dtype=torch.int64)
    _call("ahv_topk_merge", v.device, v.data_ptr(), i.data_ptr(), parts, B, k, out_v.data_ptr(), out_i.data_ptr())
    return out_v, out_i


def gather_rotations(R: torch.Tensor, idx: torch.Tensor, idx_offset: int = 0) -> torch.Tensor:
    """sampled_R[pred_index] (modules/model.py:196): [B,k,3,3]."""
    R, idx = _dev(R, "R"), _dev(idx, "idx", torch.int64)
    B, k = idx.shape
    R, per_pair, N = _rotations(R, B)
    out = torch.empty(B, k, 3, 3, device=R.device, dtype=torch.float32)
    _call("ahv_gather_rotations", R.device, R.data_ptr(), int(per_pair), idx.data_ptr(), idx_offset, B, N, k, out.data_ptr())
    return out


class HostSession:
    """Caller-owned device scratch of the host-buffer entry (`ahv_host_session_create`), reused across calls."""

    def __init__(self, device="cuda"):
        import ctypes

        self.device = torch.device(device)
        h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ahv_host_session_create(ctypes.byref(h)), "ahv_host_session_create")
        self.handle = h

    def close(self):
        if getattr(self, "handle", None) is not None:
            with torch.cuda.device(self.device):
                _lib.lib().ahv_host_session_destroy(self.handle)
            self.handle = None

    __del__ = close


def predict_host(vol_src, vol_tgt, R, W1, W2, b2, k: int = 1, math: int = MATH_TC, return_scores: bool = False,
                 device="cuda", session: HostSession | None = None, idx_offset: int = 0, peer=None):
    """HOST tensors in, HOST results out (copies inside the call): `ahv_predict_host`, or with a `session`
    (reused device scratch), bf16 source volumes, an index offset or a `peer` exchange (`R` = this rank's slice
    of a sharded rotation set; results over the whole set) `ahv_predict_host_ex`."""
    f = torch.float32
    bf16 = vol_src.dtype == torch.bfloat16
    vs, vt = (vol_src if bf16 else vol_src.to(f)).contiguous(), vol_tgt.to(f).contiguous()
    Rc = R.to(f).contiguous()
    if vs.is_cuda or vt.is_cuda or Rc.is_cuda:
        raise RuntimeError("predict_host takes host tensors")
    W1c, W2c, b2c = W1.reshape(32, 384).to(f).contiguous().cpu(), W2.reshape(32, 32).to(f).contiguous().cpu(), b2.to(f).contiguous().cpu()
    B = vs.shape[0]
    Rc, per_pair, N = _rotations(Rc, B)
    scores = torch.empty(B, N, dtype=f) if return_scores else None
    val = torch.empty(B, k, dtype=f)
    idx = torch.empty(B, k, dtype=torch.int64)
    Rb = torch.empty(B, k, 3, 3, dtype=f)
    base = base_coords()
    device = torch.device(device)
    sc = scores.data_ptr() if scores is not None else None
    extended = session is not None or bf16 or idx_offset != 0 or peer is not None
    if not extended:
        _call("ahv_predict_host", device, vs.data_ptr(), vt.data_ptr(), Rc.data_ptr(), int(per_pair), W1c.data_ptr(),
              W2c.data_ptr(), b2c.data_ptr(), base.data_ptr(), sc, val.data_ptr(), idx.data_ptr(), Rb.data_ptr(), k, B, N, math)
        return scores, val, idx, Rb
    own = session is None
    if own:
        session = HostSession(device)
    try:
        _call("ahv_predict_host_ex", device, session.handle, vs.data_ptr(), VOL_BF16 if bf16 else VOL_F32, vt.data_ptr(),
              Rc.data_ptr(), int(per_pair), W1c.data_ptr(), W2c.data_ptr(), b2c.data_ptr(), base.data_ptr(), sc, val.data_ptr(),
              idx.data_ptr(), Rb.data_ptr(), k, idx_offset, B, N, math, peer.rank if peer else 0, peer.world if peer else 1,
              _peer_array(peer) if peer else None, peer.max_pairs if peer else 0, peer.max_k if peer else 0)
    finally:
        if own:
            session.close()
    return scores, val, idx, Rb
