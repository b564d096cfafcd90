"""Training variant of the hypothesis-and-verification step (SURVEY.md §8a-8 / §8f-3).

The reference trains with `infoNCE_loss` (modules/model.py:43-63): per-pair rotation sets
`[B,N,3,3]`, `rotate_volume` -> `forward_3d2d` -> similarity -> softmax over hypotheses with
temperature 0.1, all under PyTorch autograd (≈420 KB of saved activations per hypothesis).

Here the forward scores come from the fused CUDA kernel (nothing saved), and the backward pass is ONE
fused kernel as well (`ahv_score_backward`, csrc/ahv_score_bwd.cu): per (pair, hypothesis) it recomputes
the forward in shared memory and pushes the upstream gradient back to the source volume (adjoint of the
trilinear resampling as a gather), the target features, W1, W2 and b2.  Only the B target volumes go
through PyTorch autograd (`head_torch`, negligible).  Gradients therefore flow to everything upstream of
the hot path (`forward_2d3d`, the backbone).  `fused_backward=False` selects the earlier chunked
recomputation (library `ahv_rotate_volume` / `ahv_rotate_volume_backward` + PyTorch head), kept as an
independent cross-check.

Arithmetic: with the default `math=MATH_TC` the FORWARD scores carry the tensor-core path's fp16-operand error
(~1e-4 relative) while the fused backward recomputes the forward in fp32, i.e. the gradient is that of a function
1e-4 away from the loss reported (tests/test_gpu_training.py holds the end-to-end gradients to 5e-3 of their maximum
against the reference's autograd in this mode, 2e-4 with `math=MATH_FP32`, which is 8x slower in the forward only).
By default the backward accumulates dV, dT, dW1, dW2, db2 across CTAs with float atomics, so gradients are
reproducible to rounding, not bit for bit, from run to run.  Under `torch.use_deterministic_algorithms(True)` (read when
the backward runs, as PyTorch's own ops do; Lightning's `Trainer(deterministic=True)` sets it) the fused backward runs
the deterministic form of the same kernels instead (`ahv_score_backward_det`: per-CTA partials in a workspace, summed
in a fixed order), and gradients are bit-identical from run to run on one device.  The paths that still scatter with
float atomics - `rotate_volume`'s backward w.r.t. the volume (`ahv_rotate_volume_backward`), and so
`fused_backward=False` - then follow PyTorch's convention for `F.grid_sample`'s backward: they raise a RuntimeError
naming the op, or warn under `warn_only=True`.

Fast form (`save_activations=True`, opt-in): the tensor-core forward also keeps conv1's ReLU'd output (fp16, 4 KB per
hypothesis - `ahv_score_train`), and the backward (`ahv_score_backward_saved`, csrc/ahv_score_bwd_tc.cu) reads it
instead of recomputing conv1 and runs its five contractions (conv2, dH1, dW2, dA, dW1) on tcgen05: 8.7 ms against
24.8 ms for the 12 x 9000 step.  Its gradient is that of the function the forward evaluated (the forward's ReLU
mask), with fp16 operand rounding - see `verification_scores`.

Rotation gradients: the reference's rotate_volume (F.affine_grid + F.grid_sample) is differentiable in the rotation
matrix as well, and so are `rotate_volume` and `verification_scores` here - `R.requires_grad_()` gives `R.grad`, with
ATen's convention at lattice points and at the volume's edge (DESIGN.md §4.4).  The fused backward then runs
`ahv_score_backward_ex`, the fp32 kernel with a rotation phase added; nothing changes for an R that needs no gradient.
`infonce_loss` keeps `sampled_R` as data: its positive mask is a step function of R.
"""
from __future__ import annotations

import math
import warnings

import torch
import torch.nn.functional as F

from . import ops
from ._lib import MATH_FP32, MATH_TC


def _alert_not_deterministic(op: str) -> None:
    """PyTorch's convention for an op without a deterministic implementation under
    `torch.use_deterministic_algorithms(True)`: raise, or warn with `warn_only=True`."""
    if not torch.are_deterministic_algorithms_enabled():
        return
    msg = (f"{op} does not have a deterministic implementation, but you set 'torch.use_deterministic_algorithms(True)'. "
           "You can turn off determinism just for this operation, or you can use the 'warn_only=True' option, if that's "
           "acceptable for your application. verification_scores with fused_backward=True (the default) has a "
           "deterministic backward.")
    if torch.is_deterministic_algorithms_warn_only_enabled():
        warnings.warn(msg, UserWarning, stacklevel=3)
    else:
        raise RuntimeError(msg)


class _RotateVolume(torch.autograd.Function):
    """utils.rotate_volume (utils.py:113-131) with gradients w.r.t. the volume and the rotations (F.grid_sample's
    backward through F.affine_grid: `ahv_rotate_volume_backward` and `ahv_rotate_volume_grad_R`)."""

    @staticmethod
    def forward(ctx, volume, R):
        ctx.per_rot = volume.dim() == 5
        ctx.save_for_backward(R, volume.detach() if ctx.needs_input_grad[1] else None)
        return ops.rotate_volume(volume.detach(), R)

    @staticmethod
    def backward(ctx, grad_out):
        R, volume = ctx.saved_tensors
        g = grad_out.contiguous()
        if ctx.needs_input_grad[0]:   # the adjoint scatters with float atomics; the gradient w.r.t. R has one writer
            _alert_not_deterministic("ahv_rotate_volume_backward (the backward of training.rotate_volume w.r.t. the volume)")
        g_vol = ops.rotate_volume_backward(g, R, ctx.per_rot) if ctx.needs_input_grad[0] else None
        g_R = ops.rotate_volume_grad_R(volume, g, R, ctx.per_rot) if ctx.needs_input_grad[1] else None
        return g_vol, g_R


def rotate_volume(volume: torch.Tensor, R: torch.Tensor) -> torch.Tensor:
    """Differentiable (w.r.t. `volume` and `R`) GPU rotate_volume: [16,8,8,8] or [n,16,8,8,8] with R [n,3,3]."""
    return _RotateVolume.apply(volume, R)


def head_torch(vol: torch.Tensor, W1, W2, b2) -> torch.Tensor:
    """Feature_Aligner.forward_3d2d (modules/modules.py:112-124) in differentiable torch ops."""
    m = vol.shape[0]
    x = vol.permute(0, 1, 4, 2, 3).reshape(m, 128, 8, 8)
    y = vol.permute(0, 1, 3, 2, 4).reshape(m, 128, 8, 8)
    z = vol.reshape(m, 128, 8, 8)
    t = torch.cat([x, y, z], dim=1).flatten(2)                       # [m,384,64]
    # the 1x1 convolutions as matmuls: fp32 at torch's default "highest" matmul precision (cuDNN's
    # default for convolutions would be TF32)
    t = torch.matmul(W1.reshape(32, 384), t)
    t = torch.matmul(W2.reshape(32, 32), F.relu(t)) + b2[None, :, None]
    return F.normalize(t, p=2, dim=1)


class _VerifyScores(torch.autograd.Function):
    """scores[b,n] of modules/model.py:53-56; forward fused, backward fused (exact fp32 kernel, saved-activation
    tensor-core kernel) or chunked recomputation.  R's gradient, when it needs one, comes from the fp32 kernel's
    rotation phase (`ahv_score_backward_ex`) or, chunked, through `_RotateVolume`."""

    @staticmethod
    def forward(ctx, vol_src, vol_tgt, R, W1, W2, b2, math, chunk, fused_backward, save_activations, tc_backward=True):
        tgt = ops.forward_3d2d(vol_tgt.detach().float(), W1.detach(), W2.detach(), b2.detach())
        h1 = pair_inv = None
        needs_grad = any(t.requires_grad for t in (vol_src, vol_tgt, R, W1, W2, b2))
        if save_activations and fused_backward and math == MATH_TC and needs_grad and vol_src.dtype == torch.float32:
            # tensor-core forward that keeps conv1's ReLU'd output (4 KB per item) for the backward kernel
            scores, h1, pair_inv = ops.score_train(vol_src.detach(), tgt, R, W1.detach(), W2.detach(), b2.detach())
        else:
            scores, _, _ = ops.score(vol_src.detach().float(), tgt, R, W1.detach(), W2.detach(), b2.detach(), k=0, math=math,
                                     return_scores=True)
        ctx.save_for_backward(vol_src, vol_tgt, R, W1, W2, b2, tgt, h1, pair_inv)
        ctx.chunk = chunk
        ctx.fused_backward = fused_backward
        ctx.bwd_math = MATH_TC if tc_backward else MATH_FP32
        return scores

    @staticmethod
    def backward(ctx, grad_scores):
        vol_src, vol_tgt, R, W1, W2, b2, tgt_saved, h1, pair_inv = ctx.saved_tensors
        B = vol_src.shape[0]
        per_pair = R.dim() == 4
        N = R.shape[1] if per_pair else R.shape[0]
        want_R = ctx.needs_input_grad[2]
        if ctx.fused_backward:
            # with R's gradient: ahv_score_backward_ex, the same fp32 kernel (and, with saved activations, the same kept
            # values and ReLU mask) plus its rotation phase - the tcgen05 backward has none
            g = ops.score_backward(vol_src.detach().float(), tgt_saved, R.detach(), W1.detach().float(), W2.detach().float(),
                                   b2.detach().float(), grad_scores.contiguous().float(), h1, pair_inv, ctx.bwd_math,
                                   want_grad_R=want_R, deterministic=torch.are_deterministic_algorithms_enabled())
            g_vs, g_tgt, g_w1, g_w2, g_b = g[:5]
            with torch.enable_grad():   # target side: B volumes through the differentiable head
                vt = vol_tgt.detach().float().requires_grad_(True)
                w1, w2, bb = (t.detach().float().requires_grad_(True) for t in (W1, W2, b2))
                gt = torch.autograd.grad(head_torch(vt, w1, w2, bb), [vt, w1, w2, bb], grad_outputs=g_tgt)
            return (g_vs, gt[0], g[5] if want_R else None, (g_w1 + gt[1].reshape(32, 384)).reshape(W1.shape),
                    (g_w2 + gt[2].reshape(32, 32)).reshape(W2.shape), g_b + gt[3], None, None, None, None, None)
        with torch.enable_grad():
            vs = vol_src.detach().float().requires_grad_(True)
            vt = vol_tgt.detach().float().requires_grad_(True)
            w1, w2, bb = (t.detach().float().requires_grad_(True) for t in (W1, W2, b2))
            Rl = R.detach().requires_grad_(want_R)
            tgt = head_torch(vt, w1, w2, bb)                                # [B,32,64]
            tgt_leaf = tgt.detach().requires_grad_(True)                    # cut here: tgt's own graph is walked once, below
            total = None
            for b in range(B):
                Rb = Rl[b] if per_pair else Rl
                for a in range(0, N, ctx.chunk):
                    Rc = Rb[a:a + ctx.chunk].contiguous()
                    f = head_torch(rotate_volume(vs[b], Rc), w1, w2, bb)   # recomputed, freed after this chunk
                    s = (f * tgt_leaf[b][None]).sum(dim=1).mean(dim=-1)
                    part = (s * grad_scores[b, a:a + ctx.chunk]).sum()
                    # backward per chunk keeps the live graph at chunk size
                    gs = torch.autograd.grad(part, [vs, w1, w2, bb, tgt_leaf] + ([Rl] if want_R else []), allow_unused=True)
                    total = gs if total is None else tuple(x + y if (x is not None and y is not None) else (x if y is None else y)
                                                           for x, y in zip(total, gs))
            g_vs, g_w1, g_w2, g_b, g_tgt = total[:5]
            g_R = total[5] if want_R else None
            # through the target features to vol_tgt and (again) the head weights
            gt = torch.autograd.grad(tgt, [vt, w1, w2, bb], grad_outputs=g_tgt, allow_unused=True)
            g_vt = gt[0]
            g_w1, g_w2, g_b = g_w1 + gt[1], g_w2 + gt[2], g_b + gt[3]
        return g_vs, g_vt, g_R, g_w1.reshape(W1.shape), g_w2.reshape(W2.shape), g_b, None, None, None, None, None


def verification_scores(vol_src, vol_tgt, R, W1, W2, b2, math: int = MATH_TC, chunk: int = 1024,
                        fused_backward: bool = True, save_activations: bool = False, tc_backward: bool = True) -> torch.Tensor:
    """Differentiable pred_sim [B,N] (modules/model.py:53-56 / :193).  R [N,3,3] or [B,N,3,3].
    `save_activations` (opt-in; tensor-core forward + fused backward only): the forward keeps conv1's ReLU'd output of
    every (pair, hypothesis) - 4 KB per item in fp16, against the ~420 KB per hypothesis the reference's autograd keeps -
    and the backward kernel reads it instead of recomputing conv1 in fp32 (a third of its arithmetic; 24.8 -> 20.3 ms
    for the 12 x 9000 step).  The gradient is then that of the function the forward actually evaluated: the ReLU mask
    comes from the fp16-operand conv1, so the ~0.05 % of pre-activations within 3e-4 of zero can sit on the other side
    of ReLU's kink than in an fp32 evaluation.  Gradients that do not pass through the mask (vol_tgt, W2, b2) agree
    with the default to 4e-4 of their maximum; vol_src / W1 to a few per cent at the voxels such an element feeds
    (measured 2.6 % of the maximum; tests/test_gpu_training.py).  The default recomputes and matches the reference's
    fp32 autograd to 1e-4.  With saved activations `tc_backward` (default) also moves the backward's two large
    contractions, dA = dH1 W1 and dW1 = dH1^T A, to tcgen05 with fp16 operands under power-of-two scales
    (csrc/ahv_score_bwd_tc.cu); False keeps them in fp32 FFMA.
    When `R` requires a gradient, `R.grad` is d/dR of the scores ([N,3,3] summed over pairs, or [B,N,3,3]).  The fused
    backward computes it, and the other gradients, with `ahv_score_backward_ex` in fp32 FFMA; with saved activations
    that call replaces the tcgen05 backward whatever `tc_backward` says (same kept values, same ReLU mask, fp32
    contractions).  The chunked form differentiates through `rotate_volume` instead.
    Under `torch.use_deterministic_algorithms(True)` the fused backward runs the deterministic form of whichever kernel
    the rules above pick (`ops.score_backward(..., deterministic=True)`): bit-identical gradients from run to run.  The
    chunked form (`fused_backward=False`) has none: it raises there, or warns with `warn_only=True`."""
    return _VerifyScores.apply(vol_src, vol_tgt, R.contiguous(), W1, W2, b2, math, chunk, fused_backward, save_activations,
                               tc_backward)


class _InfoNCE(torch.autograd.Function):
    """modules/model.py:43-63 given the scores: loss and d loss / d scores from ONE kernel (`ahv_infonce`)."""

    @staticmethod
    def forward(ctx, scores, sampled_R, gt_delta_R, acc_thr_deg, temperature):
        loss, grad = ops.infonce(scores.detach().float(), sampled_R, gt_delta_R, acc_thr_deg, temperature,
                                 want_grad=scores.requires_grad)
        ctx.save_for_backward(grad)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        (grad,) = ctx.saved_tensors
        return grad * grad_loss[:, None], None, None, None, None


def infonce_loss(scores: torch.Tensor, sampled_R: torch.Tensor, gt_delta_R: torch.Tensor, acc_thr_deg: float,
                 temperature: float = 0.1, fused: bool = True) -> torch.Tensor:
    """modules/model.py:43-63 given the scores: positives = hypotheses within `acc_thr_deg` of the
    ground-truth rotation; loss_b = -log(sum_pos e^{s/T} / sum_all e^{s/T}).  Returns [B].  `fused` (default): one
    kernel for the loss and its gradient; otherwise the eager torch formulation below (kept as a cross-check)."""
    if fused and scores.is_cuda:
        return _InfoNCE.apply(scores, sampled_R.contiguous(), gt_delta_R.contiguous(), float(acc_thr_deg), float(temperature))
    return infonce_loss_torch(scores, sampled_R, gt_delta_R, acc_thr_deg, temperature)


def infonce_loss_torch(scores: torch.Tensor, sampled_R: torch.Tensor, gt_delta_R: torch.Tensor, acc_thr_deg: float,
                       temperature: float = 0.1) -> torch.Tensor:
    """The same loss in eager torch ops."""
    with torch.no_grad():
        gt_sim = ((sampled_R.flatten(-2) * gt_delta_R.reshape(-1, 1, 9)).sum(-1).clamp(-1, 3) - 1) / 2
        positive = (180.0 * torch.arccos(gt_sim) / math.pi) <= acc_thr_deg
    e = torch.exp(scores / temperature)
    return -torch.log((e * positive).sum(-1) / e.sum(-1).clamp(min=1e-8))
