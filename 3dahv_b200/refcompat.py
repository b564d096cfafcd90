"""Reference-signature wrappers so call sites written against 3DAHV keep working.

    rotate_volume(volume, rotation_matrix, padding_mode='zeros')    utils.py:113
    forward_3d2d(feature_aligner, img_feat)                         modules/modules.py:112
    random_rotations(n)                                             pytorch3d (modules/model.py:184)
    verify(feature_aligner, img_feat_src, img_feat_tgt, sampled_R)  the idiom modules/model.py:186-196

All of them run on the GPU through lib3dahv_b200 and raise on CPU tensors.  `rotate_volume` and `forward_3d2d`
stay differentiable when autograd is recording and their inputs require a gradient (the reference trains through
them, modules/model.py:53-56; `rotate_volume` in the volume and in the rotation matrix, as F.grid_sample is);
otherwise they are single kernels with no autograd graph.
"""
from __future__ import annotations

import torch

from . import ops, so3
from .verify import HypothesisVerifier


def rotate_volume(volume: torch.Tensor, rotation_matrix: torch.Tensor, padding_mode: str = "zeros") -> torch.Tensor:
    """utils.py:113-131.  `volume` [N,C,D,H,W] — typically a stride-0 `expand` of
    one volume (modules/model.py:186), detected and passed once instead of N times."""
    if padding_mode != "zeros":
        raise NotImplementedError("the reference only ever uses padding_mode='zeros' (utils.py:113)")
    if volume.dim() != 5:
        raise ValueError("volume must be [N,16,8,8,8]")
    shared = volume.stride(0) == 0 or volume.shape[0] == 1
    v = volume[0].float() if shared else volume.float()
    # the reference back-propagates through this call (modules/model.py:53), to the volume and to the rotations
    if torch.is_grad_enabled() and (volume.requires_grad or rotation_matrix.requires_grad):
        from . import training
        return training.rotate_volume(v, rotation_matrix.float())
    return ops.rotate_volume(v, rotation_matrix.float())


def forward_3d2d(feature_aligner, img_feat: torch.Tensor) -> torch.Tensor:
    """Feature_Aligner.forward_3d2d (modules/modules.py:112-124): [M,16,8,8,8] -> [M,32,64]."""
    head = feature_aligner.feature_embedding_2d
    w1, w2, b2 = head[0].weight, head[2].weight, head[2].bias
    if torch.is_grad_enabled() and (img_feat.requires_grad or w1.requires_grad or w2.requires_grad or b2.requires_grad):
        from . import training   # the reference trains through this call (modules/model.py:54-55)
        return training.head_torch(img_feat.float(), w1, w2, b2)
    return ops.forward_3d2d(img_feat.float(), w1.detach(), w2.detach(), b2.detach())


def random_rotations(n: int, dtype=None, device=None) -> torch.Tensor:
    return so3.random_rotations(n, dtype=dtype, device=device)


def verify(feature_aligner, img_feat_src, img_feat_tgt, sampled_R, k: int = 1, math=None):
    """modules/model.py:186-196 in one call: returns (pred_sim [B,N], pred_index [B] or [B,k],
    pred_src_2_tgt_R [B,3,3] or [B,k,3,3])."""
    v = HypothesisVerifier.from_feature_aligner(feature_aligner, math)
    r = v.score(img_feat_src, img_feat_tgt, sampled_R, k=k, return_scores=True)
    if k == 1:
        return r.scores, r.topk_idx[:, 0], r.R_best[:, 0]
    return r.scores, r.topk_idx, r.R_best
