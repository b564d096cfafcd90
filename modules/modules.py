"""Feature_Aligner — 2D->3D lifting (PyTorch) and the 3D->2D verification head.

State-dict compatible re-implementation of `/root/reference/modules/modules.py`
(`ResNetBlock_3D` :9-47, `Feature_Aligner` :49-124, `ResNetBlock_2D` :126-164).
`forward_2d3d` stays in PyTorch (out of the hot path, SURVEY.md §8); `forward_3d2d`
— the tri-plane 1x1-conv head the hypothesis-and-verification loop calls for every
rotated volume — runs on the GPU through lib3dahv_b200 (`ahv_forward_3d2d`), and
inside the fused scorer it is never called at all.
"""
from __future__ import annotations

import importlib

import torch
import torch.nn as nn

from transformer.attention import BidirectionTransformer


def _ahv():
    return importlib.import_module("3dahv_b200")


class _ResNetBlock(nn.Module):
    """conv3 -> ReLU -> conv3 (+ 1x1 projection of the residual when shapes differ).
    `bn_down` is created but never used in forward, exactly like the reference
    (modules/modules.py:22-30): it must exist for checkpoints to load strictly."""

    def __init__(self, conv, bn, in_channels, out_channels, stride=1, BN=False):
        super().__init__()
        self.conv1 = conv(in_channels, out_channels, kernel_size=3, stride=stride, padding=1, bias=False)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = conv(out_channels, out_channels, kernel_size=3, padding=1, bias=False)
        self.bn1 = bn(out_channels) if BN else nn.Sequential()
        self.bn2 = bn(out_channels) if BN else nn.Sequential()
        self.downsample = None
        if stride != 1 or in_channels != out_channels:
            self.downsample = nn.Sequential(conv(in_channels, out_channels, kernel_size=1, stride=stride, bias=False))
            self.bn_down = bn(out_channels)

    def forward(self, x):
        out = self.bn2(self.conv2(self.relu(self.bn1(self.conv1(x)))))
        return out + (x if self.downsample is None else self.downsample(x))


class ResNetBlock_3D(_ResNetBlock):
    def __init__(self, in_channels, out_channels, stride=1, BN=False):
        super().__init__(nn.Conv3d, nn.BatchNorm3d, in_channels, out_channels, stride, BN)
        self._fusable = (in_channels, out_channels, stride, BN) == (32, 16, 1, False)   # the one shape the model uses

    def forward(self, x):
        """modules/modules.py:32-47.  Inference on the GPU at the model's shape (32 -> 16 on 8^3, :100-101): one
        cluster launch (`ahv_resblock3d`, the step right before the hypothesis-and-verification path);
        otherwise - training, CPU, other shapes - the PyTorch convolutions.  The kernel has no backward, so it runs only
        when nothing the block computes can need a gradient: grad mode off, or neither x nor any weight forward reads
        (conv1, conv2, downsample) requires one.  `bn_down` never enters forward."""
        weights = (self.conv1.weight, self.conv2.weight, self.downsample[0].weight) if self._fusable else ()
        if (self._fusable and x.is_cuda and x.dtype == torch.float32 and tuple(x.shape[1:]) == (32, 8, 8, 8)
                and not (torch.is_grad_enabled() and (x.requires_grad or any(w.requires_grad for w in weights)))):
            return _ahv().ops.resblock3d(x, self.conv1.weight.detach(), self.conv2.weight.detach(),
                                         self.downsample[0].weight.detach())
        return super().forward(x)


class ResNetBlock_2D(_ResNetBlock):
    def __init__(self, in_channels, out_channels, stride=1, BN=False):
        super().__init__(nn.Conv2d, nn.BatchNorm2d, in_channels, out_channels, stride, BN)


def random_masking(x: torch.Tensor, mask_ratio: float) -> torch.Tensor:
    """Per-sample random voxel mask used only in training (utils.py:133-160): keep
    a random (1-ratio) subset, and with probability 1/2 keep everything."""
    n, length = x.shape[0], x.flatten(2).shape[-1]
    keep = int(length * (1 - mask_ratio))
    rank = torch.rand(n, length, device=x.device).argsort(dim=1).argsort(dim=1)
    gate = torch.rand(n, 1, device=x.device) > 0.5
    return ((rank < keep) | gate).float()


class Feature_Aligner(nn.Module):
    def __init__(self, in_channel=256, mid_channel=256, out_channel=32, n_heads=4, depth=4):
        super().__init__()
        self.in_channel, self.mid_channel, self.out_channel = in_channel, mid_channel, out_channel
        self.feature_embedding = nn.Sequential(
            nn.Conv2d(in_channel, mid_channel, kernel_size=1, bias=False),
            ResNetBlock_2D(mid_channel, mid_channel, stride=1, BN=False),
        )
        self.att = BidirectionTransformer(mid_channel, n_heads=n_heads, d_head=mid_channel // n_heads, depth=depth,
                                          dropout=0.0, context_dim=mid_channel, normalize=True)
        self.feature_embedding_3d = ResNetBlock_3D(mid_channel // 8, 16, stride=1, BN=False)
        self.feature_embedding_2d = nn.Sequential(
            nn.Conv2d(3 * 8 * 16, out_channel, kernel_size=1, bias=False),
            nn.ReLU(inplace=True),
            nn.Conv2d(out_channel, out_channel, kernel_size=1),
        )

    @staticmethod
    def posemb_sincos_2d(patches, channel=128, temperature=10000, dtype=torch.float32):
        """[channel,h,w] sin/cos positional code, x-sin | x-cos | y-sin | y-cos (modules/modules.py:72-84)."""
        h, w, device = patches.shape[-2], patches.shape[-1], patches.device
        assert channel % 4 == 0, "feature dimension must be multiple of 4 for sincos emb"
        y, x = torch.meshgrid(torch.arange(h, device=device), torch.arange(w, device=device), indexing="ij")
        omega = torch.arange(channel // 4, device=device) / (channel // 4 - 1)
        omega = 1.0 / (temperature ** omega)
        y = y[None] * omega[:, None, None]
        x = x[None] * omega[:, None, None]
        return torch.cat((x.sin(), x.cos(), y.sin(), y.cos()), dim=0).type(dtype)

    def forward_2d3d(self, img_feat_src, img_feat_tgt, random_mask=True, mask_ratio=0.25):
        """[B,in,8,8] x2 -> two feature volumes [B,16,8,8,8] (modules/modules.py:86-110)."""
        bs = img_feat_src.shape[0]
        src = self.feature_embedding(img_feat_src)
        tgt = self.feature_embedding(img_feat_tgt)
        pe = self.posemb_sincos_2d(src, channel=self.mid_channel)[None]
        src, tgt = self.att(src + pe, tgt + pe)
        src = self.feature_embedding_3d(src.reshape(bs, self.mid_channel // 8, 8, 8, 8))
        tgt = self.feature_embedding_3d(tgt.reshape(bs, self.mid_channel // 8, 8, 8, 8))
        if random_mask is True:
            src = src * random_masking(src, mask_ratio).reshape(-1, 1, 8, 8, 8)
            tgt = tgt * random_masking(tgt, mask_ratio).reshape(-1, 1, 8, 8, 8)
        return src, tgt

    def forward_3d2d(self, img_feat):
        """[M,16,8,8,8] -> [M,32,64] unit feature vectors (modules/modules.py:112-124).  Inference: one kernel
        (`ahv_forward_3d2d`).  When autograd is recording and the input or the head can receive a gradient - the
        reference trains through this call (modules/model.py:53-56) - the differentiable formulation is used
        instead, so reference-style training code keeps its gradients."""
        return _ahv().refcompat.forward_3d2d(self, img_feat)
