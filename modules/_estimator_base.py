"""Shared machinery of the drop-in Estimators (modules/model.py, modules/model_co3d.py)."""
from __future__ import annotations

import importlib
import math

import torch
import torch.nn as nn

try:  # Lightning is optional: the reference subclasses pl.LightningModule (modules/model.py:28)
    import lightning.pytorch as pl

    _Base = pl.LightningModule
except Exception:  # pragma: no cover - lightning is absent in this image
    pl = None
    _Base = nn.Module

from modules._backbone import build_backbone
from modules.modules import Feature_Aligner


def _ahv():
    return importlib.import_module("3dahv_b200")


def geodesic_deg(R_a: torch.Tensor, R_b: torch.Tensor) -> torch.Tensor:
    """arccos((tr(Ra^T Rb) - 1)/2) in degrees (modules/model.py:198-200)."""
    s = ((R_a.reshape(-1, 9) * R_b.reshape(-1, 9)).sum(-1).clamp(-1, 3) - 1) / 2
    return torch.arccos(s) * 180.0 / math.pi


class EstimatorBase(_Base):
    """Constructor, attributes and `feature_extraction` of the reference Estimator
    (modules/model.py:29-41); the hypothesis-and-verification idiom of the
    inference steps is replaced by one fused GPU call (`predict_rotation`)."""

    def __init__(self, cfg, feature_extractor: nn.Module | None = None):
        super().__init__()
        self.cfg = cfg
        self.num_rota = cfg["DATA"]["NUM_ROTA"]
        self.feature_extractor = build_backbone() if feature_extractor is None else feature_extractor
        self.feature_aligner = Feature_Aligner(in_channel=768, mid_channel=256, out_channel=32, n_heads=4, depth=4)
        self.step_outputs = []
        self._verifier = None
        # training: keep conv1's output in the forward and run the backward's contractions on tcgen05 (2.7x faster
        # step; gradients of the function the tensor-core forward evaluated - 3dahv_b200.training.verification_scores).
        # Off by default: the default backward matches the reference's fp32 autograd to 1e-4.
        self.fast_backward = bool(cfg.get("TRAIN", {}).get("FAST_BACKWARD", False)) if isinstance(cfg, dict) else False

    if pl is None:
        def log(self, *args, **kwargs):  # Lightning's logger hook; a no-op without Lightning
            return None

    @classmethod
    def load_reference_checkpoint(cls, checkpoint_path, cfg=None, map_location="cpu", **kwargs):
        """What the reference's scripts do with `Estimator.load_from_checkpoint(path, cfg=cfg)` (test_co3d.py:218,
        test_objaverse.py:22) for a REFERENCE checkpoint, with or without Lightning installed: reads the checkpoint's
        `state_dict` (and `hyper_parameters["cfg"]` when `cfg` is not given) and loads it through
        `modules._backbone.load_reference_state_dict` - `feature_aligner.*` strictly by name, the MiDaS/timm
        backbone keys mapped onto the SwinV2-T stand-in.  The load report is kept in `model.load_report`."""
        from modules._backbone import load_reference_state_dict

        ckpt = torch.load(checkpoint_path, map_location=map_location, weights_only=False)
        if cfg is None:
            cfg = ckpt.get("hyper_parameters", {}).get("cfg")
        if cfg is None:
            raise ValueError("pass cfg= (the checkpoint holds no hyper_parameters['cfg'])")
        model = cls(cfg, **kwargs)
        model.load_report = load_reference_state_dict(model, ckpt)
        return model

    if pl is None:   # without Lightning the reference's spelling is this loader
        load_from_checkpoint = load_reference_checkpoint

    def feature_extraction(self, img):
        return self.feature_extractor(img)

    def verifier(self):
        """HypothesisVerifier bound to the CURRENT verification-head weights."""
        head = self.feature_aligner.feature_embedding_2d
        key = (head[0].weight.data_ptr(), head[0].weight._version, head[2].weight._version, head[2].bias._version,
               head[0].weight.device)
        if self._verifier is None or self._verifier[0] != key:
            self._verifier = (key, _ahv().HypothesisVerifier.from_feature_aligner(self.feature_aligner))
        return self._verifier[1]

    @torch.no_grad()
    def predict_rotation(self, img_feat_src, img_feat_tgt, sampled_R=None, k: int = 1):
        """modules/model.py:184-196 fused: sample (or take) the hypothesis set, score every
        hypothesis for every pair, select.  Returns (pred_sim_best [B,k], pred_index [B,k],
        pred_src_2_tgt_R [B,k,3,3], sampled_R)."""
        if sampled_R is None:
            sampled_R = _ahv().so3.random_rotations(self.num_rota, device=img_feat_src.device)
        r = self.verifier().score(img_feat_src, img_feat_tgt, sampled_R, k=k, return_scores=False)
        return r.topk_val, r.topk_idx, r.R_best, sampled_R

    @torch.no_grad()
    def predict_distribution(self, img_feat_src, img_feat_tgt, sampled_R=None, k: int = 1, min_sep_deg: float = 0.0,
                             gt_R=None, moments: bool = False):
        """`predict_rotation`'s selection (with min_sep_deg > 0: the top-k of rotations pairwise more than min_sep_deg
        apart) and the probability the model gives it: `HypothesisVerifier.posterior` at the training temperature
        T = 0.1 with radius cfg["DATA"]["ACC_THR"], so `mass[b,0]` is the model's estimate that pair b's prediction is
        correct at ACC_THR.  gt_R [B,3,3]: `log_density` [B,1] is the log-density of the ground-truth rotation (w.r.t.
        the normalised Haar measure; the set should be Haar-random or near-uniform).  moments=True: also each slot's
        mean rotation `mean_R` and spread (`spread_deg`).  Returns (Posterior, sampled_R)."""
        if sampled_R is None:
            sampled_R = _ahv().so3.random_rotations(self.num_rota, device=img_feat_src.device)
        R_query = None if gt_R is None else gt_R.reshape(-1, 1, 3, 3).float().contiguous()
        post = self.verifier().posterior(img_feat_src, img_feat_tgt, sampled_R, k=k, min_sep_deg=min_sep_deg,
                                         radius_deg=float(self.cfg["DATA"]["ACC_THR"]), temperature=0.1, R_query=R_query,
                                         moments=moments)
        return post, sampled_R

    @torch.no_grad()
    def score_rotations(self, img_feat_src, img_feat_tgt, R):
        """pred_sim for an explicit rotation set: R [N,3,3] shared or [B,N,3,3] per pair
        (the ground-truth hypothesis check of modules/model.py:137-143 is N=1 per pair)."""
        return self.verifier().score(img_feat_src, img_feat_tgt, R, k=1, return_scores=True).scores

    def infoNCE_loss(self, img_feat_1, img_feat_2, sampled_R, gt_delta_R):
        """modules/model.py:43-63 — per-pair hypothesis sets [B,N,3,3] with the ground truth at index 0.
        Differentiable: the scores come from the fused kernel, their backward pass is the fused backward kernel
        (3dahv_b200.training; `self.fast_backward` / cfg["TRAIN"]["FAST_BACKWARD"] selects the saved-activation
        tensor-core form); gradients reach the volumes (hence the lifting and the backbone) and the verification
        head.  Returns the per-sample loss [B]."""
        head = self.feature_aligner.feature_embedding_2d
        tr = _ahv().training
        scores = tr.verification_scores(img_feat_1, img_feat_2, sampled_R.contiguous(), head[0].weight, head[2].weight,
                                        head[2].bias, save_activations=self.fast_backward)
        return tr.infonce_loss(scores, sampled_R, gt_delta_R, self.cfg["DATA"]["ACC_THR"])

    def _sample_training_rotations(self, gt_R):
        """modules/model.py:101-103: B*(N-1) random rotations per batch, ground truth prepended at index 0."""
        B = gt_R.shape[0]
        with torch.no_grad():
            Rs = _ahv().so3.random_rotations(B * (self.num_rota - 1), device=gt_R.device).reshape(B, self.num_rota - 1, 3, 3)
            return torch.cat([gt_R[:, None], Rs], dim=1)

    def _optimizers(self, backbone_lr_scale: float, step_size: int):
        lr = float(self.cfg["TRAIN"]["LR"])
        opt = torch.optim.AdamW([{"params": self.feature_aligner.parameters(), "lr": lr},
                                 {"params": self.feature_extractor.parameters(), "lr": backbone_lr_scale * lr}], eps=1e-5)
        return [opt], [torch.optim.lr_scheduler.StepLR(opt, step_size=step_size, gamma=0.1)]
