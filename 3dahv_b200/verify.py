"""HypothesisVerifier — the fused hypothesis-and-verification step.

Replaces the idiom the reference pastes at modules/model.py:131-146, :184-196,
test_co3d.py:137-146 and test_linemod.py:43-63:

    rotate_volume(vol.expand(N), R) -> forward_3d2d -> (a*b[:,None]).sum(2).mean(-1)
    -> torch.max(dim=1) -> R[idx]

with one call into lib3dahv_b200 (no rotated volume, grid or feature tensor is
ever materialised).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch

from . import ops
from ._lib import MATH_FP32, MATH_TC, MATH_TC_F16GATHER

DEFAULT_MATH = MATH_TC


def _src_volume(vol_src):
    """A bf16 source volume as it is, any other as fp32: the two dtypes the scoring kernels read."""
    return vol_src if vol_src.dtype == torch.bfloat16 else vol_src.float()


def _clamp_k(k: int, R):
    """(min(k, N), N) for a rotation set R [N,3,3] (shared) or [B,N,3,3] (per pair)."""
    N = R.shape[1] if R.dim() == 4 else R.shape[0]
    return min(k, N), N


@dataclass
class VerifyResult:
    scores: torch.Tensor | None    # [B,N] pred_sim (modules/model.py:193)
    topk_val: torch.Tensor         # [B,k]
    topk_idx: torch.Tensor         # [B,k] int64, global hypothesis index
    R_best: torch.Tensor           # [B,k,3,3] sampled_R[pred_index] (:196)


@dataclass
class Posterior:
    """The selection and what the verifier's softmax p_b(n) = exp(s[b,n]/T) / Z_b says about it (`posterior`)."""
    topk_val: torch.Tensor                # [B,k]
    topk_idx: torch.Tensor                # [B,k] int64 (-1: empty distinct slot)
    R_best: torch.Tensor                  # [B,k,3,3] (NaN: empty distinct slot)
    mass: torch.Tensor                    # [B,k] probability held by each selected rotation's neighbourhood
    log_z: torch.Tensor                   # [B] log Z_b
    log_density: torch.Tensor | None      # [B,Q] log-density of R_query w.r.t. the normalised Haar measure
    mean_R: torch.Tensor | None = None    # [B,k,3,3] p-weighted mean rotation of each slot (moments=True)
    mean_cos: torch.Tensor | None = None  # [B,k] p-weighted mean of cos(angle to mean_R) over each slot
    moment: torch.Tensor | None = None    # [B,k,3,3] p-weighted mean of the slot's hypothesis matrices

    @property
    def spread_deg(self) -> torch.Tensor | None:
        """[B,k] arccos of mean_cos in degrees: each mode's width, close to the RMS angle to mean_R when the mode is
        concentrated (None without moments)."""
        if self.mean_cos is None:
            return None
        return torch.rad2deg(torch.arccos(self.mean_cos.clamp(-1.0, 1.0)))


def _posterior_radius(min_sep_deg: float, radius_deg: float | None) -> float:
    if radius_deg is not None:
        return radius_deg
    if not min_sep_deg > 0:
        raise ValueError("radius_deg is required when min_sep_deg is 0")
    return min_sep_deg


def _posterior(scores, R, k, min_sep_deg, radius_deg, temperature, s_query, moments=False) -> Posterior:
    """The selection (`ops.topk` or `ops.topk_distinct`) and `ops.posterior_mass` (with moments: `ops.posterior_moments`)
    over a whole [B,N] score matrix."""
    if min_sep_deg > 0:
        val, idx, R_best = ops.topk_distinct(scores, R, k, min_sep_deg)
    else:
        val, idx = ops.topk(scores, k)
        R_best = ops.gather_rotations(R, idx)
    mean_R = mean_cos = moment = None
    if moments:
        log_z, mass, mean_R, mean_cos, moment = ops.posterior_moments(scores, R, R_best, radius_deg, temperature)
    else:
        log_z, mass = ops.posterior_mass(scores, R, R_best, radius_deg, temperature)
    log_density = None
    if s_query is not None:
        N = scores.shape[1]
        log_density = (s_query.double() / temperature - log_z.double()[:, None] + math.log(N)).float()
    return Posterior(val, idx, R_best, mass, log_z, log_density, mean_R, mean_cos, moment)


class HypothesisVerifier:
    """Holds the verification-head weights (state-dict names
    `feature_aligner.feature_embedding_2d.{0.weight,2.weight,2.bias}`)."""

    def __init__(self, W1: torch.Tensor, W2: torch.Tensor, b2: torch.Tensor, math: int | None = None):
        self.W1 = W1.detach().reshape(32, 384).float().contiguous()
        self.W2 = W2.detach().reshape(32, 32).float().contiguous()
        self.b2 = b2.detach().float().contiguous()
        self.math = DEFAULT_MATH if math is None else math
        self._ws = None

    @classmethod
    def from_feature_aligner(cls, feature_aligner, math: int | None = None) -> "HypothesisVerifier":
        head = feature_aligner.feature_embedding_2d
        return cls(head[0].weight, head[2].weight, head[2].bias, math)

    def to(self, device) -> "HypothesisVerifier":
        self.W1, self.W2, self.b2 = self.W1.to(device), self.W2.to(device), self.b2.to(device)
        return self

    def _weights_on(self, device):
        if self.W1.device != device:
            self.to(device)
        return self.W1, self.W2, self.b2

    def target_features(self, vol_tgt: torch.Tensor) -> torch.Tensor:
        """feature_aligner.forward_3d2d(img_feat_tgt) (modules/model.py:191)."""
        W1, W2, b2 = self._weights_on(vol_tgt.device)
        return ops.forward_3d2d(vol_tgt.float(), W1, W2, b2)

    def _workspace(self, B, N, k, device):
        need = ops.workspace_bytes(B, N, max(k, 1))
        if self._ws is None or self._ws.device != device or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 16), device=device, dtype=torch.uint8)
        return self._ws

    @torch.no_grad()
    def score(self, vol_src, vol_tgt, R, k: int = 1, return_scores: bool = True, tgt_feat=None,
              idx_offset: int = 0, gather: bool = True, min_sep_deg: float = 0.0) -> VerifyResult:
        """vol_src/vol_tgt [B,16,8,8,8]; R [N,3,3] shared or [B,N,3,3] per pair.  min_sep_deg > 0 keeps the k best
        rotations that lie pairwise more than min_sep_deg apart (`ops.topk_distinct`; empty slots are -inf / -1 / NaN)."""
        dev = vol_src.device
        W1, W2, b2 = self._weights_on(dev)
        k, N = _clamp_k(k, R)
        if N == 0:
            raise ValueError("empty hypothesis set")
        vs = _src_volume(vol_src)
        ws = self._workspace(vol_src.shape[0], N, k, dev)
        if min_sep_deg > 0:   # greedy NMS does not compose from per-shard lists: no idx_offset
            if idx_offset:
                raise ValueError("min_sep_deg > 0 selects over the whole set: idx_offset must be 0")
            tf = self.target_features(vol_tgt) if tgt_feat is None else tgt_feat
            scores = ops.score(vs, tf, R, W1, W2, b2, k=0, math=self.math, workspace=ws)[0]
            val, idx, R_best = ops.topk_distinct(scores, R, k, min_sep_deg, gather=gather)
            return VerifyResult(scores if return_scores else None, val, idx, R_best)
        if tgt_feat is None:   # one C call for the whole step (2 launches when k == 1)
            scores, val, idx, R_best = ops.verify(vs, vol_tgt.float(), R, W1, W2, b2, k=k, idx_offset=idx_offset,
                                                  math=self.math, return_scores=return_scores, gather=gather,
                                                  workspace=ws)
            return VerifyResult(scores, val, idx, R_best)
        scores, val, idx = ops.score(vs, tgt_feat, R, W1, W2, b2, k=k, idx_offset=idx_offset, math=self.math,
                                     return_scores=return_scores, workspace=ws)
        R_best = ops.gather_rotations(R, idx, idx_offset) if gather else None
        return VerifyResult(scores, val, idx, R_best)

    @torch.no_grad()
    def posterior(self, vol_src, vol_tgt, R, k: int = 1, min_sep_deg: float = 0.0, radius_deg: float | None = None,
                  temperature: float = 0.1, R_query=None, moments: bool = False) -> Posterior:
        """The selection of `score` (the top-k, or with min_sep_deg > 0 the top-k of distinct rotations) and how much of
        the verifier's softmax p_b(n) = exp(s[b,n]/T) / Z_b over the set it holds.  T = 0.1 is the InfoNCE training
        temperature (modules/model.py:43-63), under which p_b is the model's own estimate of where the rotation lies.
        `mass[b,j]`: the probability of the hypotheses within radius_deg of slot j's rotation and of no earlier slot
        (`ops.posterior_mass`); radius_deg defaults to min_sep_deg, where slot j holds its winner and the hypotheses
        that winner suppressed.  With radius_deg = ACC_THR and k = 1, mass[b,0] is the model's estimate that the
        prediction is correct at ACC_THR; 1 - mass.sum(1) is the probability no slot holds.
        `R_query` [B,Q,3,3] (e.g. the ground truth as Q = 1): `log_density` [B,Q] = s_q/T - log Z_b + log N, the
        log-density of p_b at R_query w.r.t. the normalised Haar measure (SO(3) has volume 1), meaningful when the set
        is Haar-random or near-uniform.  Subtract log(pi^2) for the convention that takes the volume of SO(3) as pi^2.
        `moments=True` also fills `mean_R`, `mean_cos` and `moment` (`ops.posterior_moments`: the p-weighted mean
        rotation of each slot and the mean cosine of the angle to it; `spread_deg` is its arccos in degrees).
        vol_src/vol_tgt [B,16,8,8,8]; R [N,3,3] shared or [B,N,3,3] per pair.  No host synchronisation."""
        radius_deg = _posterior_radius(min_sep_deg, radius_deg)
        dev = vol_src.device
        W1, W2, b2 = self._weights_on(dev)
        k, N = _clamp_k(k, R)
        if N == 0:
            raise ValueError("empty hypothesis set")
        vs = _src_volume(vol_src)
        tf = self.target_features(vol_tgt)
        scores = ops.score(vs, tf, R, W1, W2, b2, k=0, math=self.math, workspace=self._workspace(vol_src.shape[0], N, 1, dev))[0]
        s_query = None
        if R_query is not None:
            s_query = ops.score(vs, tf, R_query, W1, W2, b2, k=0, math=self.math)[0]
        return _posterior(scores, R, k, min_sep_deg, radius_deg, temperature, s_query, moments)

    @torch.no_grad()
    def predict(self, vol_src, vol_tgt, R):
        """argmax hypothesis per pair: (R_best [B,3,3], score [B], index [B])."""
        r = self.score(vol_src, vol_tgt, R, k=1, return_scores=False)
        return r.R_best[:, 0], r.topk_val[:, 0], r.topk_idx[:, 0]

    @torch.no_grad()
    def refine(self, vol_src, vol_tgt, R, k: int = 32, m: int = 64, max_angle_deg: float = 5.0, seed: int = 0):
        """Two-pass selection (BASELINE config 4; extension): score the set, keep the top-k, score m local
        perturbations of each, return the best - one C call (`ahv_refine`), no torch ops in between.
        Returns (R_best [B,3,3], score [B], first pass as a VerifyResult, candidate set [B,k*m,3,3])."""
        W1, W2, b2 = self._weights_on(vol_src.device)
        k, _ = _clamp_k(k, R)
        fv, fi, fR, cand, bv, bi, bR, self._ws_refine = ops.refine(
            _src_volume(vol_src), vol_tgt.float(), R, W1, W2, b2, k=k, m=m, max_angle_deg=max_angle_deg, seed=seed,
            math=self.math, workspace=getattr(self, "_ws_refine", None))
        return bR, bv, VerifyResult(None, fv, fi, fR), cand

    @torch.no_grad()
    def refine_gradient(self, vol_src, vol_tgt, R_init, steps: int = 20, step_deg: float = 1.0):
        """Gradient refinement of given rotations (extension): backtracking Riemannian gradient ascent of the
        AHV_MATH_FP32 score on SO(3), every candidate at once.  R_init [B,3,3] or [B,k,3,3] (e.g. `VerifyResult.R_best`
        of a top-k pass).  Each step takes G = dS/dR from the fused backward's rotation phase (`ops.score_grad_R`),
        the tangent direction w_i = <G, [e_i]x R>, a trial rotation exp(theta [w/|w|]x) R, and keeps it only where it
        scores higher (theta *= 1.2 there, /= 2 elsewhere).  Candidates are scored with the fp32 kernel from start to
        end, so every returned score is >= its starting score.  A fixed number of steps, no host synchronisation:
        CUDA-graph capturable.  Returns (R_best [B,3,3], score [B], R_all [B,k,3,3], score_all [B,k]); the best is
        the per-pair arg-max over k, ties to the lowest index.
        This is the torch-op restatement of the algorithm, kept as the reference for `ascend` (one kernel, faster)."""
        dev = vol_src.device
        W1, W2, b2 = self._weights_on(dev)
        R = (R_init[:, None] if R_init.dim() == 3 else R_init).float().contiguous()
        B, k = R.shape[:2]
        vs = vol_src.float()
        tgt = ops.forward_3d2d(vol_tgt.float(), W1, W2, b2)

        def score(Rc):
            return ops.score(vs, tgt, Rc, W1, W2, b2, k=0, math=MATH_FP32)[0]

        s = score(R)
        theta = torch.full((B, k), math.radians(step_deg), device=dev)
        ones = torch.ones(B, k, device=dev)
        eye = torch.eye(3, device=dev)
        for _ in range(steps):
            G = ops.score_grad_R(vs, tgt, R, W1, W2, b2, ones)
            M = G @ R.transpose(-1, -2)                                    # <G, [e_i]x R> = <G R^T, [e_i]x>
            w = torch.stack((M[..., 2, 1] - M[..., 1, 2], M[..., 0, 2] - M[..., 2, 0], M[..., 1, 0] - M[..., 0, 1]), -1)
            u = w / w.norm(dim=-1, keepdim=True).clamp_min(1e-30)
            K = _hat(u)
            dR = eye + torch.sin(theta)[..., None, None] * K + (1.0 - torch.cos(theta))[..., None, None] * (K @ K)
            Rt = dR @ R
            Rt = 1.5 * Rt - 0.5 * Rt @ Rt.transpose(-1, -2) @ Rt           # one Newton step towards the nearest rotation
            st = score(Rt)
            acc = st > s
            R = torch.where(acc[..., None, None], Rt, R).contiguous()
            s = torch.where(acc, st, s)
            theta = torch.where(acc, theta * 1.2, theta * 0.5)
        best = torch.argmax(s, dim=1)                                      # first maximal index
        rows = torch.arange(B, device=dev)
        return R[rows, best], s[rows, best], R, s

    @torch.no_grad()
    def ascend(self, vol_src, vol_tgt, R_init, steps: int = 20, step_deg: float = 1.0):
        """`refine_gradient`'s ascent as one kernel (`ahv_gradient_ascent`): every step of every candidate runs on-chip,
        one CTA per candidate at a time, and the score is differentiated again only where a trial was accepted.
        R_init [B,3,3] or [B,k,3,3]; fp32 or bf16 source volumes.  Every returned score is the fp32 scorer's score of its
        rotation and >= its starting score.  No host synchronisation: CUDA-graph capturable.  Returns (R_best [B,3,3],
        score [B], R_all [B,k,3,3], score_all [B,k]); the best is the per-pair arg-max over k, ties to the lowest index."""
        W1, W2, b2 = self._weights_on(vol_src.device)
        R = (R_init[:, None] if R_init.dim() == 3 else R_init).float()
        R_all, s_all = ops.gradient_ascent(_src_volume(vol_src), self.target_features(vol_tgt), R, W1, W2, b2, steps=steps,
                                           step_deg=step_deg)
        val, idx = ops.topk(s_all, 1)
        return ops.gather_rotations(R_all, idx)[:, 0], val[:, 0], R_all, s_all

    @torch.no_grad()
    def refine_by_gradient(self, vol_src, vol_tgt, R, k: int = 32, steps: int = 20, step_deg: float = 1.0,
                           min_sep_deg: float = 0.0):
        """Grid pass + gradient ascent in one C call (`ahv_refine_gradient`; BASELINE config 4's accurate path): score
        the set with this verifier's math mode, keep the top-k, run `ascend` from each winner, return the best.
        min_sep_deg > 0 keeps the top-k of rotations pairwise more than min_sep_deg apart instead
        (`ahv_refine_gradient_distinct`), so the ascents start in distinct basins; slots left empty are not ascended.
        Returns (R_best [B,3,3], score [B], first pass as a VerifyResult, R_all [B,k,3,3], score_all [B,k])."""
        W1, W2, b2 = self._weights_on(vol_src.device)
        k, _ = _clamp_k(k, R)
        fv, fi, fR, Ra, sa, bv, bi, bR, self._ws_refine_gradient = ops.refine_gradient(
            _src_volume(vol_src), vol_tgt.float(), R, W1, W2, b2, k=k, steps=steps, step_deg=step_deg, math=self.math,
            workspace=getattr(self, "_ws_refine_gradient", None), min_sep_deg=min_sep_deg)
        return bR, bv, VerifyResult(None, fv, fi, fR), Ra, sa


    @torch.no_grad()
    def search(self, vol_src, vol_tgt, base_level: int = 2, levels: int = 4, k: int = 32, min_sep_deg: float = 0.0,
               beam: int = 4):
        """Coarse-to-fine rotation search on the nested Hopf x HEALPix grid (`so3.hopf_grid`) in one C call
        (`ahv_search_hierarchical`): score all 72 * 8^base_level cells of the base level with this verifier's math mode,
        keep the top-k, then `levels` times score the 8 children of each kept cell and keep the top-k of those.  It
        scores 72 * 8^base_level + levels * 8k hypotheses per pair and ends on cells of level base_level + levels, about
        (pi^2 / (72 * 8^L))^(1/3) rad across (level 6: 0.46 deg).  fp32 or bf16 source volumes; no host synchronisation.
        The defaults come from profiles/r14_hierarchical_search.jsonl (B200): base level 2 (4 608 cells of about 7.4 deg) keeps
        B = 1 at 0.18 ms, against 0.49 ms for verify(k = 1) on the 50 000-point grid, where base level 3 (36 864 cells) costs
        more than that grid; k = 32 reaches the dense grid's top-1 score on 96.5 % of 256 random pairs against 89.5 % for
        k = 8, for 6-15 % more time; four levels end on 0.46-deg cells, below the 50 000-point grid's 3.3 deg.  A coarse base
        level can miss the right basin: on near-symmetric volumes only base_level=3 with k=32 found every pair's mode.
        min_sep_deg > 0 keeps k distinct modes instead (`ops.search_modes`, `ahv_search_modes`): the base level's k winners
        pairwise more than min_sep_deg apart, each descended with a beam of its own `beam` best cells, so a second peak
        that scores a little lower is not dropped at the coarse level.  `first` then holds the distinct base winners and
        `final` the k modes ordered by score.  On near-symmetric volumes (profiles/r18_search_modes.jsonl, B200) the modes
        at (2, 4, k=8, beam=4, 30 deg) held every pair's true basin, but the top-1 was often the mirrored peak: `ascend`
        from every mode and take the best score (0.035 deg at most there).  Empty modes (fewer than k distinct winners) carry score -inf, index -1
        and NaN rotations: filter them (final.topk_idx >= 0) before passing final.R_best to `ascend`.  `beam` applies to
        min_sep_deg > 0 only.
        Returns (R_best [B,3,3], score [B], first: VerifyResult of the base level's top-k, final: VerifyResult of the
        finest level's top-k); the VerifyResults carry grid indices of their level and no scores."""
        if not min_sep_deg >= 0:
            raise ValueError("min_sep_deg must be >= 0")
        W1, W2, b2 = self._weights_on(vol_src.device)
        if min_sep_deg > 0:
            fv, fi, fR, v, i, R, self._ws_search_modes = ops.search_modes(
                _src_volume(vol_src), vol_tgt.float(), W1, W2, b2, base_level=base_level, levels=levels, k=k, beam=beam,
                min_sep_deg=min_sep_deg, math=self.math, workspace=getattr(self, "_ws_search_modes", None))
            return R[:, 0], v[:, 0], VerifyResult(None, fv, fi, fR), VerifyResult(None, v, i, R)
        if beam != 4:
            raise ValueError("beam applies to min_sep_deg > 0 only")
        fv, fi, fR, v, i, R, self._ws_search = ops.search_hierarchical(
            _src_volume(vol_src), vol_tgt.float(), W1, W2, b2, base_level=base_level, levels=levels, k=k, math=self.math,
            workspace=getattr(self, "_ws_search", None))
        return R[:, 0], v[:, 0], VerifyResult(None, fv, fi, fR), VerifyResult(None, v, i, R)


def _replay(graph, *inputs):
    """Copies each given (static buffer, new value) pair's value into its buffer, then replays `graph`."""
    for buf, x in inputs:
        if x is not None:
            buf.copy_(x, non_blocking=True)
    graph.replay()


def _hat(u: torch.Tensor) -> torch.Tensor:
    """[..., 3] -> the cross-product matrices [u]x [..., 3, 3]."""
    z = torch.zeros_like(u[..., 0])
    return torch.stack((z, -u[..., 2], u[..., 1], u[..., 2], z, -u[..., 0], -u[..., 1], u[..., 0], z), -1).reshape(*u.shape[:-1], 3, 3)


class GraphedVerifier:
    """CUDA-graph replay of one verification step for fixed (B, N, k): target
    features + fused scoring + selection + winner gather are captured once and
    replayed with a single launch, which is what bounds the B=1 latency
    (the reference's per-pair loop is batch 1, test_co3d.py:133).  Inputs are
    copied into static buffers; outputs are static tensors valid until the next
    replay."""

    def __init__(self, verifier: HypothesisVerifier, B: int, N: int, k: int = 1, per_pair_R: bool = False,
                 device="cuda", vol_dtype=torch.float32, peer=None, idx_offset: int = 0):
        """`peer` (a `dist.PeerExchange`): N is THIS rank's slice of a hypothesis set sharded over the peer
        group (global index = local + idx_offset) and the captured step is `ahv_verify_sharded` - the scoring
        kernels exchange their winners over NVLink themselves, so the multi-GPU step contains no NCCL call and
        is graph-capturable as it stands.  Every rank must replay in lockstep."""
        self.v = verifier.to(torch.device(device))
        dev = torch.device(device)
        self.vol_src = torch.zeros(B, 16, 8, 8, 8, device=dev, dtype=vol_dtype)
        self.vol_tgt = torch.zeros(B, 16, 8, 8, 8, device=dev)
        self.R = torch.eye(3, device=dev).repeat(*((B, N) if per_pair_R else (N,)), 1, 1).contiguous()
        self.k = min(k, N)
        self.peer = peer

        def run():
            if peer is None:
                return self.v.score(self.vol_src, self.vol_tgt, self.R, k=self.k, return_scores=False, idx_offset=idx_offset)
            W1, W2, b2 = self.v._weights_on(dev)
            val, idx, Rb = ops.verify_sharded(self.vol_src, self.vol_tgt, self.R, W1, W2, b2, idx_offset, peer, k=self.k,
                                              math=self.v.math, workspace=self.v._workspace(B, N, self.k, dev))
            return VerifyResult(None, val, idx, Rb)

        stream = torch.cuda.Stream(device=dev)
        stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(stream):
            for _ in range(2):                      # warm-up outside capture (module load, attributes)
                self.out = run()
        torch.cuda.current_stream(dev).wait_stream(stream)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = run()

    @torch.no_grad()
    def __call__(self, vol_src=None, vol_tgt=None, R=None) -> VerifyResult:
        _replay(self.graph, (self.vol_src, vol_src), (self.vol_tgt, vol_tgt), (self.R, R))
        return self.out

    def check(self) -> int:
        """Sharded replays only: synchronises and raises if an exchange timed out waiting for a peer (that step's
        results are NaN / index -1); returns the number of exchanges this rank has completed."""
        return self.peer.check() if self.peer is not None else 0


class GraphedRefiner:
    """CUDA-graph replay of the two-pass selection (`ahv_refine`: dense set -> top-k -> m local candidates each ->
    arg-max; BASELINE config 4) for fixed (B, N, k, m): the whole chain - target features, both scoring passes, top-k,
    candidate generation, selection - is one C call with no host step or torch op inside, so it captures as it stands.
    method="gradient" captures `ahv_refine_gradient` instead (dense set -> top-k -> `steps` steps of gradient ascent
    from each winner, starting at step_deg -> arg-max; m, max_angle_deg and seed are unused), or with min_sep_deg > 0
    `ahv_refine_gradient_distinct` (the top-k of rotations pairwise more than min_sep_deg apart).
    Outputs are static tensors valid until the next replay."""

    def __init__(self, verifier: HypothesisVerifier, B: int, N: int, k: int = 32, m: int = 64, max_angle_deg: float = 5.0,
                 seed: int = 0, device="cuda", vol_dtype=torch.float32, method: str = "perturb", steps: int = 20,
                 step_deg: float = 1.0, min_sep_deg: float = 0.0):
        if method not in ("perturb", "gradient"):
            raise ValueError('method must be "perturb" or "gradient"')
        if min_sep_deg != 0 and method != "gradient":
            raise ValueError('min_sep_deg applies to method="gradient" only')
        dev = torch.device(device)
        self.v = verifier.to(dev)
        self.vol_src = torch.zeros(B, 16, 8, 8, 8, device=dev, dtype=vol_dtype)
        self.vol_tgt = torch.zeros(B, 16, 8, 8, 8, device=dev)
        self.R = torch.eye(3, device=dev).repeat(N, 1, 1).contiguous()
        k = min(k, N)
        W1, W2, b2 = self.v._weights_on(dev)

        def run(out=None, ws=None):
            if method == "gradient":
                return ops.refine_gradient(self.vol_src, self.vol_tgt, self.R, W1, W2, b2, k=k, steps=steps, step_deg=step_deg,
                                           math=self.v.math, workspace=ws, out=out, min_sep_deg=min_sep_deg)
            return ops.refine(self.vol_src, self.vol_tgt, self.R, W1, W2, b2, k=k, m=m, max_angle_deg=max_angle_deg, seed=seed,
                              math=self.v.math, workspace=ws, out=out)

        stream = torch.cuda.Stream(device=dev)
        stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(stream):
            res = run()
            res = run(res[:-1], res[-1])           # warm-up on the buffers the graph will use
        torch.cuda.current_stream(dev).wait_stream(stream)
        torch.cuda.synchronize(dev)
        self._bufs, self._ws = res[:-1], res[-1]
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            run(self._bufs, self._ws)
        if method == "gradient":
            fv, fi, fR, self.R_all, self.score_all, self.best_val, self.best_idx, self.R_best = self._bufs
        else:
            fv, fi, fR, self.candidates, self.best_val, self.best_idx, self.R_best = self._bufs
        self.first = VerifyResult(None, fv, fi, fR)

    @torch.no_grad()
    def __call__(self, vol_src=None, vol_tgt=None, R=None):
        """Returns (R_best [B,3,3], score [B]); `.first` holds the first pass's top-k, `.candidates` the refinement set
        (method="perturb") or `.R_all` / `.score_all` the ascended top-k (method="gradient")."""
        _replay(self.graph, (self.vol_src, vol_src), (self.vol_tgt, vol_tgt), (self.R, R))
        return self.R_best, self.best_val


class GraphedTail:
    """CUDA-graph replay of everything downstream of the 2D backbone for fixed (B, N, k): `forward_2d3d`
    (1x1 conv + 2D ResNet block, bidirectional transformer, 3D ResNet block - `ahv_resblock3d` - for both views;
    modules/modules.py:86-110) followed by the fused verification step, captured once and replayed with a single
    launch.  This is the per-pair latency path of the reference's evaluation loops (test_co3d.py:133-146) minus
    the backbone.  Inputs are copied into static buffers; outputs are static tensors valid until the next replay."""

    def __init__(self, feature_aligner, B: int, N: int, k: int = 1, device="cuda", math: int | None = None,
                 in_channels: int = 768):
        dev = torch.device(device)
        self.fa = feature_aligner
        self.v = HypothesisVerifier.from_feature_aligner(feature_aligner, math).to(dev)
        self.feat_src = torch.zeros(B, in_channels, 8, 8, device=dev)
        self.feat_tgt = torch.zeros(B, in_channels, 8, 8, device=dev)
        self.R = torch.eye(3, device=dev).repeat(N, 1, 1).contiguous()
        self.k = min(k, N)

        def run():
            with torch.no_grad():
                vs, vt = self.fa.forward_2d3d(self.feat_src, self.feat_tgt, random_mask=False, mask_ratio=0.0)
                return self.v.score(vs, vt, self.R, k=self.k, return_scores=False), vs, vt

        stream = torch.cuda.Stream(device=dev)
        stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(stream):
            for _ in range(3):                      # warm-up outside capture (cuDNN/cuBLAS plans, module load)
                self.out, self.vol_src, self.vol_tgt = run()
        torch.cuda.current_stream(dev).wait_stream(stream)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out, self.vol_src, self.vol_tgt = run()

    @torch.no_grad()
    def __call__(self, feat_src=None, feat_tgt=None, R=None) -> VerifyResult:
        _replay(self.graph, (self.feat_src, feat_src), (self.feat_tgt, feat_tgt), (self.R, R))
        return self.out
