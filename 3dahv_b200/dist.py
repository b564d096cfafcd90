"""Hypothesis sharding across the GPUs of one node.

Every (pair, hypothesis) score is independent, so rank r of P scores the slice
[r*ceil(N/P), min(N,(r+1)*ceil(N/P))) of the rotation set for ALL pairs; the
only exchange is one small all-gather of the per-rank top-k lists
(B*k*12 bytes per rank) followed by a deterministic local merge, after which
every rank holds bit-identical results.  The reference has no multi-GPU
inference (it runs batch 1 on one GPU, test_co3d.py:133).
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import ops


def shard_bounds(N: int, rank: int, world: int) -> tuple[int, int]:
    per = -(-N // world)
    lo = min(N, rank * per)
    return lo, min(N, lo + per)


def all_gather_topk(val: torch.Tensor, idx: torch.Tensor, group=None):
    """[B,k] per rank -> [P,B,k] on every rank (one all-gather each for the
    fp32 values and the int64 indices)."""
    world = dist.get_world_size(group)
    val, idx = val.contiguous(), idx.contiguous()
    vals = [torch.empty_like(val) for _ in range(world)]
    idxs = [torch.empty_like(idx) for _ in range(world)]
    dist.all_gather(vals, val, group=group)
    dist.all_gather(idxs, idx, group=group)
    vals, idxs = torch.stack(vals), torch.stack(idxs)
    return vals, idxs


def pad_topk(val: torch.Tensor, idx: torch.Tensor, k: int):
    """Ranks whose slice is shorter than k pad with (-inf, -1), which the merge ignores."""
    B, have = val.shape
    if have == k:
        return val, idx
    pv = torch.full((B, k - have), float("-inf"), dtype=val.dtype, device=val.device)
    pi = torch.full((B, k - have), -1, dtype=idx.dtype, device=idx.device)
    return torch.cat([val, pv], 1), torch.cat([idx, pi], 1)


class PeerExchange:
    """Exchange buffers for the fused sharded step (`ahv_verify_sharded`): every rank allocates one buffer
    (`ahv_peer_alloc`), sends its CUDA IPC handle to the peers (one all-gather of 64 bytes at set-up) and maps
    theirs, after which the scoring kernels talk to each other through NVLink peer memory and a verification
    step involves no NCCL call at all.  One instance per process group; it serves any call with B <= max_pairs and
    k <= max_k (the entry stride depends on the capacity only, so B and k may change from step to step).
    max_hyps > 0 adds a score region (`ahv_peer_alloc_ex`, 2 * max_pairs * max_hyps * 4 bytes) through which
    `ShardedVerifier.scores` and the distinct selection all-gather [B,N] score matrices with N <= max_hyps."""

    def __init__(self, max_pairs: int, device, group=None, max_k: int = 1, max_hyps: int = 0):
        import ctypes

        from . import _lib

        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        if self.world > 8:
            raise ValueError("the peer exchange covers the GPUs of one node (<= 8)")
        if not (1 <= max_k <= 32) or max_pairs < 1:
            raise ValueError("max_pairs >= 1 and 1 <= max_k <= 32 expected")
        if not 0 <= max_hyps < 2**31:
            raise ValueError("0 <= max_hyps < 2**31 expected")
        self.max_pairs, self.max_k, self.max_hyps = max_pairs, max_k, max_hyps
        self.device = torch.device(device)
        lib = _lib.lib()
        self._lib = lib
        self.own, self.ptrs, self._opened = None, [], []
        # Every step below that can fail is local; the ranks agree on the outcome with one all-reduce at the
        # end, so a rank that cannot export or map a buffer makes ALL ranks raise instead of leaving the
        # others blocked in a collective.
        ok = True
        own = ctypes.c_void_p()
        handle = ctypes.create_string_buffer(64)
        with torch.cuda.device(self.device):
            if lib.ahv_peer_alloc_ex(max_pairs, max_k, max_hyps, ctypes.byref(own)) != 0:
                ok = False
            elif lib.ahv_peer_export(own, handle) != 0:
                ok = False
            self.own = own.value
            mine = torch.frombuffer(bytearray(handle.raw), dtype=torch.uint8).to(self.device)
            every = [torch.empty_like(mine) for _ in range(self.world)]
            dist.all_gather(every, mine, group=group)
            flag = torch.tensor([1 if ok else 0], device=self.device, dtype=torch.int32)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
            if int(flag) == 1:
                for r, h in enumerate(every):
                    if r == self.rank:
                        self.ptrs.append(self.own)
                        continue
                    p = ctypes.c_void_p()
                    if lib.ahv_peer_open(bytes(h.cpu().numpy().tobytes()), ctypes.byref(p)) != 0:
                        ok = False
                        break
                    self.ptrs.append(p.value)
                    self._opened.append(p.value)
            else:
                ok = False
            flag = torch.tensor([1 if ok else 0], device=self.device, dtype=torch.int32)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if int(flag) != 1:
            self.close()
            raise RuntimeError("peer exchange unavailable: a rank could not allocate, export or map a CUDA IPC buffer "
                               "(use the NCCL path: ShardedVerifier without `peer`)")

    def check(self) -> int:
        """Synchronises the device and raises if an exchange on this rank timed out waiting for a peer (that
        step returned NaN scores and index -1).  Returns the number of exchanges completed."""
        import ctypes

        from . import _lib

        seq, err = ctypes.c_uint32(), ctypes.c_uint32()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.ahv_peer_status(self.own, ctypes.byref(seq), ctypes.byref(err)), "ahv_peer_status")
        if err.value != 0:
            raise RuntimeError("a sharded verification step timed out waiting for a peer rank")
        return int(seq.value)

    def close(self):
        """Collective: every rank unmaps the peers' buffers before anyone frees its own."""
        if getattr(self, "own", None) is None and not getattr(self, "_opened", None):
            return
        torch.cuda.synchronize(self.device)
        with torch.cuda.device(self.device):
            for p in self._opened:
                self._lib.ahv_peer_close(p)
            if dist.is_initialized():
                dist.barrier(group=self.group)
            if self.own:
                self._lib.ahv_peer_free(self.own)
        self.own, self.ptrs, self._opened = None, [], []


class ShardedVerifier:
    """Wraps a HypothesisVerifier; `score` takes the FULL rotation set on every
    rank (36 B per hypothesis, replicated like the 40 KB/pair volumes) and
    scores only this rank's slice."""

    def __init__(self, verifier, group=None, merge=None, score_fn=None, peer: "PeerExchange | None" = None,
                 check_every: int = 0):
        self.verifier = verifier
        self.group = group
        self.peer = peer   # NVLink peer exchange by the kernels themselves (None: NCCL all-gather + merge kernel)
        self.check_every = check_every   # synchronising error check (a peer that never arrived) every so many steps
        self._steps = 0
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self._merge = merge or ops.topk_merge
        # score_fn(vol_src, vol_tgt, R_slice, k, idx_offset) -> (val [B,k'], idx [B,k'])
        self._score_fn = score_fn or self._score_local

    def _score_local(self, vol_src, vol_tgt, R_slice, k, idx_offset):
        r = self.verifier.score(vol_src, vol_tgt, R_slice, k=k, return_scores=False, idx_offset=idx_offset, gather=False)
        return r.topk_val, r.topk_idx

    def _stepped(self):
        """Counts a peer-exchanging call; every `check_every` of them, raises if one timed out."""
        self._steps += 1
        if self.check_every and self._steps % self.check_every == 0:
            self.peer.check()

    @torch.no_grad()
    def score(self, vol_src, vol_tgt, R, k: int = 1, min_sep_deg: float = 0.0):
        """Returns (topk_val [B,k], topk_idx [B,k] global, R_best [B,k,3,3]).  min_sep_deg > 0: the k best rotations
        pairwise more than min_sep_deg apart, as `HypothesisVerifier.score(min_sep_deg=...)` gives them on one GPU.
        Greedy suppression does not compose from per-shard lists, so the whole [B,N] matrix is assembled on every rank
        (`scores`) and `ops.topk_distinct` runs on every rank over the whole set."""
        per_pair = R.dim() == 4
        N = R.shape[1] if per_pair else R.shape[0]
        k = min(k, N)
        if min_sep_deg > 0:
            return ops.topk_distinct(self.scores(vol_src, vol_tgt, R), R, k, min_sep_deg)
        lo, hi = shard_bounds(N, self.rank, self.world)
        B = vol_src.shape[0]
        if (self.peer is not None and self.world > 1 and B <= self.peer.max_pairs and k <= self.peer.max_k
                and self._score_fn == self._score_local):
            # one C call: shard scoring + NVLink exchange + merge (k == 1: all inside the scoring kernel); empty
            # slices take part in the exchange with empty lists
            v = self.verifier
            W1, W2, b2 = v._weights_on(vol_src.device)
            Rs = (R[:, lo:hi] if per_pair else R[lo:hi]).contiguous()
            vs = vol_src if vol_src.dtype == torch.bfloat16 else vol_src.float()
            val, idx, Rb = ops.verify_sharded(vs, vol_tgt.float(), Rs, W1, W2, b2, lo, self.peer, k=k, math=v.math,
                                              workspace=v._workspace(B, hi - lo, k, vol_src.device))
            self._stepped()
            return val, idx, Rb
        if hi > lo:
            Rs = (R[:, lo:hi] if per_pair else R[lo:hi]).contiguous()
            val, idx = self._score_fn(vol_src, vol_tgt, Rs, min(k, hi - lo), lo)
        else:
            val = torch.empty(B, 0, dtype=torch.float32, device=vol_src.device)
            idx = torch.empty(B, 0, dtype=torch.int64, device=vol_src.device)
        val, idx = pad_topk(val, idx, k)
        if self.world > 1:
            vals, idxs = all_gather_topk(val, idx, self.group)
            val, idx = self._merge(vals, idxs)
        safe = idx.clamp_min(0)
        if per_pair:
            R_best = torch.gather(R, 1, safe[..., None, None].expand(-1, -1, 3, 3))
        else:
            R_best = R[safe]
        return val, idx, R_best

    @torch.no_grad()
    def refine(self, vol_src, vol_tgt, R, k: int = 32, m: int = 64, max_angle_deg: float = 5.0, seed: int = 0):
        """Two-pass selection (BASELINE config 4) with BOTH passes sharded: pass 1 scores this rank's slice of the
        dense set and the ranks exchange their top-k (identical on every rank afterwards, rotations included);
        every rank then builds the same k*m candidates per pair (`ahv_so3_perturb`) and pass 2 shards THOSE over the
        ranks, winners exchanged inside the scoring kernel.  With a `peer` exchange the whole thing contains no NCCL
        call.  Returns (R_best [B,3,3], score [B], (first_val, first_idx, first_R), candidates [B,k*m,3,3]) - equal
        to `HypothesisVerifier.refine` on one GPU."""
        from . import so3

        per_pair = R.dim() == 4
        k = min(k, R.shape[1] if per_pair else R.shape[0])
        first_val, first_idx, first_R = self.score(vol_src, vol_tgt, R, k=k)
        B = vol_src.shape[0]
        cand = so3.perturb_rotations(first_R.contiguous(), m, max_angle_deg, seed).reshape(B, k * m, 3, 3).contiguous()
        val, _, R_best = self.score(vol_src, vol_tgt, cand, k=1)
        return R_best[:, 0], val[:, 0], (first_val, first_idx, first_R), cand

    @torch.no_grad()
    def refine_by_gradient(self, vol_src, vol_tgt, R, k: int = 32, steps: int = 20, step_deg: float = 1.0,
                           min_sep_deg: float = 0.0):
        """`HypothesisVerifier.refine_by_gradient` over a sharded set (BASELINE config 4's accurate path on several
        GPUs): every rank passes the WHOLE set and gets the one-GPU result bit for bit.  The grid pass is sharded;
        with min_sep_deg > 0 the distinct selection runs on every rank over the assembled score matrix; each rank
        ascends its share of the B*k (pair, slot) items and the ascended slots are gathered.  With a `peer` exchange
        (max_hyps >= N for min_sep_deg > 0) the whole chain is one C call with no NCCL call
        (`ops.refine_gradient_sharded`); without, it is composed of NCCL all-gathers and the one-GPU ops.
        Returns (R_best [B,3,3], score [B], first pass as a VerifyResult, R_all [B,k,3,3], score_all [B,k])."""
        from .verify import VerifyResult, _src_volume

        v = self.verifier
        per_pair = R.dim() == 4
        N = R.shape[1] if per_pair else R.shape[0]
        k = min(k, N)
        B = vol_src.shape[0]
        if self.world == 1:
            return v.refine_by_gradient(vol_src, vol_tgt, R, k=k, steps=steps, step_deg=step_deg, min_sep_deg=min_sep_deg)
        dev = vol_src.device
        W1, W2, b2 = v._weights_on(dev)
        p = self.peer
        if (p is not None and B <= p.max_pairs and k <= p.max_k and (min_sep_deg == 0 or N <= p.max_hyps)):
            fv, fi, fR, Ra, sa, bv, bi, bR, self._ws_refine_gradient = ops.refine_gradient_sharded(
                _src_volume(vol_src), vol_tgt.float(), R, W1, W2, b2, p, k=k, steps=steps, step_deg=step_deg, math=v.math,
                workspace=getattr(self, "_ws_refine_gradient", None), min_sep_deg=min_sep_deg)
            self._stepped()
            return bR, bv, VerifyResult(None, fv, fi, fR), Ra, sa
        # NCCL composition: first pass over the whole set, this rank's share of the ascents, all-gather of the slots
        fv, fi, fR = self.score(vol_src, vol_tgt, R, k=k, min_sep_deg=min_sep_deg)
        total = B * k
        ilo, ihi = shard_bounds(total, self.rank, self.world)
        per = -(-total // self.world)
        R_part = torch.zeros(per, 9, device=dev, dtype=torch.float32)
        s_part = torch.zeros(per, device=dev, dtype=torch.float32)
        if ihi > ilo:
            pair = torch.arange(ilo, ihi, device=dev) // k
            tgt = v.target_features(vol_tgt)[pair]
            Ri, si = ops.gradient_ascent(_src_volume(vol_src)[pair], tgt, fR.reshape(total, 1, 3, 3)[ilo:ihi], W1, W2, b2,
                                         steps=steps, step_deg=step_deg)
            empty = fi.reshape(total)[ilo:ihi] < 0        # empty distinct slots are not ascended
            R_part[:ihi - ilo] = torch.where(empty[:, None], torch.full_like(Ri.reshape(-1, 9), float("nan")), Ri.reshape(-1, 9))
            s_part[:ihi - ilo] = torch.where(empty, torch.full_like(si.reshape(-1), float("-inf")), si.reshape(-1))
        Rs = [torch.empty_like(R_part) for _ in range(self.world)]
        ss = [torch.empty_like(s_part) for _ in range(self.world)]
        dist.all_gather(Rs, R_part, group=self.group)
        dist.all_gather(ss, s_part, group=self.group)
        R_all = torch.cat(Rs)[:total].reshape(B, k, 3, 3).contiguous()
        s_all = torch.cat(ss)[:total].reshape(B, k).contiguous()
        val, idx = ops.topk(s_all, 1)
        return ops.gather_rotations(R_all, idx)[:, 0], val[:, 0], VerifyResult(None, fv, fi, fR), R_all, s_all

    @torch.no_grad()
    def posterior(self, vol_src, vol_tgt, R, k: int = 1, min_sep_deg: float = 0.0, radius_deg: float | None = None,
                  temperature: float = 0.1, R_query=None, moments: bool = False):
        """`HypothesisVerifier.posterior` over a sharded set: every rank passes the WHOLE set and gets the one-GPU
        result bit for bit.  The slices' scores are assembled into the whole [B,N] on every rank (`scores`, as for the
        distinct selection), and the selection and `ops.posterior_mass` (`ops.posterior_moments` with moments) run
        replicated on every rank; R_query's few rotations are scored on every rank."""
        from .verify import _posterior, _posterior_radius, _src_volume

        radius_deg = _posterior_radius(min_sep_deg, radius_deg)
        N = R.shape[1] if R.dim() == 4 else R.shape[0]
        scores = self.scores(vol_src, vol_tgt, R)
        s_query = None
        if R_query is not None:
            v = self.verifier
            W1, W2, b2 = v._weights_on(vol_src.device)
            s_query = ops.score(_src_volume(vol_src), v.target_features(vol_tgt), R_query, W1, W2, b2, k=0, math=v.math)[0]
        return _posterior(scores, R, min(k, N), min_sep_deg, radius_deg, temperature, s_query, moments)

    @torch.no_grad()
    def scores(self, vol_src, vol_tgt, R):
        """The full pred_sim [B,N] (modules/model.py:193) of a sharded set on every rank: each rank scores its slice,
        and the slices are all-gathered - through the score region of `peer` (NVLink, no NCCL call) when it has
        max_hyps >= N and max_pairs >= B, else with one NCCL all-gather of B*N/P floats per rank (SURVEY.md §8e;
        25.6 MB per rank at B=128, N=50 000, P=8).  Only needed when the caller wants every score, or for the
        distinct selection; the plain top-k never moves them."""
        per_pair = R.dim() == 4
        N = R.shape[1] if per_pair else R.shape[0]
        B = vol_src.shape[0]
        per = -(-N // self.world)
        lo, hi = shard_bounds(N, self.rank, self.world)
        p = self.peer
        via_peer = p is not None and self.world > 1 and N <= getattr(p, "max_hyps", 0) and B <= p.max_pairs
        part = torch.zeros(B, hi - lo if via_peer else per, device=vol_src.device, dtype=torch.float32)
        if hi > lo:
            Rs = (R[:, lo:hi] if per_pair else R[lo:hi]).contiguous()
            part[:, :hi - lo] = self.verifier.score(vol_src, vol_tgt, Rs, k=1, return_scores=True).scores
        if via_peer:
            out = ops.scores_exchange(part, N, p)
            self._stepped()
            return out
        if self.world == 1:
            return part[:, :N]
        pieces = [torch.empty_like(part) for _ in range(self.world)]
        dist.all_gather(pieces, part, group=self.group)
        return torch.cat(pieces, dim=1)[:, :N]
