"""GPU: ShardedVerifier.posterior(moments=True) over a hypothesis set sharded across ranks equals
HypothesisVerifier.posterior(moments=True) on one GPU, bit for bit, on every rank.  Two or four "ranks" live in this
process on one GPU, with the harness of test_gpu_sharded_refine.py (one exchange buffer, stream and verifier per rank)."""
import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_sharded_refine import _Ranks, _assert_same, _setup  # noqa: E402

pytestmark = pytest.mark.gpu
FIELDS = ("topk_val", "topk_idx", "R_best", "mass", "log_z", "log_density", "mean_R", "mean_cos", "moment")


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_posterior_moments_equal_one_gpu(ahv, golden, world):
    dev, vs, vt, R, (W1, W2, b2) = _setup(ahv, golden)
    Rp = R.reshape(3, 1000, 3, 3).contiguous()                                   # per-pair sets
    gt = ahv.so3.sample_rotations(3, seed=4, device=dev)[:, None].contiguous()  # [B,1,3,3]
    one = ahv.HypothesisVerifier(W1, W2, b2)
    ranks = _Ranks(ahv, world, dev)
    try:
        svs = []
        for r in range(world):
            sv = ahv.dist.ShardedVerifier(ahv.HypothesisVerifier(W1, W2, b2), peer=ranks.peers[r])
            sv.rank, sv.world = r, world
            svs.append(sv)
        # (set, k, min_sep_deg, radius_deg, R_query); B, k and N change from call to call on the same buffers
        cases = [(R, 1, 0.0, 15.0, gt), (R, 8, 15.0, None, None), (R[:2999], 32, 30.0, 20.0, gt), (Rp, 4, 10.0, None, gt)]
        for Rs, k, sep, radius, Rq in cases:
            want = one.posterior(vs, vt, Rs, k=k, min_sep_deg=sep, radius_deg=radius, R_query=Rq, moments=True)
            got = ranks.run(lambda r, p: svs[r].posterior(vs, vt, Rs, k=k, min_sep_deg=sep, radius_deg=radius, R_query=Rq,
                                                          moments=True), exchanges=1)
            ranks.check_status()
            names = [f for f in FIELDS if getattr(want, f) is not None]
            assert want.mean_R is not None and want.moment is not None
            for r in range(world):
                assert all((getattr(got[r], f) is None) == (getattr(want, f) is None) for f in FIELDS)
                _assert_same([getattr(got[r], f) for f in names], [getattr(want, f) for f in names],
                             (world, tuple(Rs.shape), k, sep, radius, r))
    finally:
        ranks.close()
