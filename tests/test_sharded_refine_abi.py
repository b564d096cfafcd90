"""CPU: the sharded gradient-refinement entries (ahv_refine_gradient_sharded, ahv_scores_exchange) and the score
region of the exchange buffer reject malformed arguments before they touch a device, and a buffer without a score
region keeps ahv_peer_bytes' size."""
import ctypes
import math


def _peers(n, base=4096):
    return (ctypes.c_void_p * n)(*[base * (r + 1) for r in range(n)])


def test_peer_bytes_ex_without_scores_is_peer_bytes(ahv):
    lib = ahv._lib.lib()
    for p, k in ((1, 1), (8, 8), (128, 32), (3, 5)):
        assert lib.ahv_peer_bytes_ex(p, k, 0) == lib.ahv_peer_bytes(p, k) > 0
        # the region: two parities of [max_pairs, max_hyps] fp32 after the entries
        assert lib.ahv_peer_bytes_ex(p, k, 50000) == lib.ahv_peer_bytes(p, k) + 2 * p * 50000 * 4
    assert lib.ahv_peer_bytes_ex(0, 1, 10) == 0 and lib.ahv_peer_bytes_ex(1, 33, 10) == 0
    assert lib.ahv_peer_bytes_ex(1, 1, -1) == 0 and lib.ahv_peer_bytes_ex(1, 1, 2**31) == 0
    E = ahv._lib.AHV_EINVAL
    p = ctypes.c_void_p()
    assert lib.ahv_peer_alloc_ex(0, 1, 10, ctypes.byref(p)) == E and lib.ahv_peer_alloc_ex(1, 1, -1, ctypes.byref(p)) == E
    assert lib.ahv_peer_alloc_ex(1, 1, 10, None) == E
    i, j, h = ctypes.c_int(), ctypes.c_int(), ctypes.c_int64()
    assert lib.ahv_peer_capacity_ex(None, ctypes.byref(i), ctypes.byref(j), ctypes.byref(h)) == E


def test_refine_gradient_sharded_rejects_malformed_arguments_without_gpu(ahv):
    lib, E, EW = ahv._lib.lib(), ahv._lib.AHV_EINVAL, ahv._lib.AHV_EWORKSPACE
    one = ctypes.c_void_p(16)
    B, N, k, world = 2, 100, 4, 2
    need = lib.ahv_refine_gradient_sharded_workspace_bytes(B, N, k, world)
    assert need > 0
    assert lib.ahv_refine_gradient_sharded_workspace_bytes(B, N, k, 1) == lib.ahv_refine_gradient_workspace_bytes(B, N, k)
    assert lib.ahv_refine_gradient_sharded_workspace_bytes(B, N, k, 0) == 0
    assert lib.ahv_refine_gradient_sharded_workspace_bytes(B, N, k, 9) == 0

    # ahv_refine_gradient_sharded(vol, dtype, vol_tgt, R, r_per_pair, W1, W2, b2, base, k, steps, step_deg, min_sep_deg,
    #     first_val, first_idx, first_R, R_all, score_all, best_val, best_idx, R_best, B, N, math, workspace, ws_bytes,
    #     rank, world, peers, peer_max_pairs, peer_max_k, peer_max_hyps, stream)
    def ref(ins=(one,) * 7, outs=(one,) * 8, ws=one, dtype=0, k=k, steps=20, step_deg=1.0, sep=15.0, B=B, N=N, math_mode=0,
            nbytes=need, rank=0, world=world, peers="ok", mp=8, mk=8, mh=1000):
        vs, vt, R, W1, W2, b2, base = ins
        pp = _peers(world if world > 0 else 1) if peers == "ok" else peers
        return lib.ahv_refine_gradient_sharded(vs, dtype, vt, R, 0, W1, W2, b2, base, k, steps, step_deg, sep, *outs, B, N,
                                               math_mode, ws, nbytes, rank, world, pp, mp, mk, mh, None)

    assert ref(B=0) == E and ref(N=0) == E and ref(N=-1) == E and ref(N=2**31) == E       # shapes
    assert ref(k=0) == E and ref(k=33) == E and ref(k=5, N=4) == E                        # k outside [1, min(32, N)]
    assert ref(steps=-1) == E and ref(steps=1001) == E
    for bad in (0.0, -2.0, math.inf, math.nan):
        assert ref(step_deg=bad) == E, bad
    for bad in (-1e-3, 180.5, -math.inf, math.inf, math.nan):                             # min_sep_deg outside [0, 180]
        assert ref(sep=bad) == E, bad
    assert ref(dtype=3) == E and ref(math_mode=7) == E
    for hole in range(7):                                                                  # each null input
        ins = [one] * 7
        ins[hole] = None
        assert ref(ins=tuple(ins)) == E, hole
    for hole in range(7):                                                                  # each required output
        outs = [one] * 8
        outs[hole] = None
        assert ref(outs=tuple(outs)) == E, hole
    assert ref(ws=None) == E
    assert ref(ins=(one, one, ctypes.c_void_p(20), one, one, one, one)) == E              # misaligned R
    for pos in (2, 3, 7):                                                                  # misaligned first_R, R_all, R_best
        outs = [one] * 8
        outs[pos] = ctypes.c_void_p(24)
        assert ref(outs=tuple(outs)) == E, pos
    for rank, world in ((-1, 2), (2, 2), (0, 0), (0, 9), (3, 2)):                          # rank / world
        assert ref(rank=rank, world=world) == E, (rank, world)
    assert ref(peers=None) == E                                                            # NULL peer array
    holes = _peers(world)
    holes[1] = None
    assert ref(peers=holes) == E                                                           # a NULL peer buffer
    assert ref(mp=B - 1) == E and ref(mk=k - 1) == E and ref(mk=0) == E                   # exchange capacity
    assert ref(mh=N - 1) == E and ref(mh=-1) == E                                         # score region, distinct path
    for sep in (0.0, 15.0):
        assert ref(nbytes=need - 1, sep=sep) == EW, sep                                    # workspace too small
    assert ref(mh=0, sep=0.0, nbytes=need - 1) == EW     # the top-k path does not need a score region
    assert ref(world=1, peers=None, mp=0, mk=0, mh=0, nbytes=lib.ahv_refine_gradient_workspace_bytes(B, N, k) - 1) == EW


def test_scores_exchange_rejects_malformed_arguments_without_gpu(ahv):
    lib, E = ahv._lib.lib(), ahv._lib.AHV_EINVAL
    one = ctypes.c_void_p(16)

    # ahv_scores_exchange(part, B, N, scores, rank, world, peers, peer_max_pairs, peer_max_k, peer_max_hyps, stream)
    def ex(part=one, B=2, N=100, out=one, rank=0, world=2, peers="ok", mp=4, mk=1, mh=100):
        pp = _peers(max(world, 1)) if peers == "ok" else peers
        return lib.ahv_scores_exchange(part, B, N, out, rank, world, pp, mp, mk, mh, None)

    assert ex(B=0) == E and ex(N=0) == E and ex(N=2**31) == E and ex(out=None) == E
    assert ex(part=None) == E                                      # rank 0 owns columns [0, 50)
    for rank, world in ((-1, 2), (2, 2), (0, 1), (0, 9)):
        assert ex(rank=rank, world=world) == E, (rank, world)
    assert ex(peers=None) == E and ex(mp=1) == E and ex(mh=99) == E and ex(mh=0) == E and ex(mk=0) == E
