"""CPU: the distinct-rotation entries (ahv_topk_distinct, ahv_refine_gradient_distinct) reject malformed arguments
before they touch a device."""
import ctypes
import math


def test_topk_distinct_rejects_malformed_arguments_without_gpu(ahv):
    lib, E = ahv._lib.lib(), ahv._lib.AHV_EINVAL
    one = ctypes.c_void_p(16)

    # ahv_topk_distinct(scores, R, r_per_pair, B, N, k, min_sep_deg, topk_val, topk_idx, R_best, stream)
    def td(bufs=(one,) * 5, B=2, N=100, k=4, sep=10.0):
        sc, R, v, i, Rb = bufs
        return lib.ahv_topk_distinct(sc, R, 0, B, N, k, sep, v, i, Rb, None)

    assert td(B=-1) == E and td(N=-1) == E and td(N=2**31) == E                        # shapes
    assert td(k=0) == E and td(k=33) == E and td(k=-1) == E                            # k outside [1, 32]
    for bad in (-1e-3, 180.5, -math.inf, math.inf, math.nan):                          # min_sep_deg outside [0, 180]
        assert td(sep=bad) == E, bad
    for hole in range(4):                                                              # each required buffer (R_best may be NULL)
        bufs = [one] * 5
        bufs[hole] = None
        assert td(bufs=tuple(bufs)) == E, hole
    for pos in (1, 4):                                                                 # misaligned R, R_best
        bufs = [one] * 5
        bufs[pos] = ctypes.c_void_p(20)
        assert td(bufs=tuple(bufs)) == E, pos


def test_refine_gradient_distinct_rejects_malformed_arguments_without_gpu(ahv):
    lib, E, EW = ahv._lib.lib(), ahv._lib.AHV_EINVAL, ahv._lib.AHV_EWORKSPACE
    one = ctypes.c_void_p(16)
    B, N, k = 2, 100, 4
    need = lib.ahv_refine_gradient_workspace_bytes(B, N, k)

    # ahv_refine_gradient_distinct(vol, dtype, vol_tgt, R, r_per_pair, W1, W2, b2, base, k, steps, step_deg, min_sep_deg,
    #     first_val, first_idx, first_R, R_all, score_all, best_val, best_idx, R_best, B, N, math, workspace, ws_bytes, stream)
    def ref(ins=(one,) * 7, outs=(one,) * 8, ws=one, dtype=0, k=k, steps=20, step_deg=1.0, sep=15.0, B=B, N=N, math_mode=0,
            nbytes=need):
        vs, vt, R, W1, W2, b2, base = ins
        return lib.ahv_refine_gradient_distinct(vs, dtype, vt, R, 0, W1, W2, b2, base, k, steps, step_deg, sep, *outs, B, N,
                                                math_mode, ws, nbytes, None)

    assert ref(B=0) == E and ref(N=0) == E and ref(N=-1) == E and ref(N=2**31) == E   # shapes
    assert ref(k=0) == E and ref(k=33) == E and ref(k=5, N=4) == E                    # k outside [1, min(32, N)]
    assert ref(steps=-1) == E and ref(steps=1001) == E
    for bad in (0.0, -2.0, math.inf, math.nan):
        assert ref(step_deg=bad) == E, bad
    for bad in (-1e-3, 180.5, -math.inf, math.inf, math.nan):                         # min_sep_deg outside [0, 180]
        assert ref(sep=bad) == E, bad
    assert ref(dtype=3) == E and ref(math_mode=7) == E
    for hole in range(7):                                                              # each null input
        ins = [one] * 7
        ins[hole] = None
        assert ref(ins=tuple(ins)) == E, hole
    for hole in range(7):                                                              # each required output (R_best may be NULL)
        outs = [one] * 8
        outs[hole] = None
        assert ref(outs=tuple(outs)) == E, hole
    assert ref(ws=None) == E
    for pos in (2, 3, 7):                                                              # misaligned first_R, R_all, R_best
        outs = [one] * 8
        outs[pos] = ctypes.c_void_p(24)
        assert ref(outs=tuple(outs)) == E, pos
    assert ref(nbytes=need - 1) == EW                                                  # workspace too small
    assert ref(nbytes=need - 1, sep=0.0) == EW
