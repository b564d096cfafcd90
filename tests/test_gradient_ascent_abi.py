"""CPU: the gradient-ascent entries reject malformed arguments before they touch a device."""
import ctypes
import math


def test_gradient_ascent_rejects_malformed_arguments_without_gpu(ahv):
    lib, E = ahv._lib.lib(), ahv._lib.AHV_EINVAL
    one = ctypes.c_void_p(16)

    # ahv_gradient_ascent(vol, dtype, tgt, R_init, W1, W2, b2, base, steps, step_deg, R_out, score_out, B, K, stream)
    def asc(bufs=(one,) * 9, dtype=0, steps=20, step_deg=1.0, B=2, K=3):
        vs, tg, R, W1, W2, b2, base, Ro, so = bufs
        return lib.ahv_gradient_ascent(vs, dtype, tg, R, W1, W2, b2, base, steps, step_deg, Ro, so, B, K, None)

    assert asc(B=0) == E and asc(B=-1) == E and asc(K=0) == E                                  # shapes
    assert asc(steps=-1) == E and asc(steps=1001) == E                                         # step cap
    for bad in (0.0, -1.0, math.inf, -math.inf, math.nan):                                     # step size
        assert asc(step_deg=bad) == E, bad
    assert asc(dtype=2) == E and asc(dtype=-1) == E                                            # volume dtype
    for hole in range(9):                                                                      # each null buffer
        bufs = [one] * 9
        bufs[hole] = None
        assert asc(bufs=tuple(bufs)) == E, hole
    for pos in (2, 7):                                                                         # misaligned R_init, R_out
        bufs = [one] * 9
        bufs[pos] = ctypes.c_void_p(20)
        assert asc(bufs=tuple(bufs)) == E, pos


def test_refine_gradient_rejects_malformed_arguments_without_gpu(ahv):
    lib, E, EW = ahv._lib.lib(), ahv._lib.AHV_EINVAL, ahv._lib.AHV_EWORKSPACE
    one = ctypes.c_void_p(16)
    B, N, k = 2, 100, 4
    need = lib.ahv_refine_gradient_workspace_bytes(B, N, k)
    assert need >= lib.ahv_workspace_bytes(B, N, k) + B * 32 * 64 * 4
    assert lib.ahv_refine_gradient_workspace_bytes(B, N, 0) == 0 and lib.ahv_refine_gradient_workspace_bytes(B, N, 33) == 0

    # ahv_refine_gradient(vol, dtype, vol_tgt, R, r_per_pair, W1, W2, b2, base, k, steps, step_deg, first_val, first_idx,
    #                     first_R, R_all, score_all, best_val, best_idx, R_best, B, N, math, workspace, ws_bytes, stream)
    def ref(ins=(one,) * 7, outs=(one,) * 8, ws=one, dtype=0, k=k, steps=20, step_deg=1.0, B=B, N=N, math_mode=0, nbytes=need):
        vs, vt, R, W1, W2, b2, base = ins
        return lib.ahv_refine_gradient(vs, dtype, vt, R, 0, W1, W2, b2, base, k, steps, step_deg, *outs, B, N, math_mode, ws,
                                       nbytes, None)

    assert ref(B=0) == E and ref(N=0) == E and ref(N=-1) == E                                  # shapes
    assert ref(k=0) == E and ref(k=33) == E and ref(k=5, N=4) == E                             # k outside [1, min(32, N)]
    assert ref(steps=-1) == E and ref(steps=1001) == E
    for bad in (0.0, -2.0, math.inf, math.nan):
        assert ref(step_deg=bad) == E, bad
    assert ref(dtype=3) == E and ref(math_mode=7) == E
    for hole in range(7):                                                                      # each null input
        ins = [one] * 7
        ins[hole] = None
        assert ref(ins=tuple(ins)) == E, hole
    for hole in range(7):                                                                      # each required output (R_best may be NULL)
        outs = [one] * 8
        outs[hole] = None
        assert ref(outs=tuple(outs)) == E, hole
    assert ref(ws=None) == E
    for pos in (2, 3, 7):                                                                      # misaligned first_R, R_all, R_best
        outs = [one] * 8
        outs[pos] = ctypes.c_void_p(24)
        assert ref(outs=tuple(outs)) == E, pos
    assert ref(nbytes=need - 1) == EW                                                          # workspace too small
