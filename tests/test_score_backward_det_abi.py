"""CPU: the deterministic backward entry (ahv_score_backward_det) rejects malformed arguments before it touches a
device, and its workspace size depends on the shapes alone."""
import ctypes

import pytest

W_SLOT = 32 * 384 + 32 * 32 + 32          # floats of one CTA's weight partials
SEG_SLOT = 16 * 512 + 32 * 64             # floats of one (CTA, pair) segment: dV_b and dT_b
CAP = 160                                 # largest grid of the deterministic backward


def expected_bytes(B, N, r_per_pair, want_grad_R):
    grid = min(B * N, CAP)
    floats = grid * W_SLOT + ((grid + B - 1) * SEG_SLOT if B > 0 and grid > 0 else 0)
    if want_grad_R and not r_per_pair:
        floats += (B * N * 9 + 63) // 64 * 64
    return 4 * floats


def test_det_workspace_bytes(ahv):
    f = ahv._lib.lib().ahv_score_backward_det_workspace_bytes
    for B, N in ((1, 1), (1, 7), (3, 50), (12, 9000), (300, 3), (2, 2**31 - 1), (159, 1), (160, 1), (161, 1)):
        for per_pair in (0, 1):
            for want_R in (0, 1):
                assert f(B, N, per_pair, want_R) == expected_bytes(B, N, per_pair, want_R), (B, N, per_pair, want_R)
    assert f(12, 9000, 1, 0) == 4 * (160 * W_SLOT + 171 * SEG_SLOT) == 15_544_320   # ~15 MB at the training step's size
    assert f(0, 100, 0, 1) == 0 and f(5, 0, 0, 1) == 0                               # nothing to do
    assert f(-1, 10, 0, 0) == 0 and f(2, -1, 0, 0) == 0 and f(2, 2**31, 0, 0) == 0    # invalid
    assert ahv.ops.score_backward_det_workspace_bytes(12, 9000, True, False) == f(12, 9000, 1, 0)


def test_det_rejects_malformed_arguments_without_gpu(ahv):
    lib, E, EW = ahv._lib.lib(), ahv._lib.AHV_EINVAL, ahv._lib.AHV_EWORKSPACE
    TC, FP32 = ahv._lib.MATH_TC, ahv._lib.MATH_FP32
    one = ctypes.c_void_p(16)
    B, N = 2, 100

    # ahv_score_backward_det(vol_src, tgt_feat, R, r_per_pair, W1, W2, b2, base, grad_scores, h1_saved, pair_inv,
    #     grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2, grad_R, B, N, math_mode, workspace, workspace_bytes, stream)
    def det(ins=(one,) * 9, saved=(one, one), outs=(one,) * 5 + (None,), B=B, N=N, mode=TC, ws=one, nbytes=None,
            per_pair=0):
        if nbytes is None:
            nbytes = lib.ahv_score_backward_det_workspace_bytes(B, N, per_pair, int(outs[5] is not None))
        vs, tg, R, W1, W2, b2, base, gs = ins[:3] + ins[4:]
        return lib.ahv_score_backward_det(vs, tg, R, per_pair, W1, W2, b2, base, gs, *saved, *outs, B, N, mode, ws,
                                          nbytes, None)

    # shapes
    assert det(B=-1) == E and det(N=-1) == E and det(N=2**31) == E
    # math mode: AHV_MATH_TC or AHV_MATH_FP32 only
    for bad in (ahv._lib.MATH_TC_F16GATHER, -1, 3, 7):
        assert det(mode=bad) == E, bad
    # every gradient output NULL
    assert det(outs=(None,) * 6, mode=FP32) == E
    # grad_R with AHV_MATH_TC, saved or recomputed
    assert det(outs=(one,) * 6) == E
    assert det(outs=(one,) * 6, saved=(None, None)) == E
    assert det(outs=(None,) * 5 + (one,)) == E
    # AHV_MATH_TC with a NULL output (the tcgen05 form writes all five); AHV_MATH_FP32 accepts it up to the workspace
    for hole in range(5):
        outs = [one] * 5 + [None]
        outs[hole] = None
        assert det(outs=tuple(outs)) == E, hole
        assert det(outs=tuple(outs), mode=FP32, nbytes=0) == EW, hole
    # h1_saved without pair_inv and the reverse
    assert det(saved=(one, None)) == E and det(saved=(None, one)) == E
    # each NULL input (slot 3 of `ins` stands for r_per_pair and is not passed)
    for hole in (0, 1, 2, 4, 5, 6, 7, 8):
        ins = [one] * 9
        ins[hole] = None
        assert det(ins=tuple(ins)) == E, hole
        assert det(ins=tuple(ins), mode=FP32, saved=(None, None)) == E, hole
    # misaligned inputs, saved activations and workspace
    for pos in (0, 1, 2, 4, 5):
        ins = [one] * 9
        ins[pos] = ctypes.c_void_p(20)
        assert det(ins=tuple(ins)) == E, pos
    assert det(saved=(ctypes.c_void_p(24), one)) == E
    assert det(ws=ctypes.c_void_p(36)) == E
    # workspace: NULL, or one byte short, in every form
    for mode, saved, outs, per_pair in ((TC, (one, one), (one,) * 5 + (None,), 0),
                                        (FP32, (one, one), (one,) * 5 + (None,), 1),
                                        (FP32, (None, None), (one,) * 6, 0),
                                        (FP32, (None, None), (one,) * 6, 1),
                                        (FP32, (None, None), (None,) * 5 + (one,), 0)):
        need = lib.ahv_score_backward_det_workspace_bytes(B, N, per_pair, int(outs[5] is not None))
        assert need > 0
        assert det(mode=mode, saved=saved, outs=outs, per_pair=per_pair, ws=None) == EW
        assert det(mode=mode, saved=saved, outs=outs, per_pair=per_pair, nbytes=need - 1) == EW
    # a shared R's gradient needs its per-item slots: the size without them is short
    short = lib.ahv_score_backward_det_workspace_bytes(B, N, 0, 0)
    assert det(mode=FP32, saved=(None, None), outs=(one,) * 6, nbytes=short) == EW


@pytest.mark.parametrize("B,N", [(0, 5), (3, 0)])
def test_det_empty_call_needs_no_workspace_without_gpu(ahv, B, N):
    """An empty call checks its arguments and returns without device work or workspace (as the other entries do; on
    a machine without a device the device check answers)."""
    lib = ahv._lib.lib()
    one = ctypes.c_void_p(16)
    st = lib.ahv_score_backward_det(None, None, None, 0, None, None, None, None, None, None, None, one, one, one, one, one,
                                    None, B, N, ahv._lib.MATH_FP32, None, 0, None)
    assert st in (ahv._lib.AHV_OK, ahv._lib.AHV_ECUDA, ahv._lib.AHV_ENOTSUP)
