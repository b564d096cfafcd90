"""CPU: the rotation-gradient entries reject malformed arguments before they touch a device."""
import ctypes


def test_rotation_gradient_entries_reject_malformed_arguments_without_gpu(ahv):
    lib, E = ahv._lib.lib(), ahv._lib.AHV_EINVAL
    one = ctypes.c_void_p(16)
    # ahv_rotate_volume_grad_R(vol, per_rotation, R, base, grad_out, grad_R, n, stream)
    assert lib.ahv_rotate_volume_grad_R(one, 0, one, one, one, one, -1, None) == E            # n < 0
    for hole in range(5):                                                                      # each null buffer
        bufs = [one] * 5
        bufs[hole] = None
        v, R, base, go, gR = bufs
        assert lib.ahv_rotate_volume_grad_R(v, 0, R, base, go, gR, 3, None) == E, hole

    # ahv_score_backward_ex(vol, tgt, R, r_per_pair, W1, W2, b2, base, grad_scores, h1_saved, pair_inv,
    #                       grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2, grad_R, B, N, stream)
    def ex(inputs=(one,) * 8, h1=None, pinv=None, outs=(None,) * 5 + (one,), B=2, N=10):
        vs, tg, R, W1, W2, b2, base, gs = inputs
        return lib.ahv_score_backward_ex(vs, tg, R, 0, W1, W2, b2, base, gs, h1, pinv, *outs, B, N, None)

    assert ex(B=-1) == E and ex(N=-1) == E and ex(N=1 << 31) == E                            # shapes
    assert ex(outs=(None,) * 6) == E                                                           # every output NULL
    assert ex(h1=one) == E and ex(pinv=one) == E                                               # only one of the saved pair
    assert ex(h1=ctypes.c_void_p(24), pinv=one) == E                                           # misaligned activations
    for hole in range(8):                                                                      # each null input
        inputs = [one] * 8
        inputs[hole] = None
        assert ex(inputs=tuple(inputs)) == E, hole
