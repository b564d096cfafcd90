"""CPU: ahv_search_modes rejects malformed arguments before it touches a device, and its workspace size function."""
import ctypes
import math


def test_search_modes_rejects_malformed_arguments_without_gpu(ahv):
    lib, E, EW = ahv._lib.lib(), ahv._lib.AHV_EINVAL, ahv._lib.AHV_EWORKSPACE
    one = ctypes.c_void_p(256)
    B, base, levels, k, w = 3, 2, 4, 8, 4
    need = lib.ahv_search_modes_workspace_bytes(B, base, k, w)
    assert need > 0

    # (vol_src, vol_dtype, vol_tgt, W1, W2, b2, base, base_level, levels, k, beam, min_sep_deg, first_val, first_idx, first_R,
    #  val, idx, R_out, B, math_mode, workspace, workspace_bytes, stream); bufs = the 13 pointers in that order
    def s(bufs=(one,) * 13, dt=0, base_level=base, levels=levels, k=k, beam=w, sep=30.0, B=B, math=0, nbytes=need):
        vs, vt, w1, w2, b2, bc, fv, fi, fR, v, i, R, ws = bufs
        return lib.ahv_search_modes(vs, dt, vt, w1, w2, b2, bc, base_level, levels, k, beam, sep, fv, fi, fR, v, i, R, B, math,
                                    ws, nbytes, None)

    assert s(B=0) == E and s(B=-1) == E
    assert s(k=0) == E and s(k=33) == E and s(k=-1) == E
    assert s(beam=0) == E and s(beam=9) == E and s(beam=-1) == E
    for sep in (0.0, -1.0, 180.5, 1e9, math.nan, math.inf, -math.inf):                # a finite 0 < min_sep_deg <= 180
        assert s(sep=sep) == E, sep
    assert s(dt=2) == E and s(dt=-1) == E and s(math=3) == E and s(math=-1) == E
    assert s(base_level=-1) == E and s(base_level=7) == E
    assert s(levels=-1) == E and s(levels=15) == E                                  # base_level + levels <= 16
    for hole in range(13):                                                          # every buffer is required
        bufs = [one] * 13
        bufs[hole] = None
        assert s(bufs=tuple(bufs)) == E, hole
    for pos in (0, 1, 2, 3, 8, 11, 12):                                             # misaligned vol_src, vol_tgt, W1, W2,
        bufs = [one] * 13                                                           # first_R, R_out, workspace
        bufs[pos] = ctypes.c_void_p(260)
        assert s(bufs=tuple(bufs)) == E, pos
    assert s(nbytes=need - 1) == EW and s(nbytes=0) == EW
    # valid calls get past the checks (no device here: a CUDA error or "unsupported device", never EINVAL)
    for kw in ({}, {"levels": 0}, {"levels": 14}, {"math": 1}, {"math": 2}, {"dt": 1}, {"sep": 180.0}, {"sep": 1e-6},
               {"beam": 1}, {"k": 1, "nbytes": lib.ahv_search_modes_workspace_bytes(B, base, 1, w)}):
        assert s(**kw) not in (E, EW), kw
    big = lib.ahv_search_modes_workspace_bytes(B, base, 32, 8)
    assert s(k=32, beam=8, nbytes=big) not in (E, EW) and s(k=32, beam=8) == EW
    assert s(base_level=0, levels=16, nbytes=lib.ahv_search_modes_workspace_bytes(B, 0, k, w)) not in (E, EW)


def test_search_modes_workspace_bytes(ahv):
    lib = ahv._lib.lib()
    size = lib.ahv_search_modes_workspace_bytes
    up = lambda v: (v + 255) // 256 * 256
    for B, base, k, w in ((1, 0, 1, 1), (1, 2, 8, 4), (8, 2, 8, 4), (32, 3, 32, 8), (5, 6, 1, 2)):
        n0, nc = 72 * 8 ** base, 8 * k * w
        scoring = max(lib.ahv_workspace_bytes(B, n0, 1), lib.ahv_workspace_bytes(B, nc, 1))
        ours = (up(B * 32 * 64 * 4) + up(n0 * 36) + up(B * n0) + up(B * nc * 8) + up(B * nc * 36)
                + 2 * up(B * k * w * 8))
        assert scoring + ours >= size(B, base, k, w) > ours, (B, base, k, w)        # scoring part: ahv_score's share
    assert size(2, 3, 8, 4) > size(2, 2, 8, 4) > size(1, 2, 8, 4)
    assert size(2, 2, 8, 8) > size(2, 2, 8, 4) > size(2, 2, 8, 1)
    assert size(0, 2, 8, 4) == 0 and size(-1, 2, 8, 4) == 0
    assert size(2, -1, 8, 4) == 0 and size(2, 7, 8, 4) == 0
    assert size(2, 2, 0, 4) == 0 and size(2, 2, 33, 4) == 0
    assert size(2, 2, 8, 0) == 0 and size(2, 2, 8, 9) == 0
