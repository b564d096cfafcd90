"""CPU: ahv_so3_hopf_grid, ahv_so3_hopf_children and ahv_search_hierarchical reject malformed arguments before they touch a
device, and the search's workspace size function."""
import ctypes


def test_hopf_grid_rejects_malformed_arguments_without_gpu(ahv):
    lib, E = ahv._lib.lib(), ahv._lib.AHV_EINVAL
    one = ctypes.c_void_p(256)
    g = lambda level=2, first=0, R=one, count=10: lib.ahv_so3_hopf_grid(level, first, R, count, None)
    assert g(level=-1) == E and g(level=17) == E                                    # levels 0 .. 16
    assert g(first=-1) == E and g(count=-1) == E
    assert g(first=4608 - 9) == E and g(first=0, count=4609) == E                   # past the level's 72*8^2 cells
    assert g(level=16, first=72 * 8 ** 16 - 1, count=2) == E
    assert g(R=None) == E
    assert g(R=None, count=0) not in (E,)                                           # nothing to write needs no buffer
    assert g() != E and g(first=4608 - 10) != E and g(level=16, first=72 * 8 ** 16 - 1, count=1) != E


def test_hopf_children_rejects_malformed_arguments_without_gpu(ahv):
    lib, E = ahv._lib.lib(), ahv._lib.AHV_EINVAL
    one = ctypes.c_void_p(256)
    c = lambda level=2, bufs=(one,) * 3, n=4: lib.ahv_so3_hopf_children(level, bufs[0], n, bufs[1], bufs[2], None)
    assert c(level=-1) == E and c(level=16) == E                                    # children must exist: level <= 15
    assert c(n=-1) == E and c(n=2 ** 62) == E
    for hole in range(3):
        bufs = [one] * 3
        bufs[hole] = None
        assert c(bufs=tuple(bufs)) == E, hole
    assert c(bufs=(None,) * 3, n=0) != E
    assert c() != E and c(level=15) != E


def test_search_hierarchical_rejects_malformed_arguments_without_gpu(ahv):
    lib, E, EW = ahv._lib.lib(), ahv._lib.AHV_EINVAL, ahv._lib.AHV_EWORKSPACE
    one = ctypes.c_void_p(256)
    B, base, levels, k = 3, 2, 4, 8
    need = lib.ahv_search_hierarchical_workspace_bytes(B, base, k)
    assert need > 0

    # (vol_src, vol_dtype, vol_tgt, W1, W2, b2, base, base_level, levels, k, first_val, first_idx, first_R, val, idx, R_out,
    #  B, math_mode, workspace, workspace_bytes, stream); bufs = the 13 pointers in that order
    def s(bufs=(one,) * 13, dt=0, base_level=base, levels=levels, k=k, B=B, math=0, nbytes=need):
        vs, vt, w1, w2, b2, bc, fv, fi, fR, v, i, R, ws = bufs
        return lib.ahv_search_hierarchical(vs, dt, vt, w1, w2, b2, bc, base_level, levels, k, fv, fi, fR, v, i, R, B, math, ws,
                                           nbytes, None)

    assert s(B=0) == E and s(B=-1) == E
    assert s(k=0) == E and s(k=33) == E and s(k=-1) == E
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
    for kw in ({}, {"levels": 0}, {"levels": 14}, {"math": 1}, {"math": 2}, {"dt": 1}):
        assert s(**kw) not in (E, EW), kw
    assert s(base_level=0, levels=16, nbytes=lib.ahv_search_hierarchical_workspace_bytes(B, 0, k)) not in (E, EW)


def test_search_hierarchical_workspace_bytes(ahv):
    lib = ahv._lib.lib()
    size = lib.ahv_search_hierarchical_workspace_bytes
    up = lambda v: (v + 255) // 256 * 256
    for B, base, k in ((1, 0, 1), (1, 2, 8), (8, 2, 8), (32, 3, 32), (5, 6, 1)):
        n0, nc = 72 * 8 ** base, 8 * k
        scoring = max(lib.ahv_workspace_bytes(B, n0, k), lib.ahv_workspace_bytes(B, nc, k))
        ours = up(B * 32 * 64 * 4) + up(n0 * 36) + up(B * nc * 8) + up(B * nc * 36) + up(B * k * 4) + 2 * up(B * k * 8)
        assert scoring + ours >= size(B, base, k) > ours, (B, base, k)               # scoring part: ahv_score's share
        assert size(B, base, k) >= up(n0 * 36)
    assert size(2, 3, 8) > size(2, 2, 8) > size(1, 2, 8)
    assert size(0, 2, 8) == 0 and size(-1, 2, 8) == 0
    assert size(2, -1, 8) == 0 and size(2, 7, 8) == 0
    assert size(2, 2, 0) == 0 and size(2, 2, 33) == 0
