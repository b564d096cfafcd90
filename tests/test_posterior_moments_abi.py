"""CPU: ahv_posterior_moments rejects malformed arguments before it touches a device, and its workspace size function."""
import ctypes
import math


def test_posterior_moments_rejects_malformed_arguments_without_gpu(ahv):
    lib, E, EW = ahv._lib.lib(), ahv._lib.AHV_EINVAL, ahv._lib.AHV_EWORKSPACE
    one = ctypes.c_void_p(256)
    B, N, k = 2, 5000, 4
    need = lib.ahv_posterior_moments_workspace_bytes(B, N, k)

    # ahv_posterior_moments(scores, R, r_per_pair, centers, B, N, k, radius_deg, temperature, log_z, mass, mean_R,
    #                       mean_cos, moment, ws, ws_bytes, stream)
    def pm(bufs=(one,) * 9, B=B, N=N, k=k, radius=10.0, T=0.1, nbytes=need):
        sc, R, cen, lz, ms, mr, mc, mo, ws = bufs
        return lib.ahv_posterior_moments(sc, R, 0, cen, B, N, k, radius, T, lz, ms, mr, mc, mo, ws, nbytes, None)

    assert pm(B=-1) == E and pm(N=0) == E and pm(N=-1) == E and pm(N=2**31) == E        # shapes
    assert pm(k=0) == E and pm(k=-1) == E and pm(k=33) == E                             # k outside [1, 32]
    for bad in (-1e-3, 180.5, -math.inf, math.inf, math.nan):                           # radius outside [0, 180]
        assert pm(radius=bad) == E, bad
    for bad in (0.0, -1.0, math.inf, -math.inf, math.nan):                              # temperature finite and > 0
        assert pm(T=bad) == E, bad
    for hole in range(9):                                                               # each buffer is required
        bufs = [one] * 9
        bufs[hole] = None
        assert pm(bufs=tuple(bufs)) == E, hole
    for pos in (1, 2, 8):                                                               # misaligned R, centers, workspace
        bufs = [one] * 9
        bufs[pos] = ctypes.c_void_p(260)
        assert pm(bufs=tuple(bufs)) == E, pos
    assert pm(nbytes=need - 1) == EW                                                    # workspace too small
    assert pm(nbytes=lib.ahv_posterior_mass_workspace_bytes(B, N, k)) == EW             # the mass's is not enough
    assert pm(B=0, bufs=(None,) * 9) not in (E, EW)                                     # B == 0 needs no buffer
    # valid calls get past the checks (no device here: a CUDA error or "unsupported device", never EINVAL)
    assert pm() not in (E, EW)
    assert pm(k=32, nbytes=lib.ahv_posterior_moments_workspace_bytes(B, N, 32)) not in (E, EW)


def test_posterior_moments_workspace_bytes(ahv):
    lib = ahv._lib.lib()
    size, mass_size = lib.ahv_posterior_moments_workspace_bytes, lib.ahv_posterior_mass_workspace_bytes
    up = lambda v: (v + 255) // 256 * 256
    chunks = lambda N: -(-N // 2048)
    for B, N, k in ((1, 1, 1), (3, 2048, 1), (3, 2049, 8), (32, 50_000, 32), (1, 1_000_000, 32), (128, 50_000, 1)):
        assert size(B, N, k) == mass_size(B, N, k) + up(B * chunks(N) * k * 9 * 8), (B, N, k)
        assert size(B, N, k) >= mass_size(B, N, k)
    assert size(0, 100, 4) == 0
    assert size(-1, 100, 4) == 0 and size(2, 0, 4) == 0 and size(2, 2**31, 4) == 0
    assert size(2, 100, 0) == 0 and size(2, 100, -1) == 0 and size(2, 100, 33) == 0
