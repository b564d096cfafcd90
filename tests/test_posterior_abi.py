"""CPU: ahv_posterior_mass rejects malformed arguments before it touches a device, and its workspace size function."""
import ctypes
import math


def test_posterior_mass_rejects_malformed_arguments_without_gpu(ahv):
    lib, E, EW = ahv._lib.lib(), ahv._lib.AHV_EINVAL, ahv._lib.AHV_EWORKSPACE
    one = ctypes.c_void_p(256)
    B, N, k = 2, 5000, 4
    need = lib.ahv_posterior_mass_workspace_bytes(B, N, k)

    # ahv_posterior_mass(scores, R, r_per_pair, centers, B, N, k, radius_deg, temperature, log_z, mass, ws, ws_bytes, stream)
    def pm(bufs=(one,) * 6, B=B, N=N, k=k, radius=10.0, T=0.1, nbytes=need):
        sc, R, cen, lz, ms, ws = bufs
        return lib.ahv_posterior_mass(sc, R, 0, cen, B, N, k, radius, T, lz, ms, ws, nbytes, None)

    assert pm(B=-1) == E and pm(N=0) == E and pm(N=-1) == E and pm(N=2**31) == E        # shapes
    assert pm(k=-1) == E and pm(k=33) == E                                              # k outside [0, 32]
    for bad in (-1e-3, 180.5, -math.inf, math.inf, math.nan):                           # radius outside [0, 180]
        assert pm(radius=bad) == E, bad
    for bad in (0.0, -0.1, math.inf, -math.inf, math.nan):                              # temperature finite and > 0
        assert pm(T=bad) == E, bad
    for hole in range(6):                                                               # each required buffer
        bufs = [one] * 6
        bufs[hole] = None
        assert pm(bufs=tuple(bufs)) == E, hole
    # k == 0: centers and mass must be NULL
    assert pm(k=0) == E
    assert pm(k=0, bufs=(one, one, None, one, one, one)) == E and pm(k=0, bufs=(one, one, one, one, None, one)) == E
    for pos in (1, 2, 5):                                                               # misaligned R, centers, workspace
        bufs = [one] * 6
        bufs[pos] = ctypes.c_void_p(260)
        assert pm(bufs=tuple(bufs)) == E, pos
    assert pm(nbytes=need - 1) == EW                                                    # workspace too small
    # B == 0 needs no buffer at all
    assert pm(B=0, bufs=(None,) * 6, k=0) not in (E, EW)
    # valid calls get past the checks (no device here: a CUDA error or "unsupported device", never EINVAL)
    assert pm() not in (E, EW)
    assert pm(k=0, bufs=(one, one, None, one, None, one), nbytes=lib.ahv_posterior_mass_workspace_bytes(B, N, 0)) not in (E, EW)


def test_posterior_mass_workspace_bytes(ahv):
    size = ahv._lib.lib().ahv_posterior_mass_workspace_bytes
    up = lambda v: (v + 255) // 256 * 256
    chunks = lambda N: -(-N // 2048)
    for B, N, k in ((1, 1, 0), (3, 2048, 1), (3, 2049, 8), (32, 50_000, 32), (1, 1_000_000, 32), (128, 50_000, 0)):
        assert size(B, N, k) == up(B * chunks(N) * (k + 1) * 8) + up(B * chunks(N) * 4), (B, N, k)
    assert size(0, 100, 4) == 0
    assert size(-1, 100, 4) == 0 and size(2, 0, 4) == 0 and size(2, 2**31, 4) == 0
    assert size(2, 100, -1) == 0 and size(2, 100, 33) == 0
