"""The host-side contract of the verification entries, frozen as literals: the three workspace-size functions over a
grid of shapes, and the status every checked entry returns for each malformed argument.

Callers allocate by the size functions and branch on the statuses, so neither may drift when the host glue changes.
The CPU tests pass fake host addresses only: every call that clears an entry's argument checks reaches the device check
and returns AHV_ECUDA there, so the status tables also pin where each entry's checks end.  With a device present those
calls are skipped (they would launch on the fake addresses).  The workspace bounds that the device check hides are
checked on the GPU with real buffers."""
import ast
import ctypes
import math

import pytest

OK, EINVAL, ENOTSUP, ECUDA, EWORKSPACE = 0, -1, -2, -3, -4
P = 16                       # a fake, 16-byte aligned address
BIG = 1 << 40                # workspace bytes that pass any bound
I31, I32 = 2**31 - 1, 2**32

# ---- workspace sizes -------------------------------------------------------------------------------------------------
SIZE_B = (-1, 0, 1, 2, 32, 128)
SIZE_N = (-1, 0, 1, 31, 4095, 4096, 4097, 50000, 262144, I31)
SIZE_K = (-1, 0, 1, 8, 32, 33)
SIZE_M = (0, 1, 64)


def size_tables(lib):
    """{function: {B (, m): [[bytes for k in SIZE_K] for N in SIZE_N]}}."""
    grid = lambda f: [[int(f(N, k)) for k in SIZE_K] for N in SIZE_N]
    return {
        "ahv_workspace_bytes": {B: grid(lambda N, k: lib.ahv_workspace_bytes(B, N, k)) for B in SIZE_B},
        "ahv_refine_workspace_bytes": {(B, m): grid(lambda N, k: lib.ahv_refine_workspace_bytes(B, N, k, m))
                                       for B in SIZE_B for m in SIZE_M},
        "ahv_refine_gradient_workspace_bytes": {B: grid(lambda N, k: lib.ahv_refine_gradient_workspace_bytes(B, N, k))
                                                for B in SIZE_B},
    }


def test_workspace_sizes_are_frozen(ahv):
    assert size_tables(ahv._lib.lib()) == SIZES


# ---- argument statuses -----------------------------------------------------------------------------------------------
# Each entry: its parameters in ABI order with a valid value (P for a pointer), and the values each scalar is tried at.
# Every pointer is also tried NULL and at two misaligned addresses.
_VOL = dict(vol_dtype=(-1, 1, 2))
_MATH = dict(math_mode=(-1, 1, 2, 3))
_BN = dict(B=(-1, 0, 1), N=(-1, 0, 1, 3, I31, I31 + 1))
_K = dict(k=(-1, 0, 1, 32, 33))
_ASCENT = dict(steps=(-1, 0, 1000, 1001), step_deg=(0.0, -1.0, math.inf, math.nan))
_SEP = dict(min_sep_deg=(0.0, -1e-3, 180.0, 180.5, math.inf, math.nan))
_PEERS = dict(rank=(-1, 1), world=(0, 2, 8, 9), peer_max_pairs=(0, 1), peer_max_k=(0, 1, 33), idx_offset=(-1, I32 - 100, I32 - 99))


def _spec(params, **tries):
    value = lambda s: BIG if s == "BIG" else ast.literal_eval(s)
    return [(p.split("=")[0], value(p.split("=")[1]) if "=" in p else P) for p in params.split()], tries


_HEAD = "vol_src vol_dtype=0 vol_tgt R r_per_pair=0 W1 W2 b2 base"
ENTRIES = {
    "ahv_score": _spec("vol_src vol_dtype=0 tgt_feat R r_per_pair=0 W1 W2 b2 base scores topk_val topk_idx k=4 idx_offset=0 "
                       "B=2 N=100 math_mode=0 workspace workspace_bytes=BIG stream=None",
                       **_VOL, **_MATH, **_BN, **_K, workspace_bytes=(0,)),
    "ahv_verify": _spec(_HEAD + " scores topk_val topk_idx R_best k=4 idx_offset=0 B=2 N=100 math_mode=0 workspace "
                        "workspace_bytes=BIG stream=None", **_VOL, **_MATH, **_BN, **_K, workspace_bytes=(0,)),
    "ahv_verify_sharded": _spec(_HEAD + " topk_val topk_idx R_best k=4 idx_offset=0 B=2 N=100 math_mode=0 workspace "
                                "workspace_bytes=BIG rank=0 world=1 peers=None peer_max_pairs=4 peer_max_k=32 stream=None",
                                **_VOL, **_MATH, **_BN, **_K, **_PEERS, workspace_bytes=(0,)),
    "ahv_refine": _spec(_HEAD + " k=4 m=8 max_angle_deg=5.0 seed=0 first_val first_idx first_R cand best_val best_idx R_best "
                        "B=2 N=100 math_mode=0 workspace workspace_bytes=BIG stream=None",
                        **_VOL, **_MATH, **_BN, **_K, m=(0, 1, 2**29 - 1, 2**29), max_angle_deg=(-1.0, 180.0, 181.0, math.nan),
                        workspace_bytes=(0, "need-1", "need")),
    "ahv_refine_gradient": _spec(_HEAD + " k=4 steps=20 step_deg=1.0 first_val first_idx first_R R_all score_all best_val "
                                 "best_idx R_best B=2 N=100 math_mode=0 workspace workspace_bytes=BIG stream=None",
                                 **_VOL, **_MATH, **_BN, **_K, **_ASCENT, workspace_bytes=(0, "need-1", "need")),
    "ahv_refine_gradient_distinct": _spec(_HEAD + " k=4 steps=20 step_deg=1.0 min_sep_deg=15.0 first_val first_idx first_R R_all "
                                          "score_all best_val best_idx R_best B=2 N=100 math_mode=0 workspace workspace_bytes=BIG "
                                          "stream=None", **_VOL, **_MATH, **_BN, **_K, **_ASCENT, **_SEP,
                                          workspace_bytes=(0, "need-1", "need")),
    "ahv_score_train": _spec("vol_src tgt_feat R r_per_pair=0 W1 W2 b2 base scores h1_saved pair_inv_scale B=2 N=100 workspace "
                             "workspace_bytes=BIG stream=None", **_BN, workspace_bytes=(0,)),
    "ahv_score_backward_saved": _spec("vol_src tgt_feat R r_per_pair=0 W1 W2 b2 base grad_scores h1_saved pair_inv_scale grad_vol "
                                      "grad_tgt grad_W1 grad_W2 grad_b2 B=2 N=100 math_mode=0 stream=None", **_MATH, **_BN),
    "ahv_score_backward_ex": _spec("vol_src tgt_feat R r_per_pair=0 W1 W2 b2 base grad_scores h1_saved pair_inv_scale grad_vol "
                                   "grad_tgt grad_W1 grad_W2 grad_b2 grad_R B=2 N=100 stream=None", **_BN),
    "ahv_gradient_ascent": _spec("vol_src vol_dtype=0 tgt_feat R_init W1 W2 b2 base steps=20 step_deg=1.0 R_out score_out B=2 "
                                 "K=3 stream=None", **_VOL, **_ASCENT, B=(-1, 0, 1), K=(-1, 0, 1)),
    "ahv_predict_host_ex": _spec("session vol_src_host vol_dtype=0 vol_tgt_host R_host r_per_pair=0 W1_host W2_host b2_host "
                                 "base_host scores_host topk_val_host topk_idx_host R_best_host k=4 idx_offset=0 B=2 N=100 "
                                 "math_mode=0 rank=0 world=1 peers=None peer_max_pairs=4 peer_max_k=32 stream=None",
                                 **_VOL, **_MATH, **_BN, **_K, **_PEERS),
}
_NEED = {
    "ahv_refine": lambda lib, a: lib.ahv_refine_workspace_bytes(a["B"], a["N"], a["k"], a["m"]),
    "ahv_refine_gradient": lambda lib, a: lib.ahv_refine_gradient_workspace_bytes(a["B"], a["N"], a["k"]),
    "ahv_refine_gradient_distinct": lambda lib, a: lib.ahv_refine_gradient_workspace_bytes(a["B"], a["N"], a["k"]),
}


def _cases(name):
    """(case id, overrides) for one entry: the valid call, each scalar at each tried value, each pointer NULL and
    misaligned, every pointer NULL on an empty batch, and a two-rank peer group where the entry takes one."""
    params, tries = ENTRIES[name]
    ptrs = [p for p, v in params if v is P]
    yield "valid", {}
    for p, values in tries.items():
        for v in values:
            yield f"{p}={v}", {p: v}
    for p in ptrs:
        for v in (None, 20, 24):
            yield f"{p}={v}", {p: v}
    for p in ("B", "N"):
        if p in tries and 0 in tries[p]:
            yield f"{p}=0,all=None", {p: 0, **{q: None for q in ptrs}}
    if "peers" in dict(params):
        group = (ctypes.c_void_p * 2)(P, P)
        yield "world=2,peers", {"world": 2, "peers": group}
        yield "world=2,peers,peer_max_pairs=1", {"world": 2, "peers": group, "peer_max_pairs": 1}
        yield "world=2,peers,peer_max_k=1", {"world": 2, "peers": group, "peer_max_k": 1}
        if "scores_host" in dict(params):
            yield "world=2,peers,scores_host=None", {"world": 2, "peers": group, "scores_host": None}


def statuses(lib, name, skip_device_calls=False, frozen=None):
    """{case id: status} of one entry; with skip_device_calls only the cases `frozen` records as rejected before the
    device check are called."""
    params, _ = ENTRIES[name]
    out = {}
    for cid, over in _cases(name):
        if skip_device_calls and frozen.get(cid) == ECUDA:
            continue
        args = dict(params, **over)
        if args.get("workspace_bytes") in ("need", "need-1"):
            args["workspace_bytes"] = _NEED[name](lib, dict(params)) - (args["workspace_bytes"] == "need-1")
        out[cid] = getattr(lib, name)(*args.values())
    return out


def _unpack(table):
    return {cid: st for st, ids in table.items() for cid in ids.split()}


def _has_device():
    import torch

    return torch.cuda.is_available()


@pytest.mark.parametrize("name", sorted(ENTRIES))
def test_argument_statuses_are_frozen(ahv, name):
    frozen = _unpack(STATUSES[name])
    got = statuses(ahv._lib.lib(), name, skip_device_calls=_has_device(), frozen=frozen)
    assert got == {cid: st for cid, st in frozen.items() if cid in got}
    assert set(got) == set(frozen) or _has_device()


# ---- workspace bounds behind the device check ------------------------------------------------------------------------
SCORE_NEED_B2_N300 = 46592   # ahv_score's own bound at B = 2, N = 300: scores, top-k partials, tensor-core scratch


@pytest.mark.gpu
def test_workspace_bounds_on_the_device(ahv):
    """need - 1 bytes is AHV_EWORKSPACE and need bytes AHV_OK, on real, correctly sized buffers."""
    import torch

    lib = ahv._lib.lib()
    dev = torch.device("cuda", 0)
    B, N = 2, 300
    g = torch.Generator().manual_seed(5)
    T = lambda *s: torch.randn(*s, generator=g).to(dev)
    vs, vt, tgt = T(B, 16, 8, 8, 8), T(B, 16, 8, 8, 8), T(B, 32, 64)
    R = ahv.so3.grid_rotations(N, device=dev)
    W1, W2, b2 = T(32, 384) * 0.05, T(32, 32) * 0.2, T(32) * 0.1
    base = ahv.ops.base_coords(dev)
    f32 = lambda *s: torch.empty(*s, device=dev)
    i64 = lambda *s: torch.empty(*s, device=dev, dtype=torch.int64)
    head = (vs.data_ptr(), 0, vt.data_ptr(), R.data_ptr(), 0, W1.data_ptr(), W2.data_ptr(), b2.data_ptr(), base.data_ptr())
    stream = torch.cuda.current_stream(dev).cuda_stream

    def bounded(need, call):
        ws = torch.empty(need, device=dev, dtype=torch.uint8)
        assert call(ws.data_ptr(), need - 1) == EWORKSPACE
        assert call(ws.data_ptr(), need) == OK
        torch.cuda.synchronize(dev)

    k = 4
    val, idx, Rb, sc = f32(B, k), i64(B, k), f32(B, k, 3, 3), f32(B, N)
    bounded(SCORE_NEED_B2_N300, lambda ws, n: lib.ahv_score(
        vs.data_ptr(), 0, tgt.data_ptr(), R.data_ptr(), 0, W1.data_ptr(), W2.data_ptr(), b2.data_ptr(), base.data_ptr(),
        sc.data_ptr(), val.data_ptr(), idx.data_ptr(), k, 0, B, N, 0, ws, n, stream))
    for kk, math_mode in ((1, 0), (4, 0), (4, 1)):
        bounded(lib.ahv_workspace_bytes(B, N, kk), lambda ws, n: lib.ahv_verify(
            *head, None, val.data_ptr(), idx.data_ptr(), Rb.data_ptr(), kk, 0, B, N, math_mode, ws, n, stream))
    bounded(lib.ahv_workspace_bytes(B, N, k), lambda ws, n: lib.ahv_verify_sharded(
        *head, val.data_ptr(), idx.data_ptr(), Rb.data_ptr(), k, 0, B, N, 0, ws, n, 0, 1, None, 0, 0, stream))
    m = 8
    fv, fi, fR, cand, bv, bi, bR = f32(B, k), i64(B, k), f32(B, k, 3, 3), f32(B, k * m, 3, 3), f32(B), i64(B), f32(B, 3, 3)
    bounded(lib.ahv_refine_workspace_bytes(B, N, k, m), lambda ws, n: lib.ahv_refine(
        *head, k, m, 5.0, 0, fv.data_ptr(), fi.data_ptr(), fR.data_ptr(), cand.data_ptr(), bv.data_ptr(), bi.data_ptr(),
        bR.data_ptr(), B, N, 0, ws, n, stream))
    Ra, sa = f32(B, k, 3, 3), f32(B, k)
    outs = (fv.data_ptr(), fi.data_ptr(), fR.data_ptr(), Ra.data_ptr(), sa.data_ptr(), bv.data_ptr(), bi.data_ptr(), bR.data_ptr())
    need = lib.ahv_refine_gradient_workspace_bytes(B, N, k)
    bounded(need, lambda ws, n: lib.ahv_refine_gradient(*head, k, 5, 1.0, *outs, B, N, 0, ws, n, stream))
    bounded(need, lambda ws, n: lib.ahv_refine_gradient_distinct(*head, k, 5, 1.0, 20.0, *outs, B, N, 0, ws, n, stream))


@pytest.mark.gpu
@pytest.mark.parametrize("max_angle_deg", (-1.0, 181.0, math.nan))
def test_rejected_refine_leaves_its_outputs_untouched(ahv, max_angle_deg):
    """ahv_refine checks max_angle_deg before its first pass: a rejected call enqueues no work and writes nothing."""
    import torch

    lib = ahv._lib.lib()
    dev = torch.device("cuda", 0)
    B, N, k, m = 2, 300, 4, 8
    g = torch.Generator().manual_seed(7)
    T = lambda *s: torch.randn(*s, generator=g).to(dev)
    vs, vt = T(B, 16, 8, 8, 8), T(B, 16, 8, 8, 8)
    R = ahv.so3.grid_rotations(N, device=dev)
    W1, W2, b2 = T(32, 384) * 0.05, T(32, 32) * 0.2, T(32) * 0.1
    outs = [torch.full(s, 7.0, device=dev) for s in ((B, k), (B, k, 3, 3), (B, k * m, 3, 3), (B,), (B, 3, 3))]
    idx = [torch.full(s, 7, device=dev, dtype=torch.int64) for s in ((B, k), (B,))]
    fv, fR, cand, bv, bR = outs
    fi, bi = idx
    need = lib.ahv_refine_workspace_bytes(B, N, k, m)
    ws = torch.empty(need, device=dev, dtype=torch.uint8)
    stream = torch.cuda.current_stream(dev).cuda_stream
    st = lib.ahv_refine(vs.data_ptr(), 0, vt.data_ptr(), R.data_ptr(), 0, W1.data_ptr(), W2.data_ptr(), b2.data_ptr(),
                        ahv.ops.base_coords(dev).data_ptr(), k, m, max_angle_deg, 0, fv.data_ptr(), fi.data_ptr(), fR.data_ptr(),
                        cand.data_ptr(), bv.data_ptr(), bi.data_ptr(), bR.data_ptr(), B, N, 0, ws.data_ptr(), need, stream)
    torch.cuda.synchronize(dev)
    assert st == EINVAL
    assert all(bool((t == 7).all()) for t in outs + idx)


# ---- frozen values ---------------------------------------------------------------------------------------------------
SIZES = {
    'ahv_workspace_bytes': {
        -1: [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
        ],
        0: [
            [0, 0, 0, 0, 0, 0],
            [26880, 26880, 26880, 26880, 26880, 26880],
            [26880, 26880, 26880, 26880, 26880, 26880],
            [26880, 26880, 26880, 26880, 26880, 26880],
            [26880, 26880, 26880, 26880, 26880, 26880],
            [26880, 26880, 26880, 26880, 26880, 26880],
            [26880, 26880, 26880, 26880, 26880, 26880],
            [26880, 26880, 26880, 26880, 26880, 26880],
            [26880, 26880, 26880, 26880, 26880, 26880],
            [26880, 26880, 26880, 26880, 26880, 26880],
        ],
        1: [
            [0, 0, 0, 0, 0, 0],
            [35840, 35840, 35840, 35840, 36096, 36096],
            [36096, 36096, 36096, 36096, 36352, 36352],
            [36096, 36096, 36096, 36096, 36352, 36352],
            [52224, 52224, 52224, 52224, 52480, 52480],
            [52224, 52224, 52224, 52224, 52480, 52480],
            [52480, 52480, 52480, 52480, 52736, 52736],
            [238848, 238848, 238848, 238848, 239104, 239104],
            [1100544, 1100544, 1100544, 1100544, 1100800, 1100800],
            [8589986560, 8589986560, 8589986560, 8589986560, 8589986816, 8589986816],
        ],
        2: [
            [0, 0, 0, 0, 0, 0],
            [44288, 44288, 44288, 44288, 44800, 45056],
            [44544, 44544, 44544, 44544, 45056, 45312],
            [44544, 44544, 44544, 44544, 45056, 45312],
            [77056, 77056, 77056, 77056, 77568, 77824],
            [77056, 77056, 77056, 77056, 77568, 77824],
            [77312, 77312, 77312, 77312, 77824, 78080],
            [450048, 450048, 450048, 450048, 450560, 450816],
            [2173696, 2173696, 2173696, 2173696, 2174208, 2174464],
            [17179945728, 17179945728, 17179945728, 17179945728, 17179946240, 17179946496],
        ],
        32: [
            [0, 0, 0, 0, 0, 0],
            [298240, 298240, 298240, 300800, 310016, 310528],
            [298496, 298496, 298496, 301056, 310272, 310784],
            [302336, 302336, 302336, 304896, 314112, 314624],
            [822528, 822528, 822528, 825088, 834304, 834816],
            [822528, 822528, 822528, 825088, 834304, 834816],
            [822784, 822784, 822784, 825344, 834560, 835072],
            [6788352, 6788352, 6788352, 6790912, 6800128, 6800640],
            [34368768, 34368768, 34368768, 34371328, 34380544, 34381056],
            [274878721280, 274878721280, 274878721280, 274878723840, 274878733056, 274878733568],
        ],
        128: [
            [0, 0, 0, 0, 0, 0],
            [1111808, 1111808, 1111808, 1122560, 1159424, 1160960],
            [1112320, 1112320, 1112320, 1123072, 1159936, 1161472],
            [1127680, 1127680, 1127680, 1138432, 1175296, 1176832],
            [3208448, 3208448, 3208448, 3219200, 3256064, 3257600],
            [3208960, 3208960, 3208960, 3219712, 3256576, 3258112],
            [3209472, 3209472, 3209472, 3220224, 3257088, 3258624],
            [27072256, 27072256, 27072256, 27083008, 27119872, 27121408],
            [137393920, 137393920, 137393920, 137404672, 137441536, 137443072],
            [1099514803456, 1099514803456, 1099514803456, 1099514814208, 1099514851072, 1099514852608],
        ],
    },
    'ahv_refine_workspace_bytes': {
        (-1, 0): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
        ],
        (-1, 1): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
        ],
        (-1, 64): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
        ],
        (0, 0): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
        ],
        (0, 1): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
        ],
        (0, 64): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
            [0, 0, 53760, 53760, 53760, 0],
        ],
        (1, 0): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
        ],
        (1, 1): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 71936, 71936, 72192, 0],
            [0, 0, 72192, 72192, 72448, 0],
            [0, 0, 72192, 72192, 72448, 0],
            [0, 0, 88320, 88320, 88576, 0],
            [0, 0, 88320, 88320, 88576, 0],
            [0, 0, 88576, 88576, 88832, 0],
            [0, 0, 274944, 274944, 275200, 0],
            [0, 0, 1136640, 1136640, 1136896, 0],
            [0, 0, 8590022656, 8590022656, 8590022912, 0],
        ],
        (1, 64): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 71936, 73728, 80128, 0],
            [0, 0, 72192, 73984, 80384, 0],
            [0, 0, 72192, 73984, 80384, 0],
            [0, 0, 88320, 90112, 96512, 0],
            [0, 0, 88320, 90112, 96512, 0],
            [0, 0, 88576, 90368, 96768, 0],
            [0, 0, 274944, 276736, 283136, 0],
            [0, 0, 1136640, 1138432, 1144832, 0],
            [0, 0, 8590022656, 8590024448, 8590030848, 0],
        ],
        (2, 0): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
        ],
        (2, 1): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 88832, 88832, 89344, 0],
            [0, 0, 89088, 89088, 89600, 0],
            [0, 0, 89088, 89088, 89600, 0],
            [0, 0, 121600, 121600, 122112, 0],
            [0, 0, 121600, 121600, 122112, 0],
            [0, 0, 121856, 121856, 122368, 0],
            [0, 0, 494592, 494592, 495104, 0],
            [0, 0, 2218240, 2218240, 2218752, 0],
            [0, 0, 17179990272, 17179990272, 17179990784, 0],
        ],
        (2, 64): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 89088, 92672, 105472, 0],
            [0, 0, 89344, 92928, 105728, 0],
            [0, 0, 89344, 92928, 105728, 0],
            [0, 0, 121856, 125440, 138240, 0],
            [0, 0, 121856, 125440, 138240, 0],
            [0, 0, 122112, 125696, 138496, 0],
            [0, 0, 494848, 498432, 511232, 0],
            [0, 0, 2218496, 2222080, 2234880, 0],
            [0, 0, 17179990528, 17179994112, 17180006912, 0],
        ],
        (32, 0): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
        ],
        (32, 1): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 596736, 600064, 612352, 0],
            [0, 0, 596992, 600320, 612608, 0],
            [0, 0, 600832, 604160, 616448, 0],
            [0, 0, 1121024, 1124352, 1136640, 0],
            [0, 0, 1121024, 1124352, 1136640, 0],
            [0, 0, 1121280, 1124608, 1136896, 0],
            [0, 0, 7086848, 7090176, 7102464, 0],
            [0, 0, 34667264, 34670592, 34682880, 0],
            [0, 0, 274879019776, 274879023104, 274879035392, 0],
        ],
        (32, 64): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 604672, 664576, 870400, 0],
            [0, 0, 604928, 664832, 870656, 0],
            [0, 0, 608768, 668672, 874496, 0],
            [0, 0, 1128960, 1188864, 1394688, 0],
            [0, 0, 1128960, 1188864, 1394688, 0],
            [0, 0, 1129216, 1189120, 1394944, 0],
            [0, 0, 7094784, 7154688, 7360512, 0],
            [0, 0, 34675200, 34735104, 34940928, 0],
            [0, 0, 274879027712, 274879087616, 274879293440, 0],
        ],
        (128, 0): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
        ],
        (128, 1): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 2224128, 2238464, 2287616, 0],
            [0, 0, 2224640, 2238976, 2288128, 0],
            [0, 0, 2240000, 2254336, 2303488, 0],
            [0, 0, 4320768, 4335104, 4384256, 0],
            [0, 0, 4321280, 4335616, 4384768, 0],
            [0, 0, 4321792, 4336128, 4385280, 0],
            [0, 0, 28184576, 28198912, 28248064, 0],
            [0, 0, 138506240, 138520576, 138569728, 0],
            [0, 0, 1099515915776, 1099515930112, 1099515979264, 0],
        ],
        (128, 64): [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 2256384, 2496512, 3319808, 0],
            [0, 0, 2256896, 2497024, 3320320, 0],
            [0, 0, 2272256, 2512384, 3335680, 0],
            [0, 0, 4353024, 4593152, 5416448, 0],
            [0, 0, 4353536, 4593664, 5416960, 0],
            [0, 0, 4354048, 4594176, 5417472, 0],
            [0, 0, 28216832, 28456960, 29280256, 0],
            [0, 0, 138538496, 138778624, 139601920, 0],
            [0, 0, 1099515948032, 1099516188160, 1099517011456, 0],
        ],
    },
    'ahv_refine_gradient_workspace_bytes': {
        -1: [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
            [0, 0, 0, 0, 0, 0],
        ],
        0: [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 26880, 26880, 26880, 0],
            [0, 0, 26880, 26880, 26880, 0],
            [0, 0, 26880, 26880, 26880, 0],
            [0, 0, 26880, 26880, 26880, 0],
            [0, 0, 26880, 26880, 26880, 0],
            [0, 0, 26880, 26880, 26880, 0],
            [0, 0, 26880, 26880, 26880, 0],
            [0, 0, 26880, 26880, 26880, 0],
            [0, 0, 26880, 26880, 26880, 0],
        ],
        1: [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 44288, 44288, 44544, 0],
            [0, 0, 44544, 44544, 44800, 0],
            [0, 0, 44544, 44544, 44800, 0],
            [0, 0, 60672, 60672, 60928, 0],
            [0, 0, 60672, 60672, 60928, 0],
            [0, 0, 60928, 60928, 61184, 0],
            [0, 0, 247296, 247296, 247552, 0],
            [0, 0, 1108992, 1108992, 1109248, 0],
            [0, 0, 8589995008, 8589995008, 8589995264, 0],
        ],
        2: [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 61184, 61184, 61696, 0],
            [0, 0, 61440, 61440, 61952, 0],
            [0, 0, 61440, 61440, 61952, 0],
            [0, 0, 93952, 93952, 94464, 0],
            [0, 0, 93952, 93952, 94464, 0],
            [0, 0, 94208, 94208, 94720, 0],
            [0, 0, 466944, 466944, 467456, 0],
            [0, 0, 2190592, 2190592, 2191104, 0],
            [0, 0, 17179962624, 17179962624, 17179963136, 0],
        ],
        32: [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 568576, 571136, 580352, 0],
            [0, 0, 568832, 571392, 580608, 0],
            [0, 0, 572672, 575232, 584448, 0],
            [0, 0, 1092864, 1095424, 1104640, 0],
            [0, 0, 1092864, 1095424, 1104640, 0],
            [0, 0, 1093120, 1095680, 1104896, 0],
            [0, 0, 7058688, 7061248, 7070464, 0],
            [0, 0, 34639104, 34641664, 34650880, 0],
            [0, 0, 274878991616, 274878994176, 274879003392, 0],
        ],
        128: [
            [0, 0, 0, 0, 0, 0],
            [0, 0, 2193152, 2203904, 2240768, 0],
            [0, 0, 2193664, 2204416, 2241280, 0],
            [0, 0, 2209024, 2219776, 2256640, 0],
            [0, 0, 4289792, 4300544, 4337408, 0],
            [0, 0, 4290304, 4301056, 4337920, 0],
            [0, 0, 4290816, 4301568, 4338432, 0],
            [0, 0, 28153600, 28164352, 28201216, 0],
            [0, 0, 138475264, 138486016, 138522880, 0],
            [0, 0, 1099515884800, 1099515895552, 1099515932416, 0],
        ],
    },
}
STATUSES = {
    'ahv_gradient_ascent': {
        ECUDA: (
            'valid vol_dtype=1 steps=0 steps=1000 B=1 K=1 b2=20 b2=24 base=20 base=24 score_out=20 score_out=24 '),
        EINVAL: (
            'vol_dtype=-1 vol_dtype=2 steps=-1 steps=1001 step_deg=0.0 step_deg=-1.0 step_deg=inf step_deg=nan '
            'B=-1 B=0 K=-1 K=0 vol_src=None vol_src=20 vol_src=24 tgt_feat=None tgt_feat=20 tgt_feat=24 '
            'R_init=None R_init=20 R_init=24 W1=None W1=20 W1=24 W2=None W2=20 W2=24 b2=None base=None R_out=None '
            'R_out=20 R_out=24 score_out=None B=0,all=None '),
    },
    'ahv_predict_host_ex': {
        ECUDA: (
            'valid vol_dtype=1 math_mode=-1 math_mode=1 math_mode=2 math_mode=3 B=1 N=1 N=3 N=2147483647 '
            'N=2147483648 k=1 k=32 rank=-1 rank=1 world=0 peer_max_pairs=0 peer_max_pairs=1 peer_max_k=0 '
            'peer_max_k=1 peer_max_k=33 idx_offset=-1 idx_offset=4294967196 idx_offset=4294967197 session=20 '
            'session=24 vol_src_host=20 vol_src_host=24 vol_tgt_host=20 vol_tgt_host=24 R_host=20 R_host=24 '
            'W1_host=20 W1_host=24 W2_host=20 W2_host=24 b2_host=20 b2_host=24 base_host=20 base_host=24 '
            'scores_host=None scores_host=20 scores_host=24 topk_val_host=20 topk_val_host=24 topk_idx_host=20 '
            'topk_idx_host=24 R_best_host=None R_best_host=20 R_best_host=24 world=2,peers,scores_host=None '),
        EINVAL: (
            'vol_dtype=-1 vol_dtype=2 B=-1 B=0 N=-1 N=0 k=-1 k=0 k=33 world=2 world=8 world=9 session=None '
            'vol_src_host=None vol_tgt_host=None R_host=None W1_host=None W2_host=None b2_host=None '
            'base_host=None topk_val_host=None topk_idx_host=None B=0,all=None N=0,all=None world=2,peers '
            'world=2,peers,peer_max_pairs=1 world=2,peers,peer_max_k=1 '),
    },
    'ahv_refine': {
        EWORKSPACE: (
            'workspace_bytes=0 workspace_bytes=need-1 '),
        ECUDA: (
            'valid vol_dtype=1 math_mode=1 math_mode=2 B=1 N=2147483647 k=1 k=32 m=1 m=536870911 '
            'max_angle_deg=180.0 workspace_bytes=need '
            'b2=20 b2=24 base=20 base=24 first_val=20 first_val=24 first_idx=20 first_idx=24 first_R=20 '
            'first_R=24 best_val=20 best_val=24 best_idx=20 best_idx=24 R_best=None R_best=20 R_best=24 '),
        EINVAL: (
            'vol_dtype=-1 vol_dtype=2 math_mode=-1 math_mode=3 B=-1 B=0 N=-1 N=0 N=1 N=3 N=2147483648 k=-1 k=0 '
            'k=33 m=0 m=536870912 max_angle_deg=-1.0 max_angle_deg=181.0 max_angle_deg=nan vol_src=None '
            'vol_src=20 vol_src=24 vol_tgt=None vol_tgt=20 vol_tgt=24 R=None '
            'R=20 R=24 W1=None W1=20 W1=24 W2=None W2=20 W2=24 b2=None base=None first_val=None first_idx=None '
            'first_R=None cand=None cand=20 cand=24 best_val=None best_idx=None workspace=None workspace=20 '
            'workspace=24 B=0,all=None N=0,all=None '),
    },
    'ahv_refine_gradient': {
        EWORKSPACE: (
            'workspace_bytes=0 workspace_bytes=need-1 '),
        ECUDA: (
            'valid vol_dtype=1 math_mode=1 math_mode=2 B=1 N=2147483647 k=1 k=32 steps=0 steps=1000 '
            'workspace_bytes=need b2=20 b2=24 base=20 base=24 first_val=20 first_val=24 first_idx=20 first_idx=24 '
            'score_all=20 score_all=24 best_val=20 best_val=24 best_idx=20 best_idx=24 R_best=None '),
        EINVAL: (
            'vol_dtype=-1 vol_dtype=2 math_mode=-1 math_mode=3 B=-1 B=0 N=-1 N=0 N=1 N=3 N=2147483648 k=-1 k=0 '
            'k=33 steps=-1 steps=1001 step_deg=0.0 step_deg=-1.0 step_deg=inf step_deg=nan vol_src=None '
            'vol_src=20 vol_src=24 vol_tgt=None vol_tgt=20 vol_tgt=24 R=None R=20 R=24 W1=None W1=20 W1=24 '
            'W2=None W2=20 W2=24 b2=None base=None first_val=None first_idx=None first_R=None first_R=20 '
            'first_R=24 R_all=None R_all=20 R_all=24 score_all=None best_val=None best_idx=None R_best=20 '
            'R_best=24 workspace=None workspace=20 workspace=24 B=0,all=None N=0,all=None '),
    },
    'ahv_refine_gradient_distinct': {
        EWORKSPACE: (
            'workspace_bytes=0 workspace_bytes=need-1 '),
        ECUDA: (
            'valid vol_dtype=1 math_mode=1 math_mode=2 B=1 N=2147483647 k=1 k=32 steps=0 steps=1000 '
            'min_sep_deg=0.0 min_sep_deg=180.0 workspace_bytes=need b2=20 b2=24 base=20 base=24 first_val=20 '
            'first_val=24 first_idx=20 first_idx=24 score_all=20 score_all=24 best_val=20 best_val=24 best_idx=20 '
            'best_idx=24 R_best=None '),
        EINVAL: (
            'vol_dtype=-1 vol_dtype=2 math_mode=-1 math_mode=3 B=-1 B=0 N=-1 N=0 N=1 N=3 N=2147483648 k=-1 k=0 '
            'k=33 steps=-1 steps=1001 step_deg=0.0 step_deg=-1.0 step_deg=inf step_deg=nan min_sep_deg=-0.001 '
            'min_sep_deg=180.5 min_sep_deg=inf min_sep_deg=nan vol_src=None vol_src=20 vol_src=24 vol_tgt=None '
            'vol_tgt=20 vol_tgt=24 R=None R=20 R=24 W1=None W1=20 W1=24 W2=None W2=20 W2=24 b2=None base=None '
            'first_val=None first_idx=None first_R=None first_R=20 first_R=24 R_all=None R_all=20 R_all=24 '
            'score_all=None best_val=None best_idx=None R_best=20 R_best=24 workspace=None workspace=20 '
            'workspace=24 B=0,all=None N=0,all=None '),
    },
    'ahv_score': {
        ECUDA: (
            'valid vol_dtype=1 math_mode=1 math_mode=2 B=0 B=1 N=0 N=1 N=3 N=2147483647 k=0 k=1 k=32 '
            'workspace_bytes=0 b2=20 b2=24 base=20 base=24 scores=None scores=20 scores=24 topk_val=20 '
            'topk_val=24 topk_idx=20 topk_idx=24 workspace=None '),
        EINVAL: (
            'vol_dtype=-1 vol_dtype=2 math_mode=-1 math_mode=3 B=-1 N=-1 N=2147483648 k=-1 k=33 vol_src=None '
            'vol_src=20 vol_src=24 tgt_feat=None tgt_feat=20 tgt_feat=24 R=None R=20 R=24 W1=None W1=20 W1=24 '
            'W2=None W2=20 W2=24 b2=None base=None topk_val=None topk_idx=None workspace=20 workspace=24 '
            'B=0,all=None N=0,all=None '),
    },
    'ahv_score_backward_ex': {
        ECUDA: (
            'valid B=0 B=1 N=0 N=1 N=3 N=2147483647 vol_src=20 vol_src=24 tgt_feat=20 tgt_feat=24 R=20 R=24 W1=20 '
            'W1=24 W2=20 W2=24 b2=20 b2=24 base=20 base=24 grad_scores=20 grad_scores=24 pair_inv_scale=20 '
            'pair_inv_scale=24 grad_vol=None grad_vol=20 grad_vol=24 grad_tgt=None grad_tgt=20 grad_tgt=24 '
            'grad_W1=None grad_W1=20 grad_W1=24 grad_W2=None grad_W2=20 grad_W2=24 grad_b2=None grad_b2=20 '
            'grad_b2=24 grad_R=None grad_R=20 grad_R=24 '),
        EINVAL: (
            'B=-1 N=-1 N=2147483648 vol_src=None tgt_feat=None R=None W1=None W2=None b2=None base=None '
            'grad_scores=None h1_saved=None h1_saved=20 h1_saved=24 pair_inv_scale=None B=0,all=None N=0,all=None '),
    },
    'ahv_score_backward_saved': {
        ECUDA: (
            'valid math_mode=1 B=0 B=1 N=0 N=1 N=3 N=2147483647 vol_src=20 vol_src=24 tgt_feat=20 tgt_feat=24 '
            'R=20 R=24 W1=20 W1=24 W2=20 W2=24 b2=20 b2=24 base=20 base=24 grad_scores=20 grad_scores=24 '
            'pair_inv_scale=20 pair_inv_scale=24 grad_vol=20 grad_vol=24 grad_tgt=20 grad_tgt=24 grad_W1=20 '
            'grad_W1=24 grad_W2=20 grad_W2=24 grad_b2=20 grad_b2=24 B=0,all=None N=0,all=None '),
        EINVAL: (
            'math_mode=-1 math_mode=2 math_mode=3 B=-1 N=-1 N=2147483648 vol_src=None tgt_feat=None R=None '
            'W1=None W2=None b2=None base=None grad_scores=None h1_saved=None h1_saved=20 h1_saved=24 '
            'pair_inv_scale=None grad_vol=None grad_tgt=None grad_W1=None grad_W2=None grad_b2=None '),
    },
    'ahv_score_train': {
        ECUDA: (
            'valid B=0 B=1 N=0 N=1 N=3 N=2147483647 workspace_bytes=0 b2=20 b2=24 base=20 base=24 scores=20 '
            'scores=24 pair_inv_scale=20 pair_inv_scale=24 B=0,all=None N=0,all=None '),
        EINVAL: (
            'B=-1 N=-1 N=2147483648 vol_src=None vol_src=20 vol_src=24 tgt_feat=None tgt_feat=20 tgt_feat=24 '
            'R=None R=20 R=24 W1=None W1=20 W1=24 W2=None W2=20 W2=24 b2=None base=None scores=None h1_saved=None '
            'h1_saved=20 h1_saved=24 pair_inv_scale=None workspace=None workspace=20 workspace=24 '),
    },
    'ahv_verify': {
        ECUDA: (
            'valid vol_dtype=1 math_mode=1 math_mode=2 B=0 B=1 N=0 N=1 N=3 N=2147483647 k=1 k=32 '
            'workspace_bytes=0 b2=20 b2=24 base=20 base=24 scores=None scores=20 scores=24 topk_val=20 '
            'topk_val=24 topk_idx=20 topk_idx=24 R_best=None R_best=20 R_best=24 workspace=None B=0,all=None '
            'N=0,all=None '),
        EINVAL: (
            'vol_dtype=-1 vol_dtype=2 math_mode=-1 math_mode=3 B=-1 N=-1 N=2147483648 k=-1 k=0 k=33 vol_src=None '
            'vol_src=20 vol_src=24 vol_tgt=None vol_tgt=20 vol_tgt=24 R=None R=20 R=24 W1=None W1=20 W1=24 '
            'W2=None W2=20 W2=24 b2=None base=None topk_val=None topk_idx=None workspace=20 workspace=24 '),
    },
    'ahv_verify_sharded': {
        ECUDA: (
            'valid vol_dtype=1 math_mode=1 math_mode=2 B=1 N=0 N=1 N=3 N=2147483647 k=1 k=32 peer_max_pairs=0 '
            'peer_max_pairs=1 peer_max_k=0 peer_max_k=1 peer_max_k=33 idx_offset=4294967196 workspace_bytes=0 '
            'b2=20 b2=24 base=20 base=24 topk_val=20 topk_val=24 topk_idx=20 topk_idx=24 R_best=None R_best=20 '
            'R_best=24 workspace=None world=2,peers '),
        EINVAL: (
            'vol_dtype=-1 vol_dtype=2 math_mode=-1 math_mode=3 B=-1 B=0 N=-1 N=2147483648 k=-1 k=0 k=33 rank=-1 '
            'rank=1 world=0 world=2 world=8 world=9 idx_offset=-1 idx_offset=4294967197 vol_src=None vol_src=20 '
            'vol_src=24 vol_tgt=None vol_tgt=20 vol_tgt=24 R=None R=20 R=24 W1=None W1=20 W1=24 W2=None W2=20 '
            'W2=24 b2=None base=None topk_val=None topk_idx=None workspace=20 workspace=24 B=0,all=None '
            'N=0,all=None world=2,peers,peer_max_pairs=1 world=2,peers,peer_max_k=1 '),
    },
}
