"""ctypes binding of lib3dahv_b200.so (C ABI declared in include/ahv_b200.h).

The product path has no CPU fallback: if the shared library is missing this
module raises at import of the first op, and on a non-sm_100 device every
compute entry returns AHV_ENOTSUP which `check` turns into RuntimeError.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib3dahv_b200.so")

AHV_OK, AHV_EINVAL, AHV_ENOTSUP, AHV_ECUDA, AHV_EWORKSPACE = 0, -1, -2, -3, -4
VOL_F32, VOL_BF16 = 0, 1
MATH_TC, MATH_FP32, MATH_TC_F16GATHER = 0, 1, 2

_vp, _i, _i64, _u64, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64, ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/ahv_b200.h one to one
SIGNATURES = {
    "ahv_version": (_i, []),
    "ahv_status_string": (ctypes.c_char_p, [_i]),
    "ahv_so3_from_normals": (_i, [_vp, _vp, _i64, _vp]),
    "ahv_so3_sample": (_i, [_u64, _i64, _vp, _i64, _vp]),
    "ahv_so3_grid": (_i, [_i64, _i64, _vp, _i64, _vp]),
    "ahv_so3_perturb": (_i, [_vp, _i64, _i, ctypes.c_float, _u64, _vp, _vp]),
    "ahv_rotate_volume": (_i, [_vp, _i, _vp, _vp, _vp, _i64, _vp]),
    "ahv_rotate_volume_backward": (_i, [_vp, _i, _vp, _vp, _vp, _i64, _vp]),
    "ahv_score_backward": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "ahv_infonce": (_i, [_vp, _vp, _i, _vp, ctypes.c_float, ctypes.c_float, _vp, _vp, _i, _i64, _vp]),
    "ahv_resblock3d": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ahv_score_train": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _vp, _sz, _vp]),
    "ahv_score_backward_saved": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _vp]),
    "ahv_rotate_volume_grad_R": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ahv_score_backward_ex": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "ahv_score_backward_det_workspace_bytes": (_sz, [_i, _i64, _i, _i]),
    "ahv_score_backward_det": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i,
                                    _vp, _sz, _vp]),
    "ahv_forward_3d2d": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ahv_workspace_bytes": (_sz, [_i, _i64, _i]),
    "ahv_score": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _i64, _i, _vp, _sz, _vp]),
    "ahv_verify": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _i64, _i, _vp, _sz, _vp]),
    "ahv_refine_workspace_bytes": (_sz, [_i, _i64, _i, _i]),
    "ahv_refine": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, ctypes.c_float, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                        _i, _i64, _i, _vp, _sz, _vp]),
    "ahv_gradient_ascent": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, ctypes.c_float, _vp, _vp, _i, _i, _vp]),
    "ahv_refine_gradient_workspace_bytes": (_sz, [_i, _i64, _i]),
    "ahv_refine_gradient": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, ctypes.c_float, _vp, _vp, _vp, _vp, _vp, _vp,
                                 _vp, _vp, _i, _i64, _i, _vp, _sz, _vp]),
    "ahv_refine_gradient_distinct": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, ctypes.c_float, ctypes.c_float, _vp,
                                          _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _vp, _sz, _vp]),
    "ahv_topk_distinct": (_i, [_vp, _vp, _i, _i, _i64, _i, ctypes.c_float, _vp, _vp, _vp, _vp]),
    "ahv_topk": (_i, [_vp, _i, _i64, _i, _i64, _vp, _vp, _vp, _sz, _vp]),
    "ahv_topk_merge": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "ahv_gather_rotations": (_i, [_vp, _i, _vp, _i64, _i, _i64, _i, _vp, _vp]),
    "ahv_diag_smem_read": (_i, [_vp, _i, _i, ctypes.POINTER(ctypes.c_ulonglong), _vp]),
    "ahv_peer_bytes": (_sz, [_i, _i]),
    "ahv_peer_alloc": (_i, [_i, _i, ctypes.POINTER(ctypes.c_void_p)]),
    "ahv_peer_free": (_i, [_vp]),
    "ahv_peer_export": (_i, [_vp, ctypes.c_char_p]),
    "ahv_peer_open": (_i, [ctypes.c_char_p, ctypes.POINTER(ctypes.c_void_p)]),
    "ahv_peer_close": (_i, [_vp]),
    "ahv_peer_status": (_i, [_vp, ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint32)]),
    "ahv_peer_capacity": (_i, [_vp, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "ahv_topk_exchange": (_i, [_vp, _vp, _vp, _i, _i64, _i64, _i, _i, _vp, _vp, _vp, _i, _i, ctypes.POINTER(ctypes.c_void_p),
                               _i, _i, _vp]),
    "ahv_verify_sharded": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _i64, _i, _vp, _sz, _i, _i,
                                ctypes.POINTER(ctypes.c_void_p), _i, _i, _vp]),
    "ahv_host_session_create": (_i, [ctypes.POINTER(ctypes.c_void_p)]),
    "ahv_host_session_destroy": (_i, [_vp]),
    "ahv_predict_host_ex": (_i, [_vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _i64, _i, _i, _i,
                                 ctypes.POINTER(ctypes.c_void_p), _i, _i, _vp]),
    "ahv_predict_host": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i64, _i, _vp]),
}

_lib = None


def lib() -> ctypes.CDLL:
    """Load the library (built in-tree by `python 3dahv_b200/build.py`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python 3dahv_b200/build.py` "
                "(there is no CPU or PyTorch fallback for the 3DAHV hot path)"
            )
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(status: int, what: str = "lib3dahv_b200") -> None:
    if status != AHV_OK:
        msg = lib().ahv_status_string(status).decode()
        raise RuntimeError(f"{what} failed: {msg} (status {status})")
