"""ctypes binding of libbigru_b200.so (include/bigru_b200.h).

There is no CPU or PyTorch fallback: if the shared library cannot be loaded, or a call
returns an error code, a RuntimeError/ValueError is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbigru_b200.so")

PREC_FP32, PREC_BF16, PREC_BF16X3 = 0, 1, 2
LOSS_CE, LOSS_BCE, LOSS_MLSM = 0, 1, 2
ERR_ARG, ERR_CUDA, ERR_DEVICE, ERR_UNSUPPORTED = -1, -2, -3, -4

_vp, _i, _i64, _f, _u64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint64, C.c_double

# name -> (restype, argtypes); mirrors include/bigru_b200.h one to one
SIGNATURES = {
    "bigru_last_error": (C.c_char_p, []),
    "bigru_version": (_i, []),
    "bigru_device_check": (_i, [_i]),
    "bigru_plan_create": (_i, [_i, _i, _i, _i, _i, _i, _i, _i, C.POINTER(_vp)]),
    "bigru_plan_destroy": (_i, [_vp]),
    "bigru_param_count": (_i64, [_vp]),
    "bigru_param_offset": (_i, [_vp, _i, _i, _i, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)]),
    "bigru_workspace_bytes": (_i, [_vp, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "bigru_stash_argmax_offset": (_i, [_vp, C.POINTER(C.c_size_t)]),
    "bigru_forward": (_i, [_vp, _vp, _vp, _vp, _f, _i, _i, _u64, _vp, _vp, _vp, _vp, _vp]),
    "bigru_backward": (_i, [_vp, _vp, _vp, _vp, _f, _i, _i, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bigru_backward_layers": (_i, [_vp, _vp, _vp, _vp, _f, _i, _i, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]),
    "bigru_loss": (_i, [_i, _vp, _vp, _vp, _vp, _i, _i, _d, _vp, _vp, _vp]),
    "bigru_sqnorm": (_i, [_vp, _i64, _vp, _vp]),
    "bigru_clip_adam_step": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _f, _f, _f, _f, _f, _i, _f, _vp]),
    "bigru_adam_tick": (_i, [_vp, _vp, _vp]),
    "bigru_clip_adam_step_dev": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _f, _f, _f, _f, _f, _vp, _f, _vp]),
    "bigru_launch_count_add": (None, [C.c_longlong]),
    "bigru_window_gather_norm": (_i, [_vp, _vp, _vp, _i64, _i64, _i, _i, _i, _vp, _vp]),
    "bigru_window_targets": (_i, [_vp, _i64, _i64, _i, _i, _i, _vp, _vp]),
    "bigru_multilabel_counts": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "bigru_forward_windows": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _f, _i, _i, _u64, _vp, _vp, _vp, _vp, _vp]),
    "bigru_chunk_minmax": (_i, [_vp, _i64, _i, _i64, _i64, _vp, _vp, _vp]),
    "bigru_infer_window": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "bigru_infer_cluster_workspace_bytes": (_i, [_i, _i, _i, _i, _i, _i, C.POINTER(C.c_size_t)]),
    "bigru_infer_cluster": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "bigru_infer_cluster_geometry": (_i, [_i, _i, _i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "bigru_window_features": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, C.POINTER(_i), _i, C.POINTER(_i), _i, C.POINTER(_i), _i, _i, _f, _i,
                                   _f, _f, _vp, _vp, C.POINTER(_i), _vp]),
    "bigru_launch_count": (C.c_longlong, []),
    "bigru_prof_enable": (_i, [_i]),
    "bigru_prof_classes": (_i, []),
    "bigru_prof_class_name": (C.c_char_p, [_i]),
    "bigru_prof_report": (_i, [_i, C.POINTER(_d), C.POINTER(C.c_longlong), C.POINTER(_d), C.POINTER(_d)]),
}

_lib = None
_lock = threading.Lock()


def load():
    """Load (once) and return the ctypes handle.  Raises if the library is absent."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} is missing: build it with `python -m financial_market_data_analysis_b200.build` "
                    "(or __graft_entry__.build()). This package has no CPU/PyTorch fallback.")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)          # AttributeError here = header/library mismatch
                fn.restype, fn.argtypes = res, args
            _lib = lib
    return _lib


def check(rc: int, what: str):
    if rc == 0:
        return
    msg = load().bigru_last_error().decode("utf-8", "replace")
    if rc in (ERR_ARG, ERR_UNSUPPORTED):
        raise ValueError(f"{what}: {msg} (code {rc})")
    raise RuntimeError(f"{what}: {msg} (code {rc})")


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())
