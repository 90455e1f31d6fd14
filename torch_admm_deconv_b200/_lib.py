"""ctypes binding of libadmm_b200.so (C ABI in include/admm_b200.h).

There is deliberately no fallback: if the shared library is missing or does not export a symbol the
header declares, importing the operators fails loudly.
"""
from __future__ import annotations

import ctypes
import os

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# ADMM_B200_LIB: an alternative build of the same library (kernel-tuning experiments); never a different implementation
LIB_PATH = os.environ.get("ADMM_B200_LIB") or os.path.join(_PKG_DIR, "libadmm_b200.so")

_vp, _i, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t

# name -> (restype, argtypes); must list every symbol of include/admm_b200.h
SIGNATURES = {
    "admm_version": (_i, []),
    "admm_last_error": (ctypes.c_char_p, []),
    "admm_set_option": (_i, [ctypes.c_char_p, _i]),
    "admm_get_option": (_i, [ctypes.c_char_p, ctypes.POINTER(_i)]),
    "admm_query_workspace": (_sz, [_i] * 6),
    "admm_query_workspace_backward": (_sz, [_i] * 6),
    "admm_query_saved": (_sz, [_i] * 6),
    "admm_tv_forward": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp, _sz, _vp]),
    "admm_tv_backward": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp, _sz,
                              _vp, _vp, _vp, _vp, _vp]),
    "admm_profile_reset": (_i, []),
    "admm_profile_read": (_i, [_i, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(_i)]),
    "admm_launch_count": (ctypes.c_longlong, []),
    "admm_dbg_rows_r2c": (_i, [_vp, _vp, _i, _i, _i, _vp, _sz, _vp]),
    "admm_dbg_rows_c2r": (_i, [_vp, _vp, _i, _i, _i, _vp, _sz, _vp]),
    "admm_dbg_cols_fft": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _sz, _vp]),
}

class AdmmExt(ctypes.Structure):
    """`admm_ext` of include/admm_b200.h (fused layer prologue / epilogue, output placement, shared spectrum)."""
    _fields_ = [("struct_size", _i), ("in_dtype", _i), ("activation", _i), ("ckpt_interval", _i),
                ("out_batch_stride", ctypes.c_longlong), ("yhat_in", _vp), ("yhat_out", _vp),
                ("resid", _vp), ("resid_every", _i), ("rtol", ctypes.c_float), ("atol", ctypes.c_float),
                ("host_flag", _vp), ("iters_out", _vp)]


IN_F32, IN_U8_DIV255 = 0, 1
ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_TANH = 0, 1, 2, 3

SIGNATURES["admm_query_yhat"] = (_sz, [_i] * 3)
SIGNATURES["admm_query_resid"] = (_sz, [_i] * 6)
SIGNATURES["admm_query_saved_ex"] = (_sz, [_i] * 7)
SIGNATURES["admm_query_workspace_backward_ex"] = (_sz, [_i] * 7)
SIGNATURES["admm_tv_backward_ex"] = (_i, SIGNATURES["admm_tv_backward"][1] + [_i])
SIGNATURES["admm_spectrum_forward"] = (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _sz, _vp])
SIGNATURES["admm_tv_forward_ex"] = (_i, SIGNATURES["admm_tv_forward"][1] + [ctypes.POINTER(AdmmExt)])
# float64 solve: the float32 calls with double tensors (admm_tv_forward_f64 has no bias argument)
SIGNATURES["admm_query_workspace_f64"] = (_sz, [_i] * 6)
SIGNATURES["admm_query_workspace_backward_f64"] = (_sz, [_i] * 6)
SIGNATURES["admm_query_saved_f64"] = (_sz, [_i] * 6)
SIGNATURES["admm_tv_forward_f64"] = (_i, [_vp, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp, _sz, _vp])
SIGNATURES["admm_tv_backward_f64"] = SIGNATURES["admm_tv_backward"]

_lib = None


class AdmmLibraryError(RuntimeError):
    pass


def load():
    """Load (once) and return the ctypes handle; raises if the CUDA library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AdmmLibraryError(
            "libadmm_b200.so not found at %s -- build it with `python -m torch_admm_deconv_b200.build` "
            "(there is no CPU or PyTorch fallback for this path)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:  # pragma: no cover
            raise AdmmLibraryError("libadmm_b200.so does not export %s" % name) from e
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    msg = load().admm_last_error()
    return msg.decode() if msg else ""


def check(status, what):
    if status != 0:
        msg = last_error()
        if status == 1:
            raise ValueError("%s: %s" % (what, msg))
        raise RuntimeError("%s failed (status %d): %s" % (what, status, msg))


def set_option(key, value):
    if load().admm_set_option(key.encode(), int(value)) != 0:
        raise KeyError("unknown or invalid option %s=%r" % (key, value))


def get_option(key):
    v = ctypes.c_int(0)
    if load().admm_get_option(key.encode(), ctypes.byref(v)) != 0:
        raise KeyError(key)
    return v.value


def profile_reset():
    load().admm_profile_reset()


def profile_read(kind):
    """(total_ms, launches) of kernel class `kind` (0 rows, 1 cols, 2 other) since the last reset."""
    ms = ctypes.c_double(0.0)
    n = ctypes.c_int(0)
    check(load().admm_profile_read(int(kind), ctypes.byref(ms), ctypes.byref(n)), "admm_profile_read")
    return ms.value, n.value


def launch_count():
    return int(load().admm_launch_count())
