"""ctypes binding of the C ABI declared in include/paradis_sl.h (and the bf16 entry points of
include/paradis_sl_bf16.h, include/paradis_geocyclic.h and include/paradis_sl_tl.h, each in a table of its own).

The product has no CPU fallback: if the shared library is missing this module
raises, it never substitutes another implementation.
"""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH

OK = 0
INTERP = {"bilinear": 1, "bicubic": 2}
MATH = {"fast": 0, "exact": 1}
MAX_DISP_ROWS = 126   # PARADIS_SL_MAX_DISP_ROWS
STATUS_NAMES = {
    0: "OK", 1: "BAD_SHAPE", 2: "ODD_WIDTH", 3: "BAD_INTERP", 4: "NULL_POINTER", 5: "WORKSPACE",
    6: "CUDA", 7: "DISPLACEMENT", 8: "NO_DEVICE",
}


class Geom(C.Structure):
    """struct paradis_sl_geom"""
    _fields_ = [("H", C.c_int32), ("W", C.c_int32),
                ("sin_lat", C.c_void_p), ("cos_lat", C.c_void_p), ("lon", C.c_void_p),
                ("min_lat", C.c_float), ("d_lat", C.c_float), ("min_lon", C.c_float), ("d_lon", C.c_float),
                ("own_row0", C.c_int32), ("own_rows", C.c_int32),
                ("arr_row0", C.c_int32), ("arr_rows", C.c_int32),
                ("fld_row0", C.c_int32), ("fld_rows", C.c_int32),
                ("fld_peer_lo", C.c_void_p), ("fld_peer_hi", C.c_void_p), ("fld_peer_rows", C.c_int32),
                ("arr_peer_lo", C.c_void_p * 3), ("arr_peer_hi", C.c_void_p * 3), ("arr_peer_rows", C.c_int32)]


_lib = None

_P = C.c_void_p
_PROTOS = {
    "paradis_sl_abi_version": (C.c_int, []),
    "paradis_last_error": (C.c_char_p, []),
    "paradis_geocyclic_pad_fwd": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.c_int, C.c_int, _P]),
    "paradis_geocyclic_pad_bwd": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.c_int, C.c_int, _P]),
    "paradis_geocyclic_dwconv_fwd": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "paradis_geocyclic_dwconv_bwd_input": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "paradis_geocyclic_dwconv_wgrad_workspace": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "paradis_geocyclic_dwconv_bwd_weight": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                      _P, C.c_size_t, _P]),
    "paradis_geocyclic_avgpool5_fwd": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "paradis_halo_pack": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "paradis_sl_advect_fwd_workspace": (C.c_size_t, [C.c_int, C.c_int]),
    "paradis_sl_advect_fwd": (C.c_int, [C.POINTER(Geom), _P, _P, _P, _P, C.c_int, C.c_int, C.c_int64, C.c_int64,
                                        C.c_int64, C.c_float, C.c_int, C.c_int, C.c_int, _P, C.c_size_t, _P, _P]),
    "paradis_sl_advect_bwd_workspace": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "paradis_sl_advect_bwd": (C.c_int, [C.POINTER(Geom), _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int64,
                                        C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_float, _P, C.c_size_t, _P, _P]),
    "paradis_sl_departure_coords": (C.c_int, [C.POINTER(Geom), _P, _P, _P, C.c_int, C.c_int, C.c_int64, C.c_int64,
                                              C.c_float, C.c_int, C.c_int, _P]),
    "paradis_sl_host_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "paradis_sl_advect_fwd_bwd_host": (C.c_int, [C.POINTER(Geom), _P, _P, _P, _P, _P, _P, _P, _P, C.c_int64,
                                                 C.c_float, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, _P, C.c_size_t]),
}


# include/paradis_sl_bf16.h: bf16 storage of field, u, v and their gradients (same ABI version: entry points added)
_PROTOS_BF16 = {
    "paradis_sl_advect_fwd_bf16": (C.c_int, [C.POINTER(Geom), _P, _P, _P, _P, C.c_int, C.c_int, C.c_int64, C.c_int64,
                                             C.c_int64, C.c_float, C.c_int, C.c_int, C.c_int, _P, C.c_size_t, _P, _P]),
    "paradis_sl_advect_bwd_bf16_workspace": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "paradis_sl_advect_bwd_bf16": (C.c_int, [C.POINTER(Geom), _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int64,
                                             C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_int, C.c_int, C.c_int,
                                             C.c_int, C.c_float, _P, C.c_size_t, _P, _P]),
}


# include/paradis_geocyclic.h: bf16 storage of the padding / depthwise-convolution / downsampling ops and the
# avgpool5 adjoint (same ABI version: entry points added)
_PROTOS_GEO = {
    "paradis_geocyclic_pad_fwd_bf16": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.c_int, C.c_int, _P]),
    "paradis_geocyclic_pad_bwd_bf16": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.c_int, C.c_int, _P]),
    "paradis_geocyclic_dwconv_fwd_bf16": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "paradis_geocyclic_dwconv_bwd_input_bf16": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                          _P]),
    "paradis_geocyclic_dwconv_bwd_weight_bf16": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int,
                                                           C.c_int, _P, C.c_size_t, _P]),
    "paradis_geocyclic_avgpool5_fwd_bf16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "paradis_geocyclic_avgpool5_bwd": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "paradis_geocyclic_avgpool5_bwd_bf16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
}


# include/paradis_sl_tl.h: tangent-linear model of the advection (same ABI version: entry points added)
_PROTOS_TL = {
    "paradis_sl_advect_jvp_workspace": (C.c_size_t, [C.c_int, C.c_int]),
    "paradis_sl_advect_jvp": (C.c_int, [C.POINTER(Geom), _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int64,
                                        C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_int,
                                        C.c_int, C.c_int, _P, C.c_size_t, _P, _P]),
}


def exported_symbols():
    """The functions of include/paradis_sl.h."""
    return list(_PROTOS)


def exported_symbols_bf16():
    """The functions of include/paradis_sl_bf16.h."""
    return list(_PROTOS_BF16)


def exported_symbols_geocyclic():
    """The functions of include/paradis_geocyclic.h."""
    return list(_PROTOS_GEO)


def exported_symbols_tl():
    """The functions of include/paradis_sl_tl.h."""
    return list(_PROTOS_TL)


def lib():
    """Load (once) and return the shared library; raise if it is not built."""
    global _lib
    if _lib is None:
        path = os.environ.get("PARADIS_SL_LIB", LIB_PATH)
        build_error = None
        if not os.path.exists(path) and path == LIB_PATH:
            try:                              # a fresh checkout: compile the CUDA sources once (nvcc, sm_100a)
                from .build import build_library
                build_library()
            except Exception as exc:          # no nvcc: fail loudly below
                build_error = exc
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} is missing: build it with `python -m paradis_model_b200.build` "
                "(nvcc, sm_100a). There is no CPU or PyTorch fallback for this operator."
                + (f"\nThe automatic build failed: {build_error}" if build_error is not None else ""))
        if path == LIB_PATH:
            try:                              # never rebuilt behind the caller's back, but never silently stale either
                from .build import is_stale
                if is_stale():
                    import warnings
                    warnings.warn(f"{path} is older than its CUDA sources: rebuild with `python -m paradis_model_b200.build`")
            except Exception:
                pass
        handle = C.CDLL(path)
        for name, (res, args) in (list(_PROTOS.items()) + list(_PROTOS_BF16.items()) + list(_PROTOS_GEO.items())
                           + list(_PROTOS_TL.items())):
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        if handle.paradis_sl_abi_version() != 2 and not os.environ.get("PARADIS_SL_SKIP_ABI_CHECK"):
            raise RuntimeError("libparadis_sl.so ABI version mismatch")
        _lib = handle
    return _lib


def check(rc: int, what: str):
    if rc != OK:
        msg = lib().paradis_last_error().decode()
        raise RuntimeError(f"{what} failed [{STATUS_NAMES.get(rc, rc)}]: {msg}")
