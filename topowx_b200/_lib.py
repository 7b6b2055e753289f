"""ctypes binding of libtwxi.so (include/twxi.h).  There is no fallback: if the CUDA library is missing or
fails to load, importing this module raises."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TWXI_LIB") or os.path.join(HERE, "libtwxi.so")   # TWXI_LIB: instrumented developer builds

MEM_HOST, MEM_DEVICE = 0, 1
ST_OK, ST_NO_NNGHS, ST_NO_VARIO, ST_TOO_FEW_STNS, ST_SINGULAR, ST_FIXER_EMPTY, ST_CLIMDIV, ST_KNN_TIES, ST_LIMIT = range(9)
ST_MASKED = 255
FILL_I2, FILL_I4 = -32767, -2147483647
FILL_F4 = np.float32(9.969209968386869e+36)
FILL_F8 = 9.969209968386869e+36
INIT_NNGHS, MAX_NNGHS, MAX_STNS, MAX_RM, MAX_KRIG_NNGHS = 100, 255, 24000, 4, 168

# messages of the reference exceptions (interp_tair.py:252,829,843,192; station_select.py:164)
STATUS_MESSAGES = {
    ST_NO_NNGHS: "Cannot determine the optimal # of neighbors to use!",
    ST_NO_VARIO: "Cannot determine variogram params!",
    ST_TOO_FEW_STNS: "index out of bounds: not enough candidate stations for the requested # of neighbors",
    ST_SINGULAR: "singular or non-finite kriging/GWR system",
    ST_FIXER_EMPTY: "No valid tmin/tmax in window",
    ST_CLIMDIV: "climate division not found in station database",
    ST_KNN_TIES: "too many exact distance ties",
    ST_LIMIT: "neighbour count exceeds the kriging kernel's limit (%d)" % MAX_KRIG_NNGHS,
}


class TwxiError(RuntimeError):
    pass


class Points(C.Structure):
    _fields_ = [("npts", C.c_int32), ("lat", C.c_void_p), ("lon", C.c_void_p), ("elev", C.c_void_p),
                ("tdi", C.c_void_p), ("lst", C.c_void_p), ("rm_idx", C.c_void_p), ("n_rm", C.c_int32),
                ("rm_zero_dist", C.c_int32)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s not found: build it with `python -m topowx_b200.build` (needs nvcc). "
                          "topowx_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    sig = {
        "twxi_version": (C.c_int, []),
        "twxi_last_error": (C.c_char_p, []),
        "twxi_launch_count": (i64, [i32]),
        "twxi_set_stage_timing": (i32, [i32]),
        "twxi_get_stage_ms": (i32, [vp]),
        "twxi_get_ked_kernel_ms": (i32, [vp]),
        "twxi_ctx_create": (i32, [C.POINTER(vp), i32, i32] + [vp] * 11),
        "twxi_ctx_set_obs": (i32, [vp, vp, i32, vp, vp]),
        "twxi_ctx_set_climdivs": (i32, [vp, vp, i32]),
        "twxi_ctx_set_stream": (i32, [vp, vp]),
        "twxi_ctx_destroy": (i32, [vp]),
        "twxi_ctx_stat": (i32, [vp, i32, vp]),
        "twxi_ctx_n_stns": (i32, [vp]),
        "twxi_ctx_n_days": (i32, [vp]),
        "twxi_knn": (i32, [vp, i32, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, i32]),
        "twxi_nngh_params": (i32, [vp, C.POINTER(Points), vp, vp, vp, vp, i32]),
        "twxi_krig": (i32, [vp, C.POINTER(Points), i32, vp, vp, vp, vp, vp, i32]),
        "twxi_fit_vario": (i32, [vp, C.POINTER(Points), i32, vp, vp, vp, i32]),
        "twxi_krig_all": (i32, [vp, C.POINTER(Points), vp, vp, vp, vp, vp, i32]),
        "twxi_gwr_hat": (i32, [vp, C.POINTER(Points), i32, vp, i32, vp, vp, vp, vp, i32]),
        "twxi_gwr_mth": (i32, [vp, C.POINTER(Points), i32, vp, vp, vp, vp, i32]),
        "twxi_xval_anom": (i32, [vp, i32, vp, i32, vp, vp, vp, vp, vp, i32]),
        "twxi_interp_points": (i32, [vp, C.POINTER(Points), vp, vp, vp, vp, vp, i32]),
        "twxi_interp_cells": (i32, [vp, vp, i32] + [vp] * 9 + [i32, i32, i32] + [vp] * 8 + [i32]),
        "twxi_interp_chunk": (i32, [vp, vp, vp, i32, i32] + [vp] * 8 + [i32]),
        "twxi_interp_chunk_async": (i32, [vp, vp, vp, i32, i32] + [vp] * 8 + [i32]),
        "twxi_interp_chunk_wait": (i32, [vp, i32]),
        "twxi_tile_begin": (i32, [vp, vp, vp, i32, i32, i32]),
        "twxi_tile_days": (i32, [vp, vp, i32, vp, vp, i32]),
        "twxi_tile_days_mth": (i32, [vp, vp, i32, vp, vp, i32, vp, vp, vp, i32]),
        "twxi_tile_end": (i32, [vp, vp] + [vp] * 6 + [i32]),
        "twxi_measure_fp64_peak": (i32, [i32, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib, sorted(sig)


lib, EXPORTED = _load()


def check(rc):
    if rc != 0:
        raise TwxiError("libtwxi error %d: %s" % (rc, lib.twxi_last_error().decode()))


def ptr(a):
    """void* of a numpy array, a torch tensor (host or CUDA) or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        if not a.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):
        if not a.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return C.c_void_p(a.data_ptr())
    raise TypeError("expected numpy array or torch tensor, got %r" % type(a))


def is_device(a):
    return hasattr(a, "is_cuda") and a.is_cuda
