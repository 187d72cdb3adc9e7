"""ctypes binding of libsres_b200.so (the C ABI declared in include/sres_b200.h).

There is deliberately no fallback: if the library is missing or a call fails, an exception is
raised.  Nothing here imports the oracle.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "..", "lib", "libsres_b200.so")

SRES_OK = 0
EPI_RELU = 1
EPI_POOL = 2
EPI_DOT = 4
MAP_IDENT, MAP_SHUFFLE, MAP_UNSHUFFLE = 0, 1, 2
# SRES_RESIZE_* of include/sres_b200.h, keyed by F.interpolate's mode names
RESIZE_MODES = {"nearest": 0, "nearest-exact": 1, "bilinear": 2, "bicubic": 3, "area": 4}


class SresError(RuntimeError):
    pass


class ConvArgs(C.Structure):
    _fields_ = [
        ("in_bf16", C.c_void_p),
        ("wpack_bf16", C.c_void_p),
        ("bias", C.c_void_p),
        ("resid_f32", C.c_void_p),
        ("resid2_f32", C.c_void_p),
        ("mask_bf16", C.c_void_p),
        ("out_f32", C.c_void_p),
        ("out_bf16", C.c_void_p),
        ("pool_part", C.c_void_p),
        ("out_nchw", C.c_void_p),
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("n_out", C.c_int32), ("c_real", C.c_int32),
        ("epi_flags", C.c_uint32),
        ("map_mode", C.c_int32), ("sub_i", C.c_int32), ("sub_j", C.c_int32),
        ("shuffle_factor", C.c_int32),
        ("debug_flags", C.c_int32),
        ("debug_timeline", C.c_void_p),
    ]


class WgradJob(C.Structure):
    """sres_wgrad_job (include/sres_b200.h)."""
    _fields_ = [
        ("x_bf16", C.c_void_p), ("dy_bf16", C.c_void_p), ("dw_oihw", C.c_void_p), ("dbias", C.c_void_p),
        ("cout_total", C.c_int32), ("oc_stride", C.c_int32), ("oc_offset", C.c_int32), ("accumulate", C.c_int32),
        ("scale", C.c_float),
    ]


_lib = None


def lib():
    """Load the shared library once; raise loudly when it has not been built."""
    global _lib
    if _lib is None:
        path = os.path.abspath(LIB_PATH)
        if not os.path.exists(path):
            raise SresError(
                f"{path} not found: build it with `python super-resolution-climate_b200/build.py` "
                "(there is no CPU / PyTorch fallback for the RCAN hot path)")
        L = C.CDLL(path)
        L.sres_last_error.restype = C.c_char_p
        L.sres_ptl_rows.restype = C.c_int64
        L.sres_launch_count.restype = C.c_longlong
        L.sres_resize.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                                  C.c_double, C.c_int, C.c_void_p]
        L.sres_resize.restype = C.c_int
        _lib = L
    return _lib


def check(status, what=""):
    if status != SRES_OK:
        msg = lib().sres_last_error().decode("utf-8", "replace")
        raise SresError(f"{what} failed with status {status}: {msg}")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def cur_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
