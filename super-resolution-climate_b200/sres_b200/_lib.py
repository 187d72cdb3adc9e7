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


class ChainArgs(C.Structure):
    """sres_rcab_chain_args (include/sres_b200.h)."""
    _fields_ = [
        ("xb_bf16", C.c_void_p), ("t1_bf16", C.c_void_p), ("t2_bf16", C.c_void_p),
        ("wpack_bf16", C.c_void_p), ("params", C.c_void_p), ("x_in_f32", C.c_void_p), ("x_f32", C.c_void_p),
        ("save_mean", C.c_void_p), ("save_s", C.c_void_p), ("scratch", C.c_void_p),
        ("rcab_stride", C.c_int64), ("save_stride", C.c_int64),
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("n_blocks", C.c_int32), ("hidden", C.c_int32),
        ("xb_first", C.c_int32), ("xb_ring", C.c_int32), ("xb_count", C.c_int32),
        ("t_first", C.c_int32), ("t_fixed", C.c_int32), ("t_count", C.c_int32),
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
        L.sres_rcab_chain_scratch_bytes.restype = C.c_size_t
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
