"""ctypes loader for libssimu2_b200.so (the C ABI of include/ssimu2_b200.h).

The product path has no CPU fallback: if the shared library is missing or cannot be loaded
this module raises, and every scorer call fails with the library's error code when no
sm_100 device is present.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libssimu2_b200.so")


class Frame(C.Structure):
    """ssimu2_frame: one device (or host) frame; pitch in bytes."""
    _fields_ = [("plane", C.c_uint64 * 2), ("pitch", C.c_uint32), ("reserved", C.c_uint32)]


class Config(C.Structure):
    """ssimu2_config"""
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("format", C.c_int32),
                ("matrix", C.c_int32), ("full_range", C.c_int32), ("device", C.c_int32),
                ("batch", C.c_uint32), ("ring", C.c_uint32), ("pipeline", C.c_uint32), ("flags", C.c_uint32),
                ("input_group", C.c_uint32), ("reserved", C.c_uint32 * 5)]


class Source(C.Structure):
    """ssimu2_source: the description of the distorted frames of a mixed handle (ssimu2_create_mixed).  `width` and `height`
    (the distorted frames' size, 0 = the reference's) are the C struct's first two of the four words `reserved` views."""
    _fields_ = [("format", C.c_int32), ("matrix", C.c_int32), ("full_range", C.c_int32), ("flags", C.c_uint32),
                ("reserved", C.c_uint32 * 4)]

    @property
    def width(self) -> int:
        return self.reserved[0]

    @width.setter
    def width(self, v: int):
        self.reserved[0] = v

    @property
    def height(self) -> int:
        return self.reserved[1]

    @height.setter
    def height(self, v: int):
        self.reserved[1] = v


PIPELINE_DEFAULT, PIPELINE_SPLIT = 0, 1
FLAG_SCORE_ONLY, FLAG_NO_TIMING, FLAG_P016_DEEP = 1, 2, 4


class Info(C.Structure):
    """ssimu2_info"""
    _fields_ = [("nscales", C.c_uint32), ("width", C.c_uint32 * 6), ("height", C.c_uint32 * 6),
                ("pitch", C.c_uint32 * 6), ("batch", C.c_uint32), ("ring", C.c_uint32),
                ("alg_bytes_per_pair", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("pipeline", C.c_uint32), ("flags", C.c_uint32), ("input_group", C.c_uint32),
                ("strips_per_pair", C.c_uint32), ("io_bytes_per_pair", C.c_uint64)]


# every symbol include/ssimu2_b200.h and include/ssimu2_b200_debug.h declare: name -> (restype, argtypes)
_P = C.c_void_p
_FP = C.POINTER(Frame)
SYMBOLS = {
    "ssimu2_create": (C.c_int, [C.POINTER(_P), C.POINTER(Config)]),
    "ssimu2_create_mixed": (C.c_int, [C.POINTER(_P), C.POINTER(Config), C.POINTER(Source)]),
    "ssimu2_destroy": (C.c_int, [_P]),
    "ssimu2_mem_usage": (C.c_int, [_P, C.POINTER(C.c_size_t)]),
    "ssimu2_strerror": (C.c_char_p, [C.c_int]),
    "ssimu2_version": (C.c_uint32, []),
    "ssimu2_submit": (C.c_int, [_P, _FP, _FP, _P, C.POINTER(C.c_uint64)]),
    "ssimu2_submit_batch": (C.c_int, [_P, C.c_uint32, _FP, _FP, _P, C.POINTER(C.c_uint64)]),
    "ssimu2_flush": (C.c_int, [_P]),
    "ssimu2_wait": (C.c_int, [_P, C.c_uint64]),
    "ssimu2_completed": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "ssimu2_get_score": (C.c_int, [_P, C.c_uint64, C.POINTER(C.c_double)]),
    "ssimu2_get_scores": (C.c_int, [_P, C.c_uint64, C.c_uint32, C.POINTER(C.c_double)]),
    "ssimu2_get_norms": (C.c_int, [_P, C.c_uint64, C.POINTER(C.c_double)]),
    "ssimu2_compute_sync": (C.c_int, [_P, _FP, _FP, _P, C.POINTER(C.c_double)]),
    "ssimu2_stream_wait": (C.c_int, [_P, C.c_uint64, _P]),
    "ssimu2_stream_wait_input": (C.c_int, [_P, C.c_uint64, _P]),
    "ssimu2_submit_host": (C.c_int, [_P, _FP, _FP, C.c_size_t, C.POINTER(C.c_uint64)]),
    "ssimu2_submit_host_batch": (C.c_int, [_P, C.c_uint32, _FP, _FP, C.c_size_t, C.POINTER(C.c_uint64)]),
    "ssimu2_submit_host_sized": (C.c_int, [_P, C.c_uint32, _FP, C.c_size_t, _FP, C.c_size_t, C.POINTER(C.c_uint64)]),
    "ssimu2_scores_device": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "ssimu2_get_info": (C.c_int, [_P, C.POINTER(Info)]),
    "ssimu2_debug_read": (C.c_int, [_P, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_float), C.c_size_t]),
    "ssimu2_debug_read_partials": (C.c_int, [_P, C.c_uint64, C.POINTER(C.c_double), C.c_size_t]),
    "ssimu2_debug_strips": (C.c_int, [_P, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "ssimu2_debug_math":(C.c_int, [C.c_int, C.POINTER(C.c_float), C.c_float, C.POINTER(C.c_float), C.c_size_t]),
    "ssimu2_last_batch_ms": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "ssimu2_kernel_ms": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_int]),
    "ssimu2_shard_create": (C.c_int, [C.POINTER(_P), C.POINTER(Config), C.POINTER(C.c_int32), C.c_uint32]),
    "ssimu2_shard_create_mixed": (C.c_int, [C.POINTER(_P), C.POINTER(Config), C.POINTER(Source), C.POINTER(C.c_int32),
                                            C.c_uint32]),
    "ssimu2_shard_destroy": (C.c_int, [_P]),
    "ssimu2_shard_submit_host": (C.c_int, [_P, C.c_uint32, _FP, _FP, C.c_size_t, C.POINTER(C.c_uint64)]),
    "ssimu2_shard_submit_host_sized": (C.c_int, [_P, C.c_uint32, _FP, C.c_size_t, _FP, C.c_size_t, C.POINTER(C.c_uint64)]),
    "ssimu2_shard_submit_device": (C.c_int, [_P, C.c_uint32, _FP, _FP, C.POINTER(_P), C.POINTER(C.c_uint64)]),
    "ssimu2_shard_device_of": (C.c_int, [_P, C.c_uint64, C.POINTER(C.c_int32)]),
    "ssimu2_shard_get_scores": (C.c_int, [_P, C.c_uint64, C.c_uint32, C.POINTER(C.c_double)]),
    "ssimu2_shard_flush": (C.c_int, [_P]),
}

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)")
        l = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


class Ssimu2Error(RuntimeError):
    def __init__(self, status: int, where: str):
        self.status = status
        msg = lib().ssimu2_strerror(status)
        super().__init__(f"{where}: {msg.decode() if msg else status} ({status})")


def check(status: int, where: str) -> None:
    if status != 0:
        raise Ssimu2Error(status, where)
