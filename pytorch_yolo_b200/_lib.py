"""ctypes binding of the C-ABI library (``include/yolo_b200.h``).

There is no fallback: if ``libyolo_b200.so`` is missing it is built with nvcc, and if that is
impossible the import of any compute entry point raises.  Nothing here touches the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

MAX_SCALES = 4
MAX_ANCHORS = 8
DET_COLS = 7


class Scale(C.Structure):
    """``yolo_b200_scale``"""
    _fields_ = [("head", C.c_void_p), ("ny", C.c_int32), ("nx", C.c_int32), ("na", C.c_int32),
                ("row_off", C.c_int32), ("stride", C.c_float), ("anchor_vec", (C.c_float * 2) * MAX_ANCHORS)]


class Head(C.Structure):
    """``yolo_b200_head``"""
    _fields_ = [("x", C.c_void_p), ("weight", C.c_void_p), ("bias_host", C.POINTER(C.c_float)), ("head_out", C.c_void_p),
                ("c_in", C.c_int32), ("x_row_pitch", C.c_int32), ("negative_slope", C.c_float), ("scale", Scale)]


class NmsOpts(C.Structure):
    """``yolo_b200_nms_opts``"""
    _fields_ = [("flags", C.c_int32), ("seg_warps_per_sm", C.c_int32), ("step_seq", C.c_void_p), ("step_stamp", C.c_void_p)]


class TargetLayer(C.Structure):
    """``yolo_b200_target_layer``"""
    _fields_ = [("nx", C.c_int32), ("ny", C.c_int32), ("na", C.c_int32), ("reserved", C.c_int32),
                ("anchor_vec", (C.c_float * 2) * MAX_ANCHORS),
                ("b", C.c_void_p), ("a", C.c_void_p), ("gj", C.c_void_p), ("gi", C.c_void_p), ("tcls", C.c_void_p),
                ("txy", C.c_void_p), ("twh", C.c_void_p)]


ABI_VERSION = 3
E_UNSUPPORTED = -5
VARIANT_ACCUMULATE = 0x100
VARIANT_F16 = 0x200
VARIANT_BF16 = 0x400
HEAD_ACCUMULATE = 1
HEAD_FP32X3 = 8
HEAD_NO_CANDIDATES = 2


class YoloB200Error(RuntimeError):
    pass


_lock = threading.Lock()
_lib = None

_SIGNATURES = {
    "yolo_b200_abi_version": (C.c_int, []),
    "yolo_b200_error_string": (C.c_char_p, [C.c_int]),
    "yolo_b200_decode_dense": (C.c_int, [C.POINTER(Scale), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "yolo_b200_decode_dense_ex": (C.c_int, [C.POINTER(Scale), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "yolo_b200_decode_compact": (C.c_int, [C.POINTER(Scale), C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                                           C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "yolo_b200_decode_compact_ex": (C.c_int, [C.POINTER(Scale), C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                                              C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "yolo_b200_compact_from_dense": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int,
                                               C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "yolo_b200_pad_planes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_void_p]),
    "yolo_b200_head_supported": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "yolo_b200_head_supported_ex": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "yolo_b200_head_decode_compact": (C.c_int, [C.POINTER(Head), C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                                                C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "yolo_b200_nms_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "yolo_b200_nms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "yolo_b200_nms_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(NmsOpts),
                                   C.c_void_p]),
    "yolo_b200_build_targets": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(TargetLayer), C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
    "yolo_b200_flag_wait": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_void_p]),
    "yolo_b200_flag_post": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "yolo_b200_scale_coords": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, C.c_void_p]),
    "yolo_b200_scale_detections": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "yolo_b200_peer_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "yolo_b200_peer_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "yolo_b200_peer_close": (C.c_int, [C.c_void_p]),
    "yolo_b200_device_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "yolo_b200_device_free": (C.c_int, [C.c_void_p]),
}


def lib_path() -> str:
    # YOLO_B200_LIB selects an alternative build of the same library (kernel tuning experiments only)
    return os.environ.get("YOLO_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libyolo_b200.so")


def load():
    """Load (building first if needed) the shared library and declare every prototype."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = lib_path()
        if not os.environ.get("YOLO_B200_LIB"):
            from . import build as _build
            _build.build()       # returns at once unless a source / header changed since the library was built (content hash)
        lib = C.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError here = header and library disagree
            fn.restype = res
            fn.argtypes = args
        if lib.yolo_b200_abi_version() != ABI_VERSION:
            raise YoloB200Error("libyolo_b200.so ABI version mismatch; rebuild with python -m pytorch_yolo_b200.build --force")
        _lib = lib
        return lib


def exported_symbols():
    return list(_SIGNATURES)


def check(code: int, what: str) -> None:
    if code != 0:
        msg = load().yolo_b200_error_string(code).decode()
        raise YoloB200Error(f"{what} failed: {msg} (code {code})")
