"""ctypes binding of libfmgpu.so (include/fm_gpu.h).  No CPU fallback: a missing library or a
missing CUDA device raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libfmgpu.so")


class FmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libfmgpu error {code}: {msg}")
        self.code = code


class fm_config(C.Structure):
    _fields_ = [
        ("device", C.c_int32), ("n_streams", C.c_int32), ("frame_width", C.c_int32),
        ("frame_height", C.c_int32), ("max_frames", C.c_int32), ("fps", C.c_int32),
        ("box_size", C.c_int32), ("min_box_scale", C.c_int32), ("blur_scale", C.c_int32),
        ("threshold", C.c_int32), ("avg", C.c_double), ("min_time", C.c_double),
        ("cache_time", C.c_double), ("max_components", C.c_int32), ("flags", C.c_int32),
    ]


class fm_info(C.Structure):
    _fields_ = [
        ("proc_width", C.c_int32), ("proc_height", C.c_int32), ("gaussian", C.c_int32),
        ("min_area", C.c_int32), ("max_area", C.c_int32), ("cache_frames", C.c_int32),
        ("min_movement_frames", C.c_int32), ("words_per_row", C.c_int32), ("scale", C.c_double),
        ("front_end", C.c_int32), ("max_components", C.c_int32),
    ]


class fm_frame_stats(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_contours", "n_counted", "movement", "movement_counter",
                                         "movement_decay", "cache_len", "wrote", "n_flush")]


class fm_component(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("area_x2", "x", "y", "w", "h")]


class fm_rows_plan_info(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("usable", "band_rows", "box_rows", "chunk_cols", "seg_cols", "box_bytes",
                                         "smem_bytes", "bands", "segs", "max_groups")]


FLAG_KEEP_PLANES = 1
FLAG_NO_FUSED = 2
FLAG_NO_UMMA = 8
FLAG_UMMA_APRON = 16
FLAG_UMMA = 32
FLAG_NO_ROWS = 64
FLAG_UPSCALE = 128
FLAG_DEVICE_CLIPS = 256
FLAG_NV12 = 512
FLAG_OBJECT_PLANES = 1024
OBJECT_WIDTH = 300

# every symbol include/fm_gpu.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "fm_last_error": (C.c_char_p, []),
    "fm_version": (C.c_int, []),
    "fm_ctx_create": (C.c_int, [C.POINTER(fm_config), C.POINTER(_P)]),
    "fm_ctx_destroy": (C.c_int, [_P]),
    "fm_ctx_info": (C.c_int, [_P, C.POINTER(fm_info)]),
    "fm_ctx_set_masks": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "fm_ctx_reset": (C.c_int, [_P, C.c_int]),
    "fm_process": (C.c_int, [_P, _P, C.c_size_t, C.c_size_t, C.c_int, _P, _P]),
    "fm_process_ragged": (C.c_int, [_P, _P, C.c_size_t, C.c_size_t, C.c_int, _P, _P, _P]),
    "fm_process_clip": (C.c_int, [_P, _P, C.c_size_t, C.c_size_t, C.c_int, _P, _P, _P, _P, C.c_size_t, C.c_int]),
    "fm_object_planes": (C.c_int, [_P, _P, _P, C.c_size_t, C.c_int]),
    "fm_process_host": (C.c_int, [_P, _P, C.c_size_t, C.c_size_t, C.c_int, _P]),
    "fm_submit_host": (C.c_int, [_P, C.c_int, _P, C.c_size_t, C.c_size_t, C.c_int, _P]),
    "fm_wait": (C.c_int, [_P, C.c_int, _P]),
    "fm_submit_reset": (C.c_int, [_P, C.c_int]),
    "fm_host_alloc": (C.c_int, [C.c_int, C.c_size_t, C.POINTER(_P), C.POINTER(C.c_int)]),
    "fm_host_free": (C.c_int, [_P]),
    "fm_ctx_check": (C.c_int, [_P]),
    "fm_get_components": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.POINTER(fm_component), C.POINTER(C.c_int)]),
    "fm_debug_planes": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P]),
    "fm_debug_mask": (C.c_int, [_P, C.c_int, _P]),
    "fm_debug_components": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, C.c_int, C.POINTER(fm_component), C.POINTER(C.c_int)]),
    "fm_resize_area": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, C.c_int, _P, C.POINTER(C.c_int)]),
    "fm_debug_rows_plan": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(fm_rows_plan_info)]),
    "fm_launch_count": (C.c_uint64, []),
    "fm_timing_enable": (C.c_int, [_P, C.c_int]),
    "fm_timing_reset": (C.c_int, [_P]),
    "fm_timing_get": (C.c_int, [_P, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
}

_lib = None


def load():
    """Load libfmgpu.so (built in-tree by find_motion_b200/build.py) and bind every symbol."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FmError(-2, f"{LIB_PATH} is missing: run `python -m find_motion_b200.build` "
                          "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)       # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise FmError(rc, (load().fm_last_error() or b"").decode("utf-8", "replace"))
