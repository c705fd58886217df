"""ctypes binding of libbgsb200.so (include/bgsb200.h) -- the only way Python reaches the kernels.

There is no fallback: if the shared library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbgsb200.so")

OK, ERR_ARG, ERR_CUDA, ERR_STATE, ERR_CAPACITY = 0, 1, 2, 3, 4
ALGO_FRAME_DIFFERENCE, ALGO_WEIGHTED_MOVING_VARIANCE, ALGO_MOG2, ALGO_ADAPTIVE_BG_LEARNING = 0, 3, 5, 6
ALGO_STATIC_FRAME_DIFFERENCE, ALGO_WEIGHTED_MOVING_MEAN = 1, 2        # sibling plugins (SURVEY 8f N3)
ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING = 7
ALGO_DP_ZIVKOVIC_AGMM = 11
ALGO_DP_ADAPTIVE_MEDIAN, ALGO_DP_MEAN, ALGO_DP_WREN_GA = 9, 12, 13     # the DP package's simple per-pixel models
ALGO_DP_PRATI_MEDIOD = 14
ALGO_SIGMA_DELTA = 35
MORPH_ERODE, MORPH_DILATE = 0, 1
POOL_MASKS, POOL_DETECT = 1, 2
INPUT_BGR, INPUT_NV12, INPUT_I420 = 0, 1, 2                            # "inputFormat" (BGSB_INPUT_*)


class BgsbError(RuntimeError):
    def __init__(self, code, text):
        super().__init__("bgsb200 error %d: %s" % (code, text))
        self.code = code


class Component(C.Structure):
    _fields_ = [("label", C.c_int32), ("first_index", C.c_int32), ("x", C.c_int32), ("y", C.c_int32),
                ("w", C.c_int32), ("h", C.c_int32), ("area", C.c_int32), ("external", C.c_int32)]


class Trace(C.Structure):
    _fields_ = [("frame", C.c_int64), ("wall_ms", C.c_double), ("upload_ms", C.c_double), ("kernel_ms", C.c_double),
                ("download_ms", C.c_double), ("bands", C.c_int)]


class Blob(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("w", C.c_float), ("h", C.c_float), ("id", C.c_int32)]


u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int32)
f32p = C.POINTER(C.c_float)
intp = C.POINTER(C.c_int)
vp = C.c_void_p

# name -> (restype, argtypes); every symbol include/bgsb200.h declares
SIGNATURES = {
    "bgsb_last_error": (C.c_char_p, []),
    "bgsb_version": (C.c_char_p, []),
    "bgsb_device_count": (C.c_int, [intp]),
    "bgsb_kernel_launch_count": (C.c_uint64, []),
    "bgsb_copy_probe": (C.c_int, [C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                  C.POINTER(C.c_double)]),
    "bgsb_host_alloc": (C.c_int, [C.POINTER(vp), C.c_size_t, C.c_int]),
    "bgsb_host_free": (None, [vp]),
    "bgsb_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int]),
    "bgsb_create_group": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int]),
    "bgsb_destroy": (None, [vp]),
    "bgsb_reset": (C.c_int, [vp]),
    "bgsb_set_param": (C.c_int, [vp, C.c_char_p, C.c_double]),
    "bgsb_get_param": (C.c_int, [vp, C.c_char_p, C.POINTER(C.c_double)]),
    "bgsb_process": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_size_t, vp, C.c_size_t, vp, C.c_size_t, intp, intp]),
    "bgsb_submit": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_size_t, vp, C.c_size_t, vp, C.c_size_t, intp, intp]),
    "bgsb_wait": (C.c_int, [vp]),
    "bgsb_process_fanout": (C.c_int, [C.POINTER(vp), C.c_int, vp, C.c_int, C.c_int, C.c_size_t, C.POINTER(vp),
                                      C.POINTER(C.c_size_t), C.POINTER(vp), C.POINTER(C.c_size_t), intp, intp]),
    "bgsb_process_dev": (C.c_int, [vp, vp, C.c_int, C.c_int, vp, vp, intp, intp, vp]),
    "bgsb_process_batch_dev": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, intp, intp, vp]),
    "bgsb_trace_last": (C.c_int, [vp, C.POINTER(Trace)]),
    "bgsb_frame_count": (C.c_int, [vp, C.POINTER(C.c_int64)]),
    "bgsb_state_bytes": (C.c_int, [vp, C.POINTER(C.c_size_t)]),
    "bgsb_mog2_export_state": (C.c_int, [vp, C.c_int, f32p, u8p]),
    "bgsb_mog2_import_state": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int64, f32p, u8p]),
    "bgsb_morph_dev": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, intp, C.c_int, vp, vp]),
    "bgsb_morph": (C.c_int, [vp, C.c_int, C.c_int, C.c_size_t, intp, C.c_int, vp, C.c_size_t]),
    "bgsb_ccl_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int]),
    "bgsb_ccl_create_batch": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int]),
    "bgsb_ccl_destroy": (None, [vp]),
    "bgsb_ccl_set_param": (C.c_int, [vp, C.c_char_p, C.c_double]),
    "bgsb_ccl_label_batch_dev": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]),
    "bgsb_ccl_components_of": (C.c_int, [vp, C.c_int, C.POINTER(Component), C.c_int, intp]),
    "bgsb_ccl_label_dev": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, vp, vp]),
    "bgsb_ccl_components": (C.c_int, [vp, C.POINTER(Component), C.c_int, intp]),
    "bgsb_ccl_rect_moments": (C.c_int, [vp, i32p, C.c_int, C.POINTER(C.c_uint64)]),
    "bgsb_ccl_rect_moments_of": (C.c_int, [vp, C.c_int, i32p, C.c_int, C.POINTER(C.c_uint64)]),
    "bgsb_ccl_label": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_size_t, C.c_int, vp, C.POINTER(Component),
                                 C.c_int, intp]),
    "bgsb_blobdetector_create": (C.c_int, [C.POINTER(vp), C.c_int]),
    "bgsb_blobdetector_destroy": (None, [vp]),
    "bgsb_blobdetector_set_param": (C.c_int, [vp, C.c_char_p, C.c_double]),
    "bgsb_blobdetector_detect": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_size_t, C.POINTER(Blob), C.c_int,
                                           C.POINTER(Blob), C.c_int, intp, intp, C.POINTER(Blob), C.c_int, intp]),
    "bgsb_blobdetector_detect_dev": (C.c_int, [vp, vp, C.c_int, C.c_int, C.POINTER(Blob), C.c_int,
                                               C.POINTER(Blob), C.c_int, intp, intp, C.POINTER(Blob), C.c_int,
                                               intp, vp]),
    "bgsb_pipeline_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int]),
    "bgsb_pipeline_destroy": (None, [vp]),
    "bgsb_pipeline_bgs": (vp, [vp]),
    "bgsb_pipeline_set_morph": (C.c_int, [vp, intp, C.c_int]),
    "bgsb_pipeline_set_param": (C.c_int, [vp, C.c_char_p, C.c_double]),
    "bgsb_pipeline_process_dev": (C.c_int, [vp, vp, C.c_int, C.c_int, vp, vp, vp, intp, intp, vp]),
    "bgsb_pipeline_join_dev": (C.c_int, [vp, vp]),
    "bgsb_pipeline_components": (C.c_int, [vp, C.c_int, C.POINTER(Component), C.c_int, intp]),
    "bgsb_pipeline_tables_dev": (C.c_int, [vp, vp, C.c_int, vp]),
    "bgsb_pipeline_rect_moments": (C.c_int, [vp, C.c_int, i32p, C.c_int, C.POINTER(C.c_uint64)]),
    "bgsb_pipeline_detect": (C.c_int, [vp, C.POINTER(vp), C.POINTER(C.POINTER(Blob)), intp, C.POINTER(Blob), intp,
                                       C.POINTER(Blob), intp, intp]),
    "bgsb_pool_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, intp, C.c_int, C.c_int, C.c_int, C.c_int]),
    "bgsb_pool_destroy": (None, [vp]),
    "bgsb_pool_set_param": (C.c_int, [vp, C.c_char_p, C.c_double]),
    "bgsb_pool_set_morph": (C.c_int, [vp, intp, C.c_int]),
    "bgsb_pool_device_of": (C.c_int, [vp, C.c_int, intp]),
    "bgsb_pool_info": (C.c_int, [vp, intp, intp, intp]),
    "bgsb_pool_frame_buffer": (vp, [vp, C.c_int, C.c_int]),
    "bgsb_pool_submit": (C.c_int, [vp, C.c_int, C.c_int]),
    "bgsb_pool_wait": (C.c_int, [vp, C.c_int, intp]),
    "bgsb_pool_mask": (vp, [vp, C.c_int, C.c_int]),
    "bgsb_pool_components": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(Component), C.c_int, intp]),
    "bgsb_pool_detect": (C.c_int, [vp, C.c_int, C.POINTER(vp), C.POINTER(C.POINTER(Blob)), intp, C.POINTER(Blob), intp,
                                   C.POINTER(Blob), intp, intp]),
    "bgsb_synth_frames_dev": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, vp]),
    "bgsb_synth_churn_frames_dev": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, vp]),
}

_lib = None


def lib():
    """Load libbgsb200.so; raises (loudly) when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "tracking_b200: %s is missing -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError if the header and the library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != OK:
        raise BgsbError(rc, lib().bgsb_last_error().decode("utf-8", "replace"))


def kernel_launch_count():
    return int(lib().bgsb_kernel_launch_count())
