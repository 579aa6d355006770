"""ctypes binding of the C-ABI library (include/tsd_b200.h -> libtsd_b200.so).

Fails loudly: a missing library or a missing CUDA device raises; there is no CPU fallback and nothing here
imports the oracle.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TSD_LIB") or os.path.join(_PKG, "libtsd_b200.so")     # TSD_LIB: an alternative build (A/B experiments)

MEM_HOST, MEM_DEVICE = 0, 1
RUN_DETECT, RUN_RECOGNIZE = 1, 2
REC_GRAY, REC_KNN = 4, 8              # classifier modifiers OR-ed into RUN_RECOGNIZE (HOG + LDA without them)
HOG_LEN = 324


class TsdError(RuntimeError):
    """Raised for every non-zero status of the C ABI (the reference's drivers catch Exception and carry on)."""


class Config(C.Structure):
    _fields_ = [
        ("enlarge", C.c_double), ("aspect_lo", C.c_double), ("aspect_hi", C.c_double),
        ("window", C.c_int32), ("score_tol_hundredths", C.c_int32),
        ("hist_tol", C.c_double), ("coord_tol", C.c_double), ("merge_factor", C.c_double),
        ("red_lo", (C.c_uint8 * 3) * 2), ("red_hi", (C.c_uint8 * 3) * 2),
        ("blue_lo", C.c_uint8 * 3), ("blue_hi", C.c_uint8 * 3), ("pad_", C.c_uint8 * 6),
        ("proba_tol", C.c_double), ("knn_k", C.c_int32), ("reserved", C.c_int32),
    ]


class Detection(C.Structure):
    _fields_ = [("frame", C.c_int32), ("x1", C.c_int32), ("y1", C.c_int32), ("x2", C.c_int32), ("y2", C.c_int32),
                ("id", C.c_int32), ("hundredths", C.c_int32), ("reserved", C.c_int32)]


class FrameDesc(C.Structure):
    """tsd_frame_desc: one frame of a batch of frames of different sizes (the *_ragged entry points)."""
    _fields_ = [("offset", C.c_int64), ("row_stride", C.c_int64), ("H", C.c_int32), ("W", C.c_int32)]


FRAME_DESC_DTYPE = np.dtype([("offset", "<i8"), ("row_stride", "<i8"), ("H", "<i4"), ("W", "<i4")])

DET_DTYPE = np.dtype([("frame", "<i4"), ("x1", "<i4"), ("y1", "<i4"), ("x2", "<i4"), ("y2", "<i4"),
                      ("id", "<i4"), ("hundredths", "<i4"), ("reserved", "<i4")])

_vp, _i, _i64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_double

_SIGNATURES = {
    "tsd_config_default": (_i, [C.POINTER(Config), _i]),
    "tsd_last_error": (C.c_char_p, []),
    "tsd_version": (C.c_char_p, []),
    "tsd_device_count": (_i, []),
    "tsd_create": (_i, [C.POINTER(_vp), _i, C.POINTER(Config)]),
    "tsd_destroy": (_i, [_vp]),
    "tsd_stream": (_vp, [_vp]),
    "tsd_synchronize": (_i, [_vp]),
    "tsd_flush": (_i, [_vp]),
    "tsd_match_detections": (_i, [_vp, _vp, _i, _vp, _vp, _i, _d, _vp, _vp, _vp]),
    "tsd_match_iou": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _d, _vp, _vp]),
    "tsd_launch_count": (_i64, [_vp]),
    "tsd_mean_windows": (_i, [_vp, _vp, _vp, _i, _i, _vp, _i]),
    "tsd_score": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _i]),
    "tsd_lda_predict_tf32": (_i, [_vp, _vp, _i, _d, _i, _vp, _vp, C.POINTER(C.c_float), _i]),
    "tsd_recognize": (_i, [_vp, _vp, _i, _d, _vp, _i]),
    "tsd_set_gamma_table": (_i, [_vp, _vp]),
    "tsd_preprocess": (_i, [_vp, _vp, _i, _i, _i, _i64, _i64, _d, _i, _i, _vp, _i]),
    "tsd_host_register": (_i, [_vp, _i64]),
    "tsd_stat_hist_entries": (_i, [_vp, C.POINTER(C.c_int64)]),
    "tsd_stat_unsure_pairs": (_i, [_vp, C.POINTER(C.c_int64), _i]),
    "tsd_stat_staged_bytes": (_i, [_vp, C.POINTER(C.c_int64), _i]),
    "tsd_stat_graphs": (_i, [_vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "tsd_host_unregister": (_i, [_vp]),
    "tsd_set_templates": (_i, [_vp, _vp, _vp]),
    "tsd_set_similarity_table": (_i, [_vp, _vp, _i]),
    "tsd_set_lda": (_i, [_vp, _vp, _vp, _i]),
    "tsd_set_knn": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _i, _i]),
    "tsd_expand_boxes": (_i, [_vp, _vp, _i, _d, _vp, _vp, _i]),
    "tsd_crop_resize": (_i, [_vp, _vp, _i, _i, _i, _i64, _i64, _i, _vp, _vp, _i, _i, _vp, _i]),
    "tsd_windows": (_i, [_vp, _vp, _i, _i, _i, _i64, _i64, _vp, _vp, _d, _i, _vp, _vp, _vp, _vp, _i]),
    "tsd_crop_resize_ragged": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _i, _i, _vp, _i]),
    "tsd_windows_ragged": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _d, _i, _vp, _vp, _vp, _vp, _i]),
    "tsd_detect_frames_ragged": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _i]),
    "tsd_enqueue_frames_ragged": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _i, _i]),
    "tsd_dedup": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _d, _vp, _vp, _vp, _vp, _i]),
    "tsd_hist": (_i, [_vp, _vp, _i, _i, _vp, _i]),
    "tsd_hist_sparse": (_i, [_vp, _vp, _i, _i, _i64, _vp, _vp, _vp]),
    "tsd_color_masks": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i]),
    "tsd_bgr2hsv": (_i, [_vp, _vp, _i64, _vp, _i]),
    "tsd_score_masks": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _i]),
    "tsd_bgr2gray": (_i, [_vp, _vp, _i64, _vp, _i]),
    "tsd_hog": (_i, [_vp, _vp, _i, _vp, _i]),
    "tsd_lda_predict": (_i, [_vp, _vp, _i, _d, _vp, _vp, _i]),
    "tsd_knn_predict": (_i, [_vp, _vp, _i, _vp, _vp, _i]),
    "tsd_detect_frames": (_i, [_vp, _i, _vp, _i, _i, _i, _i64, _i64, _vp, _vp, _vp, _i, _vp, _vp, _i]),
    "tsd_enqueue_frames": (_i, [_vp, _i, _vp, _i, _i, _i, _i64, _i64, _vp, _vp, _i, _i]),
    "tsd_fetch_detections": (_i, [_vp, _vp, _i, _vp, _vp]),
    "tsd_fetch_previous": (_i, [_vp, _vp, _i, _vp, _vp]),
    "tsd_set_profiling": (_i, [_vp, _i]),
    "tsd_stage_times": (_i, [_vp, _vp, _vp, _i]),
    "tsd_timeline": (_i, [_vp, _vp, _vp, _i]),
}

EXPORTS = tuple(sorted(_SIGNATURES))


def build(force=False):
    """Compile csrc/ for sm_100a with nvcc (in-tree .so).  Cross-compiles without a GPU."""
    src_dir = os.path.join(_PKG, "csrc")
    srcs = [os.path.join(src_dir, f) for f in os.listdir(src_dir) if f.endswith((".cu", ".cuh", "Makefile"))]
    srcs.append(os.path.join(_PKG, "..", "include", "tsd_b200.h"))
    stale = not os.path.isfile(LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        subprocess.check_call(["make", "-C", src_dir, "-s"] + (["-B"] if force else []))
    return LIB_PATH


_lib = None


def lib():
    """The loaded library (ctypes.CDLL) with argtypes set.  Raises if the extension was not built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise TsdError("CUDA extension %s is missing -- run __graft_entry__.build() (nvcc, sm_100a). "
                           "There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status):
    if status != 0:
        raise TsdError("tsd_b200 error %d: %s" % (status, lib().tsd_last_error().decode(errors="replace")))


def ptr(a):
    """Host numpy array / integer device pointer / None -> void*."""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    return C.c_void_p(a.ctypes.data)
