"""ctypes binding of the C ABI (include/clfd_b200.h -> libclfd_b200.so).

This is plumbing only: every function maps 1:1 to an exported ``clfd_*`` symbol.  There is
no Python or CPU implementation behind it -- if the shared library is missing, ``lib()``
raises, and if no B200 is visible, ``clfd_context_create`` fails.
"""
from __future__ import annotations

import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CLFD_LIB") or os.path.join(_HERE, "libclfd_b200.so")   # CLFD_LIB: A/B builds of the same ABI
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "clfd_b200.h")
_lib = None


class ClfdError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"clfd status {status}: {message}")
        self.status = status


class CascadeInfo(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "win_w", "win_h", "n_stages", "n_trees", "n_nodes", "is_tree", "is_stump_based", "has_tilted",
        "n_tilted_nodes", "n_three_rect_nodes", "max_trees_per_stage", "max_nodes_per_tree",
        "dense_stages", "dense_stumps", "order_free_stages", "packed_bytes")]


class DetectorConfig(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("max_batch", C.c_int),
                ("scale_factor", C.c_double), ("min_w", C.c_int), ("min_h", C.c_int),
                ("max_w", C.c_int), ("max_h", C.c_int), ("want_codes", C.c_int),
                ("max_rects", C.c_int64), ("mode", C.c_int)]


class Rect(C.Structure):
    _fields_ = [("x", C.c_int32), ("y", C.c_int32), ("w", C.c_int32), ("h", C.c_int32),
                ("frame", C.c_int32), ("cascade", C.c_int32)]


class Level(C.Structure):
    _fields_ = [("factor", C.c_double), ("img_w", C.c_int), ("img_h", C.c_int), ("win_w", C.c_int),
                ("win_h", C.c_int), ("ystep", C.c_int), ("nx", C.c_int), ("ny", C.c_int),
                ("win_base", C.c_int64)]


class RunStats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in (
        "windows", "rects", "deep_windows", "kernel_launches", "pyramid_pixels",
        "bytes_resize", "bytes_integral", "bytes_cascade", "bytes_tilted", "exact_stage_evals", "near_threshold_events")]


def exported_symbols_in_header() -> list[str]:
    """Every function name include/clfd_b200.h declares with CLFD_API."""
    text = open(HEADER_PATH).read()
    return sorted(set(re.findall(r"CLFD_API[^;(]*?\b(clfd_\w+)\s*\(", text)))


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no fallback implementation)")
    L = C.CDLL(LIB_PATH)
    vp, ip, fp = C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_float)
    u8p = C.c_void_p  # raw host or device addresses
    L.clfd_last_error.restype = C.c_char_p
    L.clfd_version.restype = C.c_char_p
    L.clfd_device_count.argtypes = [ip]
    L.clfd_context_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.clfd_context_destroy.argtypes = [vp]
    L.clfd_context_destroy.restype = None
    L.clfd_context_device.argtypes = [vp]
    L.clfd_context_launch_count.argtypes = [vp]
    L.clfd_context_launch_count.restype = C.c_int64
    L.clfd_context_synchronize.argtypes = [vp]
    L.clfd_cascade_load_xml.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.clfd_cascade_from_arrays.argtypes = [C.c_int, C.c_int, C.c_int, ip, fp, ip, ip, ip, ip, ip, fp, fp, ip, ip, fp,
                                           C.POINTER(vp)]
    L.clfd_cascade_destroy.argtypes = [vp]
    L.clfd_cascade_destroy.restype = None
    L.clfd_cascade_id.argtypes = [vp]
    L.clfd_cascade_id.restype = C.c_uint64
    L.clfd_cascade_get_info.argtypes = [vp, C.POINTER(CascadeInfo)]
    L.clfd_cascade_get_arrays.argtypes = [vp, ip, fp, ip, ip, ip, ip, ip, ip, fp, fp, ip, ip, fp]
    L.clfd_cascade_get_hidden.argtypes = [vp, fp, ip, fp, ip]
    L.clfd_integral.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_int]
    L.clfd_resize.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p, C.c_int, C.c_int, C.c_int, C.c_int]
    L.clfd_bgr_to_gray.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, u8p, C.c_int, C.c_int]
    L.clfd_integral_image.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, u8p, C.c_int]
    L.clfd_detector_create.argtypes = [vp, C.POINTER(vp), C.c_int, C.POINTER(DetectorConfig), C.POINTER(vp)]
    L.clfd_detector_destroy.argtypes = [vp]
    L.clfd_detector_destroy.restype = None
    L.clfd_detector_num_levels.argtypes = [vp, C.c_int]
    L.clfd_detector_get_levels.argtypes = [vp, C.c_int, C.POINTER(Level), C.c_int]
    L.clfd_detector_windows_per_frame.argtypes = [vp, C.c_int]
    L.clfd_detector_windows_per_frame.restype = C.c_int64
    L.clfd_detector_enqueue.argtypes = [vp, u8p, C.c_int, C.c_size_t, C.c_int, vp]
    L.clfd_detector_fetch.argtypes = [vp, C.POINTER(Rect), C.c_int64, C.POINTER(C.c_int64), vp]
    L.clfd_detect.argtypes = [vp, u8p, C.c_int, C.c_size_t, C.c_int, C.POINTER(Rect), C.c_int64,
                              C.POINTER(C.c_int64)]
    L.clfd_group_batch.argtypes = [C.POINTER(Rect), C.c_int64, C.c_int, C.c_double, C.c_int, C.POINTER(Rect),
                                   C.POINTER(C.c_int32), C.c_int64, C.POINTER(C.c_int64)]
    L.clfd_detect_image.argtypes = [vp, u8p, C.c_int, C.c_int, C.POINTER(Rect), C.c_int64, C.POINTER(C.c_int64)]
    L.clfd_detect_submit.argtypes = [vp, u8p, C.c_int, C.c_size_t, C.c_int]
    L.clfd_detect_collect.argtypes = [vp, C.POINTER(Rect), C.c_int64, C.POINTER(C.c_int64)]
    L.clfd_detector_enqueue_color.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_size_t, C.c_int, vp]
    L.clfd_detect_submit_color.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_size_t, C.c_int]
    L.clfd_detect_color.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_size_t, C.c_int, C.POINTER(Rect), C.c_int64,
                                    C.POINTER(C.c_int64)]
    L.clfd_detector_get_codes.argtypes = [vp, C.c_int, C.POINTER(C.c_int16), C.c_int64]
    L.clfd_detector_read_level.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]
    L.clfd_detector_get_stats.argtypes = [vp, C.POINTER(RunStats)]
    L.clfd_detector_set_profiling.argtypes = [vp, C.c_int]
    L.clfd_detector_get_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
    L.clfd_group_rectangles.argtypes = [C.POINTER(C.c_int32), ip, C.c_int, C.c_double, C.POINTER(C.c_int32)]
    L.clfd_group_rectangles_roc.argtypes = [C.POINTER(C.c_int32), ip, C.c_int, C.c_double, C.POINTER(C.c_int32),
                                            C.POINTER(C.c_double)]
    L.clfd_detector_reject_levels.argtypes = [vp, C.c_int, C.POINTER(Rect), C.POINTER(C.c_int32), C.POINTER(C.c_double),
                                              C.c_int64, C.POINTER(C.c_int64)]
    _lib = L
    return L


def check(status: int) -> int:
    if status < 0:
        raise ClfdError(status, lib().clfd_last_error().decode(errors="replace"))
    return status
