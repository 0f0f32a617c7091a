"""clfacedetection_b200 -- B200-native Viola-Jones hot path behind the clif/clod API.

The product is the CUDA library ``libclfd_b200.so`` (C ABI in include/clfd_b200.h) and the
C++ clif/clod layer over it (include/clif.h, include/clod.h).  This Python package is the
thin ctypes plumbing the tests and bench.py use to drive the same ABI; it holds no compute
and no fallback path.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import abi
from .abi import ClfdError  # noqa: F401

__all__ = ["Context", "Cascade", "Detector", "group_rectangles", "group_rectangles_roc", "group_batch", "ClfdError",
           "DetectResult"]


def _ptr(a):
    """address of a numpy array / torch tensor / int"""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    raise TypeError(type(a))


class Context:
    """One per GPU (clifInitEnvironment / clodInitEnvironment, clif.cpp:80, clod.cpp:72)."""

    def __init__(self, device_index: int = 0):
        self._h = C.c_void_p()
        abi.check(abi.lib().clfd_context_create(device_index, C.byref(self._h)))
        self.device_index = device_index

    def close(self):
        if self._h:
            abi.lib().clfd_context_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self) -> int:
        return int(abi.lib().clfd_context_launch_count(self._h))

    def synchronize(self):
        abi.check(abi.lib().clfd_context_synchronize(self._h))

    # ---- clif -------------------------------------------------------------------
    def integral(self, img: np.ndarray, tilted: bool = False):
        """clifIntegral (clif.cpp:273-316): -> sum int32, sqsum uint64[, tilted int32]"""
        img = np.ascontiguousarray(img, np.uint8)
        h, w = img.shape
        s = np.empty((h + 1, w + 1), np.int32)
        q = np.empty((h + 1, w + 1), np.uint64)
        t = np.empty((h + 1, w + 1), np.int32) if tilted else None
        abi.check(abi.lib().clfd_integral(self._h, _ptr(img), w, h, img.strides[0], 0, _ptr(s), _ptr(q), _ptr(t), 0))
        return s, q, t

    def integral_image(self, img: np.ndarray, tilted: bool = False, want_gray: bool = False):
        """clifGrayscaleIntegral (clif.cpp:318-381) of one interleaved host image [H, W] or [H, W, 3 | 4] (BGR / BGRA):
        colour conversion + integral images on the device, one upload -> sum, sqsum, tilted | None[, gray]"""
        img = np.ascontiguousarray(img, np.uint8)
        h, w = img.shape[:2]
        c = 1 if img.ndim == 2 else img.shape[2]
        s = np.empty((h + 1, w + 1), np.int32)
        q = np.empty((h + 1, w + 1), np.uint64)
        t = np.empty((h + 1, w + 1), np.int32) if tilted else None
        g = np.empty((h, w), np.uint8) if want_gray else None
        abi.check(abi.lib().clfd_integral_image(self._h, _ptr(img), w, h, img.strides[0], c, _ptr(s), _ptr(q), _ptr(t),
                                                _ptr(g) if want_gray else None, w))
        return (s, q, t, g) if want_gray else (s, q, t)

    def resize(self, img: np.ndarray, dw: int, dh: int) -> np.ndarray:
        """cvResize(INTER_LINEAR) of one level (tempcv.cpp:1301)"""
        img = np.ascontiguousarray(img, np.uint8)
        h, w = img.shape
        out = np.empty((dh, dw), np.uint8)
        abi.check(abi.lib().clfd_resize(self._h, _ptr(img), w, h, img.strides[0], 0, _ptr(out), dw, dh, dw, 0))
        return out

    def bgr_to_gray(self, img: np.ndarray) -> np.ndarray:
        img = np.ascontiguousarray(img, np.uint8)
        h, w, c = img.shape
        out = np.empty((h, w), np.uint8)
        abi.check(abi.lib().clfd_bgr_to_gray(self._h, _ptr(img), w, h, img.strides[0], c, 0, _ptr(out), w, 0))
        return out


class Cascade:
    """A loaded + packed cascade (cvLoad at main.cpp:36 + the hidden cascade)."""

    def __init__(self, path: str | None = None, *, flat=None):
        self._h = C.c_void_p()
        L = abi.lib()
        if path is not None:
            abi.check(L.clfd_cascade_load_xml(path.encode(), C.byref(self._h)))
        else:
            ip, fp = C.POINTER(C.c_int), C.POINTER(C.c_float)
            f = flat
            abi.check(L.clfd_cascade_from_arrays(
                f.win_w, f.win_h, f.n_stages,
                f.st_ntrees.ctypes.data_as(ip), f.st_thr.ctypes.data_as(fp), f.st_parent.ctypes.data_as(ip),
                f.st_next.ctypes.data_as(ip), f.tr_nnodes.ctypes.data_as(ip), f.nd_tilted.ctypes.data_as(ip),
                f.nd_rect.ctypes.data_as(ip), f.nd_weight.ctypes.data_as(fp), f.nd_thr.ctypes.data_as(fp),
                f.nd_left.ctypes.data_as(ip), f.nd_right.ctypes.data_as(ip), f.alpha.ctypes.data_as(fp),
                C.byref(self._h)))
        self.info = abi.CascadeInfo()
        abi.check(L.clfd_cascade_get_info(self._h, C.byref(self.info)))

    def __del__(self):
        try:
            if self._h:
                abi.lib().clfd_cascade_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    def arrays(self) -> dict:
        i = self.info
        S, T, N = i.n_stages, i.n_trees, i.n_nodes
        out = dict(st_ntrees=np.zeros(S, np.int32), st_thr=np.zeros(S, np.float32),
                   st_parent=np.zeros(S, np.int32), st_next=np.zeros(S, np.int32), st_child=np.zeros(S, np.int32),
                   tr_nnodes=np.zeros(T, np.int32), nd_tilted=np.zeros(N, np.int32),
                   nd_rect=np.zeros((N, 3, 4), np.int32), nd_weight=np.zeros((N, 3), np.float32),
                   nd_thr=np.zeros(N, np.float32), nd_left=np.zeros(N, np.int32), nd_right=np.zeros(N, np.int32),
                   alpha=np.zeros(N + T, np.float32))
        ip, fp = C.POINTER(C.c_int), C.POINTER(C.c_float)
        order = ["st_ntrees", "st_thr", "st_parent", "st_next", "st_child", "tr_nnodes", "nd_tilted", "nd_rect",
                 "nd_weight", "nd_thr", "nd_left", "nd_right", "alpha"]
        args = [out[k].ctypes.data_as(fp if out[k].dtype == np.float32 else ip) for k in order]
        abi.check(abi.lib().clfd_cascade_get_arrays(self._h, *args))
        return out

    def hidden(self):
        i = self.info
        w = np.zeros((i.n_nodes, 3), np.float32)
        nr = np.zeros(i.n_nodes, np.int32)
        st = np.zeros(i.n_stages, np.float32)
        two = np.zeros(i.n_stages, np.int32)
        ip, fp = C.POINTER(C.c_int), C.POINTER(C.c_float)
        abi.check(abi.lib().clfd_cascade_get_hidden(self._h, w.ctypes.data_as(fp), nr.ctypes.data_as(ip),
                                                    st.ctypes.data_as(fp), two.ctypes.data_as(ip)))
        return w, nr, st, two


@dataclass
class DetectResult:
    rects: np.ndarray   # structured: x,y,w,h,frame,cascade
    stats: dict

    def frame_rects(self, frame: int, cascade: int = 0) -> np.ndarray:
        m = (self.rects["frame"] == frame) & (self.rects["cascade"] == cascade)
        r = self.rects[m]
        out = np.stack([r["x"], r["y"], r["w"], r["h"]], axis=1).astype(np.int32) if len(r) else np.zeros((0, 4), np.int32)
        return out[np.lexsort((out[:, 0], out[:, 1], out[:, 2]))] if len(out) else out


RECT_DTYPE = np.dtype([("x", "<i4"), ("y", "<i4"), ("w", "<i4"), ("h", "<i4"), ("frame", "<i4"), ("cascade", "<i4")])


class Detector:
    """clodInitBuffers + clodDetectObjects for one frame shape (clod.cpp:102, 1339)."""

    def __init__(self, ctx: Context, cascades, width: int, height: int, *, max_batch: int = 1,
                 scale_factor: float = 1.1, min_size=(0, 0), max_size=(0, 0), want_codes: bool = False,
                 max_rects: int = 0, scale_cascade: bool = False):
        """scale_cascade: CLFD_MODE_SCALE_CASCADE (one integral image, scaled features: what the
        cvHaarDetectObjects call of main.cpp:145 computes) instead of the image pyramid"""
        self.ctx = ctx
        self.cascades = list(cascades) if isinstance(cascades, (list, tuple)) else [cascades]
        cfg = abi.DetectorConfig(width, height, max_batch, scale_factor, min_size[0], min_size[1],
                                 max_size[0], max_size[1], int(want_codes), max_rects, int(scale_cascade))
        self.cfg = cfg
        arr = (C.c_void_p * len(self.cascades))(*[c._h for c in self.cascades])
        self._h = C.c_void_p()
        abi.check(abi.lib().clfd_detector_create(ctx._h, arr, len(self.cascades), C.byref(cfg), C.byref(self._h)))
        self.width, self.height, self.max_batch = width, height, max_batch
        self._rect_cap = max_rects if max_rects > 0 else 1 << 20
        self._rects = np.zeros(self._rect_cap, RECT_DTYPE)

    def close(self):
        if self._h:
            abi.lib().clfd_detector_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def levels(self, cascade: int = 0):
        n = abi.check(abi.lib().clfd_detector_num_levels(self._h, cascade))
        buf = (abi.Level * max(n, 1))()
        abi.check(abi.lib().clfd_detector_get_levels(self._h, cascade, buf, max(n, 1)))
        return list(buf[:n])

    def windows_per_frame(self, cascade: int = 0) -> int:
        return int(abi.lib().clfd_detector_windows_per_frame(self._h, cascade))

    def set_profiling(self, on: bool):
        abi.check(abi.lib().clfd_detector_set_profiling(self._h, int(on)))

    def kernel_ms(self):
        ms = (C.c_float * 8)()
        abi.check(abi.lib().clfd_detector_get_kernel_ms(self._h, ms))
        return list(ms)

    def stats(self) -> dict:
        s = abi.RunStats()
        abi.check(abi.lib().clfd_detector_get_stats(self._h, C.byref(s)))
        return {n: int(getattr(s, n)) for n, _ in abi.RunStats._fields_}

    # ---- device-resident input ---------------------------------------------------------
    def enqueue(self, frames_dev, n_frames: int, frame_stride: int, row_stride: int, stream: int = 0, channels: int = 1):
        """channels 3 / 4: interleaved BGR / BGRA frames, converted to gray on `stream` first"""
        s = C.c_void_p(stream) if stream else None
        if channels == 1:
            abi.check(abi.lib().clfd_detector_enqueue(self._h, _ptr(frames_dev), n_frames, frame_stride, row_stride, s))
        else:
            abi.check(abi.lib().clfd_detector_enqueue_color(self._h, _ptr(frames_dev), n_frames, channels, frame_stride,
                                                            row_stride, s))

    def fetch(self, stream: int = 0) -> DetectResult:
        n = C.c_int64()
        abi.check(abi.lib().clfd_detector_fetch(self._h, self._rects.ctypes.data_as(C.POINTER(abi.Rect)),
                                                self._rect_cap, C.byref(n), C.c_void_p(stream) if stream else None))
        return DetectResult(self._rects[:n.value].copy(), self.stats())

    def _geometry(self, frames):
        """(n_frames, frame stride, row stride, channels) of a uint8 [n, H, W] or [n, H, W, C] (C = 3 BGR, 4 BGRA) numpy
        array or torch tensor of this detector's shape"""
        n, H, W = frames.shape[:3]
        assert (H, W) == (self.height, self.width)
        strides = frames.strides if isinstance(frames, np.ndarray) else frames.stride()
        if frames.ndim == 3:
            return n, strides[0], strides[1], 1
        c = frames.shape[3]
        if frames.ndim != 4 or c not in (3, 4):
            raise ValueError(f"frames of shape {tuple(frames.shape)}: expected [n, H, W] or [n, H, W, 3 | 4]")
        if strides[3] != 1 or strides[2] != c:
            raise ValueError(f"colour frames need interleaved pixels (strides {tuple(strides)})")
        return n, strides[0], strides[1], c

    # ---- host input, end to end (the call a clod user makes) ----------------------------
    def detect(self, frames) -> DetectResult:
        """frames: uint8 [n,H,W], or [n,H,W,3 | 4] BGR / BGRA (numpy, or a pinned torch CPU tensor)"""
        if isinstance(frames, np.ndarray):
            if frames.ndim == 2:
                frames = frames[None]
            frames = np.ascontiguousarray(frames, np.uint8)
        n, fs, rs, c = self._geometry(frames)
        cnt = C.c_int64()
        out = self._rects.ctypes.data_as(C.POINTER(abi.Rect))
        if c == 1:
            abi.check(abi.lib().clfd_detect(self._h, _ptr(frames), n, fs, rs, out, self._rect_cap, C.byref(cnt)))
        else:
            abi.check(abi.lib().clfd_detect_color(self._h, _ptr(frames), n, c, fs, rs, out, self._rect_cap, C.byref(cnt)))
        return DetectResult(self._rects[:cnt.value].copy(), self.stats())

    # ---- host input, streaming: submit batch i+1 while batch i computes -----------------
    def submit(self, frames) -> None:
        """frames as for detect(); must stay alive (and should be pinned) until collected"""
        if isinstance(frames, np.ndarray):
            assert frames.ndim in (3, 4) and frames.dtype == np.uint8 and frames.flags.c_contiguous
        n, fs, rs, c = self._geometry(frames)
        if c == 1:
            abi.check(abi.lib().clfd_detect_submit(self._h, _ptr(frames), n, fs, rs))
        else:
            abi.check(abi.lib().clfd_detect_submit_color(self._h, _ptr(frames), n, c, fs, rs))

    def submit_views(self, first_frame, n_frames: int, frame_stride: int, row_stride: int) -> None:
        """submit n_frames frames that start frame_stride bytes apart at `first_frame` (a pinned tensor view or an
        address); frames may overlap (frame_stride = row_stride: views of one canvas, one row apart)"""
        abi.check(abi.lib().clfd_detect_submit(self._h, _ptr(first_frame), n_frames, frame_stride, row_stride))

    def collect(self) -> DetectResult:
        cnt = C.c_int64()
        abi.check(abi.lib().clfd_detect_collect(self._h, self._rects.ctypes.data_as(C.POINTER(abi.Rect)),
                                                self._rect_cap, C.byref(cnt)))
        return DetectResult(self._rects[:cnt.value].copy(), self.stats())

    def codes(self, cascade: int = 0, n_frames: int = 1) -> np.ndarray:
        wpf = self.windows_per_frame(cascade)
        out = np.zeros((n_frames, wpf), np.int16)
        abi.check(abi.lib().clfd_detector_get_codes(self._h, cascade, out.ctypes.data_as(C.POINTER(C.c_int16)), out.size))
        return out

    def reject_levels(self, cascade: int = 0):
        """Reject-level / ROC output of the last blocking detect (cvHaarDetectObjectsForROC with
        outputRejectLevels, tempcv.cpp:1084-1094) -> (rects RECT_DTYPE, levels int32, stage sums
        float64) in the reference's scan order.  Needs want_codes=True."""
        cap = 1 << 12
        while True:
            r = np.zeros(cap, RECT_DTYPE)
            lv = np.zeros(cap, np.int32)
            wt = np.zeros(cap, np.float64)
            n = C.c_int64()
            rc = abi.lib().clfd_detector_reject_levels(self._h, cascade, r.ctypes.data_as(C.POINTER(abi.Rect)),
                                                       lv.ctypes.data_as(C.POINTER(C.c_int32)),
                                                       wt.ctypes.data_as(C.POINTER(C.c_double)), cap, C.byref(n))
            if rc == -5 and n.value > cap:   # CLFD_ERR_CAPACITY: n holds the count
                cap = int(n.value)
                continue
            abi.check(rc)
            return r[:n.value].copy(), lv[:n.value].copy(), wt[:n.value].copy()

    def read_level(self, level: int, frame: int = 0, cascade: int = 0, tilted: bool = False):
        lv = self.levels(cascade)[level]
        w, h = lv.img_w, lv.img_h
        pyr = np.empty((h, w), np.uint8)
        s = np.empty((h + 1, w + 1), np.int32)
        q = np.empty((h + 1, w + 1), np.uint64)
        t = np.empty((h + 1, w + 1), np.int32) if tilted else None
        abi.check(abi.lib().clfd_detector_read_level(self._h, cascade, level, frame, _ptr(pyr), _ptr(s), _ptr(q), _ptr(t)))
        return pyr, s, q, t


def group_rectangles(rects: np.ndarray, group_threshold: int, eps: float = 0.2):
    """Host-side AgroupRectangles (tempcv.cpp:145-243) -> (rects[m,4], weights[m])"""
    r = np.ascontiguousarray(rects, np.int32).reshape(-1, 4).copy()
    n = C.c_int(len(r))
    w = np.zeros(max(len(r), 1), np.int32)
    abi.check(abi.lib().clfd_group_rectangles(r.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(n), group_threshold,
                                              eps, w.ctypes.data_as(C.POINTER(C.c_int32))))
    return r[:n.value].copy(), w[:n.value].copy()


def group_rectangles_roc(rects: np.ndarray, reject_levels: np.ndarray, level_weights: np.ndarray,
                         group_threshold: int, eps: float = 0.2):
    """AgroupRectangles, ROC variant (tempcv.cpp:255-258) -> (rects[m,4], levels[m], stage sums[m])"""
    r = np.ascontiguousarray(rects, np.int32).reshape(-1, 4).copy()
    lv = np.ascontiguousarray(reject_levels, np.int32).copy()
    wt = np.ascontiguousarray(level_weights, np.float64).copy()
    n = C.c_int(len(r))
    if len(r) == 0:
        return r, lv, wt
    abi.check(abi.lib().clfd_group_rectangles_roc(r.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(n), group_threshold, eps,
                                                  lv.ctypes.data_as(C.POINTER(C.c_int32)),
                                                  wt.ctypes.data_as(C.POINTER(C.c_double))))
    return r[:n.value].copy(), lv[:n.value].copy(), wt[:n.value].copy()


def group_batch(rects: np.ndarray, group_threshold: int, eps: float = 0.2, n_threads: int = 0):
    """Per-(frame, cascade) AgroupRectangles of a batch's raw rects (RECT_DTYPE) on host threads
    -> (grouped rects RECT_DTYPE, neighbour counts)."""
    r = np.ascontiguousarray(rects, RECT_DTYPE)
    out = np.zeros(max(len(r), 1), RECT_DTYPE)
    w = np.zeros(max(len(r), 1), np.int32)
    n = C.c_int64()
    abi.check(abi.lib().clfd_group_batch(r.ctypes.data_as(C.POINTER(abi.Rect)), len(r), group_threshold, eps, n_threads,
                                         out.ctypes.data_as(C.POINTER(abi.Rect)), w.ctypes.data_as(C.POINTER(C.c_int32)),
                                         len(out), C.byref(n)))
    return out[:n.value].copy(), w[:n.value].copy()
