"""Colour batches (clfd_detect_color / clfd_detect_submit_color / clfd_detector_enqueue_color): interleaved BGR and
BGRA frames converted on the device by k_color_to_gray must detect exactly what their gray frames detect, the gray
being OpenCV's fixed point (B*1868 + G*9617 + R*4899 + 8192) >> 14 computed here in int64.  Every comparison is an
exact equality, and every case checks that it is not vacuous: rects were found and the three channels differ."""
import ctypes as C

import numpy as np
import pytest

import clfacedetection_b200 as clfd
from clfacedetection_b200 import abi
from clfacedetection_b200.frames import octave_frame
from conftest import cascade_path, oracle_cascade

pytestmark = pytest.mark.gpu

SF = 1.2


def _sorted(r):
    r = np.asarray(r, np.int32).reshape(-1, 4)
    return r[np.lexsort((r[:, 0], r[:, 1], r[:, 2]))] if len(r) else r


def formula_gray(img):
    b, g, r = (img[..., k].astype(np.int64) for k in range(3))
    return ((b * 1868 + g * 9617 + r * 4899 + 8192) >> 14).astype(np.uint8)


def colour_frames(W, H, n, channels, first=0):
    """n frames [n, H, W, channels] whose B, G and R planes (and alpha) are octave frames of distinct seeds"""
    out = np.empty((n, H, W, channels), np.uint8)
    for i in range(n):
        for k in range(channels):
            out[i, ..., k] = octave_frame(W, H, 1000 + 4 * (first + i) + k)
    return out


def assert_channels_differ(frames):
    assert not np.array_equal(frames[..., 0], frames[..., 1])
    assert not np.array_equal(frames[..., 1], frames[..., 2])
    assert not np.array_equal(frames[..., 0], frames[..., 2])


def oracle_rects(name, gray, sf=SF):
    return _sorted(oracle_cascade(name).detect(gray, sf, want_codes=False)[0])


def detector(gpu_ctx, names, W, H, n, sf=SF, **kw):
    return clfd.Detector(gpu_ctx, [clfd.Cascade(cascade_path(nm)) for nm in names], W, H, max_batch=n,
                         scale_factor=sf, **kw)


def _rect_out(det):
    return det._rects.ctypes.data_as(C.POINTER(abi.Rect)), det._rect_cap


def detect_color_raw(det, addr, n, channels, frame_stride, row_stride):
    """clfd_detect_color on host memory at `addr` with any strides"""
    out, cap = _rect_out(det)
    cnt = C.c_int64()
    abi.check(abi.lib().clfd_detect_color(det._h, C.c_void_p(addr), n, channels, frame_stride, row_stride, out, cap,
                                          C.byref(cnt)))
    return clfd.DetectResult(det._rects[:cnt.value].copy(), det.stats())


def strided_buffer(frames, offset, frame_stride, row_stride):
    """the frames [n, H, W, C] laid out at `offset` in a byte buffer that ends right behind the last frame's last pixel"""
    n, H, W, c = frames.shape
    size = offset + (n - 1) * frame_stride + (H - 1) * row_stride + W * c
    buf = np.zeros(size, np.uint8)
    for f in range(n):
        for y in range(H):
            o = offset + f * frame_stride + y * row_stride
            buf[o:o + W * c] = frames[f, y].reshape(-1)
    return buf


# ---- 1. batch parity -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("channels", [3, 4])
def test_batch_parity_with_gray_and_oracle(gpu_ctx, channels):
    W, H, n = 640, 480, 9
    frames = colour_frames(W, H, n, channels)
    assert_channels_differ(frames)
    gray = np.stack([formula_gray(f) for f in frames])
    det = detector(gpu_ctx, ["frontalface_alt"], W, H, n)
    got = det.detect(frames)
    total = 0
    for f in range(n):
        want = oracle_rects("frontalface_alt", gray[f])
        assert np.array_equal(got.frame_rects(f), want), f
        total += len(want)
    assert total > 0
    assert np.array_equal(np.sort(got.rects, order=["frame", "w", "y", "x"]),
                          np.sort(det.detect(gray).rects, order=["frame", "w", "y", "x"]))
    if channels == 3:
        # control: the comparison tells channel orders apart -- R and B swapped give other rects
        swapped = [oracle_rects("frontalface_alt", formula_gray(f[..., ::-1])) for f in frames]
        assert any(not np.array_equal(got.frame_rects(f), swapped[f]) for f in range(n))
    det.close()
    # exit codes and reject levels of the diagnostic instantiation
    det = detector(gpu_ctx, ["frontalface_alt"], W, H, n, want_codes=True)
    c_res = det.detect(frames)
    c_codes, c_roc = det.codes(0, n), det.reject_levels()
    g_res = det.detect(gray)
    g_codes, g_roc = det.codes(0, n), det.reject_levels()
    assert len(c_res.rects) == total and len(g_res.rects) == total
    assert np.array_equal(c_codes, g_codes)
    assert len(c_roc[0]) > total
    for a, b in zip(c_roc, g_roc):
        assert np.array_equal(a, b)
    det.close()


# ---- 2. level 0 read-back --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("channels", [3, 4])
def test_level0_is_the_formula_gray(gpu_ctx, channels):
    W, H = 640, 480
    frames = colour_frames(W, H, 6, channels)
    assert_channels_differ(frames)
    for k in range(3):   # frames 0..2: only channel k is non-zero -- pins which coefficient goes with which channel
        frames[k, ..., [j for j in range(3) if j != k]] = 0
    frames[3, ..., :3] = 255 - frames[3, ..., :3]
    det = detector(gpu_ctx, ["frontalface_alt"], W, H, len(frames))
    assert det.levels()[0].img_w == W and det.levels()[0].img_h == H
    res = det.detect(frames)
    assert len(res.rects) > 0
    for f in range(len(frames)):
        assert np.array_equal(det.read_level(0, frame=f)[0], formula_gray(frames[f])), f
    det.close()


# ---- 3. geometry and alignment ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("W", [641, 1921])
@pytest.mark.parametrize("channels", [3, 4])
def test_strides_and_alignment(gpu_ctx, W, channels):
    """W * 3 is not a multiple of 4 or 16 at these widths.  Host input with row stride W*C + 13 and an odd frame
    stride; device input from a torch tensor at every row alignment (tight rows: 16-byte loads where the row allows
    them; W*C + 4: 32-bit loads; W*C + 13 and a base pointer offset by one byte: the byte path), on a user stream"""
    import torch
    H, n = 200, 3
    frames = colour_frames(W, H, n, channels, first=10)
    assert_channels_differ(frames)
    gray = np.stack([formula_gray(f) for f in frames])
    det = detector(gpu_ctx, ["frontalface_alt"], W, H, n)
    want = [oracle_rects("frontalface_alt", g) for g in gray]
    assert sum(len(w) for w in want) > 0

    def check(res, what):
        for f in range(n):
            assert np.array_equal(res.frame_rects(f), want[f]), (what, f)
            assert np.array_equal(det.read_level(0, frame=f)[0], gray[f]), (what, f)

    rs = W * channels + 13
    fs = H * rs + 7
    fs += 1 - fs % 2   # odd
    buf = strided_buffer(frames, 0, fs, rs)
    check(detect_color_raw(det, buf.ctypes.data, n, channels, fs, rs), "host")
    stream = torch.cuda.Stream()
    for rs in (W * channels, W * channels + 4, W * channels + 13):
        for offset in (0, 1):
            fs = H * rs + (offset or 16)
            dev = torch.from_numpy(strided_buffer(frames, offset, fs, rs)).cuda()
            torch.cuda.synchronize()
            with torch.cuda.stream(stream):
                det.enqueue(dev.data_ptr() + offset, n, fs, rs, stream.cuda_stream, channels=channels)
                res = det.fetch(stream.cuda_stream)
            check(res, ("device", rs, offset))
    det.close()


@pytest.mark.parametrize("channels", [3, 4])
def test_frame_stride_zero_repeats_one_frame(gpu_ctx, channels):
    import torch
    W, H, n = 640, 480, 4
    frame = colour_frames(W, H, 1, channels, first=3)
    assert_channels_differ(frame)
    det = detector(gpu_ctx, ["frontalface_alt"], W, H, n)
    one = det.detect(frame).frame_rects(0)
    assert len(one) > 0
    img = np.ascontiguousarray(frame[0])
    res = detect_color_raw(det, img.ctypes.data, n, channels, 0, W * channels)
    dev = torch.from_numpy(img).cuda()
    torch.cuda.synchronize()
    det.enqueue(dev, n, 0, W * channels, channels=channels)
    res_dev = det.fetch()
    for f in range(n):
        assert np.array_equal(res.frame_rects(f), one), f
        assert np.array_equal(res_dev.frame_rects(f), one), f
    det.close()


# ---- 4. streaming ----------------------------------------------------------------------------------------------------
def _stream_batches(W, H, n):
    """four distinct batches of n colour frames built from six octave planes (cheap at 1080p)"""
    planes = [octave_frame(W, H, 2000 + k) for k in range(6)]
    alpha = octave_frame(W, H, 2006)

    def batch(perm, channels):
        out = np.empty((n, H, W, channels), np.uint8)
        for i in range(n):
            for k in range(3):
                out[i, ..., k] = planes[(perm * i + 2 * k + perm) % 6] if k != 1 else planes[(i + perm + 1) % 6][::-1]
            if channels == 4:
                out[i, ..., 3] = alpha
        return out
    return batch


def test_streaming_overlap_and_two_in_flight(gpu_ctx, monkeypatch):
    """1080p, batch 16, one cascade the tile kernel finishes: the chunked copy + conversion and enqueue_overlapped.
    Then submit / collect with two batches in flight in the order BGR, gray, BGRA, BGR on one detector."""
    import torch
    W, H, n = 1920, 1080, 16
    batch = _stream_batches(W, H, n)
    bgr = batch(1, 3)
    assert_channels_differ(bgr)
    det = detector(gpu_ctx, ["frontalface_alt"], W, H, n)
    monkeypatch.setenv("CLFD_NO_OVERLAP", "1")
    monkeypatch.setenv("CLFD_DETECT_CHUNKS", "1")   # the serial order in one range: any cut launches more kernels
    serial = det.detect(bgr)
    launches_serial = serial.stats["kernel_launches"]
    monkeypatch.delenv("CLFD_NO_OVERLAP")
    monkeypatch.delenv("CLFD_DETECT_CHUNKS")
    assert len(serial.rects) > 0
    for f in (0, 7, 15):
        assert np.array_equal(serial.frame_rects(f), oracle_rects("frontalface_alt", formula_gray(bgr[f]))), f
    for chunks in (2, 8):
        monkeypatch.setenv("CLFD_OVERLAP_CHUNKS", str(chunks))
        got = det.detect(bgr)
        assert got.stats["kernel_launches"] > launches_serial   # the cut really happened
        for f in range(n):
            assert np.array_equal(got.frame_rects(f), serial.frame_rects(f)), (chunks, f)
    monkeypatch.delenv("CLFD_OVERLAP_CHUNKS")

    gray = np.stack([formula_gray(f) for f in batch(2, 3)])
    bgra = batch(3, 4)
    bgr2 = batch(5, 3)
    inputs = [bgr, gray, bgra, bgr2]
    want = [serial, det.detect(gray), det.detect(bgra), det.detect(bgr2)]
    assert not np.array_equal(np.sort(want[0].rects, order=["frame", "w", "y", "x"]),
                              np.sort(want[3].rects, order=["frame", "w", "y", "x"]))
    assert np.array_equal(np.sort(want[2].rects, order=["frame", "w", "y", "x"]),
                          np.sort(det.detect(np.stack([formula_gray(f) for f in bgra])).rects, order=["frame", "w", "y", "x"]))
    pinned = [torch.from_numpy(x).pin_memory() for x in inputs]
    det.submit(pinned[0])
    got = []
    for k in range(1, 4):
        det.submit(pinned[k])
        got.append(det.collect())
    got.append(det.collect())
    for k in range(4):
        for f in range(n):
            assert np.array_equal(got[k].frame_rects(f), want[k].frame_rects(f)), (k, f)
    det.close()


# ---- 5. modes and multi-cascade --------------------------------------------------------------------------------------
def test_scale_cascade_mode(gpu_ctx):
    W, H, n = 640, 480, 3
    frames = colour_frames(W, H, n, 3, first=20)
    assert_channels_differ(frames)
    det = detector(gpu_ctx, ["frontalface_alt"], W, H, n, scale_cascade=True)
    got = det.detect(frames)
    assert len(got.rects) > 0
    oc = oracle_cascade("frontalface_alt")
    for f in range(n):
        want = _sorted(oc.detect_sc(formula_gray(frames[f]), SF, want_codes=False)[0])
        assert np.array_equal(got.frame_rects(f), want), f
    det.close()


@pytest.mark.parametrize("channels", [3, 4])
def test_profileface_fullbody_sf11(gpu_ctx, channels):
    """two cascades, one with tilted features: the multi-cascade path (one range, counter hand-over)"""
    W, H, n = 640, 480, 3
    frames = colour_frames(W, H, n, channels, first=30)
    assert_channels_differ(frames)
    det = detector(gpu_ctx, ["profileface", "fullbody"], W, H, n, sf=1.1)
    got = det.detect(frames)
    want = det.detect(np.stack([formula_gray(f) for f in frames]))
    assert len(want.rects) > 0
    for f in range(n):
        for ci in range(2):
            assert np.array_equal(got.frame_rects(f, ci), want.frame_rects(f, ci)), (f, ci)
    det.close()


# ---- 6. clfd_detect_image --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("channels", [3, 4])
def test_detect_image_is_detect_color_of_one(gpu_ctx, channels):
    W, H = 640, 480
    img = np.ascontiguousarray(colour_frames(W, H, 1, channels, first=40)[0])
    assert_channels_differ(img)
    det = detector(gpu_ctx, ["frontalface_alt"], W, H, 1)
    out, cap = _rect_out(det)
    cnt = C.c_int64()
    abi.check(abi.lib().clfd_detect_image(det._h, C.c_void_p(img.ctypes.data), channels, W * channels, out, cap,
                                          C.byref(cnt)))
    single = _sorted(np.stack([det._rects[:cnt.value][k] for k in ("x", "y", "w", "h")], axis=1))
    batch = detect_color_raw(det, img.ctypes.data, 1, channels, H * W * channels, W * channels).frame_rects(0)
    assert len(batch) > 0
    assert np.array_equal(single, batch)
    assert np.array_equal(batch, oracle_rects("frontalface_alt", formula_gray(img)))
    det.close()


# ---- 7. errors -------------------------------------------------------------------------------------------------------
def test_errors_and_channels_one(gpu_ctx):
    import torch
    W, H, n = 640, 480, 2
    frames = np.ascontiguousarray(colour_frames(W, H, n, 3, first=50))
    assert_channels_differ(frames)
    det = detector(gpu_ctx, ["frontalface_alt"], W, H, n)
    L = abi.lib()
    out, cap = _rect_out(det)
    cnt = C.c_int64()
    p = C.c_void_p(frames.ctypes.data)
    fs, rs = H * W * 3, W * 3
    dev = torch.from_numpy(frames).cuda()
    torch.cuda.synchronize()
    dp = C.c_void_p(dev.data_ptr())

    def calls(count, channels, frame_stride, row_stride):
        return [L.clfd_detect_color(det._h, p, count, channels, frame_stride, row_stride, out, cap, C.byref(cnt)),
                L.clfd_detect_submit_color(det._h, p, count, channels, frame_stride, row_stride),
                L.clfd_detector_enqueue_color(det._h, dp, count, channels, frame_stride, row_stride, None)]
    for channels in (0, 2, 5):
        assert calls(n, channels, fs, rs) == [-1, -1, -1], channels
    assert calls(n, 3, fs, rs - 1) == [-1, -1, -1]
    assert calls(n, 4, fs, rs) == [-1, -1, -1]          # W * 4 bytes do not fit a row stride of W * 3
    assert calls(n + 1, 3, fs, rs) == [-1, -1, -1]
    # the device-input call refuses while a submitted batch is in flight (it shares slot 0's frame buffer)
    det.submit(frames)
    assert L.clfd_detector_enqueue_color(det._h, dp, n, 3, fs, rs, None) == -1
    assert len(det.collect().rects) > 0
    # channels == 1 is the gray call
    gray = np.ascontiguousarray(np.stack([formula_gray(f) for f in frames]))
    want = det.detect(gray)
    assert len(want.rects) > 0
    abi.check(L.clfd_detect_color(det._h, C.c_void_p(gray.ctypes.data), n, 1, H * W, W, out, cap, C.byref(cnt)))
    got = clfd.DetectResult(det._rects[:cnt.value].copy(), {})   # (the device appends rects in no fixed order)
    for f in range(n):
        assert np.array_equal(got.frame_rects(f), want.frame_rects(f)), f
    det.close()
