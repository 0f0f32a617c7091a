"""The detector's pyramid and integral images, level by level, against plain references built from the original frame.

Every level of every cascade and every frame of the last batch is read back with `Detector.read_level` and compared
with `oracle.resize_linear` for the pyramid and with numpy for the integrals: int64 cumulative sums wrapped to int32
(the reference's CV_32S integrals wrap the same way on large bright frames), exact uint64 squares (the low 32 bits in
pyramid mode, which keeps them modulo 2^32) and an int64 row recurrence for the tilted integral.  The oracle's integral
must agree as well.  The frame geometries sit at the kernels' boundaries: every thread-count class of
`k_integral_rows`, the tile edges of `k_tilt_tiles`, the row-block groups of `k_colscan`, the 65535-row limit of the
32-bit column carries, frames wider than the 8191-pixel level limit, and 8K UHD frames whose sums pass 2^31."""
import numpy as np
import pytest
import torch

import clfacedetection_b200 as clfd
import oracle
from clfacedetection_b200.frames import octave_frame, uniform_frame
from conftest import cascade_path, oracle_cascade

pytestmark = pytest.mark.gpu

SF = 1.2
STUMP, TILTED = "frontalface_alt", "lowerbody"
ENVS = {"default": {}, "sq64": {"CLFD_SQ64": "1"}, "no_di": {"CLFD_NO_DI": "1"}}
# k_integral_rows class (32 << c threads per row) of level 0 at each width of test_width_classes
WIDTH_CLASS = {255: 0, 256: 1, 511: 1, 512: 2, 1023: 2, 1024: 3, 2047: 3, 2048: 4, 4095: 4, 4096: 5, 8191: 5}


@pytest.fixture(scope="module")
def cas():
    out = {}

    def get(name):
        if name not in out:
            out[name] = clfd.Cascade(cascade_path(name))
        return out[name]
    return get


def integral_class(w):
    """the k_integral_rows class of a level w pixels wide: the smallest c with (32 << c) * 8 >= round8(w + 1)"""
    pitch = (w + 1 + 7) // 8 * 8
    return next(c for c in range(6) if (32 << c) * 8 >= pitch)


def bright(W, H, seed, offset=0):
    """a textured frame: octave noise, raised by `offset` and clipped"""
    return np.clip(octave_frame(W, H, seed).astype(np.int32) + offset, 0, 255).astype(np.uint8)


def wrap32(a):
    """int64 -> int32 modulo 2^32"""
    return (a & 0xFFFFFFFF).astype(np.uint32).view(np.int32)


def ref_sum(img):
    s = np.zeros((img.shape[0] + 1, img.shape[1] + 1), np.int64)
    s[1:, 1:] = img.astype(np.int64).cumsum(0).cumsum(1)
    return s


def ref_sqsum(img):
    q = np.zeros((img.shape[0] + 1, img.shape[1] + 1), np.uint64)
    v = img.astype(np.uint64)
    q[1:, 1:] = (v * v).cumsum(0).cumsum(1)
    return q


def ref_tilted(img):
    """tilted[Y][X] = sum of img[y][x] over y < Y, |x - (X - 1)| <= Y - 1 - y, in int64, from the up-left and up-right
    diagonal prefix sums A(y, x) = img[y][x] + A(y-1, x-1) and B(y, x) = img[y][x] + B(y-1, x+1), one row at a time"""
    h, w = img.shape
    t = np.zeros((h + 1, w + 1), np.int64)
    A = np.zeros(w + 2, np.int64)   # indexed x + 1: x = -1 and x = w are zero pads
    B = np.zeros(w + 2, np.int64)
    A1, B1 = np.zeros_like(A), np.zeros_like(B)
    for Y in range(1, h + 1):
        p = img[Y - 1].astype(np.int64)
        t[Y, 0] = t[Y - 1, 0] + B[1]
        A1[1:w + 1] = p + A[0:w]
        B1[1:w + 1] = p + B[2:w + 2]
        t[Y, 1:] = t[Y - 1, 1:] + A1[1:w + 1] + B1[1:w + 1] - p
        A, A1 = A1, A
        B, B1 = B1, B
    return t


def _same(got, want, what):
    if np.array_equal(got, want):
        return
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    y, x = np.argwhere(got != want)[0]
    n = int(np.count_nonzero(got != want))
    raise AssertionError(f"{what}: {n} of {got.size} differ, first at (y={y}, x={x}): gpu {got[y, x]} reference {want[y, x]}")


def check_levels(det, frames, *, sq_full, tilted, cascades=None, levels=None):
    """every level (`levels`: indices, default all) of every cascade and every frame of the last batch against the
    references -> (k_integral_rows classes seen, largest int64 sum or tilted value of any level)"""
    classes, peak = set(), 0
    for ci in range(len(det.cascades)) if cascades is None else cascades:
        lvs = det.levels(ci)
        for f, frame in enumerate(frames):
            for li in range(len(lvs)) if levels is None else levels:
                lv = lvs[li]
                where = f"cascade {ci} frame {f} level {li} ({lv.img_w}x{lv.img_h})"
                pyr, s, q, t = det.read_level(li, frame=f, cascade=ci, tilted=tilted)
                want_pyr = oracle.resize_linear(frame, lv.img_w, lv.img_h)
                _same(pyr, want_pyr, f"{where} pyr")
                del pyr
                os_, oq, ot = oracle.integral(want_pyr, tilted=tilted)
                rs = ref_sum(want_pyr)
                peak = max(peak, int(rs[-1, -1]))
                rs = wrap32(rs)
                _same(os_, rs, f"{where} oracle sum vs numpy")
                _same(s, rs, f"{where} sum")
                del s, os_, rs
                rq = ref_sqsum(want_pyr)
                _same(oq.astype(np.uint64), rq, f"{where} oracle sqsum vs numpy")
                del oq
                _same(q, rq if sq_full else rq & np.uint64(0xFFFFFFFF), f"{where} sqsum")
                del q, rq
                if tilted:
                    rt = ref_tilted(want_pyr)
                    peak = max(peak, int(rt.max()))
                    rt = wrap32(rt)
                    _same(ot, rt, f"{where} oracle tilted vs numpy")
                    _same(t, rt, f"{where} tilted")
                    del t, ot, rt
                classes.add(integral_class(lv.img_w))
    return classes, peak


def _env(monkeypatch, name):
    for k, v in ENVS[name].items():
        monkeypatch.setenv(k, v)


def _run(gpu_ctx, cascades, frames, **kw):
    """a detector for `frames` that has run them -> (detector, result)"""
    det = clfd.Detector(gpu_ctx, cascades, frames.shape[2], frames.shape[1], max_batch=len(frames), scale_factor=SF, **kw)
    return det, det.detect(frames)


# ---- 1. every k_integral_rows class, level 0 exact ------------------------------------------------------------------
@pytest.mark.parametrize("env", list(ENVS))
@pytest.mark.parametrize("w", [255, 256, 511, 512, 1023, 1024, 2047, 2048, 4095, 4096, 8191])
def test_width_classes(gpu_ctx, cas, monkeypatch, w, env):
    """Level 0 of a frame at either side of each class boundary of k_integral_rows (256, 512, ... 8192 columns of
    pitch); the 512- and 1024-thread classes combine warp totals across warps, and textured frames make every warp
    total different.  A stump and a tilted cascade share the detector: the 32-bit squares, the de-interleaved sum and
    the tilted kernels all run (CLFD_SQ64 / CLFD_NO_DI switch the first two off)."""
    _env(monkeypatch, env)
    H = 64
    frames = np.stack([bright(w, H, 1, 40), uniform_frame(w, H, 2)])
    det, _ = _run(gpu_ctx, [cas(STUMP), cas(TILTED)], frames)
    lvs = det.levels(0)
    assert lvs[0].img_w == w and lvs[0].ystep == 2
    classes, _ = check_levels(det, frames, sq_full=env == "sq64", tilted=True)
    assert integral_class(w) == WIDTH_CLASS[w] and WIDTH_CLASS[w] in classes
    det.close()


# ---- 2. tilted tile and resize chunk edges --------------------------------------------------------------------------
@pytest.mark.parametrize("w", [127, 128, 129, 191, 192, 383, 384])
def test_tilted_tile_and_resize_edges(gpu_ctx, cas, w):
    """k_tilt_tiles covers w + 1 columns in tiles of 192 (w = 191, 383 end exactly on a tile edge), k_resize_colsum
    in 128-column chunks per warp"""
    H = 72
    frames = np.stack([bright(w, H, 3, 30), uniform_frame(w, H, 4)])
    det, _ = _run(gpu_ctx, [cas(TILTED)], frames)
    assert det.levels(0)[0].img_w == w
    check_levels(det, frames, sq_full=False, tilted=True)
    det.close()


# ---- 3. heights -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("h", [31, 32, 33, 256, 257])
def test_heights_across_row_blocks(gpu_ctx, cas, h):
    """heights on either side of one 32-row block and of eight, the carries k_colscan scans (256 rows)"""
    W = 300
    frames = np.stack([bright(W, h, 5, 20), uniform_frame(W, h, 6)])
    det, _ = _run(gpu_ctx, [cas(STUMP), cas(TILTED)], frames)
    assert det.levels(1)[0].img_h == h
    check_levels(det, frames, sq_full=False, tilted=True)
    det.close()


@pytest.mark.parametrize("sq64", [False, True])
def test_tall_frame_column_square_carry(gpu_ctx, cas, monkeypatch, sq64):
    """64 x 65535, all 255 in every other 8-column group: a column's sum of squares reaches 65535 * 255^2 = 4.26e9,
    just under the 2^32 of the u32 column carries.  With CLFD_SQ64 the full 64-bit squares are compared."""
    if sq64:
        monkeypatch.setenv("CLFD_SQ64", "1")
    W, H = 64, 65535
    frame = bright(W, H, 7, 0)
    cols = (np.arange(W) // 8) % 2 == 0
    frame[:, cols] = 255
    frames = frame[None]
    det, _ = _run(gpu_ctx, [cas(STUMP)], frames)
    assert det.levels(0)[0].img_h == H
    assert int(ref_sqsum(frame[:, :1])[-1, -1]) == 65535 * 255 ** 2 > 2 ** 32 - 2 ** 28
    check_levels(det, frames, sq_full=sq64, tilted=False)
    det.close()


# ---- 4. wider than 8191 ---------------------------------------------------------------------------------------------
def test_wider_than_8191_with_min_size(gpu_ctx, cas):
    """12000 x 160: with a minimum window that skips every level wider than 8191 the detector is created and its levels
    match; without one, 8192 x 64 is refused with CLFD_ERR_INVALID naming the limit"""
    W, H = 12000, 160
    frames = np.stack([bright(W, H, 8, 30)])
    det, _ = _run(gpu_ctx, [cas(STUMP), cas(TILTED)], frames, min_size=(30, 30))
    lvs = det.levels(0)
    assert lvs and max(l.img_w for l in lvs) <= 8191 and lvs[0].img_w > 4096
    classes, _ = check_levels(det, frames, sq_full=False, tilted=True)
    assert 5 in classes
    det.close()
    for shape in ((8192, 64), (W, H)):
        with pytest.raises(clfd.ClfdError, match="8191") as e:
            clfd.Detector(gpu_ctx, [cas(STUMP)], shape[0], shape[1], scale_factor=SF)
        assert e.value.status == -1   # CLFD_ERR_INVALID


# ---- 5. int32 wrap at 7680 x 4320 -----------------------------------------------------------------------------------
def _sorted(r):
    r = np.asarray(r, np.int32).reshape(-1, 4)
    return r[np.lexsort((r[:, 0], r[:, 1], r[:, 2]))] if len(r) else r


@pytest.fixture(scope="module")
def uhd_frames():
    W, H = 7680, 4320
    return np.stack([bright(W, H, 9, 96), np.full((H, W), 255, np.uint8)])


def test_uhd_pyramid_wraps_int32(gpu_ctx, cas, uhd_frames):
    """8K UHD frames whose pixel totals pass 2^31: every level of a pyramid-mode detector, its exit codes and rects
    against the oracle, and the production detector's rects (the white frame takes the flat-window table)"""
    frames = uhd_frames
    oc = oracle_cascade(STUMP)
    det, res = _run(gpu_ctx, [cas(STUMP)], frames, want_codes=True)
    codes = det.codes(0, len(frames))
    orects = []
    for f in range(len(frames)):
        rects, ocodes, _, _, _ = oc.detect(frames[f], SF)
        bad = np.flatnonzero(codes[f] != ocodes)
        assert bad.size == 0, f"frame {f}: {bad.size} of {ocodes.size} exit codes differ, first at {bad[:5]} " \
                              f"gpu {codes[f][bad[:5]]} oracle {ocodes[bad[:5]]}"
        orects.append(_sorted(rects))
        assert np.array_equal(res.frame_rects(f), orects[f]), f"frame {f}: rect sets differ"
        if f == 0:
            assert len(np.unique(ocodes)) > 5 and len(rects) > 0
    del codes
    _, peak = check_levels(det, frames, sq_full=False, tilted=False)
    assert peak >= 2 ** 31 and int(frames[0].astype(np.int64).sum()) >= 2 ** 31
    det.close()
    det, got = _run(gpu_ctx, [cas(STUMP)], frames)
    for f in range(len(frames)):
        assert np.array_equal(got.frame_rects(f), orects[f]), f"production, frame {f}: rect sets differ"
    det.close()


def test_uhd_scale_cascade_wraps_int32(gpu_ctx, cas, uhd_frames):
    """the same frames in scale-cascade mode: codes and rects against the oracle, and its single image (64-bit squares)
    through read_level, which every level index reads"""
    frames = uhd_frames
    oc = oracle_cascade(STUMP)
    det, res = _run(gpu_ctx, [cas(STUMP)], frames, scale_cascade=True)
    codes = det.codes(0, len(frames))
    for f in range(len(frames)):
        rects, ocodes, _, _ = oc.detect_sc(frames[f], SF)
        bad = np.flatnonzero(codes[f] != ocodes)
        assert bad.size == 0, f"frame {f}: {bad.size} of {ocodes.size} codes differ, first at {bad[:5]} " \
                              f"gpu {codes[f][bad[:5]]} oracle {ocodes[bad[:5]]}"
        assert np.array_equal(res.frame_rects(f), _sorted(rects)), f"frame {f}: rect sets differ"
    del codes
    lvs = det.levels(0)
    assert len(lvs) > 10 and all((l.img_w, l.img_h) == frames.shape[2:0:-1] for l in lvs)
    _, peak = check_levels(det, frames, sq_full=True, tilted=False, levels=[0])
    assert peak >= 2 ** 31
    s0 = det.read_level(0, frame=1)[1]
    assert np.array_equal(det.read_level(len(lvs) - 1, frame=1)[1], s0)
    det.close()


# ---- 6. batches and input layouts -----------------------------------------------------------------------------------
def test_nine_frame_batch_every_frame(gpu_ctx, cas):
    """9 distinct frames of a cascade the tile kernel finishes: the batch runs in overlapped chunks whose pyramid,
    integral and tilted writes start at a per-chunk frame offset"""
    W, H = 1000, 300
    info = cas(TILTED).info
    assert info.dense_stages == info.n_stages and info.has_tilted
    frames = np.stack([bright(W, H, 10 + i, 10 * i) if i % 2 == 0 else uniform_frame(W, H, 10 + i) for i in range(9)])
    det, _ = _run(gpu_ctx, [cas(TILTED)], frames)
    check_levels(det, frames, sq_full=False, tilted=True)
    det.close()


@pytest.mark.parametrize("shift", [0, 1])
def test_device_input_with_odd_strides(gpu_ctx, cas, shift):
    """device-resident frames with row stride W + 13 and an odd frame stride, the first frame 4-byte aligned (the word
    path of k_resize_colsum) or one byte off (the byte path)"""
    W, H, n = 1000, 300, 2
    rs = W + 13
    fs = rs * H + 7
    frames = np.stack([bright(W, H, 20, 15), uniform_frame(W, H, 21)])
    host = np.zeros(fs * n + 16, np.uint8)
    for f in range(n):
        host[f * fs:f * fs + rs * H].reshape(H, rs)[:, :W] = frames[f]
    buf = torch.zeros(len(host) + 8, dtype=torch.uint8, device="cuda")
    buf[shift:shift + len(host)] = torch.from_numpy(host).cuda()
    torch.cuda.synchronize()
    det = clfd.Detector(gpu_ctx, [cas(STUMP), cas(TILTED)], W, H, max_batch=n, scale_factor=SF)
    det.enqueue(buf.data_ptr() + shift, n, fs, rs)
    det.fetch()
    check_levels(det, frames, sq_full=False, tilted=True, cascades=[0])
    det.close()


def test_resize_byte_path(gpu_ctx, cas, monkeypatch):
    """every level through the byte path of k_resize_colsum (CLFD_RESIZE_BYTES)"""
    monkeypatch.setenv("CLFD_RESIZE_BYTES", "1")
    W, H = 1001, 299
    frames = np.stack([bright(W, H, 22, 25)])
    det, _ = _run(gpu_ctx, [cas(STUMP), cas(TILTED)], frames)
    check_levels(det, frames, sq_full=False, tilted=True, cascades=[0])
    det.close()


# ---- 7. union pyramid -----------------------------------------------------------------------------------------------
def test_union_pyramid_every_cascade(gpu_ctx, cas):
    """frontalface_alt (20 x 20), fullbody (14 x 28) and eye (20 x 20) share one pyramid; a minimum window of 30 x 30
    drops different leading levels for the 14-pixel-wide fullbody window than for the others, so the cascades' level
    lists differ.  Every cascade's levels are read through its own index."""
    W, H = 640, 360
    frames = np.stack([bright(W, H, 30, 20), uniform_frame(W, H, 31)])
    det, _ = _run(gpu_ctx, [cas(STUMP), cas("fullbody"), cas("eye")], frames, min_size=(30, 30))
    sizes = [[(l.img_w, l.img_h) for l in det.levels(ci)] for ci in range(3)]
    assert sizes[0] != sizes[1] and all(sizes)
    check_levels(det, frames, sq_full=False, tilted=True)
    det.close()


# ---- 8. scale-cascade images ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(8191, 48), (1000, 300)])
def test_scale_cascade_image(gpu_ctx, cas, shape):
    """scale-cascade mode keeps one image with 64-bit squares and a tilted integral; read_level returns it for every
    level index"""
    W, H = shape
    frames = np.stack([bright(W, H, 40, 30), uniform_frame(W, H, 41)])
    det, _ = _run(gpu_ctx, [cas("fullbody")], frames, scale_cascade=True)
    n = len(det.levels(0))
    assert n >= 1
    classes, _ = check_levels(det, frames, sq_full=True, tilted=True, levels=[0])
    assert integral_class(W) in classes
    last = det.read_level(n - 1, frame=1, tilted=True)
    first = det.read_level(0, frame=1, tilted=True)
    for a, b in zip(last, first):
        assert np.array_equal(a, b)
    det.close()
