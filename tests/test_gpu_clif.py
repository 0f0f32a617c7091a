"""GPU parity: pyramid resize and integral images are BIT-EXACT against the oracle
(integer work; SURVEY 8-a rows a1, a2).  Called through the C ABI."""
import numpy as np
import pytest

import oracle
from clfacedetection_b200.frames import octave_frame, uniform_frame

pytestmark = pytest.mark.gpu


def _check_integral(ctx, img, tilted):
    """against the oracle and against numpy: int64 sums wrapped to int32 (the CV_32S integrals wrap once a frame's
    pixels add up to 2^31; the oracle's int32 adds alone are not relied on for that) and exact uint64 squares"""
    s, q, t = ctx.integral(img, tilted=tilted)
    os_, oq, ot = oracle.integral(img, tilted=tilted)
    assert np.array_equal(s, os_)
    assert np.array_equal(q, oq.astype(np.uint64))
    if tilted:
        assert np.array_equal(t, ot)
    ref = np.zeros(s.shape, np.int64)
    ref[1:, 1:] = img.astype(np.int64).cumsum(0).cumsum(1)
    assert np.array_equal(s, (ref & 0xFFFFFFFF).astype(np.uint32).view(np.int32))
    del ref
    sq = np.zeros(q.shape, np.uint64)
    sq[1:, 1:] = (img.astype(np.uint64) ** 2).cumsum(0).cumsum(1)
    assert np.array_equal(q, sq)


@pytest.mark.parametrize("shape", [(1, 1), (5, 7), (31, 33), (257, 64), (640, 480), (1333, 750), (1920, 1080),
                                   (4095, 33), (4096, 31), (8191, 40), (7680, 4320)])
@pytest.mark.parametrize("tilted", [False, True])
def test_integral_uniform_noise(gpu_ctx, shape, tilted):
    w, h = shape
    _check_integral(gpu_ctx, uniform_frame(w, h, 3), tilted)


def test_integral_4k_all_255_needs_64_bit(gpu_ctx):
    """UHD and DCI 4K white frames: the squares pass 2^32; at 4096 x 2160 the int32 sum passes 2^31 and wraps"""
    for w, tilted in ((3840, False), (4096, True)):
        img = np.full((2160, w), 255, np.uint8)
        s, q, _ = gpu_ctx.integral(img)
        assert int(q[-1, -1]) == 255 * 255 * w * 2160 > 2 ** 32
        total = 255 * w * 2160
        assert int(s[-1, -1]) == (total if total < 2 ** 31 else total - 2 ** 32)
        assert (total >= 2 ** 31) == (w == 4096)
        _check_integral(gpu_ctx, img, tilted)


def test_integral_all_zero_and_strided(gpu_ctx):
    _check_integral(gpu_ctx, np.zeros((480, 640), np.uint8), True)
    big = uniform_frame(700, 300, 9)
    view = big[:, :611]          # row stride > width
    s, q, _ = gpu_ctx.integral(np.ascontiguousarray(view))
    os_, oq, _ = oracle.integral(np.ascontiguousarray(view))
    assert np.array_equal(s, os_) and np.array_equal(q, oq.astype(np.uint64))


@pytest.mark.parametrize("src,dst", [((640, 480), (533, 400)), ((640, 480), (640, 480)), ((640, 480), (42, 31)),
                                     ((1920, 1080), (1600, 900)), ((1920, 1080), (926, 521)),
                                     ((1920, 1080), (42, 23)), ((3840, 2160), (3200, 1800)), ((37, 29), (20, 20))])
def test_resize_bit_exact(gpu_ctx, src, dst):
    img = octave_frame(src[0], src[1], 1) if src[0] >= 640 else uniform_frame(src[0], src[1], 1)
    got = gpu_ctx.resize(img, dst[0], dst[1])
    ref = oracle.resize_linear(img, dst[0], dst[1])
    assert np.array_equal(got, ref)


@pytest.mark.parametrize("src,dst", [((1920, 1080), (401, 227)), ((1920, 1080), (320, 180)), ((1920, 1080), (275, 155)),
                                     ((1919, 1079), (1600, 900)), ((1918, 1080), (1001, 563)), ((643, 481), (322, 241)),
                                     ((1921, 1080), (1067, 600)), ((1920, 1080), (1919, 1079)), ((645, 480), (643, 479)),
                                     ((1920, 1080), (6, 4)), ((9, 9), (7, 7)), ((4, 4), (3, 3)), ((5, 3), (1, 1))])
def test_resize_word_paths_bit_exact(gpu_ctx, src, dst):
    """k_resize_colsum reads source rows as 32-bit words where the taps of four (factor < 2) or two (factor <= 6)
    neighbouring pixels fit 8 bytes: factors on either side of those limits, widths that are no multiple of 4
    (partial pixel groups, the row's last word), tiny images"""
    img = uniform_frame(src[0], src[1], 11)
    assert np.array_equal(gpu_ctx.resize(img, dst[0], dst[1]), oracle.resize_linear(img, dst[0], dst[1]))


@pytest.mark.parametrize("w,stride", [(1919, 1919), (1918, 1918), (1917, 1921), (1920, 1920), (1920, 2048)])
def test_resize_device_source_any_alignment(gpu_ctx, w, stride):
    """frames already on the device with any row stride / base alignment: unaligned rows take the byte path"""
    import ctypes as C

    import torch
    from clfacedetection_b200 import abi
    h, dw, dh = 270, int(round(w / 1.2)), 225
    host = np.zeros((h, stride), np.uint8)
    host[:, :w] = uniform_frame(w, h, 12)
    for shift in (0, 1):   # base pointer 4-byte aligned or not
        buf = torch.zeros(h * stride + 8, dtype=torch.uint8, device="cuda")
        buf[shift:shift + h * stride] = torch.from_numpy(host.reshape(-1)).cuda()
        out = torch.zeros((dh, dw), dtype=torch.uint8, device="cuda")
        abi.check(abi.lib().clfd_resize(gpu_ctx._h, C.cast(buf.data_ptr() + shift, C.POINTER(C.c_uint8)), w, h, stride, 1,
                                        C.cast(out.data_ptr(), C.POINTER(C.c_uint8)), dw, dh, dw, 1))
        assert np.array_equal(out.cpu().numpy(), oracle.resize_linear(np.ascontiguousarray(host[:, :w]), dw, dh)), (w, stride, shift)


def test_resize_uniform_noise_1080p_levels(gpu_ctx):
    img = uniform_frame(1920, 1080, 5)
    f = 1.0
    for _ in range(6):
        f *= 1.2
        dw, dh = int(np.rint(1920 / f)), int(np.rint(1080 / f))
        assert np.array_equal(gpu_ctx.resize(img, dw, dh), oracle.resize_linear(img, dw, dh))


def test_integral_linearity_property_1080p(gpu_ctx):
    """size-independent property: integral(a) + integral(b) == integral(a+b) for a+b <= 255"""
    a = (uniform_frame(1920, 1080, 1) // 2).astype(np.uint8)
    b = (uniform_frame(1920, 1080, 2) // 2).astype(np.uint8)
    sa, _, _ = gpu_ctx.integral(a)
    sb, _, _ = gpu_ctx.integral(b)
    sab, _, _ = gpu_ctx.integral((a + b).astype(np.uint8))
    assert np.array_equal(sa.astype(np.int64) + sb, sab.astype(np.int64))
