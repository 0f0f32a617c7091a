"""The reference-facing C++ API (include/clif.h, clod.h over the C ABI) on the GPU: the demo
client examples/clod_demo and -- when it was built in the dev container -- the reference's own
main.cpp, compiled byte for byte against the shim (tests/_build/ref_main)."""
import os
import subprocess

import numpy as np
import pytest

import oracle
from conftest import cascade_path, oracle_cascade

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _write_pgm(path, img):
    with open(path, "wb") as f:
        f.write(b"P5 %d %d 255\n" % (img.shape[1], img.shape[0]))
        f.write(img.tobytes())


@pytest.mark.parametrize("min_neighbors", [0, 2])
def test_clod_demo_matches_oracle(tmp_path, min_neighbors):
    from clfacedetection_b200.frames import octave_frame
    img = octave_frame(640, 480, 0)
    pgm = str(tmp_path / "frame.pgm")
    _write_pgm(pgm, img)
    out = subprocess.run([os.path.join(ROOT, "examples", "clod_demo"), cascade_path("frontalface_default"), pgm, "1.2",
                          str(min_neighbors), "24", "24"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.strip().splitlines()
    # clifIntegral of the (gray -> BGR -> gray) frame: bottom-right corner of sum and squared sum.
    # gray replicated to BGR converts back to itself: (v*1868 + v*9617 + v*4899 + 8192) >> 14 == v
    s, q, _ = oracle.integral(img)
    assert lines[0].split() == ["integral", str(int(s[-1, -1])), str(int(q[-1, -1]))]
    n = int(lines[1].split()[1])
    got = np.array([[int(v) for v in ln.split()[:4]] for ln in lines[2:2 + n]], np.int32).reshape(-1, 4)
    rects, _, _, _, _ = oracle_cascade("frontalface_default").detect(img, 1.2, (24, 24))
    if min_neighbors:
        rects, weights = oracle.group_rectangles(rects, min_neighbors)
        w_got = [float(ln.split()[4]) for ln in lines[2:2 + n]]
        assert w_got == [float(w) for w in weights]
        assert np.array_equal(got, rects)
    else:
        key = lambda r: r[np.lexsort((r[:, 0], r[:, 1], r[:, 2]))] if len(r) else r
        assert np.array_equal(key(got), key(rects))


def test_clod_demo_scale_cascade_mode_matches_ref_sc(tmp_path):
    """clodSetDetectionMode(data, 1): the semantics of the cvHaarDetectObjects call of main.cpp:145."""
    from clfacedetection_b200.frames import octave_frame
    img = octave_frame(640, 480, 3)
    pgm = str(tmp_path / "frame.pgm")
    _write_pgm(pgm, img)
    out = subprocess.run([os.path.join(ROOT, "examples", "clod_demo"), cascade_path("frontalface_alt"), pgm, "1.2", "0", "0", "0", "1"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.strip().splitlines()
    n = int(lines[1].split()[1])
    got = np.array([[int(v) for v in ln.split()[:4]] for ln in lines[2:2 + n]], np.int32).reshape(-1, 4)
    rects, _, _, _ = oracle_cascade("frontalface_alt").detect_sc(img, 1.2)
    key = lambda r: r[np.lexsort((r[:, 0], r[:, 1], r[:, 2]))] if len(r) else r
    assert len(rects) > 0 and np.array_equal(key(got), key(rects))


def test_reference_main_runs_unchanged():
    exe = os.path.join(ROOT, "tests", "_build", "ref_main")
    if not os.path.exists(exe):
        pytest.skip("tests/_build/ref_main is built by the CPU suite where CLFD_REFERENCE_DIR names the original sources")
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr
    for label in ("OpenCV:", "OpenCL (optimized):", "OpenCL (per-stage):"):
        assert label in out.stdout


def test_blank_frame_with_grouping_returns_no_matches(tmp_path):
    """ADVICE r1 (high): zero raw detections + min_neighbors != 0 used to abort in the grouping call;
    the reference returns match_count = 0 (the most common real input: a frame without a face)."""
    pgm = str(tmp_path / "blank.pgm")
    _write_pgm(pgm, np.full((240, 320), 128, np.uint8))
    out = subprocess.run([os.path.join(ROOT, "examples", "clod_demo"), cascade_path("frontalface_alt"), pgm, "1.2", "2"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    assert out.stdout.strip().splitlines()[1] == "matches 0"


def test_release_and_reload_never_reuses_a_stale_plan(tmp_path):
    """ADVICE r1 (medium): load A, detect, release A, load B, detect on the same frame shape -- B's
    malloc'd cascade often lands on A's address; the cached plan must not be A's.  Both entry points
    (clodDetectObjects, cvHaarDetectObjects), two rounds over three cascades."""
    from clfacedetection_b200.frames import octave_frame
    img = octave_frame(480, 360, 5)
    pgm = str(tmp_path / "frame.pgm")
    _write_pgm(pgm, img)
    names = ["eye", "mcs_lefteye", "frontalface_alt2"]
    out = subprocess.run([os.path.join(ROOT, "examples", "clod_lifecycle"), pgm, "1.2", "2"] + [cascade_path(n) for n in names],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.strip().splitlines()
    want = {}
    for n in names:
        raw, _, _, _, _ = oracle_cascade(n).detect(img, 1.2)
        g, w = oracle.group_rectangles(raw, 2)
        want[cascade_path(n)] = [[int(v) for v in r] + [float(x)] for r, x in zip(g, w)]
    assert sum(len(v) for v in want.values()) > 0
    i = 0
    blocks = 0
    while i < len(lines):
        tag, rnd, path, n = lines[i].split()
        got = [[float(v) for v in ln.split()] for ln in lines[i + 1:i + 1 + int(n)]]
        assert got == [[float(v) for v in r] for r in want[path]], (tag, rnd, path)
        i += 1 + int(n)
        blocks += 1
    assert blocks == 2 * 2 * len(names)


def test_bgr_to_gray_colour_pixels(gpu_ctx):
    """SURVEY 8-f row 2: random COLOUR pixels (a gray image replicated to B, G, R converts to itself
    under any coefficient permutation) against OpenCV's fixed point (B*1868 + G*9617 + R*4899 + 8192) >> 14
    -- what OpenCV 2.4's cvCvtColor(BGR2GRAY) at tempcv.cpp:1250 / clif.cpp:249,328 computes -- and, where cv2
    is installed, within one grey level of cv2 4.x's cvtColor; 3 and 4 channels."""
    rng = np.random.default_rng(11)
    for (h, w, c) in ((37, 53, 3), (240, 321, 3), (64, 100, 4), (1, 1, 3), (1080, 1920, 3)):
        img = rng.integers(0, 256, size=(h, w + 3, c), dtype=np.uint8)[:, :w]   # row stride > w*c
        exp = ((img[..., 0].astype(np.int64) * 1868 + img[..., 1].astype(np.int64) * 9617 +
                img[..., 2].astype(np.int64) * 4899 + 8192) >> 14).astype(np.uint8)
        got = gpu_ctx.bgr_to_gray(np.ascontiguousarray(img))
        assert np.array_equal(got, exp), (h, w, c)
        try:
            import cv2
        except ImportError:
            continue
        # OpenCV 4.x moved to 15-bit coefficients (3735, 19235, 9798): same weights, one more bit, so it
        # may differ from the 2.4-era 14-bit formula by one grey level -- a sanity check, not the pin
        ref = cv2.cvtColor(np.ascontiguousarray(img), cv2.COLOR_BGR2GRAY if c == 3 else cv2.COLOR_BGRA2GRAY)
        assert np.abs(got.astype(np.int32) - ref.astype(np.int32)).max() <= 1, (h, w, c)
    # pure primaries pin which channel gets which coefficient
    prim = np.zeros((1, 3, 3), np.uint8)
    prim[0, 0, 0] = prim[0, 1, 1] = prim[0, 2, 2] = 255
    assert gpu_ctx.bgr_to_gray(prim).tolist() == [[29, 150, 76]]


def test_integral_image_colour_in_one_call(gpu_ctx):
    """clfd_integral_image (clifGrayscaleIntegral, clif.cpp:318-381): colour pixels -> gray -> integrals on the device
    == oracle integral of the fixed-point gray plane; also 1-channel input and the optional gray output"""
    rng = np.random.default_rng(8)
    for shape in ((37, 53, 3), (240, 321, 3), (100, 64, 4), (75, 90)):
        img = rng.integers(0, 256, size=shape, dtype=np.uint8)
        if img.ndim == 3:
            b, g, r = (img[..., k].astype(np.int64) for k in range(3))
            gray = ((b * 1868 + g * 9617 + r * 4899 + 8192) >> 14).astype(np.uint8)
        else:
            gray = img
        s, q, t, got_gray = gpu_ctx.integral_image(img, tilted=True, want_gray=True)
        os_, oq, ot = oracle.integral(gray, tilted=True)
        assert np.array_equal(got_gray, gray)
        assert np.array_equal(s, os_) and np.array_equal(q, oq.astype(np.uint64)) and np.array_equal(t, ot)
