"""GPU parity with the oracle for cascades of every window geometry (tests/synthetic_cascades.py): the smallest window,
tall and flat ones, the sizes where the tile kernel's ystep-2 tile stops fitting shared memory, and the 255-pixel limit
of the image-pyramid mode.  Exit codes, rects and reject levels must equal the oracle's exactly."""
import numpy as np
import pytest

import clfacedetection_b200 as clfd
import oracle
from clfacedetection_b200.frames import octave_frame, uniform_frame
from conftest import cascade_path, oracle_cascade
from synthetic_cascades import BEYOND_CASES, GEOMETRY_CASES, SPLIT_CASES, geometry_cascade

pytestmark = pytest.mark.gpu

W, H = 640, 480
PYRAMID_CASES = [c for c in GEOMETRY_CASES if c not in BEYOND_CASES]
SF = 1.2


def _sorted(r):
    r = np.asarray(r, np.int32).reshape(-1, 4)
    return r[np.lexsort((r[:, 0], r[:, 1], r[:, 2]))] if len(r) else r


def _flat_board(seed):
    """flat patches of many values with noise between them, as in test_flat_regions_take_the_table_and_equal_the_oracle"""
    board = octave_frame(W, H, seed)
    for v in range(0, 256, 2):   # 28 x 40 patches of every other value, 12 and 20 pixels of noise between them
        y, x = (v // 32) * 60, ((v // 2) % 16) * 40
        board[y:y + 40, x:x + 28] = v
    return board


def _frames(case):
    seed = GEOMETRY_CASES[case]["seed"]
    return np.stack([octave_frame(W, H, seed), uniform_frame(W, H, seed)])


def _level_of(levels, n):
    """index of the level each of the window indices `n` belongs to (windows are numbered level by level)"""
    ends = np.cumsum([l.nx * l.ny for l in levels])
    return np.searchsorted(ends, n, side="right")


def _accepted(flat, codes):
    """exit codes: the number of stages passed; for a stage tree, 2 * last stage + accepted"""
    return codes % 2 == 1 if np.any(flat.st_next >= 0) else codes == flat.n_stages


def _not_vacuous(case, flat, codes, levels):
    """the oracle's exit codes split the windows over the stages, some windows are accepted, and for the geometries
    whose ystep-2 tile does not fit, windows are accepted on the ystep-2 levels (factor <= 2)"""
    codes = np.concatenate([np.asarray(c).ravel() for c in codes])
    assert len(np.unique(codes)) * 2 >= flat.n_stages, (case, np.unique(codes))
    accepted = np.flatnonzero(_accepted(flat, codes))
    assert accepted.size > 0, case
    if case in SPLIT_CASES:
        wpf = sum(l.nx * l.ny for l in levels)
        lv = _level_of(levels, accepted % wpf)
        assert any(levels[i].factor <= 2 for i in lv), case


def _compare_diagnostic(gpu_ctx, cascades, frames):
    """want_codes detector over `cascades` (oracle cascade, clfd cascade) pairs: exit codes, rects and reject levels of
    every cascade against the oracle -> the oracle's codes per cascade"""
    n = len(frames)
    det = clfd.Detector(gpu_ctx, [c for _, c in cascades], W, H, max_batch=n, scale_factor=SF, want_codes=True)
    res = det.detect(frames)
    out = []
    for ci, (oc, _) in enumerate(cascades):
        codes = det.codes(ci, n)
        assert len(det.levels(ci)) == len(oc.plan_levels(W, H, SF))
        got_r, got_lv, got_wt = det.reject_levels(ci)
        at = 0
        ocodes_all = []
        for f in range(n):
            rects, ocodes, _, st, _ = oc.detect(frames[f], SF)
            assert st.windows == det.windows_per_frame(ci)
            bad = np.flatnonzero(codes[f] != ocodes)
            assert bad.size == 0, f"{oc.flat.name} frame {f}: {bad.size} of {ocodes.size} exit codes differ, first at " \
                                  f"{bad[:5]} gpu {codes[f][bad[:5]]} oracle {ocodes[bad[:5]]}"
            assert np.array_equal(res.frame_rects(f, ci), _sorted(rects)), f"{oc.flat.name} frame {f}: rect sets differ"
            orr, olv, owt = oc.detect_roc(frames[f], SF)
            k = len(orr)
            mine = got_r[at:at + k]
            assert np.all(mine["frame"] == f), f"{oc.flat.name} frame {f}: reject-level candidates differ"
            assert np.array_equal(np.stack([mine["x"], mine["y"], mine["w"], mine["h"]], 1).reshape(-1, 4), orr.reshape(-1, 4))
            assert np.array_equal(got_lv[at:at + k], olv)
            assert got_wt[at:at + k].tobytes() == owt.tobytes()
            at += k
            ocodes_all.append(ocodes)
        assert at == len(got_r)
        out.append(ocodes_all)
    det.close()
    return out


def _production_rects(gpu_ctx, cascades, frames, monkeypatch, env=None):
    if env:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
    det = clfd.Detector(gpu_ctx, cascades, W, H, max_batch=len(frames), scale_factor=SF)
    res = det.detect(frames)
    det.close()
    if env:
        for k in env:
            monkeypatch.delenv(k)
    return res


@pytest.mark.parametrize("case", PYRAMID_CASES)
def test_pyramid_codes_rects_and_reject_levels_equal_oracle(gpu_ctx, case):
    flat = geometry_cascade(case)
    oc = oracle.Cascade(flat)
    cas = clfd.Cascade(flat=flat)
    frames = _frames(case)
    ocodes = _compare_diagnostic(gpu_ctx, [(oc, cas)], frames)[0]
    _not_vacuous(case, flat, ocodes, oc.plan_levels(W, H, SF))


@pytest.mark.parametrize("case", PYRAMID_CASES)
def test_pyramid_production_rects_with_flat_frames_equal_oracle(gpu_ctx, monkeypatch, case):
    """the production detector (flat windows looked up in the measured table) on an all-0 frame, an all-255 frame and
    a board of flat patches with noise between them; the same with the table switched off"""
    flat = geometry_cascade(case)
    oc = oracle.Cascade(flat)
    cas = clfd.Cascade(flat=flat)
    seed = GEOMETRY_CASES[case]["seed"]
    frames = np.stack([np.zeros((H, W), np.uint8), np.full((H, W), 255, np.uint8), _flat_board(seed)])
    got = _production_rects(gpu_ctx, cas, frames, monkeypatch)
    plain = _production_rects(gpu_ctx, cas, frames, monkeypatch, {"CLFD_NO_FLAT_TABLE": "1"})
    total = 0
    for f in range(len(frames)):
        want = _sorted(oc.detect(frames[f], SF, want_codes=False)[0])
        assert np.array_equal(got.frame_rects(f), want), (case, f, len(got.frame_rects(f)), len(want))
        assert np.array_equal(plain.frame_rects(f), want), (case, f, len(plain.frame_rects(f)), len(want))
        total += len(want)
    assert total > 0


@pytest.mark.parametrize("case", list(GEOMETRY_CASES))
def test_scale_cascade_codes_and_rects_equal_oracle(gpu_ctx, case):
    flat = geometry_cascade(case)
    oc = oracle.Cascade(flat)
    cas = clfd.Cascade(flat=flat)
    frames = _frames(case)
    det = clfd.Detector(gpu_ctx, cas, W, H, max_batch=len(frames), scale_factor=SF, scale_cascade=True)
    res = det.detect(frames)
    codes = det.codes(0, len(frames))
    seen = []
    for f in range(len(frames)):
        rects, ocodes, _, levels = oc.detect_sc(frames[f], SF)
        # the oracle also lists the scales whose window grid is empty (the 3 x 3 window's last scale: 412 x 412 windows
        # at a step of 137 on a 480-row frame); the detector plans only scales that have windows
        assert [(l.nx, l.ny, l.win_w, l.win_h) for l in levels if l.nx * l.ny > 0] == \
            [(l.nx, l.ny, l.win_w, l.win_h) for l in det.levels()]
        bad = np.flatnonzero(codes[f] != ocodes)
        assert bad.size == 0, f"{case} frame {f}: {bad.size} of {ocodes.size} codes differ, first {bad[:5]} " \
                              f"gpu {codes[f][bad[:5]]} oracle {ocodes[bad[:5]]}"
        assert np.array_equal(res.frame_rects(f), _sorted(rects)), f"{case} frame {f}: rect sets differ"
        seen.append(ocodes[ocodes >= 0])
    seen = np.concatenate(seen)
    assert len(np.unique(seen)) * 2 >= flat.n_stages and _accepted(flat, seen).any(), case
    det.close()


@pytest.mark.parametrize("case", BEYOND_CASES)
def test_pyramid_mode_rejects_windows_beyond_255(gpu_ctx, case):
    """the image-pyramid kernels keep corner offsets in bytes and squared integrals modulo 2^32: a cascade whose
    window is wider or taller than 255 pixels is refused there (the scale-cascade mode takes it, see above)"""
    cas = clfd.Cascade(flat=geometry_cascade(case))
    for want_codes in (False, True):
        with pytest.raises(clfd.ClfdError, match="255") as e:
            clfd.Detector(gpu_ctx, cas, W, H, scale_factor=SF, want_codes=want_codes)
        assert e.value.status == -1   # CLFD_ERR_INVALID
    # ... also beside a cascade the mode can take
    with pytest.raises(clfd.ClfdError, match="255"):
        clfd.Detector(gpu_ctx, [clfd.Cascade(cascade_path("frontalface_alt")), cas], W, H, scale_factor=SF)


@pytest.mark.parametrize("sq64", [False, True])
def test_255_window_at_the_squared_integral_limit(gpu_ctx, monkeypatch, sq64):
    """A 255 x 255 window on an all-255 frame: its variance rectangle's sum of squares is 253^2 * 255^2 = 4.16e9, 3 %
    below 2^32; a 0/255 checkerboard puts half of that in every window.  The squared integral kept modulo 2^32 must give
    what the 64-bit one (CLFD_SQ64) and the oracle give."""
    if sq64:
        monkeypatch.setenv("CLFD_SQ64", "1")
    flat = geometry_cascade("255x255")
    oc = oracle.Cascade(flat)
    cas = clfd.Cascade(flat=flat)
    yy, xx = np.mgrid[0:H, 0:W]
    frames = np.stack([np.full((H, W), 255, np.uint8), (((yy + xx) & 1) * 255).astype(np.uint8),
                       octave_frame(W, H, 24)])
    ocodes = _compare_diagnostic(gpu_ctx, [(oc, cas)], frames)[0]
    _not_vacuous("255x255", flat, ocodes, oc.plan_levels(W, H, SF))


def test_three_geometries_share_one_pyramid(gpu_ctx, monkeypatch):
    """frontalface_alt (20 x 20, tile kernel), the 48 x 48 cascade (generic kernels) and the 3 x 3 cascade in one
    detector: one pyramid for all three, the rect count carried from one cascade to the next"""
    pairs = [(oracle_cascade("frontalface_alt"), clfd.Cascade(cascade_path("frontalface_alt")))]
    for case in ("48x48", "3x3"):
        flat = geometry_cascade(case)
        pairs.append((oracle.Cascade(flat), clfd.Cascade(flat=flat)))
    frames = np.stack([octave_frame(W, H, 31), octave_frame(W, H, 32)])
    ocodes = _compare_diagnostic(gpu_ctx, pairs, frames)
    for (oc, _), oco in zip(pairs[1:], ocodes[1:]):
        assert _accepted(oc.flat, np.concatenate(oco)).any()
    got = _production_rects(gpu_ctx, [c for _, c in pairs], frames, monkeypatch)
    for ci, (oc, _) in enumerate(pairs):
        for f in range(len(frames)):
            assert np.array_equal(got.frame_rects(f, ci), _sorted(oc.detect(frames[f], SF, want_codes=False)[0])), (ci, f)


@pytest.mark.parametrize("case", ["44x44", "48x48"])
def test_nine_frame_batch_equals_serial_order_and_oracle(gpu_ctx, monkeypatch, case):
    """Batches of 8+ frames of a cascade the tile kernel finishes run their pyramid beside the previous chunk's tile
    kernel (44 x 44); a cascade the tile kernel cannot take runs them in order (48 x 48).  Either way the rects are
    those of the serial order (CLFD_NO_OVERLAP) and of the oracle."""
    flat = geometry_cascade(case)
    oc = oracle.Cascade(flat)
    cas = clfd.Cascade(flat=flat)
    frames = np.stack([octave_frame(W, H, 40 + i) for i in range(9)])
    got = _production_rects(gpu_ctx, cas, frames, monkeypatch)
    serial = _production_rects(gpu_ctx, cas, frames, monkeypatch, {"CLFD_NO_OVERLAP": "1"})
    for f in range(9):
        assert np.array_equal(got.frame_rects(f), serial.frame_rects(f)), (case, f)
    total = 0
    for f in (0, 4, 8):
        want = _sorted(oc.detect(frames[f], SF, want_codes=False)[0])
        assert np.array_equal(got.frame_rects(f), want), (case, f, len(got.frame_rects(f)), len(want))
        total += len(want)
    assert total > 0
