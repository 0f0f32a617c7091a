"""THE PIN: oracle/vj_oracle.c (what every GPU test is compared with) against the reference's own
compiled code -- tempcv.cpp:40-1516, 1702-2089 built by oracle/build_ref.py from where the sources
lie (oracle/_ref/libtempcv_ref.so).  Everything here runs on the CPU.

Skipped where CLFD_REFERENCE_DIR does not name the original sources and oracle/_ref holds no built
library; tests/test_reference_golden.py then compares with the vectors that library produced.
"""
import os
import tempfile

import numpy as np
import pytest

import clfacedetection_b200 as clfd
import oracle
from clfacedetection_b200.frames import octave_frame, uniform_frame
from conftest import ALL_CASCADES, cascade_path, oracle_cascade
from oracle import ref

pytestmark = pytest.mark.skipif(not ref.available(), reason="no original sources (CLFD_REFERENCE_DIR) and no library in oracle/_ref")

_ref_cache = {}


def ref_cascade(name):
    if name not in _ref_cache:
        _ref_cache[name] = ref.RefCascade(cascade_path(name))
    return _ref_cache[name]


def _sorted(r):
    r = np.asarray(r, np.int32).reshape(-1, 4)
    return r[np.lexsort(r.T[::-1])] if len(r) else r


def _expected_results(cas, codes):
    """oracle exit codes -> what cvRunHaarClassifierCascadeSum returns (tempcv.cpp:857,946,971)"""
    if cas.is_tree:
        return (codes & 1).astype(np.int32)
    return np.where(codes == cas.flat.n_stages, 1, -codes.astype(np.int32))


# ---- a3: the XML reader ---------------------------------------------------------------------------
@pytest.mark.parametrize("name", ALL_CASCADES)
def test_loaders_equal_reference_reader(name):
    """icvReadHaarClassifier (tempcv.cpp:1750-2089) == oracle reader == product reader, bit for bit"""
    flat, child = ref_cascade(name).flat()
    ours = clfd.Cascade(cascade_path(name)).arrays()
    orc = oracle.load_cascade_xml(cascade_path(name))
    for k in ("st_ntrees", "st_thr", "st_parent", "st_next", "tr_nnodes", "nd_tilted", "nd_rect", "nd_weight",
              "nd_thr", "nd_left", "nd_right", "alpha"):
        a = getattr(flat, k)
        assert a.tobytes() == getattr(orc, k).tobytes(), k
        assert a.tobytes() == ours[k].tobytes(), k
    assert np.array_equal(child, ours["st_child"])


@pytest.mark.parametrize("old,new", [
    ("<size>20 20</size>", "<size>20</size>"),
    ("<_>3 7 14 4 -1.</_>", "<_>3 7 19 4 -1.</_>"),
    ("<_>3 7 14 4 -1.</_>", "<_>3 7 14 4 -1</_>"),
    ("<tilted>0</tilted>", ""),
    ("<parent>-1</parent>", "<parent>99</parent>"),
    ("<threshold>4.0141958743333817e-003</threshold>", "<threshold>4</threshold>"),
])
def test_malformed_files_same_message_as_reference_reader(old, new):
    """the product's loader fails with the reference reader's own message (tempcv.cpp:1766-2064)"""
    text = open(cascade_path("frontalface_alt"), encoding="latin-1").read()
    assert old in text
    f = tempfile.NamedTemporaryFile("w", suffix=".xml", delete=False, encoding="latin-1")
    f.write(text.replace(old, new, 1))
    f.close()
    try:
        with pytest.raises(ValueError) as eref:
            ref.RefCascade(f.name)
        with pytest.raises(clfd.ClfdError) as eours:
            clfd.Cascade(f.name)
        assert str(eref.value) in str(eours.value)
    finally:
        os.unlink(f.name)


# ---- a4 / a5: hidden cascade ---------------------------------------------------------------------
@pytest.mark.parametrize("name", ALL_CASCADES)
def test_hidden_cascade_equals_reference(name):
    """icvCreateHidHaarClassifierCascade + cvSetImagesForHaarClassifierCascade(scale 1)
    (tempcv.cpp:308-536, 549-768): weights, kept rects, biased thresholds, two_rects, flags, and the
    corner geometry (upright and tilted, tempcv.cpp:736-749)"""
    rc = ref_cascade(name)
    W = H = 96
    hid = rc.hidden(W, H, 1.0)
    oc = oracle_cascade(name)
    ow, onr, othr, otwo, _ = oc.hidden()
    pw, pnr, pthr, ptwo = clfd.Cascade(cascade_path(name)).hidden()
    for w, nr, thr, two in ((ow, onr, othr, otwo), (pw, pnr, pthr, ptwo)):
        assert hid["weights"].tobytes() == w.tobytes()
        assert np.array_equal(hid["nrects"], nr)
        assert hid["stage_thr"].tobytes() == thr.tobytes()
        assert np.array_equal(hid["two_rects"], two)
    assert hid["flags"] == (int(oc.is_tree) | 2 * int(oc.is_stump_based) | 4 * int(oc.has_tilted))
    w0, h0 = oc.win
    assert hid["inv_window_area"] == 1.0 / ((w0 - 2) * (h0 - 2))
    S = W + 1
    assert hid["eq_corners"].tolist() == [S + 1, S + 1 + w0 - 2, (1 + h0 - 2) * S + 1, (1 + h0 - 2) * S + 1 + w0 - 2]
    f = oc.flat
    for n in range(0, f.n_nodes, max(1, f.n_nodes // 200)):
        for k in range(int(hid["nrects"][n])):
            x, y, w, h = (int(v) for v in f.nd_rect[n, k])
            if f.nd_tilted[n]:
                exp = [y * S + x, (y + h) * S + x - h, (y + w) * S + x + w, (y + w + h) * S + x + w - h]
            else:
                exp = [y * S + x, y * S + x + w, (y + h) * S + x, (y + h) * S + x + w]
            assert hid["corners"][n, k].tolist() == exp, (n, k)


# ---- a6: the window evaluator --------------------------------------------------------------------
@pytest.mark.parametrize("name", ALL_CASCADES)
def test_oracle_equals_reference_evaluator(name):
    """per-window return codes of cvRunHaarClassifierCascadeSum (tempcv.cpp:795-972) == oracle exit
    codes, every window of four frames at both grid steps (all three evaluator branches: stage tree,
    stumps with and without two_rects stages, generic trees; tilted features)"""
    rc, oc = ref_cascade(name), oracle_cascade(name)
    total = 0
    for frame, ystep in ((octave_frame(400, 300, 3), 1), (octave_frame(331, 207, 4), 2),
                         (uniform_frame(160, 120, 5), 1), (np.full((90, 110), 255, np.uint8), 1),
                         (np.zeros((70, 80), np.uint8), 2)):
        res, _ = rc.eval_level(frame, ystep)
        codes, _, _ = oc.eval_level(frame, ystep)
        assert res.shape == codes.shape
        assert np.array_equal(_expected_results(oc, codes), res)
        total += res.size
    assert total > 100000


def test_stage_sums_equal_reference():
    """the stage_sum the evaluator hands back (tempcv.cpp:1084-1094 consumers): bit-equal doubles"""
    for name in ("eye", "frontalface_alt2", "mcs_nose"):
        rc, oc = ref_cascade(name), oracle_cascade(name)
        frame = octave_frame(320, 240, 21)
        r, _, lv, wt = rc.detect(frame, 1.2, 0, ref.CV_HAAR_SCALE_IMAGE, reject_levels=True)
        ro, lvo, wto = oc.detect_roc(frame, 1.2)
        assert np.array_equal(r, ro) and np.array_equal(lv, lvo) and wt.tobytes() == wto.tobytes()
        assert len(r) > 0


# ---- a1 + a2 + a6 + a7: the whole image-pyramid driver ----------------------------------------------
@pytest.mark.parametrize("name", ALL_CASCADES)
def test_whole_scale_image_driver_equals_oracle(name):
    """cvHaarDetectObjectsForROC with CV_HAAR_SCALE_IMAGE (tempcv.cpp:1257-1329 + invoker 1011-1103),
    run unmodified, returns the oracle's raw rect list (same order: level by level, raster)"""
    rc, oc = ref_cascade(name), oracle_cascade(name)
    for frame, sf, mn, mx in ((octave_frame(640, 480, 0), 1.2, (0, 0), (0, 0)),
                              (octave_frame(300, 200, 9), 1.1, (30, 30), (120, 120)),
                              (octave_frame(161, 203, 2), 1.37, (0, 0), (0, 0))):
        r, _, _, _ = rc.detect(frame, sf, 0, ref.CV_HAAR_SCALE_IMAGE, mn, mx)
        ro, _, _, _, _ = oc.detect(frame, sf, mn, mx)
        assert np.array_equal(r, ro)


# ---- a9: grouping ------------------------------------------------------------------------------------
def test_grouping_equals_reference_agrouprectangles():
    """AgroupRectangles (tempcv.cpp:145-243), several eps: oracle and the product's host grouping"""
    rng = np.random.default_rng(3)
    for it in range(150):
        k = int(rng.integers(1, 7))
        base = rng.integers(0, 400, size=(k, 2))
        n = int(rng.integers(0, 80))
        pick = rng.integers(0, k, size=n)
        size = 20 + rng.integers(0, 90, size=k)
        r = np.stack([base[pick, 0] + rng.integers(-6, 7, size=n), base[pick, 1] + rng.integers(-6, 7, size=n),
                      size[pick] + rng.integers(-4, 5, size=n), size[pick] + rng.integers(-4, 5, size=n)], 1).astype(np.int32)
        thr = int(rng.integers(0, 5))
        eps = float(rng.choice([0.2, 0.35, 0.1, 0.5, 0.7]))
        g, w = ref.group_rectangles(r, thr, eps)
        go, wo = oracle.group_rectangles(r, thr, eps)
        gp, wp = clfd.group_rectangles(r, thr, eps)
        assert np.array_equal(g, go) and np.array_equal(w, wo), (it, thr, eps)
        assert np.array_equal(g, gp) and np.array_equal(w, wp), (it, thr, eps)


def test_grouped_driver_output_equals_reference():
    """minNeighbors != 0 through the reference's driver: rects and neighbour counts"""
    for name in ("eye", "mcs_lefteye", "frontalface_default"):
        rc, oc = ref_cascade(name), oracle_cascade(name)
        frame = octave_frame(640, 480, 0)
        for mn in (1, 2, 3):
            r, nb, _, _ = rc.detect(frame, 1.2, mn, ref.CV_HAAR_SCALE_IMAGE)
            raw, _, _, _, _ = oc.detect(frame, 1.2)
            g, w = oracle.group_rectangles(raw, mn)
            assert np.array_equal(r, g) and np.array_equal(nb, w)
    # ROC grouping (tempcv.cpp:255-258)
    rc, oc = ref_cascade("eye"), oracle_cascade("eye")
    frame = octave_frame(640, 480, 0)
    r, _, lv, wt = rc.detect(frame, 1.2, 2, ref.CV_HAAR_SCALE_IMAGE, reject_levels=True)
    ro, lvo, wto = oc.detect_roc(frame, 1.2)
    g, gl, gw = oracle.group_rectangles_roc(ro, lvo, wto, 2)
    assert np.array_equal(r, g) and np.array_equal(lv[:len(g)], gl) and wt[:len(g)].tobytes() == gw.tobytes()
    gp, glp, gwp = clfd.group_rectangles_roc(ro, lvo, wto, 2)
    assert np.array_equal(r, gp) and np.array_equal(gl, glp) and gw.tobytes() == gwp.tobytes()


# ---- f3: the scale-cascade path ----------------------------------------------------------------------
@pytest.mark.parametrize("name", ALL_CASCADES)
def test_whole_scale_cascade_driver_equals_oracle(name):
    """cvHaarDetectObjectsForROC with flags = 0 (tempcv.cpp:1330-1456 + invoker 1132-1175: scaled
    features, skip rule), run unmodified, returns the REF-SC oracle's rect list"""
    rc, oc = ref_cascade(name), oracle_cascade(name)
    for frame, sf, mn in ((octave_frame(640, 480, 0), 1.2, (0, 0)), (octave_frame(300, 220, 7), 1.1, (40, 40))):
        r, _, _, _ = rc.detect(frame, sf, 0, 0, mn)
        ro, _, _, _ = oc.detect_sc(frame, sf, mn)
        assert np.array_equal(_sorted(r), _sorted(ro))


@pytest.mark.parametrize("name", ["frontalface_alt", "frontalface_alt_tree", "fullbody", "eye_tree_eyeglasses",
                                  "mcs_eyepair_small", "lowerbody"])
def test_scaled_evaluator_codes_equal_reference(name):
    """per-position results under cvSetImagesForHaarClassifierCascade(scale = factor)
    (tempcv.cpp:549-768: rounded corners, re-normalised weights, weight_0 correction) at every
    position the REF-SC oracle evaluates, every scale"""
    rc, oc = ref_cascade(name), oracle_cascade(name)
    frame = octave_frame(360, 270, 13)
    _, codes, _, levels = oc.detect_sc(frame, 1.2)
    off = 0
    checked = 0
    for lv in levels:
        n = lv.nx * lv.ny
        c = codes[off:off + n].reshape(lv.ny, lv.nx)
        off += n
        step = max(2.0, lv.factor)
        res = rc.eval_scaled(frame, lv.factor, step, lv.nx, lv.ny)
        ev = c != oracle.CODE_SKIPPED
        outside = c == oracle.CODE_OUTSIDE
        assert np.array_equal(res[outside], np.full(outside.sum(), -1))
        m = ev & ~outside
        assert np.array_equal(_expected_results(oc, c[m]), res[m])
        # the skip rule itself (tempcv.cpp:1161): a position is skipped iff its left neighbour was
        # evaluated with result 0
        for iy in range(0, lv.ny, 5):
            skip = False
            for ix in range(lv.nx):
                assert (c[iy, ix] == oracle.CODE_SKIPPED) == skip
                skip = (not skip) and res[iy, ix] == 0
        checked += int(m.sum())
    assert checked > 10000
