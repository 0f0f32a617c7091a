"""GPU parity of the cascade path against the REF-SI oracle: per-window exit codes and the
raw detection set must be IDENTICAL (the kernels reproduce the reference's arithmetic
bit for bit, so the north star's 1e-5 near-threshold tolerance is reported, not used)."""
import numpy as np
import pytest

import clfacedetection_b200 as clfd
from clfacedetection_b200.frames import octave_frame, uniform_frame
from conftest import cascade_path, oracle_cascade

pytestmark = pytest.mark.gpu


def _sorted(r):
    r = np.asarray(r, np.int32).reshape(-1, 4)
    return r[np.lexsort((r[:, 0], r[:, 1], r[:, 2]))] if len(r) else r


def _compare(gpu_ctx, names, frames, sf, min_size=(0, 0), max_size=(0, 0)):
    n, H, W = frames.shape
    cascades = [clfd.Cascade(cascade_path(nm)) for nm in names]
    det = clfd.Detector(gpu_ctx, cascades, W, H, max_batch=n, scale_factor=sf, min_size=min_size,
                        max_size=max_size, want_codes=True)
    res = det.detect(frames)
    report = {}
    near_events = 0
    for ci, nm in enumerate(names):
        oc = oracle_cascade(nm)
        codes = det.codes(ci, n)
        near_total = 0
        for f in range(n):
            rects, ocodes, near, st, levels = oc.detect(frames[f], sf, min_size, max_size)
            assert len(levels) == len(det.levels(ci))
            assert st.windows == det.windows_per_frame(ci)
            bad = np.flatnonzero(codes[f] != ocodes)
            assert bad.size == 0, f"{nm} frame {f}: {bad.size} exit codes differ, first at {bad[:5]} " \
                                  f"gpu {codes[f][bad[:5]]} oracle {ocodes[bad[:5]]}"
            assert np.array_equal(res.frame_rects(f, ci), _sorted(rects)), f"{nm} frame {f}: rect sets differ"
            near_total += st.near_stage_thr
            near_events += st.near_stage_events
        report[nm] = near_total
    # counted and reported: stage sums within 1e-5 relative of a threshold (all of them take the FP64 path of the
    # tile kernel, which counts them), and FP64 fallbacks as a whole.  Cascades the tile kernel finishes itself.
    if all(c.info.dense_stages == c.info.n_stages for c in cascades):
        assert res.stats["near_threshold_events"] == near_events, (res.stats["near_threshold_events"], near_events)
        assert res.stats["exact_stage_evals"] >= near_events
    det.close()
    return report


def test_cfg1_frontalface_alt_640x480(gpu_ctx):
    frames = np.stack([octave_frame(640, 480, 0), uniform_frame(640, 480, 0)])
    rep = _compare(gpu_ctx, ["frontalface_alt"], frames, 1.2, min_size=(24, 24))
    print("near-threshold windows (reported, none mismatched):", rep)


def test_cfg2_frontalface_default_1080p_batch(gpu_ctx):
    frames = np.stack([octave_frame(1920, 1080, i) for i in range(2)])
    _compare(gpu_ctx, ["frontalface_default"], frames, 1.2)


def test_northstar_frontalface_alt_1080p(gpu_ctx):
    frames = np.stack([octave_frame(1920, 1080, 7)])
    _compare(gpu_ctx, ["frontalface_alt"], frames, 1.2)


def test_cfg3_alt_tree_and_eye_share_pyramid(gpu_ctx):
    frames = np.stack([octave_frame(960, 540, 3)])
    _compare(gpu_ctx, ["frontalface_alt_tree", "eye"], frames, 1.2)


def test_cfg4_profileface_fullbody_sf11(gpu_ctx):
    frames = np.stack([octave_frame(640, 360, 4)])
    _compare(gpu_ctx, ["profileface", "fullbody"], frames, 1.1)


def test_cfg3_full_size_3840x2160_alt_tree_and_eye(gpu_ctx):
    """BASELINE config 3 at its real size: one 4K frame, 26 levels, 11 094 920 windows per cascade,
    the widest integral-row kernels (k_integral_rows<512/1024>)"""
    frames = np.stack([octave_frame(3840, 2160, 3)])
    _compare(gpu_ctx, ["frontalface_alt_tree", "eye"], frames, 1.2)


def test_cfg4_full_size_1080p_sf11_profileface_fullbody(gpu_ctx):
    """BASELINE config 4 at its real size: 1080p, scale 1.1 (42 / 39 levels), tilted integral"""
    frames = np.stack([octave_frame(1920, 1080, 4)])
    _compare(gpu_ctx, ["profileface", "fullbody"], frames, 1.1)


@pytest.mark.parametrize("name", ["lefteye_2splits", "righteye_2splits", "lowerbody", "upperbody", "mcs_eyepair_big",
                                  "mcs_eyepair_small", "mcs_lefteye", "mcs_mouth", "mcs_righteye", "mcs_upperbody"])
def test_the_other_ten_cascade_files(gpu_ctx, name):
    """the 10 reference cascades outside BASELINE's configs: generic row step (19x23, 22x18, 18x12 ...
    windows), wide / flat tiles (45x11, 22x5), 2-split trees with tilted features, the largest stages
    (415 trees), the lenient-XML headers"""
    frames = np.stack([octave_frame(480, 360, 5), uniform_frame(480, 360, 5)])
    _compare(gpu_ctx, [name], frames, 1.2)


@pytest.mark.parametrize("name", ["frontalface_alt2", "eye_tree_eyeglasses", "mcs_nose"])
def test_tree_nodes_tilted_and_lenient_xml(gpu_ctx, name):
    frames = np.stack([octave_frame(480, 360, 5), uniform_frame(480, 360, 5)])
    _compare(gpu_ctx, [name], frames, 1.2)


def test_edge_sizes(gpu_ctx):
    # frame barely larger than the window; min/max window limits; flat frames (sigma = 0 / 1 branch)
    _compare(gpu_ctx, ["frontalface_alt"], np.stack([uniform_frame(23, 22, 1)]), 1.2)
    _compare(gpu_ctx, ["frontalface_alt"], np.stack([uniform_frame(21, 21, 1)]), 1.2)
    _compare(gpu_ctx, ["frontalface_alt"], np.stack([octave_frame(320, 240, 2)]), 1.3, min_size=(40, 40), max_size=(120, 120))
    flat = np.stack([np.zeros((120, 160), np.uint8), np.full((120, 160), 255, np.uint8)])
    _compare(gpu_ctx, ["frontalface_alt", "frontalface_default"], flat, 1.2)


def test_device_resident_enqueue_matches_host_path(gpu_ctx):
    import torch
    frames = np.stack([octave_frame(640, 480, i) for i in range(3)])
    cas = clfd.Cascade(cascade_path("frontalface_alt"))
    det = clfd.Detector(gpu_ctx, cas, 640, 480, max_batch=3, scale_factor=1.2)
    a = det.detect(frames)
    t = torch.from_numpy(frames).cuda()
    torch.cuda.synchronize()
    det.enqueue(t, 3, t.stride(0), t.stride(1), torch.cuda.current_stream().cuda_stream)
    b = det.fetch(torch.cuda.current_stream().cuda_stream)
    for f in range(3):
        assert np.array_equal(a.frame_rects(f), b.frame_rects(f))
    assert b.stats["windows"] == 3 * det.windows_per_frame()
    det.close()


def test_fp32_filter_equals_all_fp64_evaluation(gpu_ctx, monkeypatch):
    """The tile kernel decides stumps with an FP32 filter and redoes a window's stage in FP64
    inside the guard band.  CLFD_FORCE_EXACT=1 makes every stage take the FP64 path: both
    must give the same exit codes (and both equal the oracle, checked by _compare)."""
    frames = np.stack([octave_frame(640, 480, 9), uniform_frame(640, 480, 9)])
    monkeypatch.setenv("CLFD_FORCE_EXACT", "1")
    _compare(gpu_ctx, ["frontalface_alt", "frontalface_default"], frames, 1.2)
    monkeypatch.delenv("CLFD_FORCE_EXACT")
    _compare(gpu_ctx, ["frontalface_alt", "frontalface_default"], frames, 1.2)


@pytest.mark.parametrize("nf", [0, 1, 5])
def test_any_split_between_fixed_and_compacted_stages(gpu_ctx, monkeypatch, nf):
    monkeypatch.setenv("CLFD_N_FIXED", str(nf))
    _compare(gpu_ctx, ["frontalface_alt"], np.stack([octave_frame(800, 600, 3)]), 1.2)


def test_other_window_shapes_use_the_generic_tile_kernel(gpu_ctx):
    # lowerbody-like shapes are not shipped here; fullbody (14x28) exercises the non-templated
    # row step of the tile kernel, with tilted features (second tile)
    _compare(gpu_ctx, ["fullbody"], np.stack([octave_frame(700, 500, 6)]), 1.25)


def test_full_size_properties_batch(gpu_ctx):
    """At BASELINE sizes the oracle is too slow for every frame; check size-independent
    properties instead: (i) a batch gives the same per-frame results as single-frame calls,
    (ii) duplicated frames give duplicated detections, (iii) accepted windows == rect count."""
    cas = clfd.Cascade(cascade_path("frontalface_alt"))
    frames = np.stack([octave_frame(1920, 1080, i % 3) for i in range(6)])
    det = clfd.Detector(gpu_ctx, cas, 1920, 1080, max_batch=6, scale_factor=1.2, want_codes=True)
    res = det.detect(frames)
    codes = det.codes(0, 6)
    for f in range(3):
        assert np.array_equal(res.frame_rects(f), res.frame_rects(f + 3))
        assert np.array_equal(codes[f], codes[f + 3])
    assert int((codes == cas.info.n_stages).sum()) == len(res.rects)
    single = clfd.Detector(gpu_ctx, cas, 1920, 1080, max_batch=1, scale_factor=1.2)
    for f in range(3):
        assert np.array_equal(single.detect(frames[f:f + 1]).frame_rects(0), res.frame_rects(f))
    det.close(); single.close()


@pytest.mark.parametrize("chunks", [1, 2, 3])
def test_detect_pipelined_chunks_equal_one_shot(gpu_ctx, monkeypatch, chunks):
    """clfd_detect cuts a batch into ranges whose H2D copy overlaps the previous range's compute.
    Rect frame indices, exit codes and per-frame intermediates must not depend on the cut."""
    frames = np.stack([octave_frame(640, 480, i) for i in range(9)])
    cas = clfd.Cascade(cascade_path("frontalface_alt"))
    monkeypatch.setenv("CLFD_DETECT_CHUNKS", str(chunks))
    det = clfd.Detector(gpu_ctx, cas, 640, 480, max_batch=9, scale_factor=1.2, want_codes=True)
    res = det.detect(frames)
    codes = det.codes(0, 9)
    oc = oracle_cascade("frontalface_alt")
    for f in (0, 4, 8):
        rects, ocodes, _, _, _ = oc.detect(frames[f], 1.2)
        assert np.array_equal(codes[f], ocodes)
        assert np.array_equal(res.frame_rects(f), _sorted(rects))
        _, s, _, _ = det.read_level(2, frame=f)
        import oracle
        lv = det.levels()[2]
        os_, _, _ = oracle.integral(oracle.resize_linear(frames[f], lv.img_w, lv.img_h))
        assert np.array_equal(s, os_)
    assert sorted(set(res.rects["frame"].tolist())) == sorted(f for f in range(9) if len(res.frame_rects(f)))
    det.close()


@pytest.mark.parametrize("chunks", [1, 3, 8])
def test_chunk_overlap_equals_serial_order(gpu_ctx, monkeypatch, chunks):
    """Batches of 8+ frames run their pyramid kernels on a second stream beside the previous chunk's tile kernel
    (clfd_api.cu, enqueue_overlapped).  Host path, device-resident path and the two-slot pipeline must return what
    the serial order (CLFD_NO_OVERLAP=1) and the oracle return, for any cut."""
    import torch
    batches = [np.stack([octave_frame(640, 480, 20 * b + i) for i in range(11)]) for b in range(3)]
    cas = clfd.Cascade(cascade_path("frontalface_alt"))
    det = clfd.Detector(gpu_ctx, cas, 640, 480, max_batch=11, scale_factor=1.2)
    monkeypatch.setenv("CLFD_NO_OVERLAP", "1")
    want = [det.detect(b) for b in batches]
    launches_serial = want[0].stats["kernel_launches"]
    monkeypatch.delenv("CLFD_NO_OVERLAP")
    monkeypatch.setenv("CLFD_OVERLAP_CHUNKS", str(chunks))
    oc = oracle_cascade("frontalface_alt")
    for f in (0, 5, 10):
        assert np.array_equal(want[1].frame_rects(f), _sorted(oc.detect(batches[1][f], 1.2, want_codes=False)[0]))
    # host path, blocking
    for b in range(3):
        got = det.detect(batches[b])
        if chunks > 1:
            assert got.stats["kernel_launches"] > launches_serial   # the cut really happened
        for f in range(11):
            assert np.array_equal(got.frame_rects(f), want[b].frame_rects(f)), (b, f)
    # device-resident path, twice on the same stream (the second batch's pyramid must wait for the first one's tiles)
    st = torch.cuda.current_stream().cuda_stream
    t = [torch.from_numpy(b).cuda() for b in batches]
    torch.cuda.synchronize()
    for b in (2, 0):
        det.enqueue(t[b], 11, t[b].stride(0), t[b].stride(1), st)
        got = det.fetch(st)
        for f in range(11):
            assert np.array_equal(got.frame_rects(f), want[b].frame_rects(f)), (b, f)
    # two batches in flight
    pinned = [torch.from_numpy(b).pin_memory() for b in batches]
    got = []
    det.submit(pinned[0])
    for b in (1, 2):
        det.submit(pinned[b])
        got.append(det.collect())
    got.append(det.collect())
    for b in range(3):
        for f in range(11):
            assert np.array_equal(got[b].frame_rects(f), want[b].frame_rects(f)), (b, f)
    det.close()


def _synthetic_cascade(big, n_stages=12):
    """frontalface_alt's first stages; with `big` != 0 the first stump of every stage votes +big
    and the last one -big whatever the window: the partial sums in between are rounded at the
    scale of `big`, so the stage sum depends on the summation order, the order-free proof fails
    and every order-sensitive shortcut must fall back to the reference's tree order."""
    from oracle.cascade_xml import FlatCascade, load_cascade_xml
    f = load_cascade_xml(cascade_path("frontalface_alt"))
    S = n_stages
    T = int(np.sum(f.st_ntrees[:S]))
    alpha = np.array(f.alpha[:2 * T], np.float32).copy()
    if big:
        first = np.concatenate([[0], np.cumsum(f.st_ntrees[:S])])
        for st in range(S):
            alpha[2 * first[st]:2 * first[st] + 2] = np.float32(big)
            alpha[2 * first[st + 1] - 2:2 * first[st + 1]] = np.float32(-big)
    thr = np.ascontiguousarray(f.st_thr[:S], np.float32) - np.float32(0.8 if big else 0.0)   # two stumps lost their vote
    c = np.ascontiguousarray
    return FlatCascade(name="synthetic", win_w=f.win_w, win_h=f.win_h, st_ntrees=c(f.st_ntrees[:S], np.int32),
                       st_thr=thr, st_parent=np.arange(-1, S - 1, dtype=np.int32),
                       st_next=np.full(S, -1, np.int32), tr_nnodes=np.ones(T, np.int32),
                       nd_tilted=c(f.nd_tilted[:T], np.int32), nd_rect=c(f.nd_rect[:T], np.int32),
                       nd_weight=c(f.nd_weight[:T], np.float32), nd_thr=c(f.nd_thr[:T], np.float32),
                       nd_left=c(f.nd_left[:T], np.int32), nd_right=c(f.nd_right[:T], np.int32), alpha=alpha)


@pytest.mark.parametrize("big", [0.0, 2.0 ** 30])
def test_synthetic_cascade_order_sensitive_sums(gpu_ctx, big):
    """Stage sums that are NOT exact in any order (alphas spanning > 2^29): the FP32 stage-sum
    filter and the split of a stage's stumps over lanes must still reproduce the reference's
    sequential double sum bit for bit (they fall back to dense_stage_exact).  12 stages also
    puts the last stages beyond the kernel-parameter budget (stumps read from global memory)."""
    import oracle
    flat = _synthetic_cascade(big)
    cas = clfd.Cascade(flat=flat)
    if big:
        assert cas.info.order_free_stages == 0
    assert cas.info.dense_stages == cas.info.n_stages
    oc = oracle.Cascade(flat)
    det = clfd.Detector(gpu_ctx, cas, 640, 480, max_batch=2, scale_factor=1.2, want_codes=True)
    frames = np.stack([octave_frame(640, 480, 11), uniform_frame(640, 480, 11)])
    res = det.detect(frames)
    for f in range(2):
        rects, ocodes, _, _, _ = oc.detect(frames[f], 1.2)
        assert np.array_equal(det.codes(0, 2)[f], ocodes)
        assert np.array_equal(res.frame_rects(f), _sorted(rects))
    det.close()


def _mixed_tree_cascade(stage_trees=(5, 9, 14, 20, 40, 60)):
    """Trees of 1, 2, 3 and 4 nodes (cyclically; the 4-node shape has a leaf, a chain and a fork)
    assembled from frontalface_alt's features, every stage threshold at the middle of its leaf
    values: the tile kernel pads every tree to 4 node records and tracks the node a window is at."""
    from oracle.cascade_xml import FlatCascade, load_cascade_xml
    f = load_cascade_xml(cascade_path("frontalface_alt"))
    shapes = {1: [(0, -1)], 2: [(1, 0), (-1, -2)], 3: [(1, 2), (0, -1), (-2, -3)],
              4: [(0, 1), (2, 3), (-1, -2), (-3, -4)]}   # (left, right): > 0 node, <= 0 leaf -idx
    nn, left, right, alpha, thr = [], [], [], [], []
    feat = 0
    for nt in stage_trees:
        mid = 0.0
        for t in range(nt):
            k = 1 + (len(nn) % 4)
            nn.append(k)
            for (l, r) in shapes[k]:
                left.append(l); right.append(r)
            leaves = [f.alpha[2 * (feat + i // 2) + (i & 1)] for i in range(k + 1)]
            alpha += leaves
            mid += float(np.mean(leaves))
            feat += k
        thr.append(mid - 0.05)
    N, S = feat, len(stage_trees)
    c = np.ascontiguousarray
    return FlatCascade(name="mixed-trees", win_w=f.win_w, win_h=f.win_h, st_ntrees=np.array(stage_trees, np.int32),
                       st_thr=np.array(thr, np.float32), st_parent=np.arange(-1, S - 1, dtype=np.int32),
                       st_next=np.full(S, -1, np.int32), tr_nnodes=np.array(nn, np.int32),
                       nd_tilted=c(f.nd_tilted[:N], np.int32), nd_rect=c(f.nd_rect[:N], np.int32),
                       nd_weight=c(f.nd_weight[:N], np.float32), nd_thr=c(f.nd_thr[:N], np.float32),
                       nd_left=np.array(left, np.int32), nd_right=np.array(right, np.int32), alpha=np.array(alpha, np.float32))


@pytest.mark.parametrize("hook", [None, "CLFD_FORCE_EXACT", "CLFD_NO_NODE_TILES"])
def test_synthetic_cascade_mixed_tree_shapes(gpu_ctx, monkeypatch, hook):
    import oracle
    if hook:
        monkeypatch.setenv(hook, "1")
    flat = _mixed_tree_cascade()
    cas = clfd.Cascade(flat=flat)
    assert cas.info.max_nodes_per_tree == 4 and not cas.info.is_stump_based
    assert cas.info.dense_stages == (0 if hook == "CLFD_NO_NODE_TILES" else cas.info.n_stages)
    oc = oracle.Cascade(flat)
    det = clfd.Detector(gpu_ctx, cas, 640, 480, max_batch=2, scale_factor=1.2, want_codes=True)
    frames = np.stack([octave_frame(640, 480, 12), uniform_frame(640, 480, 12)])
    res = det.detect(frames)
    seen = set()
    for f in range(2):
        rects, ocodes, _, _, _ = oc.detect(frames[f], 1.2)
        assert np.array_equal(det.codes(0, 2)[f], ocodes)
        assert np.array_equal(res.frame_rects(f), _sorted(rects))
        seen |= set(np.unique(ocodes).tolist())
    assert len(seen) >= 5, seen   # the thresholds really split the windows over the stages
    det.close()


@pytest.mark.parametrize("hook,names", [("CLFD_NO_NODE_TILES", ["frontalface_alt2", "eye_tree_eyeglasses"]),
                                        ("CLFD_NO_TREE_TILES", ["frontalface_alt_tree"]),
                                        ("CLFD_NO_TILTED_TILE", ["fullbody", "mcs_nose"])])
def test_generic_kernels_behind_the_tile_kernel(gpu_ctx, monkeypatch, hook, names):
    """The stock cascades all finish inside the tile kernel; the hooks switch its tree / stage-tree /
    tilted support off so that the mid and deep kernels (cascades with larger trees) stay covered."""
    monkeypatch.setenv(hook, "1")
    assert clfd.Cascade(cascade_path(names[0])).info.dense_stages < clfd.Cascade(cascade_path(names[0])).info.n_stages
    _compare(gpu_ctx, names, np.stack([octave_frame(480, 360, 5)]), 1.2)


@pytest.mark.parametrize("env", [{"CLFD_FORCE_EXACT": "1"}, {"CLFD_N_FIXED": "0"}, {"CLFD_N_FIXED": "5"}, {"CLFD_G1_MIN": "1"},
                                 {"CLFD_G1_MIN": "16"}, {"CLFD_TILE_H2": "32", "CLFD_NO_SMALL_TILES": "1"},
                                 {"CLFD_N_FIXED": "2"}, {"CLFD_NO_DI": "1"}])
def test_tile_kernel_variants_under_every_split(gpu_ctx, monkeypatch, env):
    """stage tree / multi-node / tilted variants of the tile kernel: all-FP64 evaluation, no, two or five
    fixed stages (the stage-tree walk starts from a dealt list when the linear prefix is all fixed:
    N_FIXED=5), thread-per-window only, the ystep-2 levels' integral in natural order (LDG + STS tile
    staging instead of the TMA copies from a column-de-interleaved integral, which every other test runs with)."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    _compare(gpu_ctx, ["frontalface_alt_tree", "frontalface_alt2", "eye_tree_eyeglasses", "fullbody", "frontalface_alt"],
             np.stack([octave_frame(400, 300, 8)]), 1.2)


@pytest.mark.parametrize("name", ["frontalface_alt", "eye", "frontalface_alt2", "frontalface_alt_tree", "fullbody", "mcs_nose"])
def test_reject_levels_equal_oracle(gpu_ctx, name):
    """SURVEY 8-f row 4: cvHaarDetectObjectsForROC with outputRejectLevels (tempcv.cpp:1084-1094).
    Candidates, their order, reject levels and the FP64 stage sums must equal the oracle's bit for bit."""
    frames = np.stack([octave_frame(640, 480, 7), uniform_frame(640, 480, 8), octave_frame(640, 480, 9)])
    cas = clfd.Cascade(cascade_path(name))
    det = clfd.Detector(gpu_ctx, cas, 640, 480, max_batch=3, scale_factor=1.2, want_codes=True)
    det.detect(frames)
    r, lv, wt = det.reject_levels()
    oc = oracle_cascade(name)
    at = 0
    total = 0
    for f in range(3):
        orr, olv, owt = oc.detect_roc(frames[f], 1.2)
        n = len(orr)
        mine = r[at:at + n]
        assert np.all(mine["frame"] == f) and (at + n == len(r) or r[at + n]["frame"] > f)
        assert np.array_equal(np.stack([mine["x"], mine["y"], mine["w"], mine["h"]], 1).reshape(-1, 4), orr.reshape(-1, 4))
        assert np.array_equal(lv[at:at + n], olv)
        assert wt[at:at + n].tobytes() == owt.tobytes()
        at += n
        total += n
    assert at == len(r)
    if name in ("frontalface_alt", "eye", "mcs_nose"):
        assert total > 10 and len(np.unique(lv)) >= 2   # rejected-late windows are really there
    det.close()


def test_reject_levels_errors(gpu_ctx):
    cas = clfd.Cascade(cascade_path("frontalface_alt"))
    frame = np.stack([octave_frame(320, 240, 1)])
    det = clfd.Detector(gpu_ctx, cas, 320, 240, max_batch=1, scale_factor=1.2)
    det.detect(frame)
    with pytest.raises(clfd.ClfdError, match="want_codes"):
        det.reject_levels()
    det.close()
    det = clfd.Detector(gpu_ctx, cas, 320, 240, max_batch=1, scale_factor=1.2, scale_cascade=True)
    det.detect(frame)
    with pytest.raises(clfd.ClfdError, match="image-pyramid"):
        det.reject_levels()
    det.close()
    det = clfd.Detector(gpu_ctx, cas, 320, 240, max_batch=1, scale_factor=1.2, want_codes=True)
    r, lv, wt = det.reject_levels()   # nothing detected yet
    assert len(r) == 0
    det.close()


def test_submit_collect_pipeline_keeps_batches_apart(gpu_ctx):
    """clfd_detect_submit / _collect: two batches in flight (the copy of batch i+1 overlaps the
    kernels of batch i).  Results must come back in submission order and equal the blocking call."""
    import torch
    cas = clfd.Cascade(cascade_path("frontalface_alt"))
    det = clfd.Detector(gpu_ctx, cas, 640, 480, max_batch=8, scale_factor=1.2)
    batches = [np.stack([octave_frame(640, 480, 10 * b + i) for i in range(8)]) for b in range(4)]
    pinned = [torch.from_numpy(b).pin_memory() for b in batches]
    want = [det.detect(b) for b in batches]
    got = []
    det.submit(pinned[0])
    for b in range(1, 4):
        det.submit(pinned[b])
        got.append(det.collect())
    got.append(det.collect())
    for b in range(4):
        assert got[b].stats["windows"] == 8 * det.windows_per_frame()
        for f in range(8):
            assert np.array_equal(got[b].frame_rects(f), want[b].frame_rects(f)), (b, f)
    with pytest.raises(Exception):
        det.collect()            # nothing in flight
    det.submit(pinned[0]); det.submit(pinned[1])
    with pytest.raises(Exception):
        det.submit(pinned[2])    # two already in flight
    det.collect(); det.collect()
    det.close()


@pytest.mark.parametrize("per_frame_ranges", [True, False])
@pytest.mark.parametrize("name,sf,shape", [("frontalface_alt", 1.2, (640, 480)), ("frontalface_alt2", 1.3, (500, 380)),
                                           ("frontalface_alt_tree", 1.25, (480, 360)), ("fullbody", 1.2, (400, 420)),
                                           ("eye_tree_eyeglasses", 1.1, (330, 250)), ("frontalface_default", 1.15, (700, 300))])
def test_scale_cascade_mode_equals_ref_sc_oracle(gpu_ctx, monkeypatch, name, sf, shape, per_frame_ranges):
    """CLFD_MODE_SCALE_CASCADE (SURVEY 8-f row 3): one integral image, features scaled per factor,
    step max(2, factor) and the skip rule of HaarDetectObjects_ScaleCascade_Invoker -- exit codes
    (including skipped / out-of-bounds markers) and the rect set identical to the REF-SC oracle.
    The batch runs as one range, or as one range per frame (the kernels see pre-offset codes, the
    survivor queues restart and the rect count carries over between ranges)."""
    W, H = shape
    frames = np.stack([octave_frame(W, H, 21), uniform_frame(W, H, 22), np.full((H, W), 255, np.uint8)])
    cas = clfd.Cascade(cascade_path(name))
    det = clfd.Detector(gpu_ctx, cas, W, H, max_batch=3, scale_factor=sf, scale_cascade=True)
    monkeypatch.setenv("CLFD_DETECT_CHUNKS", "1")
    if per_frame_ranges:
        launches_one_range = det.detect(frames).stats["kernel_launches"]
        monkeypatch.setenv("CLFD_DETECT_CHUNKS", "3")
    res = det.detect(frames)
    if per_frame_ranges:
        assert res.stats["kernel_launches"] > launches_one_range   # the batch really was cut
    codes = det.codes(0, 3)
    oc = oracle_cascade(name)
    for f in range(3):
        rects, ocodes, st, levels = oc.detect_sc(frames[f], sf)
        assert [(l.nx, l.ny, l.win_w, l.win_h) for l in levels] == [(l.nx, l.ny, l.win_w, l.win_h) for l in det.levels()]
        assert len(ocodes) == det.windows_per_frame()
        bad = np.flatnonzero(codes[f] != ocodes)
        assert bad.size == 0, f"{name} frame {f}: {bad.size} codes differ, first {bad[:5]} gpu {codes[f][bad[:5]]} oracle {ocodes[bad[:5]]}"
        assert np.array_equal(res.frame_rects(f), _sorted(rects))
    assert (codes == -32768).any()   # the skip rule fired
    det.close()


def test_scale_cascade_mode_min_size_and_batch_ranges(gpu_ctx, monkeypatch):
    monkeypatch.setenv("CLFD_DETECT_CHUNKS", "2")
    frames = np.stack([octave_frame(480, 360, i) for i in range(8)])
    cas = clfd.Cascade(cascade_path("frontalface_alt"))
    det = clfd.Detector(gpu_ctx, cas, 480, 360, max_batch=8, scale_factor=1.3, min_size=(40, 40), scale_cascade=True)
    res = det.detect(frames)
    oc = oracle_cascade("frontalface_alt")
    for f in (0, 5, 7):
        rects, ocodes, _, levels = oc.detect_sc(frames[f], 1.3, (40, 40))
        assert np.array_equal(det.codes(0, 8)[f], ocodes)
        assert np.array_equal(res.frame_rects(f), _sorted(rects))
        assert all(l.win_w >= 40 for l in det.levels())
    det.close()


def test_scale_cascade_mode_golden_fixture(gpu_ctx):
    """committed REF-SC vectors (tests/golden/refsc.npz) against the CUDA path"""
    import os, zlib
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "refsc.npz"))
    for name in ("frontalface_alt", "fullbody"):
        cas = clfd.Cascade(cascade_path(name))
        det = clfd.Detector(gpu_ctx, cas, 320, 240, max_batch=2, scale_factor=1.2, scale_cascade=True)
        frames = np.stack([octave_frame(320, 240, 21), uniform_frame(320, 240, 22)])
        res = det.detect(frames)
        codes = det.codes(0, 2)
        for fi in range(2):
            assert zlib.crc32(codes[fi].tobytes()) == int(g[f"{name}_crc_{fi}"][0])
            assert np.array_equal(res.frame_rects(fi), _sorted(g[f"{name}_rects_{fi}"]))
        det.close()


def test_empty_ragged_and_odd_inputs(gpu_ctx):
    """Frames too small for any window (no level at all), row strides larger than the width and not
    16-byte multiples, a 1-frame batch in a detector planned for more, and both modes."""
    import torch
    cas = clfd.Cascade(cascade_path("frontalface_alt"))
    # (i) smaller than the window: zero levels, zero rects, no launch failure
    for sc in (False, True):
        det = clfd.Detector(gpu_ctx, cas, 19, 18, scale_factor=1.2, scale_cascade=sc, want_codes=True)
        assert det.windows_per_frame() == 0 and len(det.levels()) == 0
        res = det.detect(np.zeros((1, 18, 19), np.uint8))
        assert len(res.rects) == 0
        det.close()
    # (ii) ragged rows: width 301 inside a 333-byte pitch, frame pitch with slack, device and host input
    W, H = 301, 233
    frame = octave_frame(W, H, 51)
    oc = oracle_cascade("frontalface_alt")
    want, ocodes, _, _, _ = oc.detect(frame, 1.2)
    want_sc, ocodes_sc, _, _ = oc.detect_sc(frame, 1.2)
    buf = np.full((3, H + 5, 333), 77, np.uint8)
    buf[:, :H, :W] = frame
    view = buf[:, :H, :W]                      # strides (frame 338*333... , row 333)
    for sc, w, c in ((False, want, ocodes), (True, want_sc, ocodes_sc)):
        det = clfd.Detector(gpu_ctx, cas, W, H, max_batch=4, scale_factor=1.2, scale_cascade=sc, want_codes=True)
        cnt = clfd.abi.C.c_int64()
        clfd.abi.check(clfd.abi.lib().clfd_detect(det._h, view.ctypes.data, 3, view.strides[0], view.strides[1],
                                                   det._rects.ctypes.data_as(clfd.abi.C.POINTER(clfd.abi.Rect)), det._rect_cap,
                                                   clfd.abi.C.byref(cnt)))
        res = clfd.DetectResult(det._rects[:cnt.value].copy(), det.stats())
        codes = det.codes(0, 3)
        for f in range(3):
            assert np.array_equal(codes[f], c)
            assert np.array_equal(res.frame_rects(f), _sorted(w))
        # the same ragged layout already on the device, through enqueue / fetch
        t = torch.from_numpy(buf).cuda()
        torch.cuda.synchronize()
        det.enqueue(t, 3, t.stride(0), t.stride(1), torch.cuda.current_stream().cuda_stream)
        res2 = det.fetch(torch.cuda.current_stream().cuda_stream)
        for f in range(3):
            assert np.array_equal(res2.frame_rects(f), _sorted(w))
        det.close()


@pytest.mark.parametrize("name", ["frontalface_alt", "frontalface_default", "frontalface_alt_tree", "frontalface_alt2", "fullbody",
                                  "mcs_nose", "eye"])
def test_flat_regions_take_the_table_and_equal_the_oracle(gpu_ctx, monkeypatch, name):
    """Flat windows (every pixel equal) are looked up in a table the detector measures at creation instead of walking one
    FP64 fallback per stage.  Frames made of flat regions of every kind -- letterbox bars, a saturated half, a board of
    flat patches of all 256 values with noise between them, all-black, all-white -- must give the oracle's rects, and the
    same rects with the table switched off (CLFD_NO_FLAT_TABLE)."""
    W, H = 640, 360
    base = octave_frame(W, H, 77)
    frames = []
    lb = base.copy(); lb[:60] = 0; lb[-60:] = 16; frames.append(lb)
    sat = base.copy(); sat[:, W // 2:] = 255; frames.append(sat)
    board = base.copy()
    for v in range(256):   # 40 x 32 patches of every value; noise strips between them
        y, x = (v // 16) * 22, (v % 16) * 40
        board[y:y + 20, x:x + 36] = v
    frames.append(board)
    big = base.copy(); big[40:200, 100:400] = 128; big[220:340, 50:300] = 3; frames.append(big)
    frames += [np.zeros((H, W), np.uint8), np.full((H, W), 255, np.uint8), np.full((H, W), 77, np.uint8)]
    frames = np.stack(frames)
    cas = clfd.Cascade(cascade_path(name))
    det = clfd.Detector(gpu_ctx, cas, W, H, max_batch=len(frames), scale_factor=1.2)
    got = det.detect(frames)
    det.close()
    monkeypatch.setenv("CLFD_NO_FLAT_TABLE", "1")
    det = clfd.Detector(gpu_ctx, cas, W, H, max_batch=len(frames), scale_factor=1.2)
    plain = det.detect(frames)
    det.close()
    oc = oracle_cascade(name)
    total = 0
    for f in range(len(frames)):
        rects, _, _, _, _ = oc.detect(frames[f], 1.2, want_codes=False)
        want = _sorted(rects)
        assert np.array_equal(got.frame_rects(f), want), (name, f)
        assert np.array_equal(plain.frame_rects(f), want), (name, f)
        total += len(want)
    assert total > 0
