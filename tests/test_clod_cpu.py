"""CLOD-CPU (oracle/clod_cpu.c), the restatement of the reference's OWN CPU detector -- clodDetectObjects(use_cl=FALSE),
clod.cpp:1339-1500, "the reference's CPU path" of BASELINE.json and the second CPU baseline of bench.py -- is held equal
to (a) golden vectors recorded from the reference's compiled code (tests/golden/make_clod_golden.py) and (b) that code
itself (oracle/_ref) where it is present."""
import os
import sys

import numpy as np
import pytest

import oracle
from clfacedetection_b200.frames import octave_frame, uniform_frame
from conftest import cascade_path

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_clod_golden import MODES, STUMP_CASCADES, clod_frames  # noqa: E402

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_clod.npz"))


@pytest.mark.parametrize("name", STUMP_CASCADES)
def test_clod_cpu_equals_reference_golden(name):
    oc = oracle.Cascade(cascade_path(name))
    total = 0
    for f, img in enumerate(clod_frames()):
        for tag, flags in MODES.items():
            r, n_win, n_eval = oc.clod_cpu_detect(img, 1.1, flags=flags)
            assert np.array_equal(r, GOLD[f"{name}/{tag}_{f}"]), (name, f, tag)
            assert n_win > 0 and n_eval >= n_win
            total += len(r)
    assert total > 0


def test_clod_cpu_equals_reference_code():
    """fresh frames, min / max window sizes, straight against the reference's compiled clodDetectObjects"""
    from oracle import ref
    if not ref.available():
        pytest.skip("no original sources (CLFD_REFERENCE_DIR) and no library in oracle/_ref")
    rng = np.random.default_rng(5)
    for name in ("frontalface_alt", "eye"):
        oc = oracle.Cascade(cascade_path(name))
        rc = ref.RefCascade(cascade_path(name))
        for k in range(3):
            W, H = int(rng.integers(90, 400)), int(rng.integers(80, 300))
            img = octave_frame(W, H, 100 + k) if k % 2 == 0 else uniform_frame(W, H, 100 + k)
            for mn, mx in (((0, 0), (0, 0)), ((30, 30), (0, 0)), ((0, 0), (60, 60))):
                for flags in MODES.values():
                    mine, _, _ = oc.clod_cpu_detect(img, 1.1, mn, mx, flags)
                    assert np.array_equal(mine, rc.clod_detect(img, flags, mn, mx)), (name, W, H, mn, mx, flags)


def test_clod_cpu_rejects_what_the_reference_cannot_run():
    """trees: the reference reads haar_feature[0] and alpha[0..1] only (clod.cpp:458,649)"""
    with pytest.raises(ValueError):
        oracle.Cascade(cascade_path("frontalface_alt2")).clod_cpu_detect(octave_frame(100, 100, 1))


def test_clod_cpu_batch_equals_single_frames():
    oc = oracle.Cascade(cascade_path("frontalface_alt"))
    frames = np.stack([octave_frame(160, 120, 40 + i) for i in range(5)])
    counts, n_win, n_eval = oc.clod_cpu_detect_batch(frames, 1.2, n_threads=3)
    one = [oc.clod_cpu_detect(f, 1.2) for f in frames]
    assert list(counts) == [len(r[0]) for r in one]
    assert n_win == sum(r[1] for r in one) and n_eval == sum(r[2] for r in one)
