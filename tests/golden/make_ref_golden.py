#!/usr/bin/env python
"""Golden vectors made BY THE REFERENCE'S OWN CODE (run with CLFD_REFERENCE_DIR naming the original
sources): oracle/build_ref.py compiles tempcv.cpp:40-1516, 1702-2089 from where they lie, and this
script records what those functions return on fixed-seed frames.

tests/golden/reference_tempcv.npz, per cascade `c` (all 19 files) and frame `f` (0: octave noise
320x240 seed 21, 1: uniform noise 320x240 seed 22):

  c/lvl_f      int8 [220|..][300|..]  raw return value of cvRunHaarClassifierCascadeSum (tempcv.cpp:795-972)
                                      at every (x, y) of the frame taken as one level at scale 1
                                      (1 accept, -i rejected by stage i, 0 stage 0 / any stage-tree reject)
  c/si_f       int32 [n][4]           cvHaarDetectObjectsForROC, CV_HAAR_SCALE_IMAGE, scale 1.2, minNeighbors 0
  c/sig_f      int32 [m][5]           same with minNeighbors 2: x, y, w, h, neighbors
  c/roc_f      float64 [k][6]         outputRejectLevels: x, y, w, h, level, stage sum
  c/sc_f       int32 [n][4]           flags 0 (scale-cascade path), scale 1.2, minNeighbors 0
  c/census     int32 [5]              win_w, win_h, stages, trees, nodes as icvReadHaarClassifier built them
  c/hid_w      float32 [N][3]         hidden-cascade weights at scale 1 (tempcv.cpp:733-760)
  c/hid_thr    float32 [S]            biased stage thresholds (tempcv.cpp:419)
  group/...                            AgroupRectangles on 40 random rect sets, eps 0.2 and 0.35

The .npz is what the CPU oracle and the CUDA path are compared with on machines that have
neither the original sources nor oracle/_ref (tests/test_reference_golden.py, test_gpu_reference_golden.py).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from clfacedetection_b200.frames import octave_frame, uniform_frame  # noqa: E402
from oracle import ref  # noqa: E402

CASCADES = ["eye", "eye_tree_eyeglasses", "frontalface_alt", "frontalface_alt2", "frontalface_alt_tree",
            "frontalface_default", "fullbody", "lefteye_2splits", "lowerbody", "mcs_eyepair_big",
            "mcs_eyepair_small", "mcs_lefteye", "mcs_mouth", "mcs_nose", "mcs_righteye", "mcs_upperbody",
            "profileface", "righteye_2splits", "upperbody"]


def golden_frames():
    return [octave_frame(320, 240, 21), uniform_frame(320, 240, 22)]


def group_inputs():
    rng = np.random.default_rng(77)
    sets = []
    for i in range(40):
        k = int(rng.integers(1, 6))
        base = rng.integers(0, 300, size=(k, 2))
        n = int(rng.integers(1, 60))
        pick = rng.integers(0, k, size=n)
        size = 30 + rng.integers(0, 40, size=k)
        r = np.stack([base[pick, 0] + rng.integers(-5, 6, size=n), base[pick, 1] + rng.integers(-5, 6, size=n),
                      size[pick] + rng.integers(-3, 4, size=n), size[pick] + rng.integers(-3, 4, size=n)], 1)
        sets.append(r.astype(np.int32))
    return sets


def main():
    from oracle import build_ref
    ref_dir = build_ref.REF
    out = {}
    for name in CASCADES:
        rc = ref.RefCascade(os.path.join(ref_dir, f"haarcascade_{name}.xml"))
        out[f"{name}/census"] = np.array([rc.win_w, rc.win_h, rc.n_stages, rc.n_trees, rc.n_nodes], np.int32)
        hid = rc.hidden(64, 64, 1.0)
        out[f"{name}/hid_w"] = hid["weights"]
        out[f"{name}/hid_thr"] = hid["stage_thr"]
        for fi, frame in enumerate(golden_frames()):
            res, _ = rc.eval_level(frame, 1)
            assert res.min() >= -127
            out[f"{name}/lvl_{fi}"] = res.astype(np.int8)
            r, _, _, _ = rc.detect(frame, 1.2, 0, ref.CV_HAAR_SCALE_IMAGE)
            out[f"{name}/si_{fi}"] = r
            r, nb, _, _ = rc.detect(frame, 1.2, 2, ref.CV_HAAR_SCALE_IMAGE)
            out[f"{name}/sig_{fi}"] = np.concatenate([r, nb[:, None]], 1).astype(np.int32)
            r, _, lv, wt = rc.detect(frame, 1.2, 0, ref.CV_HAAR_SCALE_IMAGE, reject_levels=True)
            out[f"{name}/roc_{fi}"] = np.concatenate([r.astype(np.float64), lv[:, None].astype(np.float64), wt[:, None]], 1)
            r, _, _, _ = rc.detect(frame, 1.2, 0, 0)
            out[f"{name}/sc_{fi}"] = r
        print(name, {k.split("/")[1]: len(v) for k, v in out.items() if k.startswith(name + "/") and k[-2] == "_"})
    for i, r in enumerate(group_inputs()):
        for eps in (0.2, 0.35):
            g, w = ref.group_rectangles(r, 2, eps)
            out[f"group/{i}_{eps}"] = np.concatenate([g, w[:, None]], 1).astype(np.int32)
    np.savez_compressed(os.path.join(HERE, "reference_tempcv.npz"), **out)
    print("wrote", os.path.join(HERE, "reference_tempcv.npz"), os.path.getsize(os.path.join(HERE, "reference_tempcv.npz")), "bytes")


if __name__ == "__main__":
    main()
