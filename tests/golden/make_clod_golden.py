#!/usr/bin/env python
"""Golden vectors made BY THE REFERENCE'S OWN CPU DETECTOR (run with CLFD_REFERENCE_DIR naming the original
sources): oracle/build_ref.py compiles clod.cpp:11-38, 182-357, 371-527, 580-787, 1339-1500 from where they lie,
and this script records clodDetectObjects(use_cl = FALSE, min_neighbors = 0) on fixed-seed frames.

tests/golden/reference_clod.npz, per stump cascade `c` and frame `f`:
  c/ps_f   int32 [n][4]   flags CLOD_PER_STAGE_ITERATIONS | CLOD_PRECOMPUTE_FEATURES (main.cpp:79,90), raw matches
  c/pw_f   int32 [n][4]   flags CLOD_PRECOMPUTE_FEATURES (window at a time, x step 2 after a stage-0 exit)
  c/pn_f   int32 [n][4]   flags 0 (features scaled per call, runClassifier clod.cpp:580-634)
Scale factor 1.1 (hard-coded, clod.cpp:1349).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from clfacedetection_b200.frames import octave_frame, uniform_frame  # noqa: E402
from oracle import ref  # noqa: E402

STUMP_CASCADES = ["frontalface_alt", "frontalface_default", "eye", "mcs_mouth", "upperbody"]
MODES = {"ps": (2 << 2) | (2 << 0), "pw": 2 << 0, "pn": 0}


def clod_frames():
    return [octave_frame(320, 240, 31), uniform_frame(200, 150, 32), octave_frame(417, 301, 33)]


def main():
    out = {}
    for name in STUMP_CASCADES:
        rc = ref.RefCascade(os.path.join(ROOT, "data", "haarcascades", f"haarcascade_{name}.xml"))
        for f, img in enumerate(clod_frames()):
            for tag, flags in MODES.items():
                out[f"{name}/{tag}_{f}"] = rc.clod_detect(img, flags)
    np.savez_compressed(os.path.join(HERE, "reference_clod.npz"), **out)
    print({k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    main()
