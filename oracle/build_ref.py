#!/usr/bin/env python3
"""Build oracle/_ref/libtempcv_ref.so: the REFERENCE'S OWN Haar code, compiled where it lies.

TEST INFRASTRUCTURE ONLY.  Reads tempcv.{hpp,cpp} of the original CLFaceDetection sources, from the
directory CLFD_REFERENCE_DIR names (read-only),
copies the line ranges below verbatim into oracle/_ref/*.inc (scratch files in a git-ignored
directory, deleted again as soon as the compiler has read them) and compiles them together with oracle/ref_shim/ (a test-only stand-in for the few
OpenCV 2.4 names those ranges touch) and oracle/vj_oracle.c (whose cv2-pinned resize / integral
stand in for the cvResize / cvIntegral the reference links from OpenCV's dylibs).

tempcv.cpp as a whole cannot be compiled in this image: it includes <vector.h> and seven OpenCV
2.4.2 headers (tempcv.cpp:6-18) that do not exist here, and its tail (2271-2309) is an `#if 0`
block.  The ranges taken are every function on the Haar path:

    tempcv.hpp   60- 155  CV_HAAR_* constants, CvHaarFeature/Classifier/StageClassifier/Cascade
    tempcv.cpp   40-1516  AgroupRectangles, hidden-cascade structs + builder,
                          cvSetImagesForHaarClassifierCascade, icvEvalHidHaarClassifier,
                          cvRunHaarClassifierCascadeSum, both invokers,
                          cvHaarDetectObjectsForROC, cvHaarDetectObjects
    tempcv.cpp 1702-2089  cvReleaseHaarClassifierCascade, icvReadHaarClassifier (XML reader)

and the reference's own CPU detector ("CLOD-CPU", what BASELINE.json calls the reference's CPU path;
clod.cpp as a whole needs the author's un-vendored CLUtil and <OpenCL/opencl.h>):

    clod.h       17-21, 39-47   CLOD_* flags, CLODWeightedRect, CLODDetectObjectsResult
    clod.cpp     11-38          macros, CLODOptimizedRect, CLODSubwindowData
    clod.cpp    182-357         areRectSimilar, partitionData, filterResult (compiled, never called: min_neighbors = 0)
    clod.cpp    371-527         setupScale, computeVariance, precomputeFeatures, precomputeWindows
    clod.cpp    580-787         runClassifier, runClassifierWithPrecomputedFeatures, runSubwindow, runCascade
    clod.cpp   1339-1500        clodDetectObjects

Without CLFD_REFERENCE_DIR nothing is built: a library already in oracle/_ref is used, and tests
that need it skip if there is none.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("CLFD_REFERENCE_DIR", "")   # the original CLFaceDetection sources; none by default
OUT = os.path.join(HERE, "_ref")
LIB = os.path.join(OUT, "libtempcv_ref.so")

RANGES = {
    "tempcv_hpp_extract.inc": ("tempcv.hpp", [(60, 155)]),
    "tempcv_cpp_extract.inc": ("tempcv.cpp", [(40, 1516), (1702, 2089)]),
    # the reference's own CPU detector, clodDetectObjects(use_cl = FALSE): flags and result structs; macros and list
    # structs, filterResult, setupScale .. precomputeWindows, runClassifier .. runCascade, clodDetectObjects
    "clod_h_extract.inc": ("clod.h", [(17, 21), (39, 47)]),
    "clod_cpp_extract.inc": ("clod.cpp", [(11, 38), (182, 357), (371, 527), (580, 787), (1339, 1500)]),
}
SOURCES = ("tempcv.hpp", "tempcv.cpp", "clod.h", "clod.cpp")

def reference_available() -> bool:
    return bool(REF) and all(os.path.exists(os.path.join(REF, f)) for f in SOURCES)


def _extract() -> None:
    os.makedirs(OUT, exist_ok=True)
    for out_name, (src, ranges) in RANGES.items():
        with open(os.path.join(REF, src), "rb") as f:
            raw = f.read()
        lines = raw.decode("utf-8", errors="replace").split("\n")
        parts = []
        for lo, hi in ranges:
            parts.append(f"/* ---- {src}:{lo}-{hi}, verbatim (build product, not committed) ---- */")
            parts.append(f'#line {lo} "{os.path.join(REF, src)}"')
            parts.extend(lines[lo - 1:hi])
        with open(os.path.join(OUT, out_name), "w") as f:
            f.write("\n".join(parts) + "\n")
    with open(os.path.join(OUT, "SOURCES.txt"), "w") as f:
        for src in SOURCES:
            with open(os.path.join(REF, src), "rb") as g:
                f.write(f"{hashlib.sha256(g.read()).hexdigest()}  {src}\n")


def build(force: bool = False) -> str | None:
    """Returns the path of the library, or None when neither the reference nor a prebuilt
    library is available."""
    deps = [os.path.join(HERE, "ref_shim", "cvmini.hpp"), os.path.join(HERE, "ref_shim", "ref_driver.cpp"),
            os.path.join(HERE, "ref_shim", "clod_driver.cpp"),
            os.path.join(HERE, "vj_oracle.c"), os.path.join(HERE, "vj_oracle.h"), os.path.abspath(__file__)]
    if not reference_available():
        return LIB if os.path.exists(LIB) else None
    deps += [os.path.join(REF, f) for f in SOURCES]
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= max(os.path.getmtime(d) for d in deps):
        return LIB
    _extract()
    cflags = ["-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC"]
    obj = os.path.join(OUT, "vj_oracle.o")
    subprocess.check_call(["/usr/bin/gcc", "-std=gnu11"] + cflags + ["-c", os.path.join(HERE, "vj_oracle.c"), "-o", obj])
    subprocess.check_call(["/usr/bin/g++", "-std=gnu++14", "-w"] + cflags +
                          ["-I", OUT, "-I", os.path.join(HERE, "ref_shim"), "-shared", "-o", LIB,
                           os.path.join(HERE, "ref_shim", "ref_driver.cpp"), os.path.join(HERE, "ref_shim", "clod_driver.cpp"),
                           obj, "-lm"])
    # the verbatim extracts were only needed by the compiler: nothing of the reference's text stays
    for name in list(RANGES) + ["vj_oracle.o"]:
        os.unlink(os.path.join(OUT, name))
    return LIB


if __name__ == "__main__":
    p = build(force="--force" in sys.argv)
    print(p if p else "reference sources not found and no prebuilt oracle/_ref/libtempcv_ref.so")
