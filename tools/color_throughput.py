"""Colour input throughput on one GPU: end-to-end frames/s of the streaming host API (clfd_detect_submit[_color] /
clfd_detect_collect, two batches in flight) for gray, BGR and BGRA batches of the same frames, and the time and
bandwidth of the colour conversion kernel (k_color_to_gray, clfd_detector_get_kernel_ms slot [6]).

    python tools/color_throughput.py [--steps 24] [--warmup 3] [--batch 64] [--out result.json]

Frames: 1080p, B, G and R planes from distinct octave_frame seeds (alpha from another one); the gray arm uses their
formula gray (B*1868 + G*9617 + R*4899 + 8192) >> 14.  frontalface_alt at scale 1.2, pinned host memory.  The three
arms run in one process and alternate batch by batch in one submit / collect stream: a batch's time is the interval
between the collect before it and its own collect, i.e. what it adds to a steady stream with two batches in flight.
The conversion time comes from a separate pass with profiling on (blocking calls, one range per batch, serial order).
Prints one JSON object; --out also writes it to a file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

W, H = 1920, 1080
SCALE = 1.2
CASCADE = os.path.join(ROOT, "data", "haarcascades", "haarcascade_frontalface_alt.xml")
HBM_MEASURED_GBS = 6549.4   # the project's measured B200 HBM copy bandwidth (BASELINE.md)
HBM_DATASHEET_GBS = 7700.0  # NVIDIA HGX B200 data sheet, per GPU
ARMS = (("gray", 1), ("bgr", 3), ("bgra", 4))


def formula_gray(img):
    b, g, r = (img[..., k].astype(np.int64) for k in range(3))
    return ((b * 1868 + g * 9617 + r * 4899 + 8192) >> 14).astype(np.uint8)


def sorted_rects(res):
    r = res.rects
    return np.sort(r, order=["frame", "cascade", "w", "y", "x", "h"])


def gpu_info(index):
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                          "-i", str(index)], capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=24, help="timed batches per arm (>= 20)")
    ap.add_argument("--warmup", type=int, default=3, help="untimed batches per arm first")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--unique", type=int, default=8, help="distinct frames, repeated to fill a batch")
    ap.add_argument("--prof-steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import clfacedetection_b200 as clfd
    from clfacedetection_b200.frames import octave_frame

    if not torch.cuda.is_available():
        raise SystemExit("color_throughput.py needs a CUDA device")
    B = args.batch
    uniq = np.empty((args.unique, H, W, 4), np.uint8)
    for i in range(args.unique):
        for k in range(4):
            uniq[i, ..., k] = octave_frame(W, H, 3000 + 4 * i + k)
    host = {
        "bgra": torch.empty((B, H, W, 4), dtype=torch.uint8).pin_memory(),
        "bgr": torch.empty((B, H, W, 3), dtype=torch.uint8).pin_memory(),
        "gray": torch.empty((B, H, W), dtype=torch.uint8).pin_memory(),
    }
    for i in range(B):
        f = uniq[i % args.unique]
        host["bgra"][i] = torch.from_numpy(f)
        host["bgr"][i] = torch.from_numpy(np.ascontiguousarray(f[..., :3]))
        host["gray"][i] = torch.from_numpy(formula_gray(f))

    ctx = clfd.Context(0)
    det = clfd.Detector(ctx, clfd.Cascade(CASCADE), W, H, max_batch=B, scale_factor=SCALE)

    # ---- end to end: one submit / collect stream, arms alternating batch by batch -----------------------------------
    order = [name for _ in range(args.warmup + args.steps) for name, _ in ARMS]
    times = {name: [] for name, _ in ARMS}
    first = None   # every batch holds the same frames: every arm's every batch must return these rects
    identical = True
    det.submit(host[order[0]])
    torch.cuda.synchronize()
    t_prev = time.perf_counter()
    for k in range(len(order)):
        if k + 1 < len(order):
            det.submit(host[order[k + 1]])
        res = det.collect()
        t = time.perf_counter()
        if k >= args.warmup * len(ARMS):
            times[order[k]].append(t - t_prev)
        t_prev = t
        r = sorted_rects(res)
        if first is None:
            first = r
        elif not np.array_equal(r, first):
            identical = False
    fps = {n: B / float(np.mean(times[n])) for n, _ in ARMS}

    # ---- conversion kernel time: profiling pass ------------------------------------------------------------------
    det.set_profiling(True)
    conv_ms = {}
    for name, c in ARMS:
        ms = []
        for _ in range(args.prof_steps + 1):
            det.detect(host[name])
            ms.append(det.kernel_ms()[6])
        conv_ms[name] = float(np.mean(ms[1:]))
    det.set_profiling(False)
    assert conv_ms["gray"] == 0.0, conv_ms

    kernel = {}
    for name, c in ARMS[1:]:
        alg = (c + 1) * W * H * B   # read C bytes, write 1 byte per pixel
        gbs = alg / (conv_ms[name] * 1e-3) / 1e9
        kernel[name] = {"ms_per_batch": round(conv_ms[name], 4), "algorithmic_bytes_per_batch": alg,
                        "achieved_gbs": round(gbs, 1),
                        "fraction_of_measured_hbm_6549.4_gbs": round(gbs / HBM_MEASURED_GBS, 3),
                        "fraction_of_datasheet_hbm_7700_gbs": round(gbs / HBM_DATASHEET_GBS, 3)}
    result = {
        "what": "colour vs gray input, streaming submit/collect with two batches in flight",
        "gpu": gpu_info(torch.cuda.current_device()),
        "frame": [W, H], "batch": B, "cascade": "frontalface_alt", "scale_factor": SCALE,
        "steps_per_arm": args.steps, "warmup_per_arm": args.warmup,
        "h2d_bytes_per_batch": {n: W * H * c * B for n, c in ARMS},
        "frames_per_s": {n: round(v, 1) for n, v in fps.items()},
        "ms_per_batch_median": {n: round(float(np.median(times[n])) * 1e3, 3) for n, _ in ARMS},
        "color_over_gray": {n: round(fps[n] / fps["gray"], 4) for n, _ in ARMS[1:]},
        "conversion_kernel": kernel,
        "rects_per_batch": int(len(first)),
        "rects_identical_across_arms": bool(identical),
    }
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    det.close()
    ctx.close()
    if not identical:
        raise SystemExit("the three arms returned different rects")


if __name__ == "__main__":
    main()
