#!/usr/bin/env python
"""bench.py -- 1080p frames/s (and windows/s) of the Viola-Jones hot path on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, C ABI)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (its own code from oracle/_ref,
                                                             # else the oracle port) on the host cores
    python bench.py --steps K --warmup W --dump-outputs DIR  # also DIR/rects.npy: the rects of the last timed step

A "step" is one pass of the whole hot path (pyramid resize -> integral images -> cascade ->
raw rects) over one batch of synthetic 1080p frames per GPU.  Workload = BASELINE.json's
metric configuration: haarcascade_frontalface_alt, 1920x1080, scale 1.2 (SURVEY 8-d,
"north-star" row of Appendix C: 22 levels, 2 672 451 windows/frame).

`value`  : frames/s with the batch already resident in HBM (enqueue + rect fetch per step).
`e2e`    : frames/s through clfd_detect() -- pinned HOST frames in, H2D inside the timed
           region, host rect list out.
`roofline`: the dominant kernel (cascade tile kernel) against the measured HBM peak, using the
           compulsory bytes of SURVEY 8-d (the contract's figure), plus what actually bounds it:
           the L1 data pipe (shared-memory corner loads), from the committed ncu capture in
           profiles/traffic.json.  Per-kernel numbers for resize / integral are under `kernels`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H = 1920, 1080
CASCADE = "frontalface_alt"
SCALE = 1.2
MIN_SIZE = (0, 0)
XML = [os.path.join(ROOT, "data", "haarcascades", f"haarcascade_{CASCADE}.xml")]
KERNEL_NAMES = ["resize_colsum", "colscan", "integral_rows", "tilted", "cascade_tiles", "cascade_deep"]


def kernel_source_stamp():
    """sha256 over the CUDA sources the kernels are built from: profiles/traffic.json carries the stamp of the build its
    ncu capture was taken from (profiles/make_traffic.py), and a capture of other kernels is not used"""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "clfacedetection_b200", "csrc")
    for f in ("kernels_clif.cu", "kernels_clod.cu", "kernels_sc.cu", "kernels.h", "clfd_pack.h", "clfd_internal.h"):
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def ncu_traffic():
    """per-kernel DRAM bytes per frame and L1 data-pipe utilisation from the committed ncu capture; None (and the
    ncu_* fields of the line stay out) when the capture was taken from other kernel sources than the ones in the tree"""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return None
    if t.get("kernel_source_stamp") != kernel_source_stamp():
        sys.stderr.write("bench.py: profiles/traffic.json is stale (kernel sources changed since its ncu capture): "
                         "ncu figures left out; regenerate with tools/capture_step.sh\n")
        return None
    return t


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def mark(self):
        """start of the timed region: earlier samples are dropped"""
        self.t0 = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0 = getattr(self, "t0", 0.0)
        for ts, ln in self.lines:
            if ts < t0:
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dump_rects(dirname: str, rects: np.ndarray):
    """--dump-outputs: int32 [n, 6] rects (x, y, w, h, global frame, cascade) -> dirname/rects.npy in float64, rows
    sorted by frame, cascade, y, x, w, h (the device appends them in no fixed order).  Above 1 << 20 rows (48 MiB) a
    fixed-seed sample of the rows is kept, so the file stays under 64 MB."""
    out = rects[np.lexsort(rects.T[[3, 2, 0, 1, 5, 4]])].astype(np.float64)
    cap = 1 << 20
    if len(out) > cap:
        out = out[np.sort(np.random.default_rng(0).choice(len(out), cap, replace=False))]
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "rects.npy"), out)


def cpu_reference(frames: np.ndarray, threads: int):
    """The reference's CPU path on `frames` with `threads` host threads; returns (seconds, windows, rects, kind).

    kind "reference": oracle/_ref/libtempcv_ref.so -- the reference's OWN cvHaarDetectObjects (tempcv.cpp:1188-1503,
    CV_HAAR_SCALE_IMAGE, compiled from /root/reference by oracle/build_ref.py; the prebuilt library travels to the GPU
    box), one frame per thread at a time, every thread with its own cascade (the reference mutates the hidden cascade
    per level, tempcv.cpp:549-768, so a cascade cannot be shared).
    kind "port": the REF-SI restatement (oracle/vj_oracle.c, held equal to that library by tests/), OpenMP over window
    rows -- used when the library is absent."""
    import oracle
    from oracle import ref
    if ref.available():
        from concurrent.futures import ThreadPoolExecutor
        n_thr = max(1, min(threads, len(frames)))
        cas = [[ref.RefCascade(x) for x in XML] for _ in range(n_thr)]
        wpf = sum(sum(l.nx * l.ny for l in oracle.Cascade(x).plan_levels(W, H, SCALE, MIN_SIZE)) for x in XML)

        def work(t):
            n = 0
            for i in range(t, len(frames), n_thr):   # ctypes releases the GIL for the duration of the call
                for c in cas[t]:
                    n += len(c.detect(frames[i], SCALE, 0, ref.CV_HAAR_SCALE_IMAGE, MIN_SIZE)[0])
            return n
        t0 = time.perf_counter()
        with ThreadPoolExecutor(n_thr) as ex:
            rects = sum(ex.map(work, range(n_thr)))
        return time.perf_counter() - t0, wpf * len(frames), rects, "reference"
    cascades = [oracle.Cascade(x) for x in XML]
    t0 = time.perf_counter()
    windows = rects = 0
    for f in frames:
        for cas in cascades:
            r, _, _, st, _ = cas.detect(f, SCALE, MIN_SIZE, want_codes=False, n_threads=threads)
            windows += st.windows
            rects += len(r)
    return time.perf_counter() - t0, windows, rects, "port"


def clod_cpu_baseline(frames: np.ndarray, threads: int):
    """CLOD-CPU: the reference's own detector with use_cl = FALSE (clod.cpp:1339-1500, CLOD_PER_STAGE_ITERATIONS |
    CLOD_PRECOMPUTE_FEATURES as main.cpp:79 -- "the reference's CPU path" of BASELINE.json), restated in
    oracle/clod_cpu.c (pinned to the reference's compiled code by tests/test_clod_cpu.py) with the scale factor as a
    parameter.  Different semantics from the metric's pipeline (float, scaled features, step max(2, scale)): a context
    number, not a parity target.  None for cascades it cannot run (trees)."""
    import oracle
    try:
        t0 = time.perf_counter()
        matches = windows = evals = 0
        for x in XML:
            c, w, e = oracle.Cascade(x).clod_cpu_detect_batch(frames, SCALE, threads)
            matches += int(c.sum()); windows += w; evals += e
        dt = time.perf_counter() - t0
    except ValueError:
        return None
    n = len(frames)
    return {"value": round(n / dt, 3), "unit": "frames/s", "cores": min(threads, n), "kind": "port",
            "sample": f"{n} frames, one frame per thread (the reference is single-threaded, clod.cpp:700)",
            "windows_per_frame": windows // n, "windows_per_sec": round(windows / dt, 1),
            "classifier_evals_per_sec": round(evals / dt, 1), "matches": matches,
            "what": "clodDetectObjects(use_cl=FALSE), per-stage iterations + precomputed features, float (clod.cpp:1434-1482)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from clfacedetection_b200.frames import make_frames
    cores = os.cpu_count() or 1
    per_step = args.ref_frames if args.ref_frames > 0 else max(4, min(cores, 64))
    frames = make_frames("octave", W, H, per_step)
    for _ in range(args.warmup):
        cpu_reference(frames[:min(per_step, cores)], cores)
    t_total, win_total = 0.0, 0
    for _ in range(args.steps):
        t, w, _, kind = cpu_reference(frames, cores)
        t_total += t
        win_total += w
    fps = per_step * args.steps / t_total
    # for the record: the scale-cascade formulation (REF-SC: what main.cpp:145 runs) on a few of the frames, one pass,
    # and the reference's own CPU detector (CLOD-CPU, clod.cpp:1339-1500)
    import oracle
    t0 = time.perf_counter()
    sc_windows = 0
    n_sc = min(per_step, 4)
    for f in frames[:n_sc]:
        for x in XML:
            _, _, st, _ = oracle.Cascade(x).detect_sc(f, SCALE, MIN_SIZE, want_codes=False, n_threads=cores)
            sc_windows += st.windows
    sc_fps = n_sc / (time.perf_counter() - t0)
    how = ("one frame per thread, every thread its own cascade" if kind == "reference" else "OpenMP over window rows")
    line = {
        "impl": "reference", "metric": "frames_per_sec_1080p" if (W, H) == (1920, 1080) else f"frames_per_sec_{W}x{H}", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"haarcascade_{CASCADE} {W}x{H} scale {SCALE}, {per_step} octave-noise frames per step "
                               "(bounded sample of the 64-frame GPU batch)", "frames_per_step": per_step},
        "windows_per_sec": win_total / t_total,
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": min(cores, per_step) if kind == "reference" else cores, "kind": kind,
                         "sample": f"{per_step} frames/step x {args.steps} steps, {how}",
                         "what": ("oracle/_ref/libtempcv_ref.so: the reference's own cvHaarDetectObjects (tempcv.cpp, CV_HAAR_SCALE_IMAGE) "
                                  "compiled from its sources" if kind == "reference" else "oracle/vj_oracle.c (REF-SI restatement)"),
                         "scale_cascade_formulation_value": sc_fps, "scale_cascade_windows_per_frame": sc_windows // n_sc,
                         "clod_cpu": clod_cpu_baseline(frames, cores)},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def run_stream_bench(args):
    """BASELINE.json configs[4]: a stream of N distinct 1080p frames cut over the ranks (strong scaling), host frames
    in -> one gathered rect list out.  `value`: the same stream with the frames resident in HBM."""
    import torch
    import torch.distributed as dist

    import clfacedetection_b200 as clfd
    from clfacedetection_b200 import sharding, stream

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    N, B = args.stream, args.batch
    ctx = clfd.Context(local_rank)
    cas = [clfd.Cascade(x) for x in XML]
    det = clfd.Detector(ctx, cas, W, H, max_batch=B, scale_factor=SCALE, min_size=MIN_SIZE)
    src = stream.StreamSource(W, H)
    dev_canvas = src.canvas.cuda()
    first, last = sharding.shard_range(N, rank, world)
    cuda_stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def device_pass():
        n_rects = 0
        for g0, n, _ in src.runs(first, last, B):
            k, dy, dx = src.locate(g0)
            det.enqueue(dev_canvas[k, dy:, dx:], n, src.pitch, src.pitch, cuda_stream)
            n_rects += len(det.fetch(cuda_stream).rects)
        return n_rects

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(max(args.warmup, 3)):   # warm-up: a few batches of the shard
        g0, n, view = next(src.runs(first, last, B))
        det.submit_views(view, n, src.pitch, src.pitch)
        det.collect()
    barrier()
    sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    device_pass()
    e1.record()
    barrier()
    dev_ms = e0.elapsed_time(e1)
    e2e_s, gathered = stream.timed_stream(det, src, N, rank, world, B, barrier)
    clocks = sampler.stop()
    t = torch.tensor([dev_ms, e2e_s], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)   # max over ranks
    dev_ms, e2e_s = (float(x) for x in t.tolist())
    if args.dump_outputs and rank == 0:
        dump_rects(args.dump_outputs, gathered)
    if rank == 0:
        wpf = sum(det.windows_per_frame(i) for i in range(len(cas)))
        steps = -(-(last - first) // B)
        line = {"metric": "frames_per_sec_1080p" if (W, H) == (1920, 1080) else f"frames_per_sec_{W}x{H}",
                "value": round(N / (dev_ms / 1e3), 2), "unit": "frames/s", "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3),
                "ms_per_step": round(dev_ms / steps, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"stream of {N} distinct {W}x{H} frames, haarcascade_{CASCADE} scale {SCALE}, cut into contiguous "
                                       f"chunks over {world} GPU(s) (sharding.shard_range), batches of {B}, one gather of the rects",
                           "frames": N, "frames_per_rank": last - first, "windows_per_frame": wpf,
                           "l2": "every batch is 64 new frames (133 MB) + 5.6 GB of intermediates: nothing survives in the 126 MB L2"},
                "windows_per_sec": round(N * wpf / (dev_ms / 1e3), 1),
                "e2e": {"value": round(N / e2e_s, 2), "unit": "frames/s", "h2d_bytes_per_step": int(B * W * H),
                        "d2h_bytes_per_step": int(len(gathered) * 24 // max(steps * world, 1) + 32), "seconds": round(e2e_s, 4),
                        "api": "clfd_detect_submit/_collect on pinned host views, 2 batches in flight, then ONE gather of the rect lists "
                               "(inside the timed region)"},
                "gpu_launches": int(ctx.launch_count), "rects_total": int(len(gathered)), "clocks": clocks,
                "roofline": None, "cpu_baseline": None}
        print(json.dumps(line))
    det.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    global CASCADE, XML, W, H, SCALE, MIN_SIZE
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="frames per step per GPU")
    ap.add_argument("--ref-frames", type=int, default=0, help="frames per step of the CPU reference arm (0: one per host core, 4..64)")
    ap.add_argument("--cpu-baseline-frames", type=int, default=0, help="0: one frame per host core (4..64)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--stream", type=int, default=0, help="strong scaling: a stream of this many distinct frames cut over the ranks "
                                                          "(BASELINE.json configs[4]: 8192); prints its own line")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary configs[1] measurement")
    ap.add_argument("--mode", default="pyramid", choices=["pyramid", "scale-cascade"],
                    help="pyramid = CV_HAAR_SCALE_IMAGE semantics (the metric); scale-cascade = scaled features on one "
                         "integral image (SURVEY 8-f row 3), an extra measurement, not the headline")
    ap.add_argument("--size", default=f"{W}x{H}", help="frame shape WxH (default: the metric's 1920x1080)")
    ap.add_argument("--scale", type=float, default=SCALE, help="pyramid scale factor (default: the metric's 1.2)")
    ap.add_argument("--min-size", default="0x0", help="minimum window WxH")
    ap.add_argument("--cascade", default=CASCADE, help="stock cascade name (default: the metric's frontalface_alt; "
                    "frontalface_default is BASELINE.json configs[1]); a comma list shares one pyramid (configs[2], [3])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the raw rects of the last timed step (with --stream: of the timed host-to-rects pass over "
                         "the stream) to DIR/rects.npy (float64 [n, 6]: x, y, w, h, global frame, cascade; rows sorted), "
                         "so that two builds can be compared on the same seeded frames")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs covers the GPU path (--impl native) only")
    CASCADE = args.cascade
    XML = [os.path.join(ROOT, "data", "haarcascades", f"haarcascade_{c}.xml") for c in CASCADE.split(",")]
    W, H = (int(v) for v in args.size.lower().split("x"))
    SCALE = args.scale
    MIN_SIZE = tuple(int(v) for v in args.min_size.lower().split("x"))
    if args.impl == "reference":
        return run_reference(args)
    if args.stream > 0:
        return run_stream_bench(args)

    import torch
    import torch.distributed as dist

    import clfacedetection_b200 as clfd
    from clfacedetection_b200.frames import make_frames

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    B = args.batch
    # distinct fixed-seed frames per rank (frame stream sharded frame-wise: rank r owns frames r*B..)
    uniq = min(B, 8)
    base = make_frames("octave", W, H, uniq, first=rank * uniq)
    host = torch.empty((B, H, W), dtype=torch.uint8).pin_memory()
    for i in range(B):
        host[i] = torch.from_numpy(base[i % uniq])
    dev = host.cuda()

    ctx = clfd.Context(local_rank)
    cas = [clfd.Cascade(x) for x in XML]
    det = clfd.Detector(ctx, cas, W, H, max_batch=B, scale_factor=SCALE, min_size=MIN_SIZE,
                        scale_cascade=args.mode == "scale-cascade")
    wpf = sum(det.windows_per_frame(i) for i in range(len(cas)))
    stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        det.enqueue(dev, B, dev.stride(0), dev.stride(1), stream)
        return det.fetch(stream)

    def step_e2e():
        return det.detect(host)

    sampler = ClockSampler(local_rank)
    sampler.start()   # nvidia-smi needs ~0.5 s to start: launch it before the warm-up
    for _ in range(max(args.warmup, 3)):
        res = step_device()
    n_rects = len(res.rects)

    # ---- timed: device-resident input ------------------------------------------------------
    # Production order of a step: the batch is cut into chunks, the (HBM-bound) pyramid kernels of chunk k+1 run on a
    # second stream beside the (L1-bound) tile kernel of chunk k (clfd_api.cu, enqueue_overlapped).
    launches0 = ctx.launch_count
    barrier()
    sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        res = step_device()
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    launches = ctx.launch_count - launches0
    ms = e0.elapsed_time(e1)
    # ---- per-kernel CUDA-event times: the same steps with profiling on, i.e. in SERIAL order on one stream (overlapping
    #      kernels have no separate durations); the clock sampler keeps running, so `clocks` covers both loops
    det.set_profiling(True)
    kernel_ms = np.zeros(8)
    prof_steps = max(1, min(args.steps, 10))
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(prof_steps):
        step_device()
        kernel_ms += np.array(det.kernel_ms())
    e3.record()
    barrier()
    serial_ms = e2.elapsed_time(e3) / prof_steps
    clocks = sampler.stop()
    det.set_profiling(False)
    kernel_ms /= prof_steps

    # ---- timed: end to end through the host API ----------------------------------------------
    # Every step copies its batch from pinned host memory (H2D inside the timed region) and
    # reads its rect list back to the host.  clfd_detect_submit / _collect keep two batches in
    # flight, so the copy of step i+1 overlaps the kernels of step i (a frame stream).
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    det.submit(host)
    for _ in range(args.steps - 1):
        det.submit(host)
        r = det.collect()
    r = det.collect()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    d2h = int(len(r.rects) * 24 + 32)
    # the same stream with the host-side rectangle grouping (min_neighbors 3, tempcv.cpp:1462-1472)
    # of batch i running while the GPU evaluates batch i+1 (SURVEY 8-f row 1)
    barrier()
    t0 = time.perf_counter()
    det.submit(host)
    grouped = 0
    for _ in range(args.steps - 1):
        det.submit(host)
        grouped += len(clfd.group_batch(det.collect().rects, 3, 0.2)[0])
    grouped += len(clfd.group_batch(det.collect().rects, 3, 0.2)[0])
    torch.cuda.synchronize()
    e2e_grouped_s = time.perf_counter() - t0
    # the blocking single call (one batch at a time, copy overlapped only inside the batch)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = step_e2e()
    torch.cuda.synchronize()
    e2e_blocking_s = time.perf_counter() - t0

    # ---- the single gather of detection rects (no collective in the hot loop) ---------------
    from clfacedetection_b200 import sharding
    t_g0 = time.perf_counter()
    local = sharding.rects_to_array(res.rects, frame_offset=rank * B)   # rank r owns frames [r*B, (r+1)*B)
    gathered = sharding.gather_rects(local, device="cuda")
    gather_ms = 1e3 * (time.perf_counter() - t_g0)
    total_rects = len(gathered)
    if args.dump_outputs and rank == 0:
        dump_rects(args.dump_outputs, gathered)
    if world > 1:
        t = torch.tensor([ms, e2e_s, e2e_blocking_s, e2e_grouped_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)   # timing: max over ranks
        ms, e2e_s, e2e_blocking_s, e2e_grouped_s = (float(x) for x in t.tolist())

    if rank == 0:
        stats = det.stats()
        frames_total = B * world * args.steps
        fps = frames_total / (ms / 1e3)
        peak, peak_src = measured_peak_gbs()
        alg = {"resize_colsum": stats["bytes_resize"] * B, "integral_rows": stats["bytes_integral"] * B,
               "tilted": stats["bytes_tilted"] * B, "cascade_tiles": stats["bytes_cascade"] * B}
        kernels = {}
        ncu = ncu_traffic()
        for i, nm in enumerate(KERNEL_NAMES):
            if kernel_ms[i] > 0:
                k = {"ms": round(float(kernel_ms[i]), 4), "share": round(float(kernel_ms[i] / max(kernel_ms.sum(), 1e-9)), 4)}
                if nm in alg:
                    k["algorithmic_bytes"] = int(alg[nm])
                    k["achieved_gbs"] = round(alg[nm] / (kernel_ms[i] * 1e-3) / 1e9, 1)
                    k["frac_of_hbm_peak"] = round(k["achieved_gbs"] / peak, 4)
                if ncu and nm in ncu["kernels"]:
                    k["ncu_dram_bytes"] = int(ncu["kernels"][nm]["dram_bytes_per_frame"]) * B
                    k["ncu_l1_data_pipe_pct"] = ncu["kernels"][nm]["l1_data_pipe_pct"]
                    for lvl in ("l1", "l2"):   # bytes through L1 (global) / L2 per frame in the capture over this run's kernel time
                        if ncu["kernels"][nm].get(lvl + "_bytes_per_frame") and kernel_ms[i] > 0:
                            k["ncu_%s_gbs" % lvl] = round(ncu["kernels"][nm][lvl + "_bytes_per_frame"] * B / (kernel_ms[i] * 1e-3) / 1e9, 1)
                    if "warp_execution_efficiency" in ncu["kernels"][nm]:
                        k["ncu_warp_execution_efficiency"] = ncu["kernels"][nm]["warp_execution_efficiency"]
                kernels[nm] = k
        dom = "cascade_tiles"
        roof = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": peak,
                "peak_source": peak_src, "unit": "GB/s", "frac": kernels[dom]["frac_of_hbm_peak"],
                "traffic": kernels[dom].get("ncu_dram_bytes"),
                "launches_per_step": 2,
                "note": "achieved = compulsory bytes (integral tiles read once + packed cascade) of both tile launches of a "
                        "step / their CUDA-event time; traffic = ncu DRAM bytes of the same two launches scaled to this "
                        "batch.  The kernel is NOT HBM-bound: it saturates the SM's L1 data pipe (shared-memory corner "
                        "loads, one 128-B wavefront per clock per SM), see l1_data_pipe and DESIGN.md",
                "l1_data_pipe": {"ncu_pct_of_peak": kernels[dom].get("ncu_l1_data_pipe_pct"),
                                 "source": ncu["source"] if ncu else None}}
        wf = ncu["kernels"][dom].get("l1_wavefronts_per_frame") if ncu and dom in ncu["kernels"] else None
        if wf and clocks.get("sm_mhz"):
            # live: the capture's wavefront count per frame x this run's frames / this run's kernel time,
            # against one 128-byte wavefront per clock per SM at the SM clock sampled during the run
            n_sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
            peak_wf = n_sms * clocks["sm_mhz"] * 1e6
            ach_wf = wf * B / (kernel_ms[KERNEL_NAMES.index(dom)] * 1e-3)
            roof["l1_data_pipe"].update({"achieved": round(ach_wf / 1e9, 1), "peak": round(peak_wf / 1e9, 1),
                                         "unit": "G wavefronts/s", "frac": round(ach_wf / peak_wf, 4)})
        line = {
            "metric": "frames_per_sec_1080p" if (W, H) == (1920, 1080) else f"frames_per_sec_{W}x{H}", "value": round(fps, 2), "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"haarcascade_{CASCADE} {W}x{H} scale {SCALE}, batch {B} octave-noise frames per GPU per step"
                                   + (f", min window {MIN_SIZE[0]}x{MIN_SIZE[1]}" if MIN_SIZE != (0, 0) else "")
                                   + (" [scale-cascade mode]" if args.mode == "scale-cascade" else ""),
                       "frames_per_step_per_gpu": B, "windows_per_frame": wpf, "levels": len(det.levels()),
                       "l2": f"inputs and intermediates ({B * W * H / 1e6:.0f} MB frames, {stats['bytes_integral'] * B / 1e9:.1f} GB integrals "
                             "per batch) exceed the 126 MB L2; no flush needed"},
            "windows_per_sec": round(fps * wpf, 1),
            "wall_s": round(wall, 4),
            "rects_per_step": total_rects,
            "rect_gather_ms": round(gather_ms, 3),
            "deep_windows_per_step": stats["deep_windows"],
            "e2e": {"value": round(B * world * args.steps / e2e_s, 2), "unit": "frames/s",
                    "h2d_bytes_per_step": int(B * W * H), "d2h_bytes_per_step": d2h,
                    "api": "clfd_detect_submit/_collect, 2 batches in flight",
                    "blocking_call_value": round(B * world * args.steps / e2e_blocking_s, 2),
                    "with_host_grouping_value": round(B * world * args.steps / e2e_grouped_s, 2),
                    "grouped_rects_per_step": grouped // args.steps},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "kernels": kernels,
            "kernels_note": f"per-kernel CUDA-event times of {prof_steps} further steps in serial order (profiling on, one stream: "
                            f"{serial_ms:.3f} ms per step); in the timed region the pyramid kernels of chunk k+1 run beside the tile "
                            "kernel of chunk k and have no separate durations",
            "serial_ms_per_step": round(serial_ms, 4),
        }
        if not args.no_cpu_baseline and world == 1:
            cores = os.cpu_count() or 1
            n = args.cpu_baseline_frames if args.cpu_baseline_frames > 0 else max(4, min(cores, 64))
            cpu_frames = base[:n] if n <= uniq else make_frames("octave", W, H, n)
            t, w, _, kind = cpu_reference(cpu_frames, cores)
            line["cpu_baseline"] = {"value": round(n / t, 3), "unit": "frames/s", "cores": min(cores, n) if kind == "reference" else cores,
                                    "kind": kind,
                                    "sample": (f"{n} 1080p frames of the batch's generator, the reference's own cvHaarDetectObjects "
                                               "(oracle/_ref, CV_HAAR_SCALE_IMAGE), one frame per thread" if kind == "reference" else
                                               f"{n} of the batch's 1080p frames, REF-SI oracle, OpenMP over window rows"),
                                    "windows_per_sec": round(w / t, 1),
                                    "clod_cpu": clod_cpu_baseline(cpu_frames, cores)}
        default_run = (CASCADE == "frontalface_alt" and (W, H) == (1920, 1080) and SCALE == 1.2 and args.mode == "pyramid"
                       and world == 1 and not args.no_extra)
        if args.mode == "pyramid" and not args.no_extra:
            # survivor counts per stage (north star's evidence list): the exit codes of frame 0 of the batch,
            # from a second, one-frame detector with want_codes -- outside every timed region
            try:
                d2 = clfd.Detector(ctx, cas, W, H, max_batch=1, scale_factor=SCALE, min_size=MIN_SIZE, want_codes=True)
                r2 = d2.detect(base[:1])
                # counted and reported (north star): stage sums within 1e-5 relative of a threshold, FP64 fallbacks
                line["near_threshold"] = {"frame": 0, "windows": int(r2.stats["windows"]),
                                          "stage_sums_within_1e-5_of_threshold": int(r2.stats["near_threshold_events"]),
                                          "stage_evaluations_redone_in_fp64": int(r2.stats["exact_stage_evals"]),
                                          "note": "per (window, stage); results are identical to the reference's for these windows "
                                                  "too (exact FP64 path), the tolerance is not used"}
                surv = []
                for ci, cc in enumerate(cas):
                    codes = d2.codes(ci, 1)[0].astype(np.int64)
                    S = cc.info.n_stages
                    if cc.info.is_tree:   # code = 2 * last evaluated stage + accepted
                        hist = np.bincount(codes >> 1, minlength=S)
                        surv.append({"cascade": XML[ci].split("haarcascade_")[-1][:-4], "windows": int(codes.size),
                                     "stage_tree": True, "windows_whose_last_stage_is": hist.tolist(),
                                     "accepted": int((codes & 1).sum())})
                    else:                 # code = stages passed
                        hist = np.bincount(codes, minlength=S + 1)
                        reach = hist[::-1].cumsum()[::-1]   # windows that reach stage s = exit code >= s
                        surv.append({"cascade": XML[ci].split("haarcascade_")[-1][:-4], "windows": int(codes.size),
                                     "windows_reaching_stage": reach[:S].tolist(), "accepted": int(hist[S])})
                d2.close()
                line["survivors_per_stage"] = {"frame": 0, "cascades": surv}
                # EFFICIENCY of the tile kernel's L1 data pipe (not its utilisation): the corner values the algorithm
                # needs -- 4 per rectangle of every weak classifier a window evaluates, 4 bytes each (SURVEY 8-d) --
                # over the kernel's time, against one 128-byte wavefront per clock per SM.  Linear stump cascades only
                # (a tree's evaluated nodes depend on the data).
                if all("windows_reaching_stage" in x for x in surv) and clocks.get("sm_mhz"):
                    import oracle
                    corner_bytes = evals = 0
                    for ci, x in enumerate(surv):
                        f = oracle.load_cascade_xml(XML[ci])
                        if int(f.tr_nnodes.max()) != 1:
                            corner_bytes = 0
                            break
                        first = np.concatenate([[0], np.cumsum(f.st_ntrees)])
                        nrect = (f.nd_weight != 0).sum(axis=1)
                        for st, n_win in enumerate(x["windows_reaching_stage"]):
                            corner_bytes += int(n_win) * int(nrect[first[st]:first[st + 1]].sum()) * 16
                            evals += int(n_win) * int(f.st_ntrees[st])
                    if corner_bytes:
                        n_sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
                        t_frame = kernel_ms[KERNEL_NAMES.index("cascade_tiles")] * 1e-3 / B
                        peak_bs = n_sms * 128 * clocks["sm_mhz"] * 1e6
                        roof["l1_data_pipe"]["efficiency"] = {
                            "useful_corner_bytes_per_frame": corner_bytes, "weak_classifier_evals_per_frame": evals,
                            "achieved_tbs": round(corner_bytes / t_frame / 1e12, 2), "peak_tbs": round(peak_bs / 1e12, 2),
                            "frac": round(corner_bytes / t_frame / peak_bs, 4),
                            "note": "frame 0's survivor counts x 16 bytes per rectangle of every weak classifier evaluated, over the "
                                    "tile kernel's time per frame, against SMs x 128 B x SM clock; the rest of the pipe's "
                                    "wavefronts are dead lanes of the fixed-geometry stages, bank conflicts of the compacted "
                                    "stages, stump records and staging"}
            except Exception as e:   # evidence only: never fail the headline line
                line["survivors_per_stage"] = {"error": str(e)[:200]}
        det.close()
        ctx.close()
        if default_run:
            # BASELINE.json configs[1] (frontalface_default, batch 64, 1080p) next to the metric's own
            # configuration (frontalface_alt): a separate short run of this script, reported as-is
            try:
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--cascade", "frontalface_default", "--steps", "10",
                                      "--warmup", "3", "--batch", str(B), "--no-cpu-baseline", "--no-extra"],
                                     capture_output=True, text=True, timeout=300)
                x = json.loads(out.stdout.strip().splitlines()[-1])
                line["configs_1"] = {"workload": x["config"]["workload"], "value": x["value"], "unit": x["unit"],
                                     "e2e": x["e2e"]["value"], "ms_per_step": x["ms_per_step"],
                                     "windows_per_sec": x["windows_per_sec"]}
            except Exception as e:   # the headline line must not depend on the extra run
                line["configs_1"] = {"error": str(e)[:200]}
        print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return 0
    det.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
