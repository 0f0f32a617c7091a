"""The driver's bench contract: one JSON line with the agreed keys, from both arms."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_native_arm_line():
    d = _run("--steps", "3", "--warmup", "3", "--batch", "4", "--cpu-baseline-frames", "1", "--no-extra")
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["metric"] == "frames_per_sec_1080p" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert "workload" in d["config"] and "frontalface_alt" in d["config"]["workload"]
    assert d["value"] > 0 and d["gpu_launches"] > 0
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 4 * 1920 * 1080 and e["d2h_bytes_per_step"] > 0
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3
    assert set(("sm_mhz", "sm_max_mhz", "reasons")) <= set(d["clocks"])
    c = d["cpu_baseline"]
    assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    # the reference's own CPU detector (CLOD-CPU, clod.cpp:1339-1500) beside it
    assert c["clod_cpu"]["value"] > 0 and c["clod_cpu"]["cores"] >= 1 and c["clod_cpu"]["windows_per_frame"] > 0


def test_dump_outputs_holds_the_last_steps_rects(tmp_path):
    """--dump-outputs: the rects of the last timed step, sorted, as float64; frame 0's are the oracle's"""
    import numpy as np
    from clfacedetection_b200.frames import octave_frame
    from conftest import oracle_cascade
    d = _run("--steps", "2", "--warmup", "3", "--batch", "4", "--no-cpu-baseline", "--no-extra", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 2
    r = np.load(tmp_path / "rects.npy")
    assert r.dtype == np.float64 and r.shape == (d["rects_per_step"], 6) and len(r) > 0
    assert np.array_equal(r, r[np.lexsort(r.T[[3, 2, 0, 1, 5, 4]])])
    assert set(r[:, 4].tolist()) <= {0, 1, 2, 3} and not r[:, 5].any()
    key = lambda a: a[np.lexsort(a.T[[3, 2, 0, 1]])]
    want = oracle_cascade("frontalface_alt").detect(octave_frame(1920, 1080, 0), 1.2, want_codes=False)[0]
    assert np.array_equal(key(r[r[:, 4] == 0][:, :4].astype(np.int32)), key(want))


def test_dump_outputs_of_the_stream_arm(tmp_path):
    """--stream --dump-outputs: the gathered rects of the timed pass over the whole stream; frame 70's are the oracle's"""
    import numpy as np
    from clfacedetection_b200 import stream
    from conftest import oracle_cascade
    d = _run("--stream", "96", "--batch", "32", "--size", "480x360", "--cascade", "eye", "--dump-outputs", str(tmp_path))
    r = np.load(tmp_path / "rects.npy")
    assert r.dtype == np.float64 and r.shape == (d["rects_total"], 6) and len(r) > 0
    assert np.array_equal(r, r[np.lexsort(r.T[[3, 2, 0, 1, 5, 4]])]) and r[:, 4].max() < 96
    key = lambda a: a[np.lexsort(a.T[[3, 2, 0, 1]])]
    frame = np.ascontiguousarray(stream.StreamSource(480, 360, pinned=False).frame(70))
    want = oracle_cascade("eye").detect(frame, 1.2, want_codes=False)[0]
    assert np.array_equal(key(r[r[:, 4] == 70][:, :4].astype(np.int32)), key(want))


def test_reference_arm_line():
    d = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-frames", "1")
    assert d["impl"] == "reference" and d["metric"] == "frames_per_sec_1080p" and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["gpu_launches"] == 0 and d["cpu_baseline"]["clod_cpu"]["value"] > 0
