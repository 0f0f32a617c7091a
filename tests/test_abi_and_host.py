"""The C ABI library loads without a GPU and exports every symbol the header declares; the
host-side pieces (grouping, frame sharding) behave like the reference / the oracle; compute
entry points fail loudly (no CPU fallback) when there is no CUDA device."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import clfacedetection_b200 as clfd
import oracle
from clfacedetection_b200 import abi, sharding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    names = abi.exported_symbols_in_header()
    assert len(names) >= 30
    L = C.CDLL(abi.LIB_PATH)
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing
    assert b"sm_100a" in abi.lib().clfd_version()


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible")
    with pytest.raises(clfd.ClfdError) as e:
        clfd.Context(0)
    assert e.value.status == -2 and "CUDA" in str(e.value)


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "clfacedetection_b200")):
        for fn in files:
            if fn.endswith((".py", ".cpp", ".cu", ".h")):
                text = open(os.path.join(dirpath, fn), encoding="utf-8", errors="replace").read()
                assert "import oracle" not in text and "vj_oracle" not in text and "from oracle" not in text, fn


def test_group_rectangles_equals_oracle():
    rng = np.random.default_rng(3)
    for _ in range(200):
        base = rng.integers(0, 300, size=(int(rng.integers(1, 7)), 2))
        r = np.array([[b[0] + rng.integers(-7, 8), b[1] + rng.integers(-7, 8), 30 + rng.integers(-4, 30), 30 + rng.integers(-4, 30)]
                      for b in base[rng.integers(0, len(base), size=int(rng.integers(0, 80)))]], np.int32).reshape(-1, 4)
        thr = int(rng.integers(0, 4))
        a, wa = clfd.group_rectangles(r, thr, 0.2)
        b, wb = oracle.group_rectangles(r, thr, 0.2)
        assert np.array_equal(a, b) and np.array_equal(wa, wb)


def test_shard_range_partitions_frames():
    for n in (0, 1, 7, 64, 8192):
        for world in (1, 2, 3, 8):
            spans = [sharding.shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


_WORKER = r'''
import os, sys
import numpy as np
import torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from clfacedetection_b200 import sharding
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{sys.argv[2]}", rank=int(sys.argv[3]), world_size=2)
rank = dist.get_rank()
first, last = sharding.shard_range(13, rank, 2)
rng = np.random.default_rng(100 + rank)
n = 5 if rank == 0 else 0          # ragged: one rank has nothing to report
local = np.zeros(n, dtype=[("x","<i4"),("y","<i4"),("w","<i4"),("h","<i4"),("frame","<i4"),("cascade","<i4")])
local["x"] = rng.integers(0, 100, n); local["frame"] = rng.integers(0, last - first, n) if n else 0
arr = sharding.rects_to_array(local, frame_offset=first)
allr = sharding.gather_rects(arr)
assert allr.shape == (5, 6), allr.shape
assert (allr[:, 4] < 13).all()
if rank == 1:
    assert first == 7 and last == 13
dist.barrier(); dist.destroy_process_group()
print("ok", rank)
'''


def test_gather_rects_world_size_2_gloo(tmp_path):
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(port), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all("ok" in o for o in outs)


def test_reference_main_cpp_compiles_unchanged(tmp_path):
    """SURVEY.md 8-b: the reference's own main.cpp must build against include/ + include/shim
    byte for byte.  Only possible where CLFD_REFERENCE_DIR names the original sources."""
    from oracle import build_ref
    ref = os.path.join(build_ref.REF, "main.cpp")
    if not build_ref.REF or not os.path.exists(ref):
        pytest.skip("no original main.cpp (CLFD_REFERENCE_DIR)")
    obj = tmp_path / "main.o"
    exe = os.path.join(ROOT, "tests", "_build", "ref_main")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", f"-I{ROOT}/include", f"-I{ROOT}/include/shim", "-c", ref, "-o", str(obj)])
    subprocess.check_call(["/usr/bin/g++", "-o", exe, str(obj), f"-L{ROOT}/clfacedetection_b200", "-lclfd_clod", "-lclfd_b200",
                           "-Wl,-rpath,$ORIGIN/../../clfacedetection_b200"])
    assert os.path.exists(exe)


def test_clod_demo_is_built():
    assert os.path.exists(os.path.join(ROOT, "examples", "clod_demo"))
    assert os.path.exists(os.path.join(ROOT, "clfacedetection_b200", "libclfd_clod.so"))


def test_group_batch_equals_per_frame_grouping():
    """clfd_group_batch (host threads, per (frame, cascade)) == the oracle's AgroupRectangles run
    frame by frame on the same rects, whatever order the device appended them in."""
    import clfacedetection_b200 as clfd
    import oracle
    rng = np.random.default_rng(5)
    recs = []
    for frame in range(7):
        for cascade in range(2):
            k = int(rng.integers(0, 5))
            for _ in range(k):   # k clusters of jittered rects
                cx, cy, s = rng.integers(0, 500, 2).tolist() + [int(rng.integers(20, 120))]
                for _ in range(int(rng.integers(1, 9))):
                    j = rng.integers(-2, 3, 3)
                    recs.append((cx + j[0], cy + j[1], s + j[2], s + j[2], frame, cascade))
    rects = np.array(recs, dtype=clfd.RECT_DTYPE)
    shuffled = rects[rng.permutation(len(rects))]
    for thr in (1, 3):
        got, w = clfd.group_batch(shuffled, thr, 0.2, n_threads=4)
        again, w2 = clfd.group_batch(rects, thr, 0.2, n_threads=1)
        assert np.array_equal(got, again) and np.array_equal(w, w2)   # order / thread independent
        o = 0
        for frame in range(7):
            for cascade in range(2):
                m = (rects["frame"] == frame) & (rects["cascade"] == cascade)
                r = rects[m]
                r = r[np.lexsort((r["x"], r["y"], r["w"]))]
                xywh = np.stack([r["x"], r["y"], r["w"], r["h"]], axis=1).astype(np.int32) if len(r) else np.zeros((0, 4), np.int32)
                want, ww = oracle.group_rectangles(xywh, thr, 0.2)
                n = len(want)
                g = got[o:o + n]
                assert np.array_equal(np.stack([g["x"], g["y"], g["w"], g["h"]], axis=1), want.reshape(-1, 4))
                assert np.all(g["frame"] == frame) and np.all(g["cascade"] == cascade)
                assert np.array_equal(w[o:o + n], ww)
                o += n
        assert o == len(got)
    empty, _ = clfd.group_batch(rects[:0], 3)
    assert len(empty) == 0


def test_tile_kernel_register_budget():
    """The headline instantiations of k_cascade_tiles (plain stump cascades) must stay at 64 registers:
    at 256 threads that is 4 CTAs per SM; a stray launch-bounds argument once let ptxas take 88
    (2 CTAs per SM, -20 % frames/s).  cuobjdump -res-usage is the authority (tools/regs.sh)."""
    import re
    import shutil
    import subprocess
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("no cuobjdump")
    from clfacedetection_b200 import abi
    out = subprocess.run([exe, "-res-usage", abi.LIB_PATH], capture_output=True, text=True).stdout
    regs = {}
    name = None
    for line in out.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            name = m.group(1)
        m = re.search(r"REG:(\d+)", line)
        if m and name:
            regs[name] = int(m.group(1))
    tiles = {k: v for k, v in regs.items() if "k_cascade_tilesILi" in k}
    assert len(tiles) >= 12, sorted(regs)
    # plain stump cascades, 24- and 32-row tiles (the 16-row tiles of tilted cascades are bound to 2-3 CTAs per SM by
    # their two shared-memory tiles anyway); both the production and the counting instantiation
    # (the TRACK instantiations -- last template flag set, sentinel-leaf cascades such as haarcascade_mcs_* only --
    # carry one more accumulator per window and may take more)
    track = {k for k in tiles if re.search(r"Lb1EEEvNS", k)}
    plain = {k: v for k, v in tiles.items() if ("ELb0ELb0ELi24E" in k or "ELb0ELb0ELi32E" in k) and k not in track}
    assert len(plain) >= 8 and all(v <= 64 for v in plain.values()), plain
    assert track, "no TRACK instantiation found"
    assert all(v <= 80 for v in tiles.values()), tiles


def test_grouping_an_empty_list_is_not_an_error():
    """ADVICE r1 (high): a frame without detections hands clfd_group_rectangles n = 0 and the NULL
    data() of an empty std::vector; the reference returns match_count = 0 there (tempcv.cpp:147)."""
    import ctypes as C
    from clfacedetection_b200 import abi
    L = abi.lib()
    n = C.c_int(0)
    assert L.clfd_group_rectangles(None, C.byref(n), 2, 0.2, None) == 0 and n.value == 0
    n = C.c_int(3)
    assert L.clfd_group_rectangles(None, C.byref(n), 2, 0.2, None) < 0      # rects missing for n > 0
    n = C.c_int(-1)
    assert L.clfd_group_rectangles(None, C.byref(n), 2, 0.2, None) < 0


def test_cascade_ids_are_never_reused():
    """ADVICE r1 (medium): plan caches are keyed by clfd_cascade_id, which -- unlike the address of a
    released cascade -- is never handed out twice."""
    import clfacedetection_b200 as clfd
    from clfacedetection_b200 import abi
    from conftest import cascade_path
    seen = set()
    for _ in range(6):
        c = clfd.Cascade(cascade_path("lefteye_2splits"))
        cid = int(abi.lib().clfd_cascade_id(c._h))
        assert cid > 0 and cid not in seen
        seen.add(cid)
        del c


def test_broken_tree_links_are_rejected():
    """ADVICE r1 (low): through clfd_cascade_from_arrays an out-of-range parent, a backward node link or
    a stage-tree cycle must fail cleanly (the XML reader rejects the first two itself)."""
    import copy
    import clfacedetection_b200 as clfd
    import oracle
    from conftest import cascade_path
    flat = oracle.load_cascade_xml(cascade_path("frontalface_alt2"))   # 2-node trees
    bad = copy.deepcopy(flat)
    bad.st_parent = bad.st_parent.copy(); bad.st_parent[3] = 999
    with pytest.raises(clfd.ClfdError, match="parent must be integer number"):
        clfd.Cascade(flat=bad)
    bad = copy.deepcopy(flat)
    n = int(np.flatnonzero(flat.nd_left > 0)[0]) if (flat.nd_left > 0).any() else int(np.flatnonzero(flat.nd_right > 0)[0])
    bad.nd_left = bad.nd_left.copy(); bad.nd_left[n + 1] = 1   # node 1 of the tree links back to itself
    with pytest.raises(clfd.ClfdError, match="Tree structure is broken"):
        clfd.Cascade(flat=bad)
    tree = oracle.load_cascade_xml(cascade_path("frontalface_alt_tree"))
    bad = copy.deepcopy(tree)
    bad.st_next = bad.st_next.copy(); bad.st_next[6] = 5       # 5 -> 6 -> 5
    with pytest.raises(clfd.ClfdError, match="not a forest"):
        clfd.Cascade(flat=bad)
    clfd.Cascade(flat=tree)   # the stock stage tree passes


def test_stream_source_is_a_function_of_the_global_frame_index():
    """bench.py --stream / tests/test_gpu_multi.py: any sharding of the stream tiles it exactly, a batch's
    overlapping canvas views are the frames, and the frames are distinct"""
    from clfacedetection_b200 import sharding, stream
    src = stream.StreamSource(160, 120, n_canvases=2, pinned=False)
    N = 300
    for world in (1, 3, 8):
        seen = []
        for r in range(world):
            f, l = sharding.shard_range(N, r, world)
            for g0, n, view in src.runs(f, l, 16):
                assert 1 <= n <= 16
                for j in (0, n - 1):
                    assert np.array_equal(view[j:j + 120, :160].numpy(), src.frame(g0 + j))
                seen += list(range(g0, g0 + n))
        assert seen == list(range(N))
    assert len({src.frame(g).tobytes() for g in range(N)}) == N
