"""The CPU oracle and the product's host code against tests/golden/reference_tempcv.npz -- vectors
recorded from the REFERENCE'S OWN compiled functions (tempcv.cpp:40-1516, 1702-2089) by
tests/golden/make_ref_golden.py.  Needs neither the original sources nor oracle/_ref, so it runs on every
machine; the CUDA path is compared with the same file in tests/test_gpu_reference_golden.py."""
import os

import numpy as np
import pytest

import clfacedetection_b200 as clfd
import oracle
from clfacedetection_b200.frames import octave_frame, uniform_frame
from conftest import ALL_CASCADES, cascade_path, oracle_cascade

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_tempcv.npz")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def golden_frames():
    return [octave_frame(320, 240, 21), uniform_frame(320, 240, 22)]


def expected_results(cas, codes):
    if cas.is_tree:
        return (codes & 1).astype(np.int32)
    return np.where(codes == cas.flat.n_stages, 1, -codes.astype(np.int32))


def test_golden_file_covers_every_cascade(gold):
    names = {k.split("/")[0] for k in gold.files} - {"group"}
    assert names == set(ALL_CASCADES)


@pytest.mark.parametrize("name", ALL_CASCADES)
def test_census_and_hidden_weights_equal_reference(gold, name):
    c = clfd.Cascade(cascade_path(name))
    i = c.info
    assert [i.win_w, i.win_h, i.n_stages, i.n_trees, i.n_nodes] == gold[f"{name}/census"].tolist()
    w, _, thr, _ = c.hidden()
    assert w.tobytes() == gold[f"{name}/hid_w"].tobytes() and thr.tobytes() == gold[f"{name}/hid_thr"].tobytes()
    ow, _, othr, _, _ = oracle_cascade(name).hidden()
    assert ow.tobytes() == gold[f"{name}/hid_w"].tobytes() and othr.tobytes() == gold[f"{name}/hid_thr"].tobytes()


@pytest.mark.parametrize("name", ALL_CASCADES)
def test_oracle_equals_reference_vectors(gold, name):
    oc = oracle_cascade(name)
    for fi, frame in enumerate(golden_frames()):
        codes, _, _ = oc.eval_level(frame, 1)
        assert np.array_equal(expected_results(oc, codes), gold[f"{name}/lvl_{fi}"].astype(np.int32))
        raw, _, _, _, _ = oc.detect(frame, 1.2)
        assert np.array_equal(raw, gold[f"{name}/si_{fi}"])
        g, w = oracle.group_rectangles(raw, 2)
        assert np.array_equal(np.concatenate([g, w[:, None]], 1), gold[f"{name}/sig_{fi}"].reshape(-1, 5))
        r, lv, wt = oc.detect_roc(frame, 1.2)
        roc = gold[f"{name}/roc_{fi}"].reshape(-1, 6)
        assert np.array_equal(r, roc[:, :4].astype(np.int32)) and np.array_equal(lv, roc[:, 4].astype(np.int32))
        assert wt.tobytes() == np.ascontiguousarray(roc[:, 5]).tobytes()
        sc, _, _, _ = oc.detect_sc(frame, 1.2)
        a, b = sc, gold[f"{name}/sc_{fi}"].reshape(-1, 4)
        assert np.array_equal(a[np.lexsort(a.T[::-1])] if len(a) else a, b[np.lexsort(b.T[::-1])] if len(b) else b)


def test_host_grouping_equals_reference_vectors(gold):
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(GOLD)))
    from make_ref_golden import group_inputs
    for i, r in enumerate(group_inputs()):
        for eps in (0.2, 0.35):
            exp = gold[f"group/{i}_{eps}"].reshape(-1, 5)
            for fn in (oracle.group_rectangles, clfd.group_rectangles):
                g, w = fn(r, 2, eps)
                assert np.array_equal(np.concatenate([g, w[:, None]], 1), exp), (i, eps, fn.__module__)
