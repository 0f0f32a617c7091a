"""Which kernels take a cascade, by window geometry (no GPU needed): the tile kernel takes a cascade only when the tiles
of BOTH row steps fit shared memory, and the stock cascades' packing stays as it is."""
import pytest

import clfacedetection_b200 as clfd
from conftest import ALL_CASCADES, cascade_path
from synthetic_cascades import GEOMETRY_CASES, SPLIT_CASES, geometry_cascade, make_cascade

# info.dense_stages: the stages the tile kernel evaluates (every stage of these cascades is one it can take), or 0
# where a tile does not fit: then the generic kernels evaluate the whole cascade on every level
DENSE_STAGES = {
    "3x3": 6, "5x40": 6, "40x5": 6, "20x20": 6, "24x24": 6, "44x44": 6,
    "44x44-trees": 0, "45x45": 0, "48x48": 0, "64x64": 0, "64x64-tilted": 0, "120x20": 0, "200x12": 0,
    "12x200": 0, "255x255": 0, "256x20": 0, "300x300": 0,
}

# (dense_stages, dense_stumps) of the 19 stock cascades
STOCK_DENSE = {
    "frontalface_alt": (22, 2135),
    "frontalface_default": (25, 2913),
    "frontalface_alt_tree": (47, 8468),
    "eye": (24, 1066),
    "profileface": (26, 2609),
    "fullbody": (30, 1464),
    "frontalface_alt2": (20, 2094),
    "eye_tree_eyeglasses": (30, 2553),
    "mcs_nose": (20, 3365),
    "lefteye_2splits": (20, 732),
    "righteye_2splits": (20, 736),
    "lowerbody": (27, 1221),
    "upperbody": (30, 2423),
    "mcs_eyepair_big": (19, 748),
    "mcs_eyepair_small": (17, 860),
    "mcs_lefteye": (14, 1648),
    "mcs_mouth": (17, 1515),
    "mcs_righteye": (18, 2942),
    "mcs_upperbody": (19, 3224),
}


def test_every_case_has_an_expectation():
    assert set(DENSE_STAGES) == set(GEOMETRY_CASES)
    assert set(STOCK_DENSE) == set(ALL_CASCADES)


@pytest.mark.parametrize("case", list(GEOMETRY_CASES))
def test_dense_stages_by_window_geometry(case):
    flat = geometry_cascade(case)
    info = clfd.Cascade(flat=flat).info
    assert (info.win_w, info.win_h) == (flat.win_w, flat.win_h)
    assert info.dense_stages == DENSE_STAGES[case]
    if info.dense_stages == 0:
        assert info.dense_stumps == 0


@pytest.mark.parametrize("case", SPLIT_CASES)
def test_split_geometries_leave_no_tile_blob_behind(case, monkeypatch):
    """32-row ystep-2 tiles (CLFD_TILE_H2=32) do not fit either: still no tile kernel"""
    monkeypatch.setenv("CLFD_TILE_H2", "32")
    assert clfd.Cascade(flat=geometry_cascade(case)).info.dense_stages == 0


@pytest.mark.parametrize("win,dense", [((44, 44), 4), ((45, 45), 0), ((100, 20), 4), ((120, 20), 0), ((12, 12), 4),
                                       ((254, 3), 0)])
def test_tile_limit_of_a_plain_stump_cascade(win, dense):
    """the last window sizes that keep the tile kernel and the first ones that lose it, 4-stage stump cascade"""
    info = clfd.Cascade(flat=make_cascade(5, win)).info
    assert info.dense_stages == dense


@pytest.mark.parametrize("name", ALL_CASCADES)
def test_stock_cascades_keep_their_tile_prefix(name):
    info = clfd.Cascade(cascade_path(name)).info
    assert (info.dense_stages, info.dense_stumps) == STOCK_DENSE[name]


def test_generator_covers_the_edges():
    """every feature edge the generator promises is present in the cases the GPU tests run"""
    import numpy as np
    seen = set()
    for case in GEOMETRY_CASES:
        f = geometry_cascade(case)
        W, H = f.win_w, f.win_h
        for n in range(f.n_nodes):
            nr = 3 if f.nd_weight[n, 2] != 0 else 2
            seen.add(f"rects{nr}")
            for x, y, w, h in f.nd_rect[n, :nr]:
                if f.nd_tilted[n]:
                    assert x - h >= 0 and x + w <= W and y >= 0 and y + w + h <= H
                    seen |= {k for k, c in (("t_x_minus_h", x - h == 0), ("t_bottom", y + w + h == H),
                                            ("t_right", x + w == W), ("t_top", y == 0)) if c}
                else:
                    assert x >= 0 and y >= 0 and x + w <= W and y + h <= H
                    seen |= {k for k, c in (("left", x == 0), ("right", x + w == W), ("top", y == 0),
                                            ("bottom", y + h == H), ("pixel", w == 1 and h == 1)) if c}
        seen |= {f"nodes{k}" for k in np.unique(f.tr_nnodes)}
        if np.any(f.st_next >= 0):
            seen.add("stage_tree")
        if np.abs(f.alpha).max() > 64:
            seen.add("sentinel")
    assert seen >= {"rects2", "rects3", "t_x_minus_h", "t_bottom", "t_right", "t_top", "left", "right", "top", "bottom",
                    "pixel", "nodes1", "nodes2", "nodes3", "nodes4", "stage_tree", "sentinel"}, seen
