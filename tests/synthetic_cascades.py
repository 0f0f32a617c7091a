"""Synthetic Haar cascades of any window geometry, for the parity tests of the kernels against the oracle.

The stock cascade files all have windows of 45 pixels or less.  The host code picks a cascade's kernels from its
window size (the tile kernel only while a tile of windows fits in shared memory; byte-sized corner offsets in the
generic kernels), so the tests need cascades of every size, built from a seed.  Every cascade covers the places
where feature evaluation goes wrong:

- rectangles flush with each border of the window, and 1-pixel rectangles;
- tilted rectangles (a rectangle rotated by 45 degrees, stored as Haar cascades store it: the top corner at (x, y),
  w pixels down-right and h pixels down-left) at their limits x - h == 0 and y + w + h == win_h;
- features of 2 and of 3 rectangles;
- trees of 1, 2, 3 and 4 nodes; a stage tree (``st_parent`` / ``st_next``) in one variant;
- a leaf value far above 64 in one variant, which puts the cascade on the kernels' ``track_abs`` instantiation.

Stage thresholds follow the leaf values: the sum of every tree's mean leaf, lowered by ``offset`` times the spread
of the stage sum, so that a fair share of the windows passes every stage.
"""
from __future__ import annotations

import numpy as np

from oracle.cascade_xml import FlatCascade

# (left, right) of each node: > 0 a node index, <= 0 the leaf -index.  The 4-node shape has a leaf, a chain and a fork.
TREE_SHAPES = {1: [(0, -1)], 2: [(1, 0), (-1, -2)], 3: [(1, 2), (0, -1), (-2, -3)],
               4: [(0, 1), (2, 3), (-1, -2), (-3, -4)]}

# forced placements, cycled through so that every cascade of a few dozen nodes has each of them
_UPRIGHT_EDGES = ("left", "right", "top", "bottom", "pixel", "whole", "free")
_TILTED_EDGES = ("x_minus_h", "bottom", "right", "top", "pixel", "free")

SENTINEL = 1000.0


def _upright_rect(rng, W, H, edge):
    if edge == "pixel":
        return int(rng.integers(0, W)), int(rng.integers(0, H)), 1, 1
    if edge == "whole":
        return 0, 0, W, H
    w, h = int(rng.integers(1, W + 1)), int(rng.integers(1, H + 1))
    x, y = int(rng.integers(0, W - w + 1)), int(rng.integers(0, H - h + 1))
    if edge == "left":
        x = 0
    elif edge == "right":
        x = W - w
    elif edge == "top":
        y = 0
    elif edge == "bottom":
        y = H - h
    return x, y, w, h


def _tilted_rect(rng, W, H, edge):
    """x - h >= 0, x + w <= W, y >= 0, y + w + h <= H (the bounds check of build_hidden / tempcv.cpp:365-387)"""
    m = min(W, H)
    if edge == "pixel":
        w = h = 1
    else:
        w = int(rng.integers(1, m))
        h = int(rng.integers(1, m - w + 1))
    x, y = int(rng.integers(h, W - w + 1)), int(rng.integers(0, H - w - h + 1))
    if edge == "x_minus_h":
        x = h
    elif edge == "right":
        x = W - w
    elif edge == "top":
        y = 0
    elif edge == "bottom":
        y = H - w - h
    return x, y, w, h


def make_cascade(seed: int, win: tuple[int, int], stage_trees=(3, 5, 8, 12), node_counts=(1,), tilted: bool = False,
                 stage_tree: bool = False, sentinel: bool = False, three_rects: float = 0.3,
                 offset: float = 0.5, name: str | None = None) -> FlatCascade:
    """A cascade of len(stage_trees) stages for a win = (w, h) window, stage i holding stage_trees[i] trees.

    node_counts: the tree sizes, cycled through tree by tree (1 = stumps).  tilted: every other node is a tilted
    feature.  stage_tree: stage 1 gets a `next` alternative (stage 2), so a window failing stage 1 or one of its
    descendants continues at stage 2; the other stages stay a chain.  sentinel: the first tree of stage 1 has a right
    leaf of SENTINEL.  three_rects: share of the nodes with a third rectangle.  offset: how far below the mean leaf sum
    the stage thresholds sit, in units of the stage sum's spread."""
    W, H = win
    assert W > 2 and H > 2
    rng = np.random.default_rng(seed)
    S = len(stage_trees)
    tr_nnodes, nd_tilted, nd_rect, nd_weight, nd_thr, nd_left, nd_right, alpha, st_thr = ([] for _ in range(9))
    n_nodes = 0
    t_all = 0
    for s, nt in enumerate(stage_trees):
        mean_sum, var_sum = 0.0, 0.0
        for t in range(nt):
            k = int(node_counts[t_all % len(node_counts)])
            t_all += 1
            tr_nnodes.append(k)
            for (l, r) in TREE_SHAPES[k]:
                nd_left.append(l)
                nd_right.append(r)
                tl = bool(tilted and n_nodes % 2 == 1)
                edges = _TILTED_EDGES if tl else _UPRIGHT_EDGES
                make = _tilted_rect if tl else _upright_rect
                rects = np.zeros((3, 4), np.int32)
                weights = np.zeros(3, np.float32)
                nr = 3 if rng.random() < three_rects else 2
                for q in range(nr):
                    rects[q] = make(rng, W, H, edges[(3 * n_nodes + q) % len(edges)])
                weights[:nr] = [-1.0, 2.0, -2.0 if rng.random() < 0.5 else 3.0][:nr]
                nd_tilted.append(int(tl))
                nd_rect.append(rects)
                nd_weight.append(weights)
                # the feature is a difference of means normalised by the window's sigma, scaled by the rectangles'
                # share of the window: thresholds around zero at that scale split the windows
                share = float(rects[1, 2] * rects[1, 3]) / (W * H)
                nd_thr.append(np.float32(rng.normal(0.0, 0.3) * share))
                n_nodes += 1
            leaves = rng.uniform(-1.0, 1.0, k + 1).astype(np.float32)
            if sentinel and s == 1 and t == 0:
                leaves[-1] = np.float32(SENTINEL)
            alpha += leaves.tolist()
            mean_sum += float(np.mean(leaves))
            var_sum += float(np.var(leaves))
        st_thr.append(np.float32(mean_sum - offset * np.sqrt(var_sum)))
    st_parent = np.arange(-1, S - 1, dtype=np.int32)
    st_next = np.full(S, -1, np.int32)
    if stage_tree:
        assert S >= 4
        # 0 -> 1 -> 3 -> 4 ...; stage 2 is the `next` of stage 1 (same parent, 0) and a leaf of the tree
        st_parent[2] = 0
        st_next[1] = 2
        st_parent[3] = 1
    return FlatCascade(name=name or f"synthetic-{W}x{H}-{seed}", win_w=W, win_h=H,
                       st_ntrees=np.array(stage_trees, np.int32), st_thr=np.array(st_thr, np.float32),
                       st_parent=st_parent, st_next=st_next, tr_nnodes=np.array(tr_nnodes, np.int32),
                       nd_tilted=np.array(nd_tilted, np.int32), nd_rect=np.ascontiguousarray(np.stack(nd_rect), np.int32),
                       nd_weight=np.ascontiguousarray(np.stack(nd_weight), np.float32),
                       nd_thr=np.array(nd_thr, np.float32), nd_left=np.array(nd_left, np.int32),
                       nd_right=np.array(nd_right, np.int32), alpha=np.array(alpha, np.float32))


STAGES = (3, 5, 8, 12, 16, 20)
MIXED = (1, 2, 3, 4)

# The window geometries the tests run, with the cascade variant each one gets.  Where the kernels change:
#   3x3          the smallest window a cascade may have
#   5x40, 40x5   tall and flat windows
#   20x20, 24x24 the two window heights with their own templated row step in the tile kernel
#   44x44        the largest square window whose tile fits shared memory at both row steps (stumps: 24-row ystep-2
#                tiles); with trees of several nodes (32-row tiles) the ystep-2 tile no longer fits
#   45x45, 48x48, 64x64, tilted 64x64, 120x20, 200x12
#                the ystep-1 tile fits, the ystep-2 tile does not: the generic kernels take these cascades whole
#   12x200       no tile fits
#   255x255      the largest window of the image-pyramid mode (byte-sized corner offsets, squared integral mod 2^32)
#   256x20       beyond it: the scale-cascade mode only
#   300x300
GEOMETRY_CASES = {
    "3x3": dict(win=(3, 3), seed=11, node_counts=MIXED),
    "5x40": dict(win=(5, 40), seed=12, node_counts=MIXED, tilted=True),
    "40x5": dict(win=(40, 5), seed=13, node_counts=(1, 2)),
    "20x20": dict(win=(20, 20), seed=14, stage_tree=True),
    "24x24": dict(win=(24, 24), seed=15, node_counts=(1, 2), sentinel=True),
    "44x44": dict(win=(44, 44), seed=16),
    "44x44-trees": dict(win=(44, 44), seed=27, node_counts=MIXED),
    "45x45": dict(win=(45, 45), seed=17),
    "48x48": dict(win=(48, 48), seed=18),
    "64x64": dict(win=(64, 64), seed=19, stage_tree=True),
    "64x64-tilted": dict(win=(64, 64), seed=20, tilted=True),
    "120x20": dict(win=(120, 20), seed=21, node_counts=MIXED),
    "200x12": dict(win=(200, 12), seed=22, sentinel=True),
    "12x200": dict(win=(12, 200), seed=23, tilted=True),
    "255x255": dict(win=(255, 255), seed=24, node_counts=(1, 3)),
    "256x20": dict(win=(256, 20), seed=25),
    "300x300": dict(win=(300, 300), seed=26, tilted=True),
}
# the ystep-1 tile fits shared memory, the ystep-2 tile does not
SPLIT_CASES = ("44x44-trees", "45x45", "48x48", "64x64", "64x64-tilted", "120x20", "200x12")
# windows wider or taller than 255 pixels: scale-cascade mode only
BEYOND_CASES = ("256x20", "300x300")


def geometry_cascade(case: str) -> FlatCascade:
    kw = dict(GEOMETRY_CASES[case])
    return make_cascade(kw.pop("seed"), kw.pop("win"), stage_trees=STAGES, name=f"synthetic-{case}", **kw)
