// haar_pack.cpp -- hidden-cascade construction and device packing.
//
// build_hidden restates, for scale = 1 (the only scale REF-SI uses, tempcv.cpp:1321):
//   * icvCreateHidHaarClassifierCascade (tempcv.cpp:308-467): rectangle bounds checks,
//     stage threshold bias (-0.0001f, :419), two_rects (:421,453-458), isStumpBased (:465),
//     is_tree (:431), has_tilted_features (:371);
//   * cvSetImagesForHaarClassifierCascade (tempcv.cpp:549-768): weight_k =
//     (float)(xml_weight_k * inv_area * (tilted ? 0.5 : 1)) (:733,752) and weight_0 =
//     (float)(-sum_{k>=1} weight_k*w_k*h_k / (w_0*h_0)) (:754-760), C expression types kept.
// This replaces the per-scale precomputeKernelCascade of clod.cpp:529-578: in the pyramid
// formulation the packed cascade is scale independent and is built once per cascade.
//
// This translation unit must be compiled with -ffp-contract=off.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "clfd_pack.h"

namespace clfd {

static thread_local char g_error[1024] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof g_error, fmt, ap);
    va_end(ap);
}
const char *get_error() { return g_error; }

#define FMT_FAIL(...) do { set_error(__VA_ARGS__); return CLFD_ERR_FORMAT; } while (0)

int build_hidden(HostCascade &c) {
    const int S = c.n_stages();
    if (S <= 0) FMT_FAIL("Number of stages should be positive");
    if (c.win_w <= 2 || c.win_h <= 2) FMT_FAIL("cascade window %dx%d is too small", c.win_w, c.win_h);
    if ((int)c.st_thr.size() != S || (int)c.st_parent.size() != S || (int)c.st_next.size() != S)
        FMT_FAIL("stage arrays have inconsistent sizes");
    c.st_first_tree.assign(S + 1, 0);
    for (int i = 0; i < S; i++) {
        if (c.st_ntrees[i] <= 0)
            FMT_FAIL("header of the stage classifier #%d is invalid (has null pointers or non-positive classfier count)", i);
        c.st_first_tree[i + 1] = c.st_first_tree[i] + c.st_ntrees[i];
    }
    const int T = c.st_first_tree[S];
    if ((int)c.tr_nnodes.size() != T) FMT_FAIL("tree count does not match the stage headers");
    c.tr_first_node.assign(T + 1, 0);
    for (int t = 0; t < T; t++) {
        if (c.tr_nnodes[t] <= 0) FMT_FAIL("Tree node is not a valid sequence. (tree %d)", t);
        c.tr_first_node[t + 1] = c.tr_first_node[t] + c.tr_nnodes[t];
    }
    const int N = c.tr_first_node[T];
    if ((int)c.nodes.size() != N) FMT_FAIL("node count does not match the tree headers");
    if ((int)c.alpha.size() != N + T) FMT_FAIL("alpha count does not match the tree headers");

    for (int i = 0; i < S; i++) {   // the reader's range checks (tempcv.cpp:2054-2071), before any use as an index
        if (c.st_parent[i] < -1 || c.st_parent[i] >= S) FMT_FAIL("parent must be integer number. (stage %d)", i);
        if (c.st_next[i] < -1 || c.st_next[i] >= S) FMT_FAIL("next must be integer number. (stage %d)", i);
    }
    // A stage tree is walked pass -> child, fail -> `next` of the nearest ancestor-or-self that has one
    // (tempcv.cpp:839-860).  That terminates iff the links form a forest whose `next` chains run through
    // later siblings; the reference's reader only range-checks them and its evaluator would spin on a
    // cycle, so anything else is rejected here (no stock cascade is affected).
    {
        bool any_next = false;
        for (int i = 0; i < S; i++) any_next |= c.st_next[i] != -1;
        for (int i = 0; any_next && i < S; i++) {
            if (c.st_parent[i] >= i) FMT_FAIL("stage tree is not a forest: parent of stage %d is %d", i, c.st_parent[i]);
            const int nx = c.st_next[i];
            if (nx != -1 && (nx <= i || c.st_parent[nx] != c.st_parent[i]))
                FMT_FAIL("stage tree is not a forest: next of stage %d is %d", i, nx);
        }
    }
    if ((int)c.st_child.size() != S) {  // derive child links (tempcv.cpp:2076-2083)
        c.st_child.assign(S, -1);
        for (int i = 0; i < S; i++) {
            int p = c.st_parent[i];
            if (p != -1 && c.st_child[p] == -1) c.st_child[p] = i;
        }
    }

    c.is_tree = false; c.is_stump_based = true; c.has_tilted = false;
    c.hid_weight.assign((size_t)N * 3, 0.f);
    c.hid_nrects.assign(N, 2);
    c.hid_thr.assign(S, 0.f);
    c.two_rects.assign(S, 1);
    c.order_free.assign(S, 0);

    const float stage_threshold_bias = 0.0001f;  // tempcv.cpp:262
    const int eq_w = c.win_w - 2, eq_h = c.win_h - 2;  // equRect at scale 1 (tempcv.cpp:614-616)
    const double weight_scale = 1. / (eq_w * eq_h);    // :617

    for (int i = 0; i < S; i++) {
        if (c.st_parent[i] < -1 || c.st_parent[i] >= S) FMT_FAIL("parent must be integer number. (stage %d)", i);
        if (c.st_next[i] < -1 || c.st_next[i] >= S) FMT_FAIL("next must be integer number. (stage %d)", i);
        c.hid_thr[i] = c.st_thr[i] - stage_threshold_bias;  // float - float, :419
        c.is_tree |= c.st_next[i] != -1;                    // :431
        for (int t = c.st_first_tree[i]; t < c.st_first_tree[i + 1]; t++) {
            const int cnt = c.tr_nnodes[t];
            c.is_stump_based &= cnt == 1;  // :465
            for (int l = 0; l < cnt; l++) {
                const int n = c.tr_first_node[t] + l;
                const HostNode &nd = c.nodes[n];
                // a link to another node must lead FORWARD (tempcv.cpp:1981-1982, 2019-2020: "<= k" is
                // rejected): a back edge would make the device tree walk loop forever
                if (nd.left >= cnt || nd.right >= cnt || -nd.left > cnt || -nd.right > cnt ||
                    (nd.left > 0 && nd.left <= l) || (nd.right > 0 && nd.right <= l))
                    FMT_FAIL("Tree structure is broken (stage %d, tree %d, node %d)", i, t - c.st_first_tree[i], l);
                for (int k = 0; k < 3; k++) {  // :365-387
                    const int *r = nd.rect[k];
                    if (!r[2]) continue;
                    c.has_tilted |= nd.tilted != 0;
                    if (r[2] < 0 || r[3] < 0 || r[1] < 0 || r[0] + r[2] > c.win_w ||
                        (!nd.tilted && (r[0] < 0 || r[1] + r[3] > c.win_h)) ||
                        (nd.tilted && (r[0] - r[3] < 0 || r[1] + r[2] + r[3] > c.win_h)))
                        FMT_FAIL("rectangle #%d of the classifier #%d of the stage classifier #%d is not inside "
                                 "the reference (original) cascade window", k, t - c.st_first_tree[i], i);
                }
                int nr = 3;  // :453-458
                if (fabs(nd.weight[2]) < DBL_EPSILON || nd.rect[2][2] == 0 || nd.rect[2][3] == 0)
                    nr = 2;
                else
                    c.two_rects[i] = 0;
                c.hid_nrects[n] = nr;
                if (nd.rect[0][2] <= 0 || nd.rect[0][3] <= 0 || nd.rect[1][2] <= 0 || nd.rect[1][3] <= 0)
                    FMT_FAIL("node needs at least two rectangles (stage %d, tree %d, node %d)", i, t - c.st_first_tree[i], l);
                // scale-1 weights, tempcv.cpp:692-760 (tr == r at scale 1)
                double sum0 = 0, area0 = 0;
                float *hw = &c.hid_weight[(size_t)n * 3];
                const double correction_ratio = weight_scale * (!nd.tilted ? 1 : 0.5);  // :733
                for (int k = 0; k < nr; k++) {
                    const int tw = nd.rect[k][2], th = nd.rect[k][3];
                    hw[k] = (float)(nd.weight[k] * correction_ratio);  // :752
                    if (k == 0)
                        area0 = tw * th;
                    else
                        sum0 += hw[k] * tw * th;  // float*int*int evaluated in float, :757
                }
                hw[0] = (float)(-sum0 / area0);  // :760
            }
        }
        // Is the stage's alpha sum exact in double whatever the order?  Every alpha is a
        // multiple of 2^(e_min-23); if sum|alpha| < 2^53 * 2^(e_min-23) every partial sum of
        // any subset is representable, so a parallel reduction equals the sequential one.
        {
            int e_min = 1 << 20;
            double abs_sum = 0;
            bool ok = true;
            for (int t = c.st_first_tree[i]; t < c.st_first_tree[i + 1]; t++) {
                const int a0 = c.tr_first_node[t] + t, a1 = a0 + c.tr_nnodes[t] + 1;
                float amax = 0;
                for (int a = a0; a < a1; a++) {
                    float v = c.alpha[a];
                    if (!std::isfinite(v)) { ok = false; continue; }
                    if (v == 0.f) continue;
                    int e;
                    frexpf(fabsf(v), &e);  // |v| = m * 2^e, m in [0.5,1): multiple of 2^(e-24)
                    if (e - 24 < e_min) e_min = e - 24;
                    if (fabsf(v) > amax) amax = fabsf(v);
                }
                abs_sum += amax;  // one leaf per tree contributes
            }
            if (ok) {
                if (e_min == (1 << 20)) c.order_free[i] = 1;  // all zeros
                else c.order_free[i] = abs_sum < ldexp(1.0, 52 + e_min) ? 1 : 0;
            }
        }
    }
    return 0;
}

// ------------------------------------------------------------------------------------
// device packing
// ------------------------------------------------------------------------------------
static void corner_coords(const HostNode &nd, int k, int dx[4], int dy[4]) {
    const int x = nd.rect[k][0], y = nd.rect[k][1], w = nd.rect[k][2], h = nd.rect[k][3];
    if (!nd.tilted) {  // tempcv.cpp:738-741
        dy[0] = y;     dx[0] = x;
        dy[1] = y;     dx[1] = x + w;
        dy[2] = y + h; dx[2] = x;
        dy[3] = y + h; dx[3] = x + w;
    } else {           // tempcv.cpp:745-749
        dy[0] = y;         dx[0] = x;
        dy[1] = y + h;     dx[1] = x - h;
        dy[2] = y + w;     dx[2] = x + w;
        dy[3] = y + w + h; dx[3] = x + w - h;
    }
}

int dense_tile_cols(int win_w, int ystep) { return ((kTileW - 1) * ystep + win_w + 1 + 3) & ~3; }
int dense_tile_rows(int win_h, int ystep, int tile_h) { return (tile_h - 1) * ystep + win_h + 1; }
int dense_tile_half(int win_w, int ystep) {
    // ystep 2: word offset of a row's odd columns.  A multiple of 4 words, so that both halves of a tile row are 16-byte
    // aligned destinations of a TMA bulk copy (whose size is rounded up to 16 bytes as well: the even half may run
    // up to `half` words, never into the odd half).
    if (ystep == 1) return 0;
    return (dense_tile_cols(win_w, ystep) / 2 + 3) & ~3;
}
int dense_tile_stride(int win_w, int ystep) {
    // ystep 1: natural layout, stride >= cols.  ystep 2: even columns at the start of a row, odd columns
    // `half` words behind them, stride >= 2 * half.  In both the word distance
    // between consecutive WINDOW rows, ystep * stride, is 8 (mod 32) and the stride is a
    // multiple of 4 words (16-byte rows / halves for the TMA bulk copies).
    const int cols = dense_tile_cols(win_w, ystep);
    int s = ystep == 1 ? cols : 2 * dense_tile_half(win_w, ystep);
    s = (s + 3) & ~3;
    while ((ystep * s) % 32 != 8) s += 4;
    return s;
}

static inline int cv_round_d(double v) { return (int)lrint(v); }   // cvRound: round half to even

void pack_sc_level(const HostCascade &c, double scale, int pitch, ScLevel &L, ScNode *out) {
    // tempcv.cpp:614-618
    const int ex = cv_round_d(scale), ey = ex;
    const int ew = cv_round_d((c.win_w - 2) * scale), eh = cv_round_d((c.win_h - 2) * scale);
    const double weight_scale = 1. / (ew * eh);
    L.inv_area = weight_scale;
    L.eq_off[0] = ey * pitch + ex; L.eq_off[1] = ey * pitch + ex + ew;
    L.eq_off[2] = (ey + eh) * pitch + ex; L.eq_off[3] = (ey + eh) * pitch + ex + ew;
    for (int n = 0; n < c.n_nodes(); n++) {   // tempcv.cpp:636-760; the flagx / flagy branch is dead (kx, ky >= 1)
        const HostNode &nd = c.nodes[n];
        ScNode &d = out[n];
        memset(&d, 0, sizeof d);
        const int nr = c.hid_nrects[n];
        double sum0 = 0, area0 = 0;
        const double correction_ratio = weight_scale * (!nd.tilted ? 1 : 0.5);   // :733
        for (int k = 0; k < nr; k++) {
            const int tx = cv_round_d(nd.rect[k][0] * scale), tw = cv_round_d(nd.rect[k][2] * scale);   // :704-716
            const int ty = cv_round_d(nd.rect[k][1] * scale), th = cv_round_d(nd.rect[k][3] * scale);
            int dy[4], dx[4];
            if (!nd.tilted) {   // :738-741
                dy[0] = ty;      dx[0] = tx;
                dy[1] = ty;      dx[1] = tx + tw;
                dy[2] = ty + th; dx[2] = tx;
                dy[3] = ty + th; dx[3] = tx + tw;
            } else {            // :745-749
                dy[2] = ty + tw;      dx[2] = tx + tw;
                dy[3] = ty + tw + th; dx[3] = tx + tw - th;
                dy[0] = ty;           dx[0] = tx;
                dy[1] = ty + th;      dx[1] = tx - th;
            }
            for (int q = 0; q < 4; q++) d.off[k * 4 + q] = dy[q] * pitch + dx[q];
            d.w[k] = (float)(nd.weight[k] * correction_ratio);   // :752
            if (k == 0) area0 = tw * th;
            else sum0 += d.w[k] * tw * th;   // float*int*int evaluated in float, :757
        }
        d.w[0] = (float)(-sum0 / area0);   // :760
        d.thr = nd.threshold;
        d.left = nd.left; d.right = nd.right;
        d.flags = (nd.tilted ? 1 : 0) | (nr << 8);
    }
}

// Tile-kernel blobs.  `elig` = leading stages the tile kernel can evaluate: one-node upright
// trees, and in a stage tree only the unconditional linear prefix (stage i the single child
// of stage i-1 with no `next` alternative).  Every eligible stump gets a TailStump record
// (global memory, warp-autonomous phase); the stumps of the first n_fixed stages are also
// parameter resident (DenseStump, fixed-geometry phase).
// allow_tiles = false: no stage for the tile kernel (tail_stages = exec_stages = 0), the generic kernels take the cascade.
static void pack_dense_one(const HostCascade &c, int ystep, DenseParams &P, std::vector<TailStump> &tail,
                           std::vector<DenseStage> &stage_tab, int &dense_stumps, bool allow_tiles = true) {
    const int S = c.n_stages(), T = c.n_trees();
    memset(&P, 0, sizeof P);
    P.total_stages = S;
    P.win_w = c.win_w; P.win_h = c.win_h;
    P.tile_stride = dense_tile_stride(c.win_w, ystep);
    P.tile_half = dense_tile_half(c.win_w, ystep);
    P.is_tree = c.is_tree ? 1 : 0;
    P.ystep = ystep;
    P.filter_eps = 9.5367431640625e-07f;  // 2^-20
    if (const char *e = getenv("CLFD_FORCE_EXACT")) P.force_exact = atoi(e) != 0;   // test hook: bypass the FP32 filters
    P.inv_area = 1. / ((c.win_w - 2) * (c.win_h - 2));
    P.eq_x = 1; P.eq_y = 1; P.eq_w = c.win_w - 2; P.eq_h = c.win_h - 2;   // equRect at scale 1 (tempcv.cpp:614-616)
    // a cascade with tilted features keeps a second tile (the tilted integral) behind the first; on
    // ystep-2 levels (more integral rows per tile) the tiles are half as high then, or the two tiles
    // leave room for only one or two CTAs per SM
    P.tilted_tile = c.has_tilted && !getenv("CLFD_NO_TILTED_TILE") ? 1 : 0;
    P.tile_h = kTileH;
    if (P.tilted_tile && ystep == 2 && !c.is_tree && !getenv("CLFD_NO_SMALL_TILES")) P.tile_h = kTileHSmall;
    // plain stump cascades on ystep-2 levels: 24-row tiles bring the tile under 56 KB, i.e. 4 CTAs per SM
    // instead of 3 (+1 % frontalface_alt, +2 % frontalface_default, measured); CLFD_TILE_H2=32 switches it off
    if (ystep == 2 && !P.tilted_tile && !c.is_tree && c.is_stump_based) {
        const char *e = getenv("CLFD_TILE_H2");
        if (!e || atoi(e) == 24) P.tile_h = 24;
    }
    const size_t tile_bytes = (size_t)dense_tile_rows(c.win_h, ystep, P.tile_h) * P.tile_stride * 4;
    const size_t tilt_base = (tile_bytes + 127) & ~(size_t)127;
    const bool dense_ok = allow_tiles && tile_bytes <= 65536 && (!P.tilted_tile || 2 * tilt_base <= 160 * 1024) && c.win_w <= 255 && c.win_h <= 255;
    // multi-node trees (<= kMaxTreeNodes nodes, children after their parent) are evaluated node by node
    // with a per-window "node I am at" state; every tree is padded to npt = the cascade's largest tree
    int npt = 1;
    for (int t = 0; t < T; t++) npt = std::max(npt, c.tr_nnodes[t]);
    if (getenv("CLFD_NO_NODE_TILES") && npt > 1) npt = kMaxTreeNodes + 1;   // test hook: leave trees to the mid / deep kernels
    P.npt = npt <= kMaxTreeNodes ? npt : 1;
    auto stage_ok = [&](int i) {   // tilted only with the second tile
        for (int t = c.st_first_tree[i]; t < c.st_first_tree[i + 1]; t++) {
            if (c.tr_nnodes[t] > P.npt) return false;
            for (int j = 0; j < c.tr_nnodes[t]; j++) {
                const HostNode &nd = c.nodes[c.tr_first_node[t] + j];
                if (!P.tilted_tile && nd.tilted) return false;
                if ((nd.left > 0 && (nd.left <= j || nd.left >= c.tr_nnodes[t])) ||
                    (nd.right > 0 && (nd.right <= j || nd.right >= c.tr_nnodes[t])))
                    return false;
            }
        }
        return true;
    };
    int elig = 0;   // the linear prefix
    while (dense_ok && elig < S && elig < kMaxDenseStages) {
        if (c.is_tree && (c.st_next[elig] != -1 || c.st_parent[elig] != elig - 1 ||
                          (elig > 0 && c.st_child[elig - 1] != elig)))
            break;
        if (!stage_ok(elig)) break;
        elig++;
    }
    // A stage tree of stumps is walked by the tile kernel itself (tempcv.cpp:834-861): the stages in
    // depth-first preorder (a stage, its child subtree, then its `next` alternative) -- both the
    // stage a passing window goes to (child) and the one a failing window goes to (the `next` of the
    // nearest ancestor-or-self that has one) lie later in that order, so one sweep over the order
    // with a per-window target position evaluates every window's path.
    std::vector<int> order;
    if (c.is_tree && P.npt == 1 && dense_ok && elig > 0 && elig < S && S < (int)kRouteReject && !getenv("CLFD_NO_TREE_TILES")) {
        std::vector<int> stack{0};
        std::vector<char> seen(S, 0);
        bool ok = true;
        while (!stack.empty() && ok) {
            const int i = stack.back();
            stack.pop_back();
            ok = !seen[i] && stage_ok(i);
            seen[i] = 1;
            order.push_back(i);
            if (c.st_next[i] >= 0) stack.push_back(c.st_next[i]);
            if (c.st_child[i] >= 0) stack.push_back(c.st_child[i]);
        }
        if (!ok || (int)order.size() != S) order.clear();
        for (int e = 0; e < elig && !order.empty(); e++) if (order[e] != e) order.clear();
    }
    const bool walk_tree = !order.empty();
    if (!walk_tree) { order.resize(elig); for (int e = 0; e < elig; e++) order[e] = e; }
    const int E = (int)order.size();
    std::vector<int> pos(S, -1);
    for (int e = 0; e < E; e++) pos[order[e]] = e;
    P.tail_stages = elig;
    P.exec_stages = E;
    P.g1_min = 12;   // measured: 8, 12, 16 within 0.6 % of each other, 12 best
    if (const char *e = getenv("CLFD_G1_MIN")) P.g1_min = std::max(1, std::min(16, atoi(e)));
    int n_elig_stumps = 0;
    for (int e = 0; e < E; e++) n_elig_stumps += c.st_ntrees[order[e]] * P.npt;
    dense_stumps = n_elig_stumps;
    tail.assign(n_elig_stumps, TailStump());
    stage_tab.assign(walk_tree ? E : 0, DenseStage());
    auto tile_offset = [&](int dy, int dx) {
        const int word = ystep == 1 ? dy * P.tile_stride + dx
                                    : dy * P.tile_stride + (dx & 1) * P.tile_half + (dx >> 1);
        return (uint32_t)(word * 4);
    };
    int tail_at = 0;   // records in execution order (== tree order for the linear prefix)
    for (int e = 0; e < E; e++) {
        const int i = order[e];
        DenseStage ds;
        memset(&ds, 0, sizeof ds);
        bool any3 = false;
        double abs_sum = 0;
        ds.tail_first = (uint32_t)tail_at;
        for (int t = c.st_first_tree[i]; t < c.st_first_tree[i + 1]; t++) {
            const int a = c.tr_first_node[t] + t;            // alpha base of tree t
            double amax = 0;
            for (int j = 0; j < P.npt; j++) {
                TailStump &ts = tail[tail_at++];
                memset(&ts, 0, sizeof ts);
                if (j >= c.tr_nnodes[t]) { ts.meta = kNodePad | (kNodeLeaf << 8) | (kNodeLeaf << 16); continue; }
                const int n = c.tr_first_node[t] + j;
                const HostNode &nd = c.nodes[n];
                any3 |= c.hid_nrects[n] == 3;
                for (int k = 0; k < c.hid_nrects[n]; k++) {
                    int dx[4], dy[4];
                    corner_coords(nd, k, dx, dy);
                    for (int q = 0; q < 4; q++) ts.off[k * 4 + q] = tile_offset(dy[q], dx[q]) + (nd.tilted ? (uint32_t)tilt_base : 0u);
                    ts.w[k] = c.hid_weight[(size_t)n * 3 + k];
                }
                ts.thr = nd.threshold;
                ts.a0 = nd.left <= 0 ? c.alpha[a + (-nd.left)] : 0.f;     // sum <  t -> left  (tempcv.cpp:788)
                ts.a1 = nd.right <= 0 ? c.alpha[a + (-nd.right)] : 0.f;   // sum >= t -> right
                ts.meta = (uint32_t)j | ((nd.left > 0 ? (uint32_t)nd.left : kNodeLeaf) << 8) |
                          ((nd.right > 0 ? (uint32_t)nd.right : kNodeLeaf) << 16);
                amax = fmax(amax, fmax(fabs((double)ts.a0), fabs((double)ts.a1)));
            }
            abs_sum += amax;
        }
        ds.first = 0; ds.count = (uint16_t)(c.st_ntrees[i] * P.npt);   // records
        ds.thr = c.hid_thr[i];
        // double products only on the reference's stump fast path (tempcv.cpp:862,872)
        ds.flags = ((!c.is_tree && c.is_stump_based && c.two_rects[i]) ? 1u : 0u) | (any3 ? 2u : 0u) |
                   (c.order_free[i] ? 4u : 0u);
        // FP32 summation of n alphas in any order: |error| <= (n-1) 2^-24 sum|alpha|; 2x slack
        const double er = (double)(c.st_ntrees[i] * P.npt) * ldexp(1.0, -23) * abs_sum;
        ds.sum_eps = std::isfinite(er) ? (float)(er * 1.0000002) + FLT_MIN : INFINITY;
        // + 1e-5 |thr|: windows whose stage sum lies within the north star's tolerance of the threshold all take the
        // FP64 path, where they are counted exactly (clfd_run_stats::near_threshold_events); ~1e-4 of the windows
        ds.sum_eps += 1.0001e-5f * std::fabs(ds.thr);
        if (walk_tree) {
            const uint32_t pass = c.st_child[i] >= 0 ? (uint32_t)pos[c.st_child[i]] : kRouteAccept;
            int p = i;
            while (p >= 0 && c.st_next[p] < 0) p = c.st_parent[p];   // tempcv.cpp:853-855
            const uint32_t fail = p >= 0 ? (uint32_t)pos[c.st_next[p]] : kRouteReject;
            ds.flags |= ((uint32_t)i << 8) | (pass << 16) | (fail << 24);
            stage_tab[e] = ds;
        }
        if (e < elig) P.stage[e] = ds;
    }
    // parameter-resident copy of the leading stages that fit the kernel-parameter budget.  Inside a
    // stage the copy is REORDERED (the FP32 filters do not depend on the order; the exact fallback
    // reads the global records, which stay in tree order): first the two-rect stumps whose rects have
    // two corners in common -- the usual edge feature, a rectangle and one of its halves -- in a
    // six-offset form E0,E1,F0,F1,G0,G1 with rect0 = (E0-E1)+(F0-F1), rect1 = (E0-E1)+(G0-G1): six
    // corner loads instead of eight.  With p0,p3 entering a rect sum with + and p1,p2 with -, the
    // common pair can only be (p0,p2), (p3,p1), (p0,p1) or (p3,p2).
    const bool share_corners = !getenv("CLFD_NO_SHARED_CORNERS");   // test hook
    int ns = 0, nstump = 0;
    while (ns < elig && nstump + c.st_ntrees[ns] * P.npt <= kMaxDenseStumps) {
        P.stage[ns].first = (uint16_t)nstump;
        std::vector<DenseStump> six, rest;
        for (int t = c.st_first_tree[ns] * P.npt; t < c.st_first_tree[ns + 1] * P.npt; t++) {
            DenseStump st = tail[t];
            bool shared = false;
            if (share_corners && P.npt == 1 && c.hid_nrects[c.tr_first_node[t]] == 2) {   // (multi-node trees keep their order)
                const uint32_t *A = st.off, *B = st.off + 4;
                static const int pairs[4][2] = {{0, 2}, {3, 1}, {0, 1}, {3, 2}};   // (plus, minus) corner
                for (const auto &pr : pairs) {
                    const int pl = pr[0], mi = pr[1];
                    if (A[pl] != B[pl] || A[mi] != B[mi]) continue;
                    const int opl = pl == 0 ? 3 : 0, omi = mi == 1 ? 2 : 1;   // the other plus / minus corner
                    const uint32_t o[6] = {A[pl], A[mi], A[opl], A[omi], B[opl], B[omi]};
                    for (int q = 0; q < 12; q++) st.off[q] = q < 6 ? o[q] : 0;
                    shared = true;
                    break;
                }
            }
            (shared ? six : rest).push_back(st);
        }
        P.stage[ns].n_shared = (uint32_t)six.size();
        for (const auto &st : six) P.stump[nstump++] = st;
        for (const auto &st : rest) P.stump[nstump++] = st;
        ns++;
    }
    P.n_stages = ns;
    // the global records go into blocks of 32 stumps with the five 16-byte chunks of a record 512 bytes apart
    // (kernels_clod.cu, stump_from_global): chunk q of a stage's record j at (j / 32) * 160 + q * 32 + j % 32;
    // every stage starts a new block, tail_first (in records) is remapped
    {
        static_assert(sizeof(TailStump) == 80, "five 16-byte chunks per record");
        struct Chunk { uint32_t v[4]; };
        std::vector<TailStump> blocked;
        const Chunk *src = reinterpret_cast<const Chunk *>(tail.data());
        int at = 0;
        for (int e = 0; e < E; e++) {
            const int count = c.st_ntrees[order[e]] * P.npt;
            const size_t first = blocked.size();
            blocked.resize(first + (size_t)((count + 31) / 32) * 32);
            Chunk *blk = reinterpret_cast<Chunk *>(blocked.data() + first);
            for (int j = 0; j < count; j++)
                for (int q = 0; q < 5; q++) blk[(size_t)(j >> 5) * 160 + q * 32 + (j & 31)] = src[(size_t)(at + j) * 5 + q];
            if (e < elig) P.stage[e].tail_first = (uint32_t)first;
            if (walk_tree) stage_tab[e].tail_first = (uint32_t)first;
            at += count;
        }
        tail.swap(blocked);
    }
    // sentinel leaf values (haarcascade_mcs_upperbody has one of 2.2e6 in stage 2): sum_eps, built from the largest
    // leaf of every stump, would exceed any real distance to the stage threshold and send every window of the stage
    // through the FP64 path; such cascades use the kernel instantiation that bounds the FP32 sum by what was added
    P.track_abs = 0;
    for (float v : c.alpha)
        if (std::fabs(v) > 64.f) P.track_abs = 1;
    if (getenv("CLFD_NO_TRACK_ABS")) P.track_abs = 0;   // A/B hook
    // stages run in fixed geometry before the first compaction (tunable for experiments)
    int nf = 3;
    if (const char *e = getenv("CLFD_N_FIXED")) nf = atoi(e);
    P.n_fixed = nf < 0 ? 0 : (nf > ns ? ns : nf);
}

void pack_cascade(const HostCascade &c, PackedCascade &out) {
    const int S = c.n_stages(), T = c.n_trees(), N = c.n_nodes();
    out.deep_stages.resize(S);
    out.deep_nodes.resize(N);
    out.tree_first_node = c.tr_first_node;
    out.alpha = c.alpha;
    for (int i = 0; i < S; i++) {
        DeepStage &s = out.deep_stages[i];
        memset(&s, 0, sizeof s);
        s.first_tree = c.st_first_tree[i];
        s.ntrees = c.st_ntrees[i];
        s.thr = c.hid_thr[i];
        bool stumps = true;
        for (int t = s.first_tree; t < s.first_tree + s.ntrees; t++) stumps &= c.tr_nnodes[t] == 1;
        // double products only on the reference's stump fast path (tempcv.cpp:862,872); stage trees
        // and multi-node cascades go through icvEvalHidHaarClassifier (float products, :782-786)
        const bool dbl = !c.is_tree && c.is_stump_based && c.two_rects[i];
        s.flags = (dbl ? 1 : 0) | (c.order_free[i] ? 2 : 0) | (stumps ? 4 : 0);
        s.parent = c.st_parent[i]; s.next = c.st_next[i]; s.child = c.st_child[i];
    }
    for (int n = 0; n < N; n++) {
        DeepNode &d = out.deep_nodes[n];
        memset(&d, 0, sizeof d);
        const HostNode &nd = c.nodes[n];
        for (int k = 0; k < c.hid_nrects[n]; k++) {
            int dx[4], dy[4];
            corner_coords(nd, k, dx, dy);
            for (int q = 0; q < 4; q++) { d.dx[k * 4 + q] = (uint8_t)dx[q]; d.dy[k * 4 + q] = (uint8_t)dy[q]; }
            d.w[k] = c.hid_weight[(size_t)n * 3 + k];
        }
        d.thr = nd.threshold;
        d.left = nd.left; d.right = nd.right;
        d.flags = (nd.tilted ? 1 : 0) | (c.hid_nrects[n] << 8);
    }

    for (int yi = 0; yi < 2; yi++) pack_dense_one(c, yi + 1, out.dense[yi], out.tail[yi], out.stage_tab[yi], out.dense_stumps);
    // Both blobs hand the tile kernel the same stages.  The host code decides from dense[0] alone whether a cascade has a
    // tile prefix, whether the tile kernel finishes it (no mid / deep kernels then, chunk overlap, the flat-window table:
    // enqueue_range, overlap_applies, build_flat_table in clfd_api.cu), but launches the ystep-2 levels' tiles with
    // dense[1].  The ystep-2 tile spans twice the rows and columns of windows, so it stops fitting shared memory at a
    // smaller window (45 x 45 for a plain stump cascade, 44 x 44 fits): when either tile does not fit, neither row step
    // uses the tile kernel and the generic kernels take the whole cascade on every level.
    if (out.dense[0].tail_stages != out.dense[1].tail_stages || out.dense[0].exec_stages != out.dense[1].exec_stages)
        for (int yi = 0; yi < 2; yi++)
            pack_dense_one(c, yi + 1, out.dense[yi], out.tail[yi], out.stage_tab[yi], out.dense_stumps, false);
}

// Tile-kernel blob of ONE scale of the scale-cascade mode, for the scales whose window step is
// exactly 2 (factor <= 2, tempcv.cpp:1365): on the full-resolution integral image those windows
// are a ystep-2 level like any other, with the cascade's rectangles scaled and its weights
// re-normalised for this scale (cvSetImagesForHaarClassifierCascade, tempcv.cpp:614-618, 636-760
// -- the same arithmetic as pack_sc_level).  Built by packing a scaled copy of the cascade whose
// "window" is the extent the scaled rectangles reach (cvRound(x*s) + cvRound(w*s) may exceed
// cvRound((x+w)*s) by one), then putting this scale's variance rectangle and area in.
bool pack_sc_dense(const HostCascade &c, double scale, DenseParams &P, std::vector<TailStump> &tail,
                   std::vector<DenseStage> &stage_tab) {
    HostCascade s = c;
    const int ex = cv_round_d(scale), ey = ex;
    const int ew = cv_round_d((c.win_w - 2) * scale), eh = cv_round_d((c.win_h - 2) * scale);
    const double weight_scale = 1. / (ew * eh);
    int ext_w = std::max(cv_round_d(c.win_w * scale), ex + ew), ext_h = std::max(cv_round_d(c.win_h * scale), ey + eh);
    for (int n = 0; n < c.n_nodes(); n++) {
        const HostNode &nd = c.nodes[n];
        HostNode &d = s.nodes[n];
        const int nr = c.hid_nrects[n];
        double sum0 = 0, area0 = 0;
        const double correction_ratio = weight_scale * (!nd.tilted ? 1 : 0.5);   // :733
        for (int k = 0; k < nr; k++) {
            d.rect[k][0] = cv_round_d(nd.rect[k][0] * scale); d.rect[k][2] = cv_round_d(nd.rect[k][2] * scale);   // :704-716
            d.rect[k][1] = cv_round_d(nd.rect[k][1] * scale); d.rect[k][3] = cv_round_d(nd.rect[k][3] * scale);
            int dx[4], dy[4];
            corner_coords(d, k, dx, dy);
            for (int q = 0; q < 4; q++) {
                if (dx[q] < 0 || dy[q] < 0) return false;
                ext_w = std::max(ext_w, dx[q]); ext_h = std::max(ext_h, dy[q]);
            }
            float &w = s.hid_weight[(size_t)n * 3 + k];
            w = (float)(nd.weight[k] * correction_ratio);   // :752
            if (k == 0) area0 = d.rect[k][2] * d.rect[k][3];
            else sum0 += w * d.rect[k][2] * d.rect[k][3];   // float*int*int evaluated in float, :757
        }
        s.hid_weight[(size_t)n * 3] = (float)(-sum0 / area0);   // :760
    }
    s.win_w = ext_w; s.win_h = ext_h;
    int dense_stumps = 0;
    pack_dense_one(s, 2, P, tail, stage_tab, dense_stumps);
    P.inv_area = weight_scale;
    P.eq_x = ex; P.eq_y = ey; P.eq_w = ew; P.eq_h = eh;
    return P.tail_stages > 0 && P.exec_stages == P.total_stages;
}

}  // namespace clfd
