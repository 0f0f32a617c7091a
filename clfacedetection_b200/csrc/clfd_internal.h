// clfd_internal.h -- structures shared by the host side (loader, packer, planner) and the
// CUDA kernels.  Not part of the ABI (include/clfd_b200.h is).
#pragma once

#include <cstdint>
#include <string>
#include <vector>

#include "clfd_b200.h"

namespace clfd {

// ------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------
void set_error(const char *fmt, ...) __attribute__((format(printf, 1, 2)));

// ------------------------------------------------------------------------------------
// Host cascade: CvHaarClassifierCascade content (tempcv.hpp:70-112) + hidden cascade
// ------------------------------------------------------------------------------------
struct HostNode {
    int tilted;
    int rect[3][4];   // x,y,w,h
    float weight[3];  // as in the XML
    float threshold;
    int left, right;
};

struct HostCascade {
    std::string name;
    int win_w = 0, win_h = 0;
    std::vector<int> st_ntrees, st_parent, st_next, st_child;
    std::vector<float> st_thr;
    std::vector<int> tr_nnodes;
    std::vector<HostNode> nodes;
    std::vector<float> alpha;
    // hidden cascade (filled by build_hidden)
    bool is_tree = false, is_stump_based = true, has_tilted = false;
    std::vector<float> hid_weight;  // [N][3]
    std::vector<int> hid_nrects;    // [N]
    std::vector<float> hid_thr;     // [S]  xml - 0.0001f
    std::vector<int> two_rects;     // [S]
    std::vector<int> order_free;    // [S]  alpha sum exact in any order
    std::vector<int> st_first_tree; // [S+1]
    std::vector<int> tr_first_node; // [T+1]
    int n_stages() const { return (int)st_ntrees.size(); }
    int n_trees() const { return (int)tr_nnodes.size(); }
    int n_nodes() const { return (int)nodes.size(); }
};

// haar_xml.cpp: restates icvReadHaarClassifier (tempcv.cpp:1750-2089). 0 or clfd_status.
int load_cascade_xml(const char *path, HostCascade &out);
// haar_pack.cpp: validation + icvCreateHidHaarClassifierCascade + scale-1 weights.
int build_hidden(HostCascade &c);

// ------------------------------------------------------------------------------------
// Device blobs
// ------------------------------------------------------------------------------------
// Tile geometry of the smem-tile ("dense") cascade kernel: TW x TH windows per CTA.
constexpr int kTileW = 64;
constexpr int kTileH = 32;
constexpr int kTileHSmall = 16;
constexpr int kTileWindows = kTileW * kTileH;
constexpr int kDenseThreads = 256;
constexpr int kDenseWarps = kDenseThreads / 32;
constexpr int kDenseSlots = kTileWindows / kDenseThreads;   // windows per thread (8)
constexpr int kMaxDenseStumps = 392;   // parameter-resident stumps (constant bank): the leading stages that fit
constexpr int kMaxDenseStages = 32;    // stages the tile kernel can evaluate (a cascade with more keeps a deep tail)

// One stump of the tile kernel, 80 B = 5 x 16 B.  The leading stages' stumps are parameter
// resident (constant bank: a warp whose lanes all evaluate the same stump reads it with LDC,
// off the L1 data pipe the corner loads saturate); every tile-evaluated stump also has a copy
// in global memory (lanes on different stumps, stages beyond the parameter budget).
struct alignas(16) DenseStump {
    uint32_t off[12];  // BYTE offsets into the smem tile: p0..p3 of rect 0,1,2 (rect 2: zeros if absent)
    float w[3];        // hidden weights (w[2] = 0 if absent)
    float thr;
    float a0, a1;      // alpha[0] (sum < t), alpha[1] (sum >= t); 0 where that branch leads to another node
    uint32_t meta;     // multi-node trees: node index in its tree | node to go to if sum < t << 8 | if sum >= t << 16
                       // (kNodeLeaf: a leaf, the tree is done); padding records have index kNodePad
    float pad;
};
typedef DenseStump TailStump;
constexpr uint32_t kRouteAccept = 255, kRouteReject = 254;
constexpr uint32_t kNodeLeaf = 255, kNodePad = 254;
constexpr int kMaxTreeNodes = 4;   // trees the tile kernel evaluates have at most this many nodes
struct DenseStage {
    uint16_t first, count;   // first: index into DenseParams::stump (stages < n_stages only)
    float thr;               // biased threshold
    uint32_t flags;          // bit0 double-product stage (two_rects fast path), bit1 any 3-rect stump,
                             // bit2 alpha sum exact in any order (HostCascade::order_free);
                             // stage trees (stage_g): bits 8-15 the stage's index in the file, bits 16-23 / 24-31 the
                             // execution position a window goes to when it passes / fails (kRouteAccept, kRouteReject)
    uint32_t tail_first;     // index of the stage's first stump in the global TailStump array
    float sum_eps;           // bound on the error of an FP32 sum of the stage's alphas in any order
    uint32_t n_shared;       // parameter-resident copy only: the first n_shared stumps of the stage are two-rect
                             // stumps whose rects share two corners, stored in six-offset form (see haar_pack.cpp)
};
// Two blobs per cascade: [0] for ystep-1 levels (natural tile layout, addr = y*S + x) and
// [1] for ystep-2 levels (columns de-interleaved: addr = y*S + (x&1)*tile_half + (x>>1)), so that in
// both a window's base word is  ystep*wy*S + wx  with ystep*S = 8 (mod 32): the bank of every
// corner load is (wx + 8*wy + const) mod 32, so lanes whose windows have distinct
// (wx + 8*wy) mod 32 never conflict, and a compact blob of survivors spreads over the banks.
struct DenseParams {
    int n_stages;       // stages whose stumps are parameter resident (>= n_fixed)
    int total_stages;   // stages in the whole cascade
    int tile_stride;    // ints per smem tile row (ystep * stride = 8 mod 32)
    int tile_half;      // ystep-2 blob: word offset of a row's odd columns (a multiple of 4: both halves of a row are
                        // 16-byte aligned for the TMA bulk copies from a column-de-interleaved integral); 0 in the ystep-1 blob
    int win_w, win_h;
    int is_tree;        // stage-tree cascade: exit codes are 2*last_stage (+accept)
    int ystep;          // 1 or 2
    int force_exact;    // test hook: skip the FP32 filter, evaluate every stage in FP64
    float filter_eps;   // FP32 filter guard band (2^-20), see kernels_clod.cu
    int n_fixed;        // leading stages run in fixed geometry (no compaction), <= n_stages
    int tail_stages;    // leading stages the tile kernel evaluates (upright stumps, linear): == total_stages
                        // when it finishes the cascade itself, otherwise survivors go to the deep kernel
    int g1_min;         // phase 2: more than this many windows in a warp -> thread per window (G = 1), max 16
    int tilted_tile;    // the cascade has tilted features: a second smem tile holds the tilted integral, right
                        // behind the first (tilted nodes' offsets already point into it)
    int exec_stages;    // == tail_stages, or for a stage tree the tile kernel walks itself: all stages, in
                        // execution order (stage_g; the first tail_stages of them are the linear prefix)
    int npt;            // records per tree: 1 = stumps; 2..4 = multi-node trees, every tree padded to npt node records
    int tile_h;         // window rows per tile: kTileH; kTileHSmall where two tiles (tilted) would leave one CTA per SM;
                        // 24 for plain stump cascades on ystep-2 levels
    int eq_x, eq_y, eq_w, eq_h;   // the variance rectangle inside the window (tempcv.cpp:614-616): (1, 1, w-2, h-2) at scale 1
    int track_abs;      // some leaf value is a sentinel (|alpha| > 64: haarcascade_mcs_*): the static sum_eps of such a stage
                        // would send every window through the FP64 path; stage verdicts bound the FP32 sum by the
                        // magnitudes actually added instead (kernels_clod.cu, stage_verdict<TRACK>)
    double inv_area;
    const TailStump *tail;   // device, layout of this blob's ystep (patched in by the detector)
    const struct DenseStage *stage_g;   // device: stage table in execution order (stage trees only)
    const int16_t *flat_code;           // device, 256 entries or NULL: the exit code of a FLAT window (every pixel = the index),
                                        // measured once per detector with the detector's own kernels (clfd_api.cu, build_flat_table)
    DenseStage stage[kMaxDenseStages];
    DenseStump stump[kMaxDenseStumps];
};

// Generic ("deep") cascade in global memory: any tree shape, tilted, stage tree.
struct DeepNode {          // 64 B
    uint8_t dx[12], dy[12];  // corner coordinates of p0..p3 of rect 0,1,2 relative to the window
    float w[3];
    float thr;
    int left, right;         // >0 node index in tree, <=0 leaf -idx
    int flags;               // bit0 tilted, bits 8.. nrects
    int pad[3];
};
struct DeepStage {         // 32 B
    int first_tree, ntrees;
    float thr;
    int flags;               // bit0 two_rects, bit1 order_free, bit2 all trees are stumps
    int parent, next, child;
    int pad;
};
struct DeepCascadeDev {
    const DeepStage *stages;
    const int *tree_first_node;  // [T+1]; alpha base of tree t = tree_first_node[t] + t
    const DeepNode *nodes;
    const float *alpha;
    int n_stages, is_tree, has_tilted, win_w, win_h;
    int mid_begin, mid_end;      // stages the thread-per-window mid kernel evaluates (equal: none)
    double inv_area;
};

// Pyramid level (shared by all cascades of a detector)
struct PyrLevel {
    int w, h;
    int pyr_pitch;       // bytes, multiple of 16
    int sum_pitch;       // elements, multiple of 8 (>= w+1)
    int nrb;             // row blocks of kRowBlock rows
    int xtab_off, ytab_off;
    int resize_mode;     // kResize*: how k_resize_colsum reads the source rows of this level
    int di;              // the int32 integral of this level is stored column-DE-INTERLEAVED: row y holds its even columns
                         // at [y*sum_pitch, +sum_pitch/2) and its odd columns behind them (element (y, x) at
                         // y*sum_pitch + (x&1)*sum_pitch/2 + (x>>1)), which is the layout the tile kernel wants in shared
                         // memory on ystep-2 levels -- a tile row is then two TMA bulk copies (kernels_clod.cu)
    long long pyr_off;   // byte offset inside a frame's pyramid block
    long long sum_off;   // element offset inside a frame's sum / sqsum / tilted block
    long long col_off;   // element offset inside a frame's column-sum block
};
constexpr int kRowBlock = 32;
// k_resize_colsum: byte loads (any factor / alignment); word loads with the taps of four (factors < 2) or two
// (factors up to 6) neighbouring pixels inside 8 source bytes
constexpr int kResizeBytes = 0, kResizeQuad = 1, kResizePair = 2;

// Per cascade, per level it evaluates
struct CasLevel {
    int pyr_level;
    int nx, ny, ystep;
    int win_w, win_h;     // output rect size
    int tiles_x, tiles_y, tile_base;
    int pad;
    long long win_base;
    double factor;
};

// Scale-cascade mode (REF-SC, tempcv.cpp:1330-1456): one full-frame integral image, the
// FEATURES scaled per factor (cvSetImagesForHaarClassifierCascade, tempcv.cpp:549-768).
struct alignas(16) ScNode {   // 80 B: one tree node with its rects scaled for one factor
    int off[12];            // element offsets dy*pitch + dx of p0..p3 of rect 0,1,2 in the frame's integral
    float w[3];
    float thr;
    int left, right;        // >0 node index in tree, <=0 leaf -idx
    int flags;              // bit0 tilted, bits 8.. nrects
    int pad;
};
struct ScLevel {          // one scale
    double factor, ystep, inv_area;
    int win_w, win_h, nx, ny;   // nx, ny = endX, endY of the invoker's grid
    int eq_off[4];              // equRect corners as element offsets
    int node_base;              // first ScNode of this scale
    int row_base;               // first grid row of this scale among all rows of a frame
    long long win_base;         // first window of this scale among all windows of a frame
};
constexpr int kScCodeSkipped = -32768;   // grid position the skip rule never evaluates (tempcv.cpp:1161)
constexpr int kScCodeOutside = -32767;   // window rejected by the bounds check (tempcv.cpp:817-820, result -1)

struct QueueItem {        // survivor handed to the deep kernel
    uint32_t key;           // frame << 16 | cas_level << 8 | next_stage
    uint32_t xy;            // y << 16 | x   (window origin, pixels of the level)
};

struct DevRect {
    int x, y, w, h, frame, cascade;
};
// one candidate of the reject-level (ROC) output; `win` = window index in the frame: the scan order
struct RocItem {
    DevRect r;
    int level, pad;
    long long win;
    double weight;
};

}  // namespace clfd
