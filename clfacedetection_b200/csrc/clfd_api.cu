// clfd_api.cu -- implementation of the C ABI (include/clfd_b200.h): contexts, cascade
// objects, the pyramid / integral plan, the detector plan and its enqueue / fetch calls.
// Host-side planning restates the level loop of cvHaarDetectObjectsForROC's
// CV_HAAR_SCALE_IMAGE branch (tempcv.cpp:1230-1234,1268-1288) and the window grid of its
// invoker (tempcv.cpp:1013-1021); all pixel work is in kernels_clif.cu / kernels_clod.cu.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <vector>

#include "clfd_pack.h"
#include "kernels.h"

using namespace clfd;

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            set_error("CUDA error %s (%s) at %s:%d: %s", cudaGetErrorName(e_), cudaGetErrorString(e_), \
                      __FILE__, __LINE__, #call);                                                  \
            return CLFD_ERR_CUDA;                                                                  \
        }                                                                                          \
    } while (0)
#define INVALID(...) do { set_error(__VA_ARGS__); return CLFD_ERR_INVALID; } while (0)

static inline int cv_round(double v) { return (int)lrint(v); }
static inline int cv_floor(double v) { int i = (int)v; return i - (i > v); }
static inline size_t round_up(size_t v, size_t m) { return (v + m - 1) / m * m; }

constexpr int kMaxPyramidWindow = 255;   // largest cascade window (either side) of the image-pyramid mode

// ------------------------------------------------------------------------------------
// objects
// ------------------------------------------------------------------------------------
struct clfd_context {
    int device = 0;
    int n_sms = 0;
    cudaStream_t stream = nullptr;
    int64_t launches = 0;
    struct PyramidPlan *scratch = nullptr;   // cached plan of clfd_integral / clfd_resize
};

// Reference counted: a detector keeps the cascades of its plan alive, so destroying a cascade
// before its detectors is safe.  `id` is unique per process (never reused, unlike the address).
struct clfd_cascade {
    HostCascade host;
    PackedCascade packed;
    std::atomic<int> refs{1};
    uint64_t id = 0;
};
static std::atomic<uint64_t> g_next_cascade_id{1};
static void cascade_release(const clfd_cascade *c) {
    if (c && const_cast<clfd_cascade *>(c)->refs.fetch_sub(1) == 1) delete c;
}

template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t count) {
        if (p) { cudaFree(p); p = nullptr; }
        n = count;
        if (count == 0) return 0;
        CK(cudaMalloc((void **)&p, count * sizeof(T)));
        return 0;
    }
    int upload(const std::vector<T> &v, cudaStream_t s) {
        int rc = alloc(v.size());
        if (rc) return rc;
        if (!v.empty()) CK(cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, s));
        return 0;
    }
};

// element `at` of a squared integral that holds 64-bit or (sq32) 32-bit elements, as the pointer the kernels take
static inline unsigned long long *sq_at(unsigned long long *base, size_t at, bool sq32) {
    return sq32 ? reinterpret_cast<unsigned long long *>(reinterpret_cast<uint32_t *>(base) + at) : base + at;
}

// Pyramid + integral plan for frames of W x H and a list of level sizes.
struct PyramidPlan {
    int W = 0, H = 0, max_batch = 0;
    bool want_tilted = false;
    bool sq32 = false;   // squared integral modulo 2^32 (pyramid-mode detectors; set before build())
    std::vector<char> di_levels;   // per level (set before build(); empty: none): store the int32 integral column-de-interleaved (PyrLevel::di)
    std::vector<PyrLevel> levels;
    size_t pyr_frame_stride = 0, sum_frame_stride = 0, col_frame_stride = 0, col_plane_stride = 0;
    int max_level_w = 0;
    int64_t pyramid_pixels = 0, bytes_resize = 0, bytes_integral = 0, bytes_tilted = 0;
    DevBuf<uint8_t> pyr;
    DevBuf<int32_t> sum, tilted;
    DevBuf<unsigned long long> sq;
    DevBuf<uint32_t> col;
    DevBuf<PyrLevel> d_levels;
    DevBuf<int> xofs, yofs;
    DevBuf<short2> xalpha, ybeta;
    DevBuf<int4> resize_items, colscan_items, integral_items[6], tilt_tile_items, tilt_diag_items, tilt_tc_items;
    DevBuf<int32_t> tcar;   // tilted integral: six carry planes per frame

    int build(int W_, int H_, const std::vector<std::pair<int, int>> &sizes, int batch, bool tilt, cudaStream_t s);
    void fill_args(PyramidArgs &a, const uint8_t *frames, size_t frame_stride, int row_stride, int n_frames) const;
    // frames: first frame of the range; frame_base: index of that frame in the per-frame device buffers
    int run(const uint8_t *frames, size_t frame_stride, int row_stride, int frame_base, int n_frames, cudaStream_t s,
            cudaEvent_t *ev, int *n_launch);
};

int PyramidPlan::build(int W_, int H_, const std::vector<std::pair<int, int>> &sizes, int batch, bool tilt,
                       cudaStream_t s) {
    W = W_; H = H_; max_batch = batch; want_tilted = tilt;
    levels.clear();
    std::vector<int> h_xofs, h_yofs;
    std::vector<short2> h_xalpha, h_ybeta;
    std::vector<int4> h_resize, h_colscan, h_integral[6], h_tilt_tile, h_tilt_diag, h_tilt_tc;
    size_t pyr_off = 0, sum_off = 0, col_off = 0;
    max_level_w = 0; pyramid_pixels = 0; bytes_resize = 0; bytes_integral = 0; bytes_tilted = 0;
    for (size_t li = 0; li < sizes.size(); li++) {
        const int w = sizes[li].first, h = sizes[li].second;
        if (w <= 0 || h <= 0) INVALID("pyramid level %zu has empty size %dx%d", li, w, h);
        PyrLevel L;
        memset(&L, 0, sizeof L);
        L.w = w; L.h = h;
        L.pyr_pitch = (int)round_up(w, 16);
        L.sum_pitch = (int)round_up(w + 1, 8);
        L.nrb = (h + kRowBlock - 1) / kRowBlock;
        L.di = li < di_levels.size() && di_levels[li] ? 1 : 0;
        L.xtab_off = (int)h_xofs.size(); L.ytab_off = (int)h_yofs.size();
        L.pyr_off = (long long)pyr_off; L.sum_off = (long long)sum_off; L.col_off = (long long)col_off;
        pyr_off += round_up((size_t)L.pyr_pitch * h, 256);
        sum_off += round_up((size_t)L.sum_pitch * (h + 1), 64);
        col_off += (size_t)L.nrb * L.sum_pitch;
        max_level_w = std::max(max_level_w, w);
        pyramid_pixels += (int64_t)w * h;
        // algorithmic bytes (SURVEY 8-d): resize min(W*H, 4*w*h) + w*h ; integral w*h + (w+1)(h+1)(4+8+4T)
        bytes_resize += std::min<int64_t>((int64_t)W * H, 4ll * w * h) + (int64_t)w * h;
        bytes_integral += (int64_t)w * h + (int64_t)(w + 1) * (h + 1) * (4 + (sq32 ? 4 : 8));
        if (tilt) bytes_tilted += (int64_t)w * h + (int64_t)(w + 1) * (h + 1) * 4;   // the tilted kernels read the level again

        // cv::resize INTER_LINEAR coefficient tables (OpenCV imgproc, SURVEY Appendix A.2)
        const double scale_x = 1. / ((double)w / W), scale_y = 1. / ((double)h / H);
        for (int dx = 0; dx < w; dx++) {
            float fx = (float)((dx + 0.5) * scale_x - 0.5);
            int sx = cv_floor(fx);
            fx -= sx;
            if (sx < 0) { fx = 0; sx = 0; }
            if (sx >= W - 1) { fx = 0; sx = W - 1; }
            h_xofs.push_back(sx);
            h_xalpha.push_back(make_short2((short)lrintf((1.f - fx) * 2048), (short)lrintf(fx * 2048)));
        }
        {   // which source-row access of k_resize_colsum this level's tap positions allow (kernels_clif.cu)
            const int *sx = h_xofs.data() + L.xtab_off;
            bool quad = true, pair = true;
            for (int x = 0; x < w; x += 4) {
                if (sx[std::min(x + 3, w - 1)] - sx[x] > 6) quad = false;
                for (int j = 0; j < 4 && x + j < w; j += 2)
                    if (sx[std::min(x + j + 1, w - 1)] - sx[x + j] > 6) pair = false;
            }
            L.resize_mode = quad ? kResizeQuad : pair ? kResizePair : kResizeBytes;
            if (const char *e = getenv("CLFD_RESIZE_BYTES")) if (atoi(e)) L.resize_mode = kResizeBytes;   // test hook
        }
        for (int dy = 0; dy < h; dy++) {
            float fy = (float)((dy + 0.5) * scale_y - 0.5);
            int sy = cv_floor(fy);
            fy -= sy;
            h_yofs.push_back(sy);
            h_ybeta.push_back(make_short2((short)lrintf((1.f - fy) * 2048), (short)lrintf(fy * 2048)));
        }
        const int xspan = std::max(L.pyr_pitch, L.sum_pitch);
        for (int rb = 0; rb < L.nrb; rb++)
            for (int c = 0; c * 128 < xspan; c++) h_resize.push_back(make_int4((int)li, rb, c, 0));   // one per warp
        for (int c = 0; c * 512 < L.sum_pitch; c++) h_colscan.push_back(make_int4((int)li, c, 0, 0));
        int cls = 0;
        while (cls < 6 && (32 << cls) * 8 < L.sum_pitch) cls++;
        if (cls >= 6) INVALID("level width %d exceeds the supported maximum of 8191 pixels", w);
        for (int rb = 0; rb < L.nrb; rb++) h_integral[cls].push_back(make_int4((int)li, rb, 0, 0));
        if (tilt) {
            const int interior = tilt_tile_interior();
            for (int rb = 0; rb < L.nrb; rb++)
                for (int t = 0; t * interior < w + 1; t++) h_tilt_tile.push_back(make_int4((int)li, rb, t, 0));
            for (int c = 0; c * 256 <= w + (L.nrb - 1) * kRowBlock; c++) h_tilt_diag.push_back(make_int4((int)li, c, 0, 0));
            for (int c = 0; c * 256 < L.sum_pitch; c++) h_tilt_tc.push_back(make_int4((int)li, c, 0, 0));
        }
        levels.push_back(L);
    }
    pyr_frame_stride = round_up(pyr_off, 256);
    sum_frame_stride = round_up(sum_off + 1024, 64);   // slack: tile rows may read past a level's last row
    col_plane_stride = round_up(col_off, 8);
    col_frame_stride = 2 * col_plane_stride;

    int rc = 0;
    if ((rc = pyr.alloc(pyr_frame_stride * batch + 256))) return rc;
    if ((rc = sum.alloc(sum_frame_stride * batch + 4096))) return rc;
    if ((rc = sq.alloc((sum_frame_stride * batch + 4096) / (sq32 ? 2 : 1)))) return rc;
    if (tilt && (rc = tilted.alloc(sum_frame_stride * batch + 4096))) return rc;
    if (tilt && (rc = tcar.alloc(6 * col_plane_stride * batch + 64))) return rc;
    if ((rc = col.alloc(col_frame_stride * batch + 64))) return rc;
    if ((rc = d_levels.upload(levels, s))) return rc;
    if ((rc = xofs.upload(h_xofs, s)) || (rc = yofs.upload(h_yofs, s))) return rc;
    if ((rc = xalpha.upload(h_xalpha, s)) || (rc = ybeta.upload(h_ybeta, s))) return rc;
    while (h_resize.size() % 4) h_resize.push_back(make_int4(-1, 0, 0, 0));   // whole CTAs of four warps
    if ((rc = resize_items.upload(h_resize, s)) || (rc = colscan_items.upload(h_colscan, s))) return rc;
    if (tilt && ((rc = tilt_tile_items.upload(h_tilt_tile, s)) || (rc = tilt_diag_items.upload(h_tilt_diag, s)) ||
                 (rc = tilt_tc_items.upload(h_tilt_tc, s))))
        return rc;
    // carry entries beyond a level's last column are read as zeros and never written
    if (tilt) CK(cudaMemsetAsync(tcar.p, 0, tcar.n * sizeof(int32_t), s));
    for (int k = 0; k < 6; k++)
        if ((rc = integral_items[k].upload(h_integral[k], s))) return rc;
    // the slack regions are read (never used) by TMA row copies: keep them defined
    CK(cudaMemsetAsync(sum.p, 0, sum.n * sizeof(int32_t), s));
    CK(cudaStreamSynchronize(s));   // host vectors go out of scope
    return 0;
}

void PyramidPlan::fill_args(PyramidArgs &a, const uint8_t *frames, size_t frame_stride, int row_stride,
                            int n_frames) const {
    memset(&a, 0, sizeof a);
    a.frames = frames; a.frame_stride = frame_stride; a.row_stride = row_stride; a.W = W; a.H = H;
    a.n_frames = n_frames;
    a.pyr = pyr.p; a.pyr_frame_stride = pyr_frame_stride;
    a.col = col.p; a.col_frame_stride = col_frame_stride; a.col_plane_stride = col_plane_stride;
    a.sum = sum.p; a.sq = sq.p; a.tilted = want_tilted ? tilted.p : nullptr;
    a.sum_frame_stride = sum_frame_stride; a.sq32 = sq32 ? 1 : 0;
    a.levels = d_levels.p; a.n_levels = (int)levels.size();
    a.xofs = xofs.p; a.xalpha = xalpha.p; a.yofs = yofs.p; a.ybeta = ybeta.p;
    a.resize_items = resize_items.p; a.n_resize_items = (int)resize_items.n;
    a.colscan_items = colscan_items.p; a.n_colscan_items = (int)colscan_items.n;
    for (int k = 0; k < 6; k++) { a.integral_items[k] = integral_items[k].p; a.n_integral_items[k] = (int)integral_items[k].n; }
    a.tcar = tcar.p; a.tcar_frame_stride = 6 * col_plane_stride;
    a.tilt_tile_items = tilt_tile_items.p; a.n_tilt_tile_items = want_tilted ? (int)tilt_tile_items.n : 0;
    a.tilt_diag_items = tilt_diag_items.p; a.n_tilt_diag_items = (int)tilt_diag_items.n;
    a.tilt_tc_items = tilt_tc_items.p; a.n_tilt_tc_items = (int)tilt_tc_items.n;
    a.max_level_w = max_level_w;
}

// ev (optional): 5 events recorded before K1, K2, K3, K4 and after K4; *n_launch: the kernels enqueued
int PyramidPlan::run(const uint8_t *frames, size_t frame_stride, int row_stride, int frame_base, int n_frames,
                     cudaStream_t s, cudaEvent_t *ev, int *n_launch) {
    if (n_frames <= 0 || frame_base < 0 || frame_base + n_frames > max_batch)
        INVALID("frames %d..%d outside 0..%d", frame_base, frame_base + n_frames, max_batch);
    if (row_stride < W) INVALID("row stride %d smaller than the frame width %d", row_stride, W);
    PyramidArgs a;
    fill_args(a, frames, frame_stride, row_stride, n_frames);
    // the kernels index the per-frame buffers with the frame number inside the launch
    a.pyr += (size_t)frame_base * a.pyr_frame_stride;
    a.col += (size_t)frame_base * a.col_frame_stride;
    a.sum += (size_t)frame_base * a.sum_frame_stride;
    a.sq = sq_at(a.sq, (size_t)frame_base * a.sum_frame_stride, sq32);
    if (a.tilted) { a.tilted += (size_t)frame_base * a.sum_frame_stride; a.tcar += (size_t)frame_base * a.tcar_frame_stride; }
    int nint = 0, ntilt = 0;
    if (ev) CK(cudaEventRecord(ev[0], s));
    CK(launch_resize_colsum(a, s));
    if (ev) CK(cudaEventRecord(ev[1], s));
    CK(launch_colscan(a, s));
    if (ev) CK(cudaEventRecord(ev[2], s));
    CK(launch_integral_rows(a, s, &nint));
    if (ev) CK(cudaEventRecord(ev[3], s));
    if (want_tilted) CK(launch_tilted(a, s, &ntilt));
    if (ev) CK(cudaEventRecord(ev[4], s));
    *n_launch = 2 + nint + ntilt;
    return 0;
}

// device counters per cascade and slot: [0] rects [1] queue items [2] rect overflow [3] queue overflow
// [4] stage evaluations redone in FP64 (exact path of the tile kernel) [5] of those, stage sums within 1e-5 relative of the threshold
constexpr int kCnt = 8;

struct CascadePlan {
    const clfd_cascade *cascade = nullptr;   // retained
    ~CascadePlan() { cascade_release(cascade); }
    std::vector<CasLevel> levels;   // the tile kernel's levels (scale-cascade mode: its scales of window step 2)
    std::vector<clfd_level> pub_levels;
    int n_tiles = 0;
    int n_tiles_y2 = 0;   // tiles of the ystep-2 levels (they come first)
    long long windows_per_frame = 0;
    int64_t bytes_cascade = 0;
    DevBuf<CasLevel> d_levels;
    DevBuf<DeepStage> d_stages;
    DevBuf<DeepNode> d_nodes;
    DevBuf<int> d_tree_first;
    DevBuf<float> d_alpha;
    // scale-cascade mode
    std::vector<ScLevel> sc_levels;
    DevBuf<ScLevel> d_sc_levels;
    DevBuf<ScNode> d_sc_nodes;
    int sc_rows = 0;
    // scales with window step 2 run through the tile kernel (pack_sc_dense): one blob + launch per scale, grid levels[i]
    struct ScTile { DenseParams P; DevBuf<TailStump> tail; DevBuf<DenseStage> stage_tab; int tile_base = 0, n_tiles = 0; };
    std::vector<std::unique_ptr<ScTile>> sc_tiles;
    long long sc_tile_windows = 0;   // grid positions [0, sc_tile_windows) of a frame belong to those scales
    DevBuf<TailStump> d_tail[2];   // warp-per-window tail records of the tile kernel, [ystep-1]
    DevBuf<DenseStage> d_stage_tab[2];   // stage trees: stage table in execution order
    DevBuf<int16_t> d_flat_code;         // exit codes of flat windows by pixel value (DenseParams::flat_code), see build_flat_table
    DenseParams dense[2];          // the cascade's parameter blobs with this detector's tail pointers
    DevBuf<int16_t> d_codes;
    DevBuf<unsigned long long> d_counters;
    DevBuf<unsigned long long> d_count_b;   // second-queue counter, one per slot
    int mid_begin = 0, mid_end = 0;         // image-pyramid mode: stages of the k_generic_pass passes (equal: none)
    std::vector<int> pass_cuts;   // stage bounds of the k_generic_pass passes
    int sc_deep_from = 0;                   // scale-cascade mode: first stage of the k_generic_deep pass (n_stages: none)
};

constexpr int kMaxChunks = 8;
constexpr int kSlots = 2;            // batches in flight through clfd_detect_submit / _collect
constexpr int kEagerRects = 1 << 16; // rects copied back with the counters; more cost one extra copy

// One batch in flight through clfd_detect_submit / _collect.  Slot 0's rects are allocated with the detector, the pinned
// ones for rect_cap (clfd_detector_fetch copies through them); slot 1's at its first submit, the pinned ones for kEagerRects.
struct BatchSlot {
    DevBuf<uint8_t> frames;    // gray staging for host input (clfd_detect / clfd_detect_submit)
    DevBuf<uint8_t> color;     // interleaved colour staging of clfd_detect_submit_color, allocated at first use
    DevBuf<DevRect> rects;
    DevRect *h_rects = nullptr;                 // pinned
    unsigned long long *h_counters = nullptr;   // pinned, kCnt per cascade, 16 cascades
    cudaEvent_t done = nullptr;
    int n_frames = 0;
    ~BatchSlot() {
        if (h_rects) cudaFreeHost(h_rects);
        if (h_counters) cudaFreeHost(h_counters);
        if (done) cudaEventDestroy(done);
    }
};

struct clfd_detector {
    clfd_context *ctx = nullptr;
    clfd_detector_config cfg;
    PyramidPlan pyr;
    std::vector<std::unique_ptr<CascadePlan>> cas;
    // the kernels of one cascade for one range of frames (enqueue_range): enqueue_sc_cascade or enqueue_pyramid_cascade
    int (*enqueue_cascade)(clfd_detector *, const CascadePlan &, CascadeArgs &, int, cudaStream_t, cudaEvent_t *, int *) = nullptr;
    DevBuf<QueueItem> queue, queue_b;
    BatchSlot slot[kSlots];
    DevBuf<RocItem> roc;                  // candidates of clfd_detector_reject_levels
    DevBuf<unsigned long long> roc_count;
    long long n_submitted = 0, n_collected = 0;
    unsigned long long rect_cap = 0, queue_cap = 0;
    int last_frames = 0;
    clfd_run_stats stats;
    bool profiling = false;
    cudaEvent_t ev[16] = {nullptr};
    float kernel_ms[8] = {0};
    bool have_events = false;
    bool color_events = false;   // ev[8] / ev[9] bracket the colour conversion of the last batch (kernel_ms[6])
    bool sum_di = false;   // the ystep-2 levels of pyr.sum are column-de-interleaved (PyrLevel::di)
    // clfd_detect pipelines the H2D copy of a batch with its own compute, chunk by chunk
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t copied[kMaxChunks] = {nullptr};
    // chunk overlap (enqueue_overlapped): the HBM-bound pyramid kernels of chunk k+1 run beside the L1-bound tile
    // kernel of chunk k
    cudaStream_t pyr_stream = nullptr, tile_stream[2] = {nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_pyr[kMaxChunks] = {nullptr}, ev_tile[2] = {nullptr, nullptr};
    ~clfd_detector() {
        for (auto &e : ev) if (e) cudaEventDestroy(e);
        for (auto &e : copied) if (e) cudaEventDestroy(e);
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (ev_fork) cudaEventDestroy(ev_fork);
        for (auto &e : ev_pyr) if (e) cudaEventDestroy(e);
        for (auto &e : ev_tile) if (e) cudaEventDestroy(e);
        if (pyr_stream) cudaStreamDestroy(pyr_stream);
        for (auto &t : tile_stream) if (t) cudaStreamDestroy(t);
    }
};

// k_generic_pass for each pass of cp.pass_cuts, ping-ponging between det->queue (counter counters[1], the first pass's
// input if from_queue, else the grid) and det->queue_b (counter d_count_b[slot]).  A counter is cleared before a pass
// writes its queue unless this range has not written that queue yet.  *p: the input of the pass after the chain.
template <class Args>
static int run_pass_chain(const clfd_detector *det, const CascadePlan &cp, const Args &a, int slot, bool from_queue,
                          cudaStream_t s, int *launches, PassArgs *p) {
    QueueItem *const items[2] = {det->queue.p, det->queue_b.p};
    unsigned long long *const count[2] = {cp.d_counters.p + kCnt * slot + 1, cp.d_count_b.p + slot};
    bool written[2] = {from_queue, false};
    memset(p, 0, sizeof *p);
    if (from_queue) { p->in = items[0]; p->in_count = count[0]; }
    for (size_t k = 0, out = from_queue; k + 1 < cp.pass_cuts.size(); k++, out ^= 1) {
        if (written[out]) CK(cudaMemsetAsync(count[out], 0, sizeof(unsigned long long), s));   // holds an older pass
        p->stage_begin = cp.pass_cuts[k]; p->stage_end = cp.pass_cuts[k + 1];
        p->out = items[out]; p->out_count = count[out];
        CK(launch_generic_pass(a, *p, det->ctx->n_sms, s));
        (*launches)++;
        written[out] = true;
        p->in = items[out]; p->in_count = count[out];
    }
    return 0;
}

// ------------------------------------------------------------------------------------
// misc
// ------------------------------------------------------------------------------------
extern "C" {

const char *clfd_last_error(void) { return get_error(); }
const char *clfd_version(void) { return "clfd_b200 0.1 (sm_100a)"; }

int clfd_device_count(int *count) {
    if (!count) INVALID("count is NULL");
    CK(cudaGetDeviceCount(count));
    return 0;
}

int clfd_context_create(int device_index, clfd_context **out) {
    if (!out) INVALID("out is NULL");
    *out = nullptr;
    int n = 0;
    CK(cudaGetDeviceCount(&n));
    if (n <= 0) { set_error("no CUDA device is visible: this library has no CPU fallback"); return CLFD_ERR_CUDA; }
    if (device_index < 0 || device_index >= n) INVALID("device index %d outside 0..%d", device_index, n - 1);
    CK(cudaSetDevice(device_index));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device_index));
    if (prop.major < 10) {
        set_error("device %d (%s) is sm_%d%d; this library is built for sm_100a only", device_index, prop.name,
                  prop.major, prop.minor);
        return CLFD_ERR_CUDA;
    }
    std::unique_ptr<clfd_context> ctx(new clfd_context());
    ctx->device = device_index;
    ctx->n_sms = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    *out = ctx.release();
    return 0;
}

void clfd_context_destroy(clfd_context *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    delete ctx->scratch;
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int clfd_context_device(const clfd_context *ctx) { return ctx ? ctx->device : -1; }
int64_t clfd_context_launch_count(const clfd_context *ctx) { return ctx ? ctx->launches : 0; }
int clfd_context_synchronize(clfd_context *ctx) {
    if (!ctx) INVALID("ctx is NULL");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// ------------------------------------------------------------------------------------
// cascades
// ------------------------------------------------------------------------------------
// a validated HostCascade (hidden cascade built) -> packed device blobs (uploaded per detector, upload_cascade) + its id
static int publish_cascade(std::unique_ptr<clfd_cascade> c, clfd_cascade **out) {
    pack_cascade(c->host, c->packed);
    c->id = g_next_cascade_id.fetch_add(1);
    *out = c.release();
    return 0;
}

int clfd_cascade_load_xml(const char *path, clfd_cascade **out) {
    if (!path || !out) INVALID("NULL argument");
    *out = nullptr;
    std::unique_ptr<clfd_cascade> c(new clfd_cascade());
    int rc = load_cascade_xml(path, c->host);
    if (rc) return rc;
    return publish_cascade(std::move(c), out);
}

int clfd_cascade_from_arrays(int win_w, int win_h, int n_stages, const int *st_ntrees, const float *st_thr,
                             const int *st_parent, const int *st_next, const int *tr_nnodes,
                             const int *nd_tilted, const int *nd_rect, const float *nd_weight,
                             const float *nd_thr, const int *nd_left, const int *nd_right, const float *alpha,
                             clfd_cascade **out) {
    if (!out || !st_ntrees || !st_thr || !st_parent || !st_next || !tr_nnodes || !nd_tilted || !nd_rect ||
        !nd_weight || !nd_thr || !nd_left || !nd_right || !alpha)
        INVALID("NULL argument");
    *out = nullptr;
    if (n_stages <= 0) { set_error("Number of stages should be positive"); return CLFD_ERR_FORMAT; }
    std::unique_ptr<clfd_cascade> c(new clfd_cascade());
    HostCascade &h = c->host;
    h.win_w = win_w; h.win_h = win_h;
    long T = 0, N = 0;
    for (int i = 0; i < n_stages; i++) {
        if (st_ntrees[i] <= 0) { set_error("header of the stage classifier #%d is invalid", i); return CLFD_ERR_FORMAT; }
        T += st_ntrees[i];
    }
    for (long t = 0; t < T; t++) {
        if (tr_nnodes[t] <= 0) { set_error("Tree node is not a valid sequence. (tree %ld)", t); return CLFD_ERR_FORMAT; }
        N += tr_nnodes[t];
    }
    h.st_ntrees.assign(st_ntrees, st_ntrees + n_stages);
    h.st_thr.assign(st_thr, st_thr + n_stages);
    h.st_parent.assign(st_parent, st_parent + n_stages);
    h.st_next.assign(st_next, st_next + n_stages);
    h.tr_nnodes.assign(tr_nnodes, tr_nnodes + T);
    h.nodes.resize(N);
    for (long n = 0; n < N; n++) {
        HostNode &nd = h.nodes[n];
        nd.tilted = nd_tilted[n] != 0;
        for (int k = 0; k < 3; k++) {
            for (int q = 0; q < 4; q++) nd.rect[k][q] = nd_rect[(n * 3 + k) * 4 + q];
            nd.weight[k] = nd_weight[n * 3 + k];
        }
        nd.threshold = nd_thr[n];
        nd.left = nd_left[n]; nd.right = nd_right[n];
    }
    h.alpha.assign(alpha, alpha + N + T);
    int rc = build_hidden(h);
    if (rc) return rc;
    return publish_cascade(std::move(c), out);
}

void clfd_cascade_destroy(clfd_cascade *c) { cascade_release(c); }
uint64_t clfd_cascade_id(const clfd_cascade *c) { return c ? c->id : 0; }

int clfd_cascade_get_info(const clfd_cascade *c, clfd_cascade_info *info) {
    if (!c || !info) INVALID("NULL argument");
    const HostCascade &h = c->host;
    memset(info, 0, sizeof *info);
    info->win_w = h.win_w; info->win_h = h.win_h;
    info->n_stages = h.n_stages(); info->n_trees = h.n_trees(); info->n_nodes = h.n_nodes();
    info->is_tree = h.is_tree; info->is_stump_based = h.is_stump_based; info->has_tilted = h.has_tilted;
    for (int n = 0; n < h.n_nodes(); n++) {
        info->n_tilted_nodes += h.nodes[n].tilted != 0;
        info->n_three_rect_nodes += h.hid_nrects[n] == 3;
    }
    for (int v : h.st_ntrees) info->max_trees_per_stage = std::max(info->max_trees_per_stage, v);
    for (int v : h.tr_nnodes) info->max_nodes_per_tree = std::max(info->max_nodes_per_tree, v);
    info->dense_stages = c->packed.dense[0].exec_stages;
    info->dense_stumps = c->packed.dense_stumps;
    for (int v : h.order_free) info->order_free_stages += v;
    info->packed_bytes = (int)(c->packed.deep_stages.size() * sizeof(DeepStage) + c->packed.deep_nodes.size() * sizeof(DeepNode) +
                               c->packed.tree_first_node.size() * 4 + c->packed.alpha.size() * 4 + sizeof(DenseParams));
    return 0;
}

int clfd_cascade_get_arrays(const clfd_cascade *c, int *st_ntrees, float *st_thr, int *st_parent, int *st_next,
                            int *st_child, int *tr_nnodes, int *nd_tilted, int *nd_rect, float *nd_weight,
                            float *nd_thr, int *nd_left, int *nd_right, float *alpha) {
    if (!c) INVALID("NULL cascade");
    const HostCascade &h = c->host;
    const int S = h.n_stages(), T = h.n_trees(), N = h.n_nodes();
    if (st_ntrees) memcpy(st_ntrees, h.st_ntrees.data(), S * sizeof(int));
    if (st_thr) memcpy(st_thr, h.st_thr.data(), S * sizeof(float));
    if (st_parent) memcpy(st_parent, h.st_parent.data(), S * sizeof(int));
    if (st_next) memcpy(st_next, h.st_next.data(), S * sizeof(int));
    if (st_child) memcpy(st_child, h.st_child.data(), S * sizeof(int));
    if (tr_nnodes) memcpy(tr_nnodes, h.tr_nnodes.data(), T * sizeof(int));
    for (int n = 0; n < N; n++) {
        const HostNode &nd = h.nodes[n];
        if (nd_tilted) nd_tilted[n] = nd.tilted;
        if (nd_rect) memcpy(nd_rect + (size_t)n * 12, nd.rect, 12 * sizeof(int));
        if (nd_weight) memcpy(nd_weight + (size_t)n * 3, nd.weight, 3 * sizeof(float));
        if (nd_thr) nd_thr[n] = nd.threshold;
        if (nd_left) nd_left[n] = nd.left;
        if (nd_right) nd_right[n] = nd.right;
    }
    if (alpha) memcpy(alpha, h.alpha.data(), (size_t)(N + T) * sizeof(float));
    return 0;
}

int clfd_cascade_get_hidden(const clfd_cascade *c, float *node_weights, int *node_nrects, float *stage_thr,
                            int *stage_two_rects) {
    if (!c) INVALID("NULL cascade");
    const HostCascade &h = c->host;
    if (node_weights) memcpy(node_weights, h.hid_weight.data(), h.hid_weight.size() * sizeof(float));
    if (node_nrects) memcpy(node_nrects, h.hid_nrects.data(), h.hid_nrects.size() * sizeof(int));
    if (stage_thr) memcpy(stage_thr, h.hid_thr.data(), h.hid_thr.size() * sizeof(float));
    if (stage_two_rects) memcpy(stage_two_rects, h.two_rects.data(), h.two_rects.size() * sizeof(int));
    return 0;
}

// ------------------------------------------------------------------------------------
// clif: stand-alone integral / resize / gray
// ------------------------------------------------------------------------------------
static int scratch_plan(clfd_context *ctx, int W, int H, int lw, int lh, bool tilt, PyramidPlan **out) {
    PyramidPlan *p = ctx->scratch;
    if (!p || p->W != W || p->H != H || p->levels.size() != 1 || p->levels[0].w != lw || p->levels[0].h != lh ||
        (tilt && !p->want_tilted)) {
        delete ctx->scratch;
        ctx->scratch = nullptr;
        p = new PyramidPlan();
        int rc = p->build(W, H, {{lw, lh}}, 1, tilt, ctx->stream);
        if (rc) { delete p; return rc; }
        ctx->scratch = p;
    }
    *out = p;
    return 0;
}

// k_color_to_gray of n_frames interleaved frames into gray frames of W x H with a 16-byte row pitch, frames pitch * H apart
static ColorArgs color_args(const uint8_t *src, int n_frames, size_t frame_stride, int row_stride, int channels, int W, int H,
                            uint8_t *dst) {
    ColorArgs a;
    a.src = src; a.frame_stride = frame_stride; a.row_stride = row_stride; a.channels = channels;
    a.W = W; a.H = H; a.n_frames = n_frames;
    a.dst = dst; a.dst_pitch = (int)round_up(W, 16); a.dst_frame_stride = (size_t)a.dst_pitch * H;
    return a;
}

// copies a host or device 8-bit image into a fresh device buffer when it lives on the host
struct InputImage {
    const uint8_t *dev = nullptr;
    uint8_t *owned = nullptr;
    int stride = 0;
    ~InputImage() { if (owned) cudaFree(owned); }
    int set(const uint8_t *img, int wbytes, int h, int stride_, int on_device, cudaStream_t s) {
        if (on_device) { dev = img; stride = stride_; return 0; }
        stride = (int)round_up(wbytes, 16);
        CK(cudaMalloc((void **)&owned, (size_t)stride * h + 16));
        CK(cudaMemcpy2DAsync(owned, stride, img, stride_, wbytes, h, cudaMemcpyHostToDevice, s));
        dev = owned;
        return 0;
    }
};

int clfd_integral(clfd_context *ctx, const uint8_t *img, int w, int h, int stride, int img_on_device,
                  int32_t *sum, uint64_t *sqsum, int32_t *tilted, int out_on_device) {
    if (!ctx || !img) INVALID("NULL argument");
    if (w <= 0 || h <= 0 || stride < w) INVALID("bad image geometry %dx%d stride %d", w, h, stride);
    CK(cudaSetDevice(ctx->device));
    PyramidPlan *p = nullptr;
    int rc = scratch_plan(ctx, w, h, w, h, tilted != nullptr, &p);
    if (rc) return rc;
    InputImage in;
    if ((rc = in.set(img, w, h, stride, img_on_device, ctx->stream))) return rc;
    const bool keep_tilt = p->want_tilted;
    p->want_tilted = tilted != nullptr;
    int launches = 0;
    rc = p->run(in.dev, 0, in.stride, 0, 1, ctx->stream, nullptr, &launches);
    p->want_tilted = keep_tilt;
    if (rc) return rc;
    ctx->launches += launches;
    const PyrLevel &L = p->levels[0];
    const cudaMemcpyKind kind = out_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    const size_t W1 = (size_t)w + 1;
    if (sum) CK(cudaMemcpy2DAsync(sum, W1 * 4, p->sum.p + L.sum_off, (size_t)L.sum_pitch * 4, W1 * 4, h + 1, kind, ctx->stream));
    if (sqsum) CK(cudaMemcpy2DAsync(sqsum, W1 * 8, p->sq.p + L.sum_off, (size_t)L.sum_pitch * 8, W1 * 8, h + 1, kind, ctx->stream));
    if (tilted) CK(cudaMemcpy2DAsync(tilted, W1 * 4, p->tilted.p + L.sum_off, (size_t)L.sum_pitch * 4, W1 * 4, h + 1, kind, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int clfd_resize(clfd_context *ctx, const uint8_t *src, int sw, int sh, int sstride, int src_on_device,
                uint8_t *dst, int dw, int dh, int dstride, int dst_on_device) {
    if (!ctx || !src || !dst) INVALID("NULL argument");
    if (sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0 || sstride < sw || dstride < dw) INVALID("bad geometry");
    CK(cudaSetDevice(ctx->device));
    PyramidPlan *p = nullptr;
    int rc = scratch_plan(ctx, sw, sh, dw, dh, false, &p);
    if (rc) return rc;
    InputImage in;
    if ((rc = in.set(src, sw, sh, sstride, src_on_device, ctx->stream))) return rc;
    PyramidArgs a;
    p->fill_args(a, in.dev, 0, in.stride, 1);
    CK(launch_resize_colsum(a, ctx->stream));
    ctx->launches++;
    const PyrLevel &L = p->levels[0];
    CK(cudaMemcpy2DAsync(dst, dstride, p->pyr.p + L.pyr_off, L.pyr_pitch, dw, dh,
                         dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int clfd_bgr_to_gray(clfd_context *ctx, const uint8_t *bgr, int w, int h, int stride, int channels,
                     int src_on_device, uint8_t *gray, int gstride, int dst_on_device) {
    if (!ctx || !bgr || !gray) INVALID("NULL argument");
    if (w <= 0 || h <= 0 || (channels != 3 && channels != 4) || stride < w * channels || gstride < w)
        INVALID("bad geometry");
    CK(cudaSetDevice(ctx->device));
    InputImage in;
    int rc = in.set(bgr, w * channels, h, stride, src_on_device, ctx->stream);
    if (rc) return rc;
    // the kernel writes 16-byte rows (zero padding behind the last pixel): a buffer of that pitch, then the caller's rows
    const int ostride = (int)round_up(w, 16);
    DevBuf<uint8_t> tmp;
    if ((rc = tmp.alloc((size_t)ostride * h))) return rc;
    CK(launch_color_to_gray(color_args(in.dev, 1, 0, in.stride, channels, w, h, tmp.p), ctx->stream));
    ctx->launches++;
    CK(cudaMemcpy2DAsync(gray, gstride, tmp.p, ostride, w, h, dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                         ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// clifGrayscaleIntegral (clif.cpp:318-381) in one call: the interleaved frame goes to the device once, the gray plane is
// made there (and stays there) and feeds the integral kernels; the gray plane comes back only if asked for.
int clfd_integral_image(clfd_context *ctx, const uint8_t *img, int w, int h, int stride, int channels, int32_t *sum,
                        uint64_t *sqsum, int32_t *tilted, uint8_t *gray, int gstride) {
    if (!ctx || !img) INVALID("NULL argument");
    if (channels == 1) {
        if (gray) {
            if (gstride < w) INVALID("bad gray stride");
            for (int y = 0; y < h; y++) memcpy(gray + (size_t)y * gstride, img + (size_t)y * stride, (size_t)w);
        }
        return clfd_integral(ctx, img, w, h, stride, 0, sum, sqsum, tilted, 0);
    }
    if (w <= 0 || h <= 0 || (channels != 3 && channels != 4) || stride < w * channels || (gray && gstride < w))
        INVALID("bad geometry");
    CK(cudaSetDevice(ctx->device));
    InputImage in;
    int rc = in.set(img, w * channels, h, stride, 0, ctx->stream);
    if (rc) return rc;
    DevBuf<uint8_t> g;
    const int dstride = (int)round_up(w, 16);
    if ((rc = g.alloc((size_t)dstride * h + 16))) return rc;
    CK(launch_color_to_gray(color_args(in.dev, 1, 0, in.stride, channels, w, h, g.p), ctx->stream));
    ctx->launches++;
    if (gray) CK(cudaMemcpy2DAsync(gray, gstride, g.p, dstride, w, h, cudaMemcpyDeviceToHost, ctx->stream));
    return clfd_integral(ctx, g.p, w, h, dstride, 1, sum, sqsum, tilted, 0);   // (synchronises the stream before it returns)
}

// ------------------------------------------------------------------------------------
// detector
// ------------------------------------------------------------------------------------
// The exit code of a FLAT window (every pixel equal) depends on the pixel value alone: rect sums are value x area, sigma
// follows from value and area.  The tile kernel looks such windows up instead of walking them through one FP64 fallback
// per stage (kernels_clod.cu, flat_window_code).  The table is MEASURED, not derived: a 16 x 16 board of flat patches, one
// per pixel value and a little larger than the window, goes through a diagnostic detector of the same cascade (want_codes:
// the instantiation that evaluates flat windows like any other) at the unscaled level, and the exit code of the window
// inside patch v is entry v.
static int build_flat_table(clfd_context *ctx, CascadePlan &cp) {
    const HostCascade &hc = cp.cascade->host;
    const DenseParams &P0 = cp.dense[0];
    // only where the tile kernel takes a window all the way (every stock cascade): codes then are final verdicts
    if (!(P0.tail_stages == P0.total_stages || P0.exec_stages > P0.tail_stages) || P0.total_stages <= 0) return 0;
    const int pw = (hc.win_w + 4 + 1) & ~1, ph = (hc.win_h + 4 + 1) & ~1;   // even: patch origins on the step-2 window grid
    clfd_detector_config cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.width = 16 * pw; cfg.height = 16 * ph; cfg.max_batch = 1;
    cfg.scale_factor = 1000.0;   // one level: the frame itself
    cfg.want_codes = 1; cfg.max_rects = 4096; cfg.mode = CLFD_MODE_SCALE_IMAGE;
    clfd_detector *probe = nullptr;
    const clfd_cascade *one = cp.cascade;
    int rc = clfd_detector_create(ctx, &one, 1, &cfg, &probe);
    if (rc) return rc;
    std::unique_ptr<clfd_detector, void (*)(clfd_detector *)> guard(probe, clfd_detector_destroy);
    std::vector<uint8_t> board((size_t)cfg.width * cfg.height);
    for (int y = 0; y < cfg.height; y++)
        for (int x = 0; x < cfg.width; x++) board[(size_t)y * cfg.width + x] = (uint8_t)((y / ph) * 16 + x / pw);
    int64_t n = 0;
    if ((rc = clfd_detect(probe, board.data(), 1, board.size(), cfg.width, nullptr, 0, &n)) && rc != CLFD_ERR_CAPACITY) return rc;
    const CascadePlan &pc = *probe->cas[0];
    if (pc.levels.empty() || pc.levels[0].ystep != 2 || pc.levels[0].win_base != 0) return 0;   // (cannot happen at factor 1)
    std::vector<int16_t> codes((size_t)pc.windows_per_frame);
    if ((rc = clfd_detector_get_codes(probe, 0, codes.data(), (int64_t)codes.size()))) return rc;
    std::vector<int16_t> table(256);
    const int nx = pc.levels[0].nx;
    for (int v = 0; v < 256; v++) {
        const int x = (v % 16) * pw + 2, y = (v / 16) * ph + 2;   // the window [x, x + w) x [y, y + h) lies inside patch v
        table[v] = codes[(size_t)(y / 2) * nx + x / 2];
    }
    if ((rc = cp.d_flat_code.upload(table, ctx->stream))) return rc;
    CK(cudaStreamSynchronize(ctx->stream));
    for (int yi = 0; yi < 2; yi++) cp.dense[yi].flat_code = cp.d_flat_code.p;
    return 0;
}

// A detector's copy of its cascade on the device: the generic kernels' global-memory blob and the tile kernel's
// parameter blobs with this copy's device pointers patched in.
static int upload_cascade(CascadePlan &cp, cudaStream_t s) {
    const PackedCascade &pk = cp.cascade->packed;
    int rc;
    if ((rc = cp.d_stages.upload(pk.deep_stages, s)) || (rc = cp.d_nodes.upload(pk.deep_nodes, s)) ||
        (rc = cp.d_tree_first.upload(pk.tree_first_node, s)) || (rc = cp.d_alpha.upload(pk.alpha, s)))
        return rc;
    for (int yi = 0; yi < 2; yi++) {
        cp.dense[yi] = pk.dense[yi];
        if (!pk.tail[yi].empty() && (rc = cp.d_tail[yi].upload(pk.tail[yi], s))) return rc;
        cp.dense[yi].tail = cp.d_tail[yi].p;
        if (!pk.stage_tab[yi].empty() && (rc = cp.d_stage_tab[yi].upload(pk.stage_tab[yi], s))) return rc;
        cp.dense[yi].stage_g = cp.d_stage_tab[yi].p;
    }
    return 0;
}

// the tile kernel's grid over one level: kTileW x tile_h windows per CTA, tiles numbered from tile_base -> tile count
static int plan_tiles(CasLevel &CL, int tile_h, int tile_base) {
    CL.tiles_x = (CL.nx + kTileW - 1) / kTileW; CL.tiles_y = (CL.ny + tile_h - 1) / tile_h;
    CL.tile_base = tile_base;
    return CL.tiles_x * CL.tiles_y;
}

// Scale-cascade mode, one cascade: its scales over the frame itself (tempcv.cpp:1344-1380) with their ScNode
// tables, the tile-kernel route of the leading scales of window step 2, and the schedule of the survivor passes.
static int plan_sc_cascade(CascadePlan &cp, const clfd_detector_config &cfg, cudaStream_t s) {
    const HostCascade &hc = cp.cascade->host;
    const int W = cfg.width, H = cfg.height, pitch = (int)round_up(W + 1, 8);
    int n_factors = 0;   // tempcv.cpp:1344-1350
    double factor = 1;
    for (; factor * hc.win_w < W - 10 && factor * hc.win_h < H - 10; factor *= cfg.scale_factor) n_factors++;
    factor = 1;
    for (; n_factors-- > 0; factor *= cfg.scale_factor) {   // tempcv.cpp:1361-1380
        const double ystep = std::max(2., factor);
        const int win_w = cv_round(hc.win_w * factor), win_h = cv_round(hc.win_h * factor);
        const int endX = cv_round((W - win_w) / ystep), endY = cv_round((H - win_h) / ystep);
        if (win_w < cfg.min_w || win_h < cfg.min_h) continue;
        if (endX <= 0 || endY <= 0) continue;
        if (cp.sc_levels.size() >= 255) INVALID("more than 255 scales");
        ScLevel L;
        memset(&L, 0, sizeof L);
        L.factor = factor; L.ystep = ystep; L.win_w = win_w; L.win_h = win_h; L.nx = endX; L.ny = endY;
        L.node_base = (int)(cp.sc_levels.size() * hc.n_nodes());
        L.row_base = cp.sc_rows; L.win_base = cp.windows_per_frame;
        cp.sc_rows += endY;
        cp.windows_per_frame += (long long)endX * endY;
        cp.sc_levels.push_back(L);
        clfd_level pl;
        pl.factor = factor; pl.img_w = W; pl.img_h = H; pl.win_w = win_w; pl.win_h = win_h;
        pl.ystep = 0; pl.nx = endX; pl.ny = endY; pl.win_base = L.win_base;
        cp.pub_levels.push_back(pl);
    }
    std::vector<ScNode> nodes(cp.sc_levels.size() * (size_t)hc.n_nodes());
    for (size_t li = 0; li < cp.sc_levels.size(); li++)
        pack_sc_level(hc, cp.sc_levels[li].factor, pitch, cp.sc_levels[li], nodes.data() + li * hc.n_nodes());
    int rc;
    if ((rc = cp.d_sc_levels.upload(cp.sc_levels, s)) || (rc = cp.d_sc_nodes.upload(nodes, s))) return rc;
    CK(cudaStreamSynchronize(s));   // `nodes` goes out of scope
    // the leading scales whose window step is exactly 2 (factor <= 2): tile kernel
    int tile_base = 0;
    for (size_t li = 0; li < cp.sc_levels.size(); li++) {
        const ScLevel &L = cp.sc_levels[li];
        if (L.ystep != 2.0 || L.win_base != cp.sc_tile_windows) break;
        std::unique_ptr<CascadePlan::ScTile> t(new CascadePlan::ScTile);
        std::vector<TailStump> tail;
        std::vector<DenseStage> stab;
        if (!pack_sc_dense(hc, L.factor, t->P, tail, stab)) break;
        if ((rc = t->tail.upload(tail, s)) || (!stab.empty() && (rc = t->stage_tab.upload(stab, s)))) return rc;
        CK(cudaStreamSynchronize(s));
        t->P.tail = t->tail.p; t->P.stage_g = t->stage_tab.p;
        CasLevel CL;
        memset(&CL, 0, sizeof CL);
        CL.pyr_level = 0; CL.nx = L.nx; CL.ny = L.ny; CL.ystep = 2; CL.win_w = L.win_w; CL.win_h = L.win_h;
        CL.win_base = L.win_base; CL.factor = L.factor;
        t->tile_base = tile_base; t->n_tiles = plan_tiles(CL, t->P.tile_h, tile_base);
        tile_base += t->n_tiles;
        cp.levels.push_back(CL);
        cp.sc_tiles.push_back(std::move(t));
        cp.sc_tile_windows = L.win_base + (long long)L.nx * L.ny;
    }
    cp.bytes_cascade += (int64_t)(W + 1) * (H + 1) * (4 + 8 + (hc.has_tilted ? 4 : 0)) + nodes.size() * sizeof(ScNode);
    // k_generic_pass passes over growing stage ranges (cumulative trees >= 10, 40, 90, 160, ... per pass), survivors
    // re-compacted through the two queues in between; a stage tree runs as one pass.  From the first stage after stage 0
    // that has >= 50 trees on, the survivors are finished one warp per position (k_generic_deep).
    static const int limit[7] = {10, 40, 90, 160, 300, 500, 800};
    cp.pass_cuts.assign(1, 0);
    cp.sc_deep_from = hc.n_stages();
    for (int st = 0, acc = 0; st < hc.n_stages() && !hc.is_tree; st++) {
        if (st > 0 && hc.st_ntrees[st] >= 50) { cp.sc_deep_from = st; break; }
        acc += hc.st_ntrees[st];
        if (cp.pass_cuts.size() <= 7 && acc >= limit[cp.pass_cuts.size() - 1] && st + 1 < hc.n_stages()) { cp.pass_cuts.push_back(st + 1); acc = 0; }
    }
    if (cp.pass_cuts.back() != cp.sc_deep_from) cp.pass_cuts.push_back(cp.sc_deep_from);
    return 0;
}

// Scale-cascade mode, one cascade: the tile kernel over the step-2 scales (exit codes only), the k_generic_pass
// passes, k_generic_deep and k_sc_rows.  ev (cascade 0, profiling): ev[5] before the first kernel, ev[6] and ev[7] after the last.
static int enqueue_sc_cascade(clfd_detector *det, const CascadePlan &cp, CascadeArgs &a, int slot, cudaStream_t s,
                              cudaEvent_t *ev, int *launches) {
    const int n_stages = cp.cascade->host.n_stages();
    ScArgs sa;
    memset(&sa, 0, sizeof sa);
    static_cast<CascadeArgs &>(sa) = a;
    const PyrLevel &L0 = det->pyr.levels[0];
    sa.sum = a.sum + L0.sum_off; sa.sq = a.sq + L0.sum_off; sa.tilted = a.tilted ? a.tilted + L0.sum_off : nullptr;
    sa.codes = cp.d_codes.p + (size_t)a.frame_base * cp.windows_per_frame;
    sa.pitch = L0.sum_pitch; sa.W = det->cfg.width; sa.H = det->cfg.height;
    sa.scales = cp.d_sc_levels.p; sa.nodes = cp.d_sc_nodes.p;
    sa.n_scales = (int)cp.sc_levels.size(); sa.rows_per_frame = cp.sc_rows;
    sa.first_window = cp.sc_tile_windows;
    if (ev) CK(cudaEventRecord(ev[5], s));
    CascadeArgs ta = a;   // the tile kernel, one launch per scale of window step 2
    ta.codes = sa.codes; ta.rects = nullptr; ta.rect_cap = 0;
    for (auto &t : cp.sc_tiles) { CK(launch_cascade_tiles(t->P, ta, t->tile_base, t->n_tiles, s)); (*launches)++; }
    PassArgs p;
    if (int rc = run_pass_chain(det, cp, sa, slot, false, s, launches, &p)) return rc;
    if (cp.sc_deep_from < n_stages) {
        p.stage_begin = cp.sc_deep_from; p.stage_end = n_stages;
        CK(launch_generic_deep(sa, p, det->ctx->n_sms, s)); (*launches)++;
    }
    CK(launch_sc_rows(sa, s)); (*launches)++;
    if (ev) { CK(cudaEventRecord(ev[6], s)); CK(cudaEventRecord(ev[7], s)); }
    return 0;
}

// Image-pyramid mode: the level loop, all cascades in lock step over the shared factor sequence.  sizes: the union
// pyramid; sizes_y2: whether a level's windows are 2 pixels apart (factor <= 2).
static int plan_pyramid_levels(clfd_detector *det, std::vector<std::pair<int, int>> &sizes, std::vector<char> &sizes_y2) {
    const clfd_detector_config &cfg = det->cfg;
    const int W = cfg.width, H = cfg.height;
    int max_w = cfg.max_w, max_h = cfg.max_h;
    if (max_h == 0 || max_w == 0) { max_h = H; max_w = W; }   // tempcv.cpp:1230-1234
    std::map<int, int> pyr_index;                    // factor index -> pyramid level
    std::vector<bool> done(det->cas.size(), false);
    double factor = 1;
    for (int k = 0;; k++, factor *= cfg.scale_factor) {
        bool all_done = true;
        if (k >= 255) INVALID("more than 255 pyramid levels");
        const int sz_w = cv_round(W / factor), sz_h = cv_round(H / factor);
        for (size_t ci = 0; ci < det->cas.size(); ci++) {
            if (done[ci]) continue;
            CascadePlan &cp = *det->cas[ci];
            const HostCascade &hc = cp.cascade->host;
            const int win_w = cv_round(hc.win_w * factor), win_h = cv_round(hc.win_h * factor);
            const int sz1_w = sz_w - hc.win_w + 1, sz1_h = sz_h - hc.win_h + 1;
            if (sz1_w <= 0 || sz1_h <= 0) { done[ci] = true; continue; }                 // :1283
            if (win_w > max_w || win_h > max_h) { done[ci] = true; continue; }           // :1285
            all_done = false;
            if (win_w < cfg.min_w || win_h < cfg.min_h) continue;                        // :1287
            const int ystep = factor > 2 ? 1 : 2;                                        // :1021
            const int xe = sz_w - hc.win_w, ye = sz_h - hc.win_h;                        // :1015-1020
            const int nx = xe > 0 ? (xe + ystep - 1) / ystep : 0, ny = ye > 0 ? (ye + ystep - 1) / ystep : 0;
            if (nx == 0 || ny == 0) continue;
            if (!pyr_index.count(k)) { pyr_index[k] = (int)sizes.size(); sizes.push_back({sz_w, sz_h}); sizes_y2.push_back(ystep == 2); }
            CasLevel CL;
            memset(&CL, 0, sizeof CL);
            CL.pyr_level = pyr_index[k];
            CL.nx = nx; CL.ny = ny; CL.ystep = ystep; CL.win_w = win_w; CL.win_h = win_h;
            const int tile_h = cp.cascade->packed.dense[ystep - 1].tile_h > 0 ? cp.cascade->packed.dense[ystep - 1].tile_h : kTileH;
            CL.win_base = cp.windows_per_frame; CL.factor = factor;
            cp.n_tiles += plan_tiles(CL, tile_h, cp.n_tiles);
            if (ystep == 2) cp.n_tiles_y2 = cp.n_tiles;
            cp.windows_per_frame += (long long)nx * ny;
            cp.bytes_cascade += (int64_t)(sz_w + 1) * (sz_h + 1) * (4 + 8 + (hc.has_tilted ? 4 : 0));
            if (cp.levels.size() >= 255) INVALID("more than 255 levels");
            cp.levels.push_back(CL);
            clfd_level pl;
            pl.factor = factor; pl.img_w = sz_w; pl.img_h = sz_h; pl.win_w = win_w; pl.win_h = win_h;
            pl.ystep = ystep; pl.nx = nx; pl.ny = ny; pl.win_base = CL.win_base;
            cp.pub_levels.push_back(pl);
        }
        if (all_done) break;
    }
    return 0;
}

// Image-pyramid mode, k_generic_pass: the stages right after the tile prefix of a LINEAR cascade whose trees the tile
// kernel cannot take, while they are too small for a warp per window (< 24 trees), at most 8.  Passes: the first ends
// once it holds >= 10 trees, the later ones >= 30 (lanes are re-compacted between passes).
static void plan_mid_passes(CascadePlan &cp) {
    const HostCascade &hc = cp.cascade->host;
    const DenseParams &P0 = cp.cascade->packed.dense[0];
    if (hc.is_tree || P0.tail_stages >= P0.total_stages) return;
    cp.mid_begin = cp.mid_end = P0.tail_stages;
    while (cp.mid_end < hc.n_stages() && cp.mid_end - cp.mid_begin < 8 && hc.st_ntrees[cp.mid_end] < 24) cp.mid_end++;
    cp.pass_cuts.assign(1, cp.mid_begin);
    for (int st = cp.mid_begin, acc = 0; st < cp.mid_end; st++) {
        acc += hc.st_ntrees[st];
        if (acc >= (cp.pass_cuts.size() == 1 ? 10 : 30) || st + 1 == cp.mid_end) { cp.pass_cuts.push_back(st + 1); acc = 0; }
    }
}

// Image-pyramid mode, one cascade: the tile kernel, the k_generic_pass passes and k_generic_deep.  ev (cascade
// 0, profiling): ev[5] before the first kernel, ev[6] after the tile kernel, ev[7] after the last.
static int enqueue_pyramid_cascade(clfd_detector *det, const CascadePlan &cp, CascadeArgs &a, int slot, cudaStream_t s,
                                   cudaEvent_t *ev, int *launches) {
    const DenseParams &P0 = cp.cascade->packed.dense[0];
    if (ev) CK(cudaEventRecord(ev[5], s));
    if (P0.tail_stages > 0) {
        // ystep-2 levels (de-interleaved tile layout) and ystep-1 levels (natural layout)
        if (cp.n_tiles_y2 > 0) { CK(launch_cascade_tiles(cp.dense[1], a, 0, cp.n_tiles_y2, s)); (*launches)++; }
        if (cp.n_tiles > cp.n_tiles_y2) {
            CK(launch_cascade_tiles(cp.dense[0], a, cp.n_tiles_y2, cp.n_tiles - cp.n_tiles_y2, s));
            (*launches)++;
        }
    }
    if (ev) CK(cudaEventRecord(ev[6], s));
    // cascades the tile kernel finishes itself (tail_stages == total_stages) never fill the queue
    const bool tiles_finish = P0.tail_stages > 0 && P0.exec_stages == P0.total_stages;
    if (!tiles_finish) {
        // without a tile prefix, the first pass (or the deep kernel) walks the window grid itself
        PassArgs p;
        if (int rc = run_pass_chain(det, cp, a, slot, P0.tail_stages > 0, s, launches, &p)) return rc;
        if (cp.mid_end < P0.total_stages) {
            p.stage_begin = cp.mid_end; p.stage_end = P0.total_stages;   // (queue items carry their first stage)
            CK(launch_generic_deep(a, p, det->ctx->n_sms, s)); (*launches)++;
        }
    }
    if (ev) CK(cudaEventRecord(ev[7], s));
    return 0;
}

int clfd_detector_create(clfd_context *ctx, const clfd_cascade *const *cascades, int n_cascades,
                         const clfd_detector_config *cfg, clfd_detector **out) {
    if (!ctx || !cascades || !cfg || !out) INVALID("NULL argument");
    *out = nullptr;
    if (n_cascades <= 0 || n_cascades > 16) INVALID("n_cascades %d outside 1..16", n_cascades);
    if (cfg->width <= 0 || cfg->height <= 0 || cfg->max_batch <= 0 || cfg->max_batch > 65535)
        INVALID("bad frame geometry / batch");
    if (!(cfg->scale_factor > 1)) INVALID("scale factor must be > 1");   // tempcv.cpp:1224-1225
    if (cfg->width > 65535 || cfg->height > 65535) INVALID("frame too large");
    CK(cudaSetDevice(ctx->device));
    std::unique_ptr<clfd_detector> det(new clfd_detector());
    det->ctx = ctx; det->cfg = *cfg;
    memset(&det->stats, 0, sizeof det->stats);
    const int W = cfg->width, H = cfg->height;

    if (cfg->mode != CLFD_MODE_SCALE_IMAGE && cfg->mode != CLFD_MODE_SCALE_CASCADE) INVALID("unknown mode %d", cfg->mode);
    const bool scale_cascade = cfg->mode == CLFD_MODE_SCALE_CASCADE;
    bool any_tilted = false;
    for (int ci = 0; ci < n_cascades; ci++) {
        if (!cascades[ci]) INVALID("cascade %d is NULL", ci);
        // the image-pyramid kernels keep a window's corner offsets in bytes (DeepNode) and its squared integral modulo
        // 2^32, exact while (w - 2)(h - 2) * 255^2 < 2^32; the scale-cascade mode has neither limit
        const HostCascade &hc = cascades[ci]->host;
        if (!scale_cascade && (hc.win_w > kMaxPyramidWindow || hc.win_h > kMaxPyramidWindow))
            INVALID("cascade %d: window %dx%d is larger than %d pixels, the limit of the image-pyramid mode (the "
                    "scale-cascade mode takes it)", ci, hc.win_w, hc.win_h, kMaxPyramidWindow);
        det->cas.emplace_back(new CascadePlan());
        det->cas.back()->cascade = cascades[ci];
        const_cast<clfd_cascade *>(cascades[ci])->refs.fetch_add(1);   // released by ~CascadePlan
        any_tilted |= cascades[ci]->host.has_tilted;
    }
    cudaStream_t s = ctx->stream;
    int rc = 0;
    std::vector<std::pair<int, int>> sizes;          // union pyramid
    std::vector<char> sizes_y2;                      // ... and whether a level's windows are 2 pixels apart (factor <= 2)
    if (scale_cascade) {
        // one "pyramid level": the frame itself (a same-size INTER_LINEAR resize is the identity)
        sizes.push_back({W, H});
        for (auto &cpp : det->cas)
            if ((rc = plan_sc_cascade(*cpp, *cfg, s))) return rc;
    } else {
        if ((rc = plan_pyramid_levels(det.get(), sizes, sizes_y2))) return rc;
        for (auto &cpp : det->cas) plan_mid_passes(*cpp);
    }
    det->enqueue_cascade = scale_cascade ? enqueue_sc_cascade : enqueue_pyramid_cascade;
    // pyramid mode: every sum of squares the kernels form is a cascade window's (< 2^32), so the squared integral is
    // kept modulo 2^32 -- a third less integral traffic; the scale-cascade mode's windows grow with the scale: 64 bits
    det->pyr.sq32 = !scale_cascade && !getenv("CLFD_SQ64");
    // pyramid mode: the int32 integral of the ystep-2 levels is written column-de-interleaved -- the layout their tiles have
    // in shared memory -- so that the tile kernel stages a tile row with two TMA bulk copies instead of LDG.128 + 2 x STS.64
    // through the L1 data pipe it is bound by; the generic kernels (mid / deep / reject levels) address it through PyrLevel::di
    det->sum_di = !scale_cascade && !getenv("CLFD_NO_DI");
    if (det->sum_di) det->pyr.di_levels = sizes_y2;
    if (!sizes.empty() && (rc = det->pyr.build(W, H, sizes, cfg->max_batch, any_tilted, s))) return rc;
    else if (sizes.empty()) { det->pyr.W = W; det->pyr.H = H; det->pyr.max_batch = cfg->max_batch; }

    long long max_wpf = 0;
    bool need_queue_b = scale_cascade;
    for (auto &cpp : det->cas) {
        CascadePlan &cp = *cpp;
        if ((rc = cp.d_levels.upload(cp.levels, s)) || (rc = upload_cascade(cp, s))) return rc;
        if ((rc = cp.d_counters.alloc(kCnt * kSlots)) || (rc = cp.d_count_b.alloc(kSlots))) return rc;
        need_queue_b |= cp.mid_end > cp.mid_begin;
        if ((cfg->want_codes || scale_cascade) && (rc = cp.d_codes.alloc((size_t)std::max<long long>(cp.windows_per_frame, 1) * cfg->max_batch)))
            return rc;
        max_wpf = std::max(max_wpf, cp.windows_per_frame);
        cp.bytes_cascade += cp.cascade->packed.deep_nodes.size() * sizeof(DeepNode);
    }
    det->queue_cap = (unsigned long long)std::max<long long>(max_wpf, 1) * cfg->max_batch;
    det->rect_cap = cfg->max_rects > 0 ? (unsigned long long)cfg->max_rects : (1ull << 20);
    if ((rc = det->queue.alloc(det->queue_cap)) || (rc = det->slot[0].rects.alloc(det->rect_cap))) return rc;
    if (need_queue_b && (rc = det->queue_b.alloc(det->queue_cap))) return rc;
    CK(cudaMallocHost((void **)&det->slot[0].h_rects, det->rect_cap * sizeof(DevRect)));
    for (auto &sl : det->slot) CK(cudaMallocHost((void **)&sl.h_counters, kCnt * 16 * sizeof(unsigned long long)));
    CK(cudaStreamSynchronize(s));
    det->stats.pyramid_pixels = det->pyr.pyramid_pixels;
    det->stats.bytes_resize = det->pyr.bytes_resize;
    det->stats.bytes_integral = det->pyr.bytes_integral;
    det->stats.bytes_tilted = det->pyr.bytes_tilted;
    for (auto &cpp : det->cas) det->stats.bytes_cascade += cpp->bytes_cascade;
    // production detectors of the pyramid mode look flat windows up (the diagnostic ones, want_codes, measure the table)
    if (!scale_cascade && !cfg->want_codes && !getenv("CLFD_NO_FLAT_TABLE"))
        for (auto &cpp : det->cas)
            if ((rc = build_flat_table(ctx, *cpp))) return rc;
    *out = det.release();
    return 0;
}

void clfd_detector_destroy(clfd_detector *det) {
    if (!det) return;
    cudaSetDevice(det->ctx->device);
    cudaDeviceSynchronize();
    delete det;
}

int clfd_detector_num_levels(const clfd_detector *det, int cascade) {
    if (!det || cascade < 0 || cascade >= (int)det->cas.size()) return CLFD_ERR_INVALID;
    return (int)det->cas[cascade]->pub_levels.size();
}

int clfd_detector_get_levels(const clfd_detector *det, int cascade, clfd_level *levels, int max_levels) {
    if (!det || !levels || cascade < 0 || cascade >= (int)det->cas.size()) INVALID("bad argument");
    const auto &v = det->cas[cascade]->pub_levels;
    if ((int)v.size() > max_levels) { set_error("need room for %zu levels", v.size()); return CLFD_ERR_CAPACITY; }
    memcpy(levels, v.data(), v.size() * sizeof(clfd_level));
    return (int)v.size();
}

int64_t clfd_detector_windows_per_frame(const clfd_detector *det, int cascade) {
    if (!det || cascade < 0 || cascade >= (int)det->cas.size()) return CLFD_ERR_INVALID;
    return det->cas[cascade]->windows_per_frame;
}

int clfd_detector_set_profiling(clfd_detector *det, int enable) {
    if (!det) INVALID("NULL detector");
    CK(cudaSetDevice(det->ctx->device));
    det->profiling = enable != 0;
    if (det->profiling)
        for (auto &e : det->ev)
            if (!e) CK(cudaEventCreate(&e));
    return 0;
}

// What every cascade kernel reads for frames [frame_base, frame_base + n_frames): the detector's integral images
// (pre-offset to frame_base), the cascade's level table and its global-memory blob.
static CascadeArgs cascade_args(const clfd_detector *det, const CascadePlan &cp, int ci, int frame_base, int n_frames) {
    const PyramidPlan &pyr = det->pyr;
    const HostCascade &hc = cp.cascade->host;
    const size_t fo = (size_t)frame_base * pyr.sum_frame_stride;
    CascadeArgs a;
    memset(&a, 0, sizeof a);
    a.sum = pyr.sum.p + fo; a.sq = sq_at(pyr.sq.p, fo, pyr.sq32); a.sq32 = pyr.sq32 ? 1 : 0;
    a.tilted = pyr.want_tilted ? pyr.tilted.p + fo : nullptr;
    a.sum_frame_stride = pyr.sum_frame_stride;
    a.sum_di = det->sum_di ? 1 : 0;
    a.levels = pyr.d_levels.p; a.cas_levels = cp.d_levels.p;
    a.n_cas_levels = (int)cp.levels.size(); a.n_tiles = cp.n_tiles; a.n_frames = n_frames;
    a.frame_base = frame_base;
    a.cascade_index = ci; a.windows_per_frame = cp.windows_per_frame;
    a.deep.stages = cp.d_stages.p; a.deep.tree_first_node = cp.d_tree_first.p;
    a.deep.nodes = cp.d_nodes.p; a.deep.alpha = cp.d_alpha.p;
    a.deep.n_stages = hc.n_stages(); a.deep.is_tree = hc.is_tree; a.deep.has_tilted = hc.has_tilted;
    a.deep.win_w = hc.win_w; a.deep.win_h = hc.win_h;
    a.deep.inv_area = cp.cascade->packed.dense[0].inv_area;
    return a;
}

// Enqueue every kernel for frames [frame_base, frame_base + n_frames) of the current batch.
// `first` resets the batch's rect / overflow counters; the kernels see frame numbers relative
// to the range (the per-frame buffers are passed pre-offset) and add frame_base to the frame
// index of the rects they emit.
// parts: which halves of the range's work go onto stream s (enqueue_overlapped puts them on different streams)
enum { kPartPyramid = 1, kPartCascades = 2, kPartCounters = 4, kPartAll = 7 };
static int enqueue_range(clfd_detector *det, const uint8_t *frames_dev, int frame_base, int n_frames, size_t frame_stride,
                         int row_stride, cudaStream_t s, bool first, int *n_launches, int slot = 0, int parts = kPartAll) {
    clfd_context *ctx = det->ctx;
    int launches = 0;
    cudaEvent_t *ev = det->profiling ? det->ev : nullptr;
    if (!det->pyr.levels.empty() && (parts & kPartPyramid)) {
        int rc = det->pyr.run(frames_dev, frame_stride, row_stride, frame_base, n_frames, s, ev, &launches);
        if (rc) return rc;
    }
    if (parts & kPartCounters)
        for (auto &cpp : det->cas) {
            if (first) CK(cudaMemsetAsync(cpp->d_counters.p + kCnt * slot, 0, kCnt * sizeof(unsigned long long), s));
            else CK(cudaMemsetAsync(cpp->d_counters.p + kCnt * slot + 1, 0, sizeof(unsigned long long), s));   // the queue is per range
            CK(cudaMemsetAsync(cpp->d_count_b.p + slot, 0, sizeof(unsigned long long), s));
        }
    if (parts & kPartCascades) {
        for (size_t ci = 0; ci < det->cas.size(); ci++) {
            const CascadePlan &cp = *det->cas[ci];
            if (cp.windows_per_frame > 0) {
                CascadeArgs a = cascade_args(det, cp, (int)ci, frame_base, n_frames);
                a.codes = det->cfg.want_codes ? cp.d_codes.p + (size_t)frame_base * cp.windows_per_frame : nullptr;
                a.count_exact = det->cfg.want_codes ? 1 : 0;
                a.queue = det->queue.p; a.queue_cap = det->queue_cap;
                a.rects = det->slot[slot].rects.p; a.rect_cap = det->rect_cap;
                a.counters = cp.d_counters.p + kCnt * slot;
                int rc = det->enqueue_cascade(det, cp, a, slot, s, ci == 0 ? ev : nullptr, &launches);
                if (rc) return rc;
            }
            // all cascades append to one rect buffer: carry the rect count over
            if (ci + 1 < det->cas.size())
                CK(cudaMemcpyAsync(det->cas[ci + 1]->d_counters.p + kCnt * slot, cp.d_counters.p + kCnt * slot, sizeof(unsigned long long),
                                   cudaMemcpyDeviceToDevice, s));
        }
        det->have_events = ev != nullptr;
    }
    ctx->launches += launches;
    *n_launches += launches;
    return 0;
}

// Chunk overlap.  The pyramid kernels are HBM-bound and the tile kernel is bound by the SMs' L1 data pipe, so they
// overlap well: the batch is cut into chunks, the pyramid of chunk k+1 runs on a high-priority stream while the tile
// kernel of chunk k runs (the per-frame buffers of different chunks are disjoint), and the tile launches of consecutive
// chunks alternate between two streams so that one chunk's last wave overlaps the next chunk's first.  Forked from and
// joined back into the caller's stream s.  Only for detectors whose (single) cascade the tile kernel finishes itself
// (no survivor queue, no counter hand-over between cascades); profiling runs keep the serial order so that the
// per-kernel event times mean something.  copied: per-chunk events of the host-to-device copies, or nullptr.
static bool overlap_applies(const clfd_detector *det, int n_frames) {
    if (det->profiling || det->cfg.mode == CLFD_MODE_SCALE_CASCADE || det->pyr.levels.empty() || det->cas.size() != 1) return false;
    if (n_frames < 8 || getenv("CLFD_NO_OVERLAP")) return false;
    const CascadePlan &cp = *det->cas[0];
    const PackedCascade &pk = cp.cascade->packed;
    return cp.windows_per_frame > 0 && pk.dense[0].tail_stages > 0 && pk.dense[0].exec_stages == pk.dense[0].total_stages;
}
static int overlap_chunks(int n_frames) {
    int n = n_frames >= 32 ? 8 : 4;
    if (const char *e = getenv("CLFD_OVERLAP_CHUNKS")) n = atoi(e);
    return std::max(1, std::min({n, kMaxChunks, n_frames}));
}
static int overlap_setup(clfd_detector *det) {
    if (det->pyr_stream) return 0;
    int lo = 0, hi = 0;
    CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));   // hi: the numerically lowest value = the highest priority
    CK(cudaStreamCreateWithPriority(&det->pyr_stream, cudaStreamNonBlocking, hi));
    for (auto &t : det->tile_stream) CK(cudaStreamCreateWithPriority(&t, cudaStreamNonBlocking, lo));
    CK(cudaEventCreateWithFlags(&det->ev_fork, cudaEventDisableTiming));
    for (auto &e : det->ev_pyr) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto &e : det->ev_tile) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    return 0;
}
static int enqueue_overlapped(clfd_detector *det, const uint8_t *frames_dev, int n_frames, size_t frame_stride, int row_stride,
                              cudaStream_t s, int n_chunks, const cudaEvent_t *copied, int *n_launches, int slot) {
    int rc = overlap_setup(det);
    if (rc) return rc;
    rc = enqueue_range(det, frames_dev, 0, n_frames, frame_stride, row_stride, s, true, n_launches, slot, kPartCounters);
    if (rc) return rc;
    CK(cudaEventRecord(det->ev_fork, s));
    CK(cudaStreamWaitEvent(det->pyr_stream, det->ev_fork, 0));
    for (auto &t : det->tile_stream) CK(cudaStreamWaitEvent(t, det->ev_fork, 0));
    for (int k = 0; k < n_chunks; k++) {
        const int f0 = (int)((long long)n_frames * k / n_chunks), f1 = (int)((long long)n_frames * (k + 1) / n_chunks);
        if (f1 <= f0) continue;
        const uint8_t *src = frames_dev + (size_t)f0 * frame_stride;
        if (copied) CK(cudaStreamWaitEvent(det->pyr_stream, copied[k], 0));
        rc = enqueue_range(det, src, f0, f1 - f0, frame_stride, row_stride, det->pyr_stream, false, n_launches, slot, kPartPyramid);
        if (rc) return rc;
        CK(cudaEventRecord(det->ev_pyr[k], det->pyr_stream));
        cudaStream_t t = det->tile_stream[k & 1];
        CK(cudaStreamWaitEvent(t, det->ev_pyr[k], 0));
        rc = enqueue_range(det, src, f0, f1 - f0, frame_stride, row_stride, t, false, n_launches, slot, kPartCascades);
        if (rc) return rc;
    }
    for (int i = 0; i < 2; i++) {
        CK(cudaEventRecord(det->ev_tile[i], det->tile_stream[i]));
        CK(cudaStreamWaitEvent(s, det->ev_tile[i], 0));
    }
    return 0;
}

int clfd_detector_enqueue(clfd_detector *det, const uint8_t *frames_dev, int n_frames, size_t frame_stride,
                          int row_stride, void *cuda_stream) {
    if (!det || !frames_dev) INVALID("NULL argument");
    clfd_context *ctx = det->ctx;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    if (n_frames <= 0 || n_frames > det->cfg.max_batch) INVALID("n_frames %d outside 1..%d", n_frames, det->cfg.max_batch);
    det->last_frames = n_frames;
    int launches = 0;
    int rc = overlap_applies(det, n_frames)
                 ? enqueue_overlapped(det, frames_dev, n_frames, frame_stride, row_stride, s, overlap_chunks(n_frames), nullptr, &launches, 0)
                 : enqueue_range(det, frames_dev, 0, n_frames, frame_stride, row_stride, s, true, &launches);
    if (rc) return rc;
    det->stats.kernel_launches = launches;
    det->color_events = false;
    return 0;
}

// What the colour entry points accept besides channels == 1 (which they hand to the gray calls).
static int check_color_batch(const clfd_detector *det, int n_frames, int channels, int row_stride) {
    if (channels != 3 && channels != 4) INVALID("channels %d: must be 1 (gray), 3 (BGR) or 4 (BGRA)", channels);
    if (n_frames <= 0 || n_frames > det->cfg.max_batch) INVALID("n_frames %d outside 1..%d", n_frames, det->cfg.max_batch);
    if ((long long)row_stride < (long long)det->cfg.width * channels)
        INVALID("row stride %d smaller than %d pixels of %d channels", row_stride, det->cfg.width, channels);
    return 0;
}

// Colour -> gray of a batch into the detector's gray frame layout (16-byte row pitch) on stream s.  With profiling on,
// ev[8] / ev[9] bracket the conversion (clfd_detector_get_kernel_ms [6]).
static int enqueue_color_to_gray(clfd_detector *det, const uint8_t *src, int n_frames, int channels, size_t frame_stride,
                                 int row_stride, uint8_t *dst, cudaStream_t s) {
    if (det->profiling) CK(cudaEventRecord(det->ev[8], s));
    CK(launch_color_to_gray(color_args(src, n_frames, frame_stride, row_stride, channels, det->cfg.width, det->cfg.height, dst), s));
    if (det->profiling) CK(cudaEventRecord(det->ev[9], s));
    det->ctx->launches++;
    return 0;
}

int clfd_detector_enqueue_color(clfd_detector *det, const uint8_t *frames_dev, int n_frames, int channels,
                                size_t frame_stride, int row_stride, void *cuda_stream) {
    if (!det || !frames_dev) INVALID("NULL argument");
    if (channels == 1) return clfd_detector_enqueue(det, frames_dev, n_frames, frame_stride, row_stride, cuda_stream);
    int rc = check_color_batch(det, n_frames, channels, row_stride);
    if (rc) return rc;
    if (det->n_submitted != det->n_collected)
        INVALID("clfd_detector_enqueue_color while submitted batches are in flight (they may still read its frame buffer)");
    clfd_context *ctx = det->ctx;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    const size_t dstride = round_up(det->cfg.width, 16), dframe = dstride * det->cfg.height;
    if (!det->slot[0].frames.p && (rc = det->slot[0].frames.alloc(dframe * det->cfg.max_batch + 64))) return rc;
    if ((rc = enqueue_color_to_gray(det, frames_dev, n_frames, channels, frame_stride, row_stride, det->slot[0].frames.p, s))) return rc;
    if ((rc = clfd_detector_enqueue(det, det->slot[0].frames.p, n_frames, dframe, (int)dstride, cuda_stream))) return rc;
    det->stats.kernel_launches += 1;
    det->color_events = det->profiling;
    return 0;
}

// The device counters of one finished batch (kCnt per cascade at hc, copied back) -> det->stats and the rect count;
// fails on a survivor-queue or rect-buffer overflow.
static int take_counters(clfd_detector *det, const unsigned long long *hc, int n_frames, int64_t *n_rects) {
    const int nc = (int)det->cas.size();
    const unsigned long long total = hc[kCnt * (nc - 1)];   // all cascades append to one rect buffer
    unsigned long long deep = 0, rect_over = 0, queue_over = 0;
    for (int ci = 0; ci < nc; ci++) {
        deep += hc[kCnt * ci + 1];
        rect_over += hc[kCnt * ci + 2];
        queue_over += hc[kCnt * ci + 3];
    }
    if (queue_over) { set_error("survivor queue overflow (%llu windows dropped)", queue_over); return CLFD_ERR_CAPACITY; }
    det->stats.rects = (int64_t)total;
    det->stats.deep_windows = (int64_t)deep;
    det->stats.exact_stage_evals = det->stats.near_threshold_events = det->cfg.want_codes ? 0 : -1;   // -1: not counted
    for (int ci = 0; ci < nc && det->cfg.want_codes; ci++) {
        det->stats.exact_stage_evals += (int64_t)hc[kCnt * ci + 4];
        det->stats.near_threshold_events += (int64_t)hc[kCnt * ci + 5];
    }
#ifdef CLFD_TILE_TIMING   // diagnostic build: the tile kernel's warp-slot accounting in place of the three counters
    det->stats.exact_stage_evals = (int64_t)hc[4];
    det->stats.near_threshold_events = (int64_t)hc[5];
    det->stats.deep_windows = (int64_t)hc[6];
#endif
    det->stats.windows = 0;
    for (auto &cpp : det->cas) det->stats.windows += cpp->windows_per_frame * n_frames;
    *n_rects = (int64_t)total;
    if (rect_over || total > det->rect_cap) {
        set_error("device rect buffer overflow: %llu accepted windows, capacity %llu (raise max_rects)", total, det->rect_cap);
        return CLFD_ERR_CAPACITY;
    }
    return 0;
}

// event times of the last batch -> det->kernel_ms (clfd_detector_get_kernel_ms)
static void read_kernel_ms(clfd_detector *det) {
    // [0] resize+colsum [1] colscan [2] integral rows [3] tilted [4] tile kernel [5] deep kernel [6] colour conversion
    cudaEventElapsedTime(&det->kernel_ms[0], det->ev[0], det->ev[1]);
    cudaEventElapsedTime(&det->kernel_ms[1], det->ev[1], det->ev[2]);
    cudaEventElapsedTime(&det->kernel_ms[2], det->ev[2], det->ev[3]);
    cudaEventElapsedTime(&det->kernel_ms[3], det->ev[3], det->ev[4]);
    cudaEventElapsedTime(&det->kernel_ms[4], det->ev[5], det->ev[6]);
    cudaEventElapsedTime(&det->kernel_ms[5], det->ev[6], det->ev[7]);
    det->kernel_ms[6] = 0;
    if (det->color_events) cudaEventElapsedTime(&det->kernel_ms[6], det->ev[8], det->ev[9]);
    (void)cudaGetLastError();   // an event a batch did not record fails its query: not an error of the next launch
}

int clfd_detector_fetch(clfd_detector *det, clfd_rect *rects, int64_t cap, int64_t *n_rects, void *cuda_stream) {
    if (!det || !n_rects) INVALID("NULL argument");
    clfd_context *ctx = det->ctx;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    BatchSlot &sl = det->slot[0];   // the slot of clfd_detector_enqueue
    for (size_t ci = 0; ci < det->cas.size(); ci++)
        CK(cudaMemcpyAsync(sl.h_counters + kCnt * ci, det->cas[ci]->d_counters.p, kCnt * sizeof(unsigned long long),
                           cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    int rc = take_counters(det, sl.h_counters, det->last_frames, n_rects);
    if (rc) return rc;
    const unsigned long long total = (unsigned long long)*n_rects;
    if (det->have_events) read_kernel_ms(det);
    if (total == 0 || !rects) return 0;
    if ((int64_t)total > cap) { set_error("rect buffer too small: need %llu, have %lld", total, (long long)cap); return CLFD_ERR_CAPACITY; }
    CK(cudaMemcpyAsync(sl.h_rects, sl.rects.p, total * sizeof(DevRect), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    static_assert(sizeof(DevRect) == sizeof(clfd_rect), "rect layout");
    memcpy(rects, sl.h_rects, total * sizeof(DevRect));
    return 0;
}

// Host input, asynchronous: copy + enqueue one batch into the next free slot.
//   * the batch is cut into ranges; range k+1 is copied on the copy stream while the kernels of
//     range k run on the compute stream (pinned host memory; pageable memory degrades to a
//     serial copy).  Multi-cascade detectors carry their rect count from one cascade to the
//     next inside a range, so they run as one range;
//   * counters and the first kEagerRects rects are copied back behind the kernels and an event
//     marks the slot done, so the NEXT batch's host-to-device copy overlaps this batch's compute.
//   * colour batches (channels 3 / 4) go to a per-slot colour staging buffer instead, and the conversion of each range
//     runs on the copy stream behind its copy, into the slot's gray frames: from there on the batch is a gray batch.
static int submit_batch(clfd_detector *det, const uint8_t *frames_host, int n_frames, int channels, size_t frame_stride,
                        int row_stride) {
    if (!det || !frames_host) INVALID("NULL argument");
    clfd_context *ctx = det->ctx;
    CK(cudaSetDevice(ctx->device));
    const int W = det->cfg.width, H = det->cfg.height;
    if (n_frames <= 0 || n_frames > det->cfg.max_batch) INVALID("n_frames %d outside 1..%d", n_frames, det->cfg.max_batch);
    if (row_stride < W) INVALID("row stride %d smaller than the frame width %d", row_stride, W);
    if (det->n_submitted - det->n_collected >= kSlots) INVALID("%d batches already in flight: collect one first", kSlots);
    const int slot = (int)(det->n_submitted % kSlots);
    BatchSlot &sl = det->slot[slot];
    const size_t dstride = round_up(W, 16), dframe = dstride * H;
    int rc;
    if (!sl.frames.p && (rc = sl.frames.alloc(dframe * det->cfg.max_batch + 64))) return rc;
    // colour staging: rows of W * channels bytes at a 16-byte pitch.  The slot's last batch has been collected, so the
    // buffer may grow here
    const size_t cstride = round_up((size_t)W * channels, 16), cframe = cstride * H;
    if (channels != 1 && sl.color.n < cframe * det->cfg.max_batch && (rc = sl.color.alloc(cframe * det->cfg.max_batch)))
        return rc;
    if (!sl.rects.p && (rc = sl.rects.alloc(det->rect_cap))) return rc;   // slot 1 (slot 0's come with the detector)
    if (!sl.h_rects) CK(cudaMallocHost((void **)&sl.h_rects, (size_t)kEagerRects * sizeof(DevRect)));
    int n_chunks = 1;
    if (n_frames >= 8) n_chunks = n_frames >= 32 ? 4 : 2;
    // with a batch already in flight the whole copy overlaps THAT batch's compute: no need to
    // pay the extra kernel boundaries of a cut
    if (det->n_submitted > det->n_collected) n_chunks = 1;
    if (const char *e = getenv("CLFD_DETECT_CHUNKS")) n_chunks = std::max(1, std::min({atoi(e), kMaxChunks, n_frames}));
    if (det->cas.size() != 1) n_chunks = 1;
    const bool overlap = overlap_applies(det, n_frames);
    if (overlap) n_chunks = overlap_chunks(n_frames);   // the compute chunks are the copy chunks
    if (channels != 1 && det->profiling) n_chunks = 1;  // one pair of events brackets the whole conversion
    if (!det->copy_stream) CK(cudaStreamCreateWithFlags(&det->copy_stream, cudaStreamNonBlocking));
    for (int k = 0; k < n_chunks; k++)
        if (!det->copied[k]) CK(cudaEventCreateWithFlags(&det->copied[k], cudaEventDisableTiming));
    for (auto &b : det->slot) if (!b.done) CK(cudaEventCreateWithFlags(&b.done, cudaEventDisableTiming));
    // The slot's staging buffer was last read by the batch submitted kSlots submits ago, which has
    // been collected (its done event was synchronised), so the copy may start right away -- while
    // the previous batch still computes.
    det->last_frames = n_frames;
    sl.n_frames = n_frames;
    int launches = 0;
    cudaStream_t cs = det->copy_stream;
    // nf frames of `wbytes` bytes per row from the host to d (pitch dpitch, frames dfr apart); nothing behind the last
    // row's last pixel is read
    auto h2d = [&](uint8_t *d, size_t dpitch, size_t dfr, const uint8_t *src, size_t wbytes, int nf) -> int {
        if ((size_t)row_stride == dpitch && frame_stride == dfr) {
            CK(cudaMemcpyAsync(d, src, dfr * nf - (dpitch - wbytes), cudaMemcpyHostToDevice, cs));
        } else if (frame_stride == (size_t)row_stride * H) {
            CK(cudaMemcpy2DAsync(d, dpitch, src, row_stride, wbytes, (size_t)H * nf, cudaMemcpyHostToDevice, cs));
        } else {
            for (int f = 0; f < nf; f++)
                CK(cudaMemcpy2DAsync(d + f * dfr, dpitch, src + f * frame_stride, row_stride, wbytes, H,
                                     cudaMemcpyHostToDevice, cs));
        }
        return 0;
    };
    for (int k = 0; k < n_chunks; k++) {
        const int f0 = (int)((long long)n_frames * k / n_chunks), f1 = (int)((long long)n_frames * (k + 1) / n_chunks);
        const int nf = f1 - f0;
        if (nf <= 0) continue;
        uint8_t *dst = sl.frames.p + (size_t)f0 * dframe;
        const uint8_t *src = frames_host + (size_t)f0 * frame_stride;
        if (channels == 1) {
            if ((rc = h2d(dst, dstride, dframe, src, W, nf))) return rc;
        } else {
            uint8_t *stage = sl.color.p + (size_t)f0 * cframe;
            if ((rc = h2d(stage, cstride, cframe, src, (size_t)W * channels, nf))) return rc;
            if ((rc = enqueue_color_to_gray(det, stage, nf, channels, cframe, (int)cstride, dst, cs))) return rc;
            launches++;
        }
        CK(cudaEventRecord(det->copied[k], cs));
        if (overlap) continue;
        CK(cudaStreamWaitEvent(ctx->stream, det->copied[k], 0));
        rc = enqueue_range(det, dst, f0, nf, dframe, (int)dstride, ctx->stream, k == 0, &launches, slot);
        if (rc) return rc;
    }
    if (overlap) {   // pyramid of chunk k+1 beside the tile kernel of chunk k, each pyramid behind its chunk's copy
        rc = enqueue_overlapped(det, sl.frames.p, n_frames, dframe, (int)dstride, ctx->stream, n_chunks, det->copied,
                                &launches, slot);
        if (rc) return rc;
    }
    det->stats.kernel_launches = launches;
    // results: counters of every cascade + the first rects, behind the kernels
    const int nc = (int)det->cas.size();
    for (int ci = 0; ci < nc; ci++)
        CK(cudaMemcpyAsync(sl.h_counters + kCnt * ci, det->cas[ci]->d_counters.p + kCnt * slot, kCnt * sizeof(unsigned long long),
                           cudaMemcpyDeviceToHost, ctx->stream));
    const size_t eager = (size_t)std::min<unsigned long long>(det->rect_cap, kEagerRects);
    CK(cudaMemcpyAsync(sl.h_rects, sl.rects.p, eager * sizeof(DevRect), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(sl.done, ctx->stream));
    det->color_events = channels != 1 && det->profiling;
    det->n_submitted++;
    return 0;
}

int clfd_detect_submit(clfd_detector *det, const uint8_t *frames_host, int n_frames, size_t frame_stride, int row_stride) {
    return submit_batch(det, frames_host, n_frames, 1, frame_stride, row_stride);
}

int clfd_detect_submit_color(clfd_detector *det, const uint8_t *frames_host, int n_frames, int channels, size_t frame_stride,
                             int row_stride) {
    if (!det || !frames_host) INVALID("NULL argument");
    if (channels != 1) {
        int rc = check_color_batch(det, n_frames, channels, row_stride);
        if (rc) return rc;
    }
    return submit_batch(det, frames_host, n_frames, channels, frame_stride, row_stride);
}

// Wait for the oldest submitted batch and hand out its rects.
int clfd_detect_collect(clfd_detector *det, clfd_rect *rects, int64_t cap, int64_t *n_rects) {
    if (!det || !n_rects) INVALID("NULL argument");
    if (det->n_collected >= det->n_submitted) INVALID("no batch in flight");
    clfd_context *ctx = det->ctx;
    CK(cudaSetDevice(ctx->device));
    BatchSlot &sl = det->slot[det->n_collected % kSlots];
    det->n_collected++;
    CK(cudaEventSynchronize(sl.done));
    if (det->have_events && det->n_collected == det->n_submitted) read_kernel_ms(det);   // the events are this batch's
    int rc = take_counters(det, sl.h_counters, sl.n_frames, n_rects);
    if (rc) return rc;
    const unsigned long long total = (unsigned long long)*n_rects;
    if (total == 0 || !rects) return 0;
    if ((int64_t)total > cap) { set_error("rect buffer too small: need %llu, have %lld", total, (long long)cap); return CLFD_ERR_CAPACITY; }
    static_assert(sizeof(DevRect) == sizeof(clfd_rect), "rect layout");
    const unsigned long long eager = std::min<unsigned long long>(total, kEagerRects);
    memcpy(rects, sl.h_rects, eager * sizeof(DevRect));
    if (total > eager)   // rare: the slot's device buffer is untouched until the slot is submitted again
        CK(cudaMemcpy(rects + eager, sl.rects.p + eager, (total - eager) * sizeof(DevRect), cudaMemcpyDeviceToHost));
    return 0;
}

// Host input end to end, synchronous: the call a clod user makes.
int clfd_detect(clfd_detector *det, const uint8_t *frames_host, int n_frames, size_t frame_stride, int row_stride,
                clfd_rect *rects, int64_t cap, int64_t *n_rects) {
    if (!det) INVALID("NULL argument");
    if (det->n_submitted != det->n_collected) INVALID("clfd_detect while submitted batches are in flight");
    int rc = clfd_detect_submit(det, frames_host, n_frames, frame_stride, row_stride);
    if (rc) return rc;
    return clfd_detect_collect(det, rects, cap, n_rects);
}

// A batch of interleaved BGR / BGRA frames from the host, synchronous: the colour form of clfd_detect.
int clfd_detect_color(clfd_detector *det, const uint8_t *frames_host, int n_frames, int channels, size_t frame_stride,
                      int row_stride, clfd_rect *rects, int64_t cap, int64_t *n_rects) {
    if (!det) INVALID("NULL argument");
    if (det->n_submitted != det->n_collected) INVALID("clfd_detect_color while submitted batches are in flight");
    int rc = clfd_detect_submit_color(det, frames_host, n_frames, channels, frame_stride, row_stride);
    if (rc) return rc;
    return clfd_detect_collect(det, rects, cap, n_rects);
}

// One interleaved 8-bit image (1, 3 = BGR or 4 = BGRA channels) from the host: a batch of one frame.
int clfd_detect_image(clfd_detector *det, const uint8_t *img_host, int channels, int stride, clfd_rect *rects, int64_t cap,
                      int64_t *n_rects) {
    if (!det || !img_host) INVALID("NULL argument");
    return clfd_detect_color(det, img_host, 1, channels, (size_t)stride * det->cfg.height, stride, rects, cap, n_rects);
}

int clfd_detector_get_codes(clfd_detector *det, int cascade, int16_t *codes, int64_t cap) {
    if (!det || !codes || cascade < 0 || cascade >= (int)det->cas.size()) INVALID("bad argument");
    if (!det->cfg.want_codes && det->cfg.mode != CLFD_MODE_SCALE_CASCADE) INVALID("detector was created without want_codes");
    CK(cudaSetDevice(det->ctx->device));
    CascadePlan &cp = *det->cas[cascade];
    const int64_t n = cp.windows_per_frame * det->last_frames;
    if (n > cap) { set_error("codes buffer too small: need %lld", (long long)n); return CLFD_ERR_CAPACITY; }
    CK(cudaDeviceSynchronize());
    if (n > 0) CK(cudaMemcpy(codes, cp.d_codes.p, n * sizeof(int16_t), cudaMemcpyDeviceToHost));
    return 0;
}

// Reject levels of the last batch (tempcv.cpp:1084-1094): a pass over the exit codes, see k_roc_collect.
int clfd_detector_reject_levels(clfd_detector *det, int cascade, clfd_rect *rects, int32_t *reject_levels,
                                double *level_weights, int64_t cap, int64_t *n_out) {
    if (!det || !n_out || cascade < 0 || cascade >= (int)det->cas.size() || cap < 0 ||
        (cap > 0 && (!rects || !reject_levels || !level_weights)))
        INVALID("bad argument");
    *n_out = 0;
    if (det->cfg.mode == CLFD_MODE_SCALE_CASCADE) INVALID("reject levels are defined on the image-pyramid path only (tempcv.cpp:1084)");
    if (!det->cfg.want_codes) INVALID("detector was created without want_codes");
    if (det->n_submitted != det->n_collected) INVALID("clfd_detector_reject_levels while submitted batches are in flight");
    CascadePlan &cp = *det->cas[cascade];
    if (det->last_frames == 0 || cp.windows_per_frame == 0) return 0;
    clfd_context *ctx = det->ctx;
    CK(cudaSetDevice(ctx->device));
    int rc;
    const unsigned long long roc_cap = 1ull << 20;
    if (!det->roc.p && ((rc = det->roc.alloc(roc_cap)) || (rc = det->roc_count.alloc(1)))) return rc;
    CascadeArgs a = cascade_args(det, cp, cascade, 0, det->last_frames);
    a.codes = cp.d_codes.p;
    CK(cudaMemsetAsync(det->roc_count.p, 0, sizeof(unsigned long long), ctx->stream));
    CK(launch_roc_collect(a, det->roc.p, roc_cap, det->roc_count.p, ctx->stream));
    ctx->launches++;
    unsigned long long n = 0;
    CK(cudaMemcpyAsync(&n, det->roc_count.p, sizeof n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (n > roc_cap) { set_error("more than %llu reject-level candidates", roc_cap); return CLFD_ERR_CAPACITY; }
    *n_out = (int64_t)n;
    if ((int64_t)n > cap) { set_error("reject-level buffers too small: need %llu", n); return CLFD_ERR_CAPACITY; }
    std::vector<RocItem> items(n);
    if (n) CK(cudaMemcpy(items.data(), det->roc.p, n * sizeof(RocItem), cudaMemcpyDeviceToHost));
    std::sort(items.begin(), items.end(), [](const RocItem &p, const RocItem &q) {   // the reference's scan order
        return p.r.frame != q.r.frame ? p.r.frame < q.r.frame : p.win < q.win;
    });
    for (size_t i = 0; i < items.size(); i++) {
        const DevRect &r = items[i].r;
        rects[i].x = r.x; rects[i].y = r.y; rects[i].w = r.w; rects[i].h = r.h; rects[i].frame = r.frame; rects[i].cascade = r.cascade;
        reject_levels[i] = items[i].level;
        level_weights[i] = items[i].weight;
    }
    return 0;
}

int clfd_detector_read_level(clfd_detector *det, int cascade, int level, int frame, uint8_t *pyr, int32_t *sum,
                             uint64_t *sqsum, int32_t *tilted) {
    if (!det || cascade < 0 || cascade >= (int)det->cas.size()) INVALID("bad argument");
    CascadePlan &cp = *det->cas[cascade];
    // pub_levels: the scale-cascade planner lists only its tile-kernel scales in `levels`; every scale reads pyramid level 0
    if (level < 0 || level >= (int)cp.pub_levels.size()) INVALID("level %d outside 0..%zu", level, cp.pub_levels.size());
    if (frame < 0 || frame >= det->last_frames) INVALID("frame %d outside the last batch", frame);
    if (tilted && !det->pyr.want_tilted) INVALID("detector has no tilted integral (no cascade with tilted features)");
    CK(cudaSetDevice(det->ctx->device));
    CK(cudaDeviceSynchronize());
    const bool scale_cascade = det->cfg.mode == CLFD_MODE_SCALE_CASCADE;
    const PyrLevel &L = det->pyr.levels[scale_cascade ? 0 : cp.levels[level].pyr_level];
    const size_t W1 = (size_t)L.w + 1;
    const size_t so = (size_t)frame * det->pyr.sum_frame_stride + L.sum_off;
    if (pyr) CK(cudaMemcpy2D(pyr, L.w, det->pyr.pyr.p + (size_t)frame * det->pyr.pyr_frame_stride + L.pyr_off, L.pyr_pitch, L.w, L.h, cudaMemcpyDeviceToHost));
    if (sum && L.di) {   // stored column-de-interleaved on the device (PyrLevel::di): back to the natural order
        std::vector<int32_t> rows((size_t)L.sum_pitch * (L.h + 1));
        CK(cudaMemcpy(rows.data(), det->pyr.sum.p + so, rows.size() * 4, cudaMemcpyDeviceToHost));
        for (int y = 0; y <= L.h; y++)
            for (size_t x = 0; x < W1; x++) sum[y * W1 + x] = rows[(size_t)y * L.sum_pitch + (x & 1) * (L.sum_pitch / 2) + (x >> 1)];
    } else if (sum) {
        CK(cudaMemcpy2D(sum, W1 * 4, det->pyr.sum.p + so, (size_t)L.sum_pitch * 4, W1 * 4, L.h + 1, cudaMemcpyDeviceToHost));
    }
    if (sqsum && det->pyr.sq32) {   // kept modulo 2^32 on the device: the low words, widened
        std::vector<uint32_t> low(W1 * (L.h + 1));
        CK(cudaMemcpy2D(low.data(), W1 * 4, reinterpret_cast<const uint32_t *>(det->pyr.sq.p) + so, (size_t)L.sum_pitch * 4, W1 * 4,
                        L.h + 1, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < low.size(); i++) sqsum[i] = low[i];
    } else if (sqsum) {
        CK(cudaMemcpy2D(sqsum, W1 * 8, det->pyr.sq.p + so, (size_t)L.sum_pitch * 8, W1 * 8, L.h + 1, cudaMemcpyDeviceToHost));
    }
    if (tilted) CK(cudaMemcpy2D(tilted, W1 * 4, det->pyr.tilted.p + so, (size_t)L.sum_pitch * 4, W1 * 4, L.h + 1, cudaMemcpyDeviceToHost));
    return 0;
}

int clfd_detector_get_stats(clfd_detector *det, clfd_run_stats *stats) {
    if (!det || !stats) INVALID("NULL argument");
    *stats = det->stats;
    return 0;
}

int clfd_detector_get_kernel_ms(clfd_detector *det, float ms[8]) {
    if (!det || !ms) INVALID("NULL argument");
    if (!det->have_events) INVALID("profiling was not enabled for the last enqueue");
    memcpy(ms, det->kernel_ms, sizeof det->kernel_ms);
    return 0;
}

}  // extern "C"
