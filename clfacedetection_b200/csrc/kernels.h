// kernels.h -- launchers of the sm_100a kernels (kernels_*.cu).  Every launcher enqueues
// on `stream` and returns the cudaError_t of the launch.
#pragma once
#include <atomic>
#include <mutex>
#include <cuda_runtime.h>

#include "clfd_internal.h"

namespace clfd {

// ---- pyramid + integral (clif) ------------------------------------------------------
struct PyramidArgs {
    const uint8_t *frames;      // device, n_frames x (H rows of row_stride bytes), frame_stride apart
    size_t frame_stride;
    int row_stride, W, H, n_frames;
    uint8_t *pyr;  size_t pyr_frame_stride;     // bytes
    uint32_t *col; size_t col_frame_stride;     // elements; plane 0 = sums, plane 1 = squares
    size_t col_plane_stride;                    // elements
    int32_t *sum; unsigned long long *sq; int32_t *tilted;   // tilted may be NULL
    size_t sum_frame_stride;                    // elements (same for sum / sq / tilted)
    int sq32;                                   // the squared integral is kept modulo 2^32 (uint32 elements at `sq`, same
                                                // element offsets): every difference the detector forms is a window's sum of
                                                // squares < 255^2 x 257^2 < 2^32, so the low words give it exactly
    const PyrLevel *levels;                     // device
    int n_levels;
    const int *xofs; const short2 *xalpha; const int *yofs; const short2 *ybeta;   // device tables
    const int4 *resize_items; int n_resize_items;      // (level, row block, 128-column chunk, -), one per warp; padded with level -1 to a multiple of 4
    const int4 *colscan_items; int n_colscan_items;    // (level, column chunk, -, -)
    // integral row-block items grouped by CTA width class: class k uses 32<<k threads
    const int4 *integral_items[6]; int n_integral_items[6];
    // tilted integral: carry planes (kernels_clif.cu, K4), laid out like one plane of `col` each
    int32_t *tcar; size_t tcar_frame_stride;           // elements
    const int4 *tilt_tile_items; int n_tilt_tile_items;   // (level, row block, column tile, -), one warp each
    const int4 *tilt_diag_items; int n_tilt_diag_items;   // (level, chunk of 256 diagonals, -, -)
    const int4 *tilt_tc_items; int n_tilt_tc_items;       // (level, chunk of 8 x 32 columns, -, -)
    int max_level_w;
};

// Raises a kernel's dynamic shared-memory limit when a launch needs more than any earlier one on
// the CURRENT device (the attribute is per device; several host threads may launch at once).
struct SmemLimitCache {
    std::atomic<size_t> configured[64];
    std::mutex lock;
    SmemLimitCache() { for (auto &c : configured) c.store(0); }
    template <typename Kernel>
    cudaError_t ensure(Kernel kernel, size_t smem) {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        std::atomic<size_t> &c = configured[dev & 63];
        if (smem <= c.load(std::memory_order_acquire)) return cudaSuccess;
        std::lock_guard<std::mutex> g(lock);
        if (smem <= c.load(std::memory_order_relaxed)) return cudaSuccess;
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) c.store(smem, std::memory_order_release);
        return e;
    }
};

cudaError_t launch_resize_colsum(const PyramidArgs &a, cudaStream_t stream);
cudaError_t launch_colscan(const PyramidArgs &a, cudaStream_t stream);
// these two enqueue several kernels: *n_launches is how many
cudaError_t launch_integral_rows(const PyramidArgs &a, cudaStream_t stream, int *n_launches);
cudaError_t launch_tilted(const PyramidArgs &a, cudaStream_t stream, int *n_launches);
int tilt_tile_interior();    // output columns per warp tile of k_tilt_tiles

// BGR / BGRA -> gray of n_frames interleaved frames (kernels_clif.cu, k_color_to_gray)
struct ColorArgs {
    const uint8_t *src;         // device, n_frames x (H rows of row_stride bytes), frame_stride apart (any alignment)
    size_t frame_stride;        // bytes; may be smaller than H * row_stride, or 0
    int row_stride, channels;   // channels 3 (BGR) or 4 (BGRA, alpha ignored); row_stride >= W * channels
    int W, H, n_frames;
    uint8_t *dst;               // device, 16-byte aligned; written up to round_up(W, 16) per row (zero padding)
    size_t dst_frame_stride;    // bytes, a multiple of 16
    int dst_pitch;              // bytes, a multiple of 16 and >= round_up(W, 16)
};
cudaError_t launch_color_to_gray(const ColorArgs &a, cudaStream_t stream);

// ---- cascade (clod) -----------------------------------------------------------------
struct CascadeArgs {
    const int32_t *sum; const unsigned long long *sq; const int32_t *tilted;
    size_t sum_frame_stride;
    int sq32;                       // `sq` holds uint32 elements (squared integral modulo 2^32, PyramidArgs::sq32)
    int sum_di;                     // the ystep-2 levels of `sum` are stored column-de-interleaved (PyrLevel::di): the tile
                                    // kernel stages their tiles with TMA bulk copies; nothing else may read `sum` then
    const PyrLevel *levels;         // device
    const CasLevel *cas_levels;     // device
    int n_cas_levels, n_tiles, n_frames, cascade_index;
    int frame_base;                 // added to the frame index of emitted rects (ranges of a batch)
    int count_exact;                // tile kernel: the instantiation that counts FP64 fallbacks / near-threshold sums (counters[4], [5])
    long long windows_per_frame;
    int16_t *codes;                 // device, [n_frames][windows_per_frame] or NULL
    QueueItem *queue; unsigned long long queue_cap;   // written by the tile kernel / k_enqueue_all, counted in counters[1]
    // mid kernel pass: input queue (NULL = every grid window) -> output queue
    const QueueItem *mid_in; const unsigned long long *mid_in_count;
    QueueItem *mid_out; unsigned long long *mid_out_count;
    const QueueItem *deep_in; const unsigned long long *deep_count;   // what the deep kernel reads
    DevRect *rects; unsigned long long rect_cap;
    unsigned long long *counters;   // [0] rects  [1] queue items  [2] rect overflow [3] queue overflow
    DeepCascadeDev deep;
};
// dense tile kernel (+ hand-off of survivors to the queue)
// tiles [tile0, tile0 + n_tiles) must all belong to levels with ystep == P.ystep
cudaError_t launch_cascade_tiles(const DenseParams &P, const CascadeArgs &a, int tile0, int n_tiles, cudaStream_t stream);
// fill the queue with every window (cascades without a dense prefix)
cudaError_t launch_enqueue_all(const CascadeArgs &a, cudaStream_t stream);
// thread-per-window evaluation of stages [deep.mid_begin, deep.mid_end) (generic trees), survivors -> queue_b
cudaError_t launch_cascade_mid(const CascadeArgs &a, int n_sms, cudaStream_t stream);
// warp-per-window evaluation of the queue
cudaError_t launch_cascade_deep(const CascadeArgs &a, int n_sms, cudaStream_t stream);
// reject-level output: scans the exit codes of n_frames frames, appends the candidates of
// tempcv.cpp:1084-1094 (count at counter[0]) with the exact stage sum of their last stage
cudaError_t launch_roc_collect(const CascadeArgs &a, RocItem *out, unsigned long long cap, unsigned long long *counter, cudaStream_t stream);

// ---- scale-cascade mode (kernels_sc.cu) -----------------------------------------------
struct ScArgs {
    const int32_t *sum; const unsigned long long *sq; const int32_t *tilted;   // full-frame integrals (level 0)
    size_t sum_frame_stride;
    int pitch, W, H;                // elements per integral row, frame size
    const ScLevel *levels;          // device
    const ScNode *nodes;            // device, n_levels x n_nodes
    int n_levels, rows_per_frame, n_frames, cascade_index, frame_base;
    long long windows_per_frame;
    long long first_window;         // grid positions below this one are evaluated by the tile kernel (step-2 scales)
    int16_t *codes;                 // device, [n_frames][windows_per_frame] (always present in this mode)
    DevRect *rects; unsigned long long rect_cap;
    unsigned long long *counters;   // [0] rects [2] rect overflow [3] queue overflow
    DeepCascadeDev deep;            // stages / tree_first_node / alpha (scale independent)
    // one evaluation pass: stages [stage_begin, stage_end) of the positions in `in` (NULL = every grid
    // position); survivors of a non-final pass go to `out`
    int stage_begin, stage_end;
    const QueueItem *in; const unsigned long long *in_count;
    QueueItem *out; unsigned long long *out_count;
    unsigned long long queue_cap;
};
// one evaluation pass over the grid / a survivor queue (k_sc_eval)
cudaError_t launch_sc_eval(const ScArgs &a, int n_sms, cudaStream_t stream);
// final pass, warp per survivor: stages [stage_begin, n_stages) of a linear cascade (k_sc_deep)
cudaError_t launch_sc_deep(const ScArgs &a, int n_sms, cudaStream_t stream);
// the invoker's skip rule + rect emission over the finished exit codes (k_sc_rows)
cudaError_t launch_sc_rows(const ScArgs &a, cudaStream_t stream);

}  // namespace clfd
