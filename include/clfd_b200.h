/*
 * clfd_b200.h -- C ABI of the B200-native Viola-Jones hot path
 * (pyramid downscale -> integral / squared-integral [/ tilted] images -> cascade
 * evaluation -> raw detection rects).
 *
 * This is the drop-in boundary: plain C, pointers and sizes only, no torch / OpenCV
 * types.  The reference-facing host API (include/clif.h, include/clod.h -- same names
 * and signatures as the reference's clif.h:43-73 and clod.h:61-81) is a thin C++ layer
 * over these entry points; INTEGRATION.md shows the binding a maintainer of the
 * reference would add.  Every call returns 0 on success or a negative clfd_status;
 * clfd_last_error() returns the message of the calling thread's last failure.  There is
 * NO CPU fallback behind any entry point: without a CUDA device they fail.
 *
 * Reference citations are file:line under CLFaceDetection/ of the reference repo.
 */
#ifndef CLFD_B200_H
#define CLFD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define CLFD_API __attribute__((visibility("default")))
#else
#define CLFD_API
#endif

typedef enum clfd_status {
    CLFD_OK = 0,
    CLFD_ERR_INVALID = -1,   /* bad argument */
    CLFD_ERR_CUDA = -2,      /* CUDA runtime/driver failure (message has the CUDA error) */
    CLFD_ERR_FORMAT = -3,    /* malformed cascade file / structure */
    CLFD_ERR_IO = -4,        /* file could not be read */
    CLFD_ERR_CAPACITY = -5   /* caller buffer too small */
} clfd_status;

typedef struct clfd_context clfd_context;   /* one per (host thread, GPU) */
typedef struct clfd_cascade clfd_cascade;   /* host-side cascade + packed device blobs */
typedef struct clfd_detector clfd_detector; /* plan + device buffers for one frame shape */

CLFD_API const char *clfd_last_error(void);
CLFD_API const char *clfd_version(void);

/* ---- environment --------------------------------------------------------------------
 * Replaces clifInitEnvironment / clodInitEnvironment (clif.cpp:80-118, clod.cpp:72-100:
 * device list, context, queue, runtime kernel build) and the *ReleaseEnvironment pair
 * (clif.cpp:226-238, clod.cpp:172-180).  device_index is honoured (the reference ignores
 * it for clif, clod.cpp:76). */
CLFD_API int clfd_device_count(int *count);
CLFD_API int clfd_context_create(int device_index, clfd_context **out);
CLFD_API void clfd_context_destroy(clfd_context *ctx);
CLFD_API int clfd_context_device(const clfd_context *ctx);
/* number of kernels this context has launched since creation */
CLFD_API int64_t clfd_context_launch_count(const clfd_context *ctx);
CLFD_API int clfd_context_synchronize(clfd_context *ctx);

/* ---- cascade loading / packing -------------------------------------------------------
 * clfd_cascade_load_xml replaces cvLoad(file_xml) (main.cpp:36), i.e. OpenCV's
 * icvReadHaarClassifier (tempcv.cpp:1750-2089) for "opencv-haar-classifier" files.
 * clfd_cascade_from_arrays takes the same content as flat arrays (what the clod layer
 * extracts from a CvHaarClassifierCascade, tempcv.hpp:70-112).  Both then build the
 * hidden cascade (icvCreateHidHaarClassifierCascade, tempcv.cpp:308-467) and the
 * scale-1 weights (cvSetImagesForHaarClassifierCascade, tempcv.cpp:549-768) and pack
 * them for the device (replacing precomputeKernelCascade, clod.cpp:529-578).
 *   st_*      : per stage (threshold as in the XML, bias not applied)
 *   tr_nnodes : nodes per tree;  nd_* per node;  nd_rect [N][3][4]=x,y,w,h; nd_weight [N][3]
 *   nd_left/right : >0 node index within the tree, <=0 leaf alpha[-idx]
 *   alpha     : (nnodes+1) per tree */
CLFD_API int clfd_cascade_load_xml(const char *path, clfd_cascade **out);
CLFD_API int clfd_cascade_from_arrays(int win_w, int win_h, int n_stages,
                                      const int *st_ntrees, const float *st_thr,
                                      const int *st_parent, const int *st_next,
                                      const int *tr_nnodes, const int *nd_tilted,
                                      const int *nd_rect, const float *nd_weight,
                                      const float *nd_thr, const int *nd_left,
                                      const int *nd_right, const float *alpha,
                                      clfd_cascade **out);
/* Cascades are reference counted: detectors created from a cascade keep it alive, so it may be
 * destroyed before them (cvReleaseHaarClassifierCascade, tempcv.cpp:1702-1719, has no such
 * ordering rule either). */
CLFD_API void clfd_cascade_destroy(clfd_cascade *c);
/* Unique per process and never reused (an address can be): the key for caches of detector plans. */
CLFD_API uint64_t clfd_cascade_id(const clfd_cascade *c);

typedef struct clfd_cascade_info {
    int win_w, win_h;
    int n_stages, n_trees, n_nodes;
    int is_tree;            /* stage tree (alt_tree)            tempcv.cpp:431 */
    int is_stump_based;     /* every tree has one node          tempcv.cpp:465 */
    int has_tilted;         /* some feature is tilted           tempcv.cpp:371 */
    int n_tilted_nodes, n_three_rect_nodes, max_trees_per_stage, max_nodes_per_tree;
    int dense_stages;       /* leading stages evaluated by the smem-tile kernel (0 = none) */
    int dense_stumps;       /* stumps in those stages */
    int order_free_stages;  /* stages whose alpha sum is exact in any order */
    int packed_bytes;       /* size of the device blob */
} clfd_cascade_info;
CLFD_API int clfd_cascade_get_info(const clfd_cascade *c, clfd_cascade_info *info);
/* copy the parsed arrays back out (any pointer may be NULL); sizes from clfd_cascade_info */
CLFD_API int clfd_cascade_get_arrays(const clfd_cascade *c, int *st_ntrees, float *st_thr,
                                     int *st_parent, int *st_next, int *st_child,
                                     int *tr_nnodes, int *nd_tilted, int *nd_rect,
                                     float *nd_weight, float *nd_thr, int *nd_left,
                                     int *nd_right, float *alpha);
/* hidden-cascade values the device blob encodes: scale-1 rect weights [N][3], kept rects
 * per node [N], biased stage thresholds [S], two_rects flag per stage [S] */
CLFD_API int clfd_cascade_get_hidden(const clfd_cascade *c, float *node_weights,
                                     int *node_nrects, float *stage_thr, int *stage_two_rects);

/* ---- clif: integral images -----------------------------------------------------------
 * Replaces clifIntegral's device branch (clif.cpp:273-316: upload, integralImageSumRows,
 * integralImageSumCols, two blocking maps) and cvIntegral at tempcv.cpp:1302.
 * img is 8-bit single channel, `stride` bytes per row.  Outputs are dense
 * (h+1) x (w+1): sum int32, sqsum uint64 (the reference's cl_ulong payload, clif.cpp:305),
 * tilted int32 (NULL to skip).  *_on_device selects host or device pointers. */
CLFD_API int clfd_integral(clfd_context *ctx, const uint8_t *img, int w, int h, int stride,
                           int img_on_device, int32_t *sum, uint64_t *sqsum, int32_t *tilted,
                           int out_on_device);
/* One pyramid level: cvResize(img, level, CV_INTER_LINEAR) at tempcv.cpp:1301. */
CLFD_API int clfd_resize(clfd_context *ctx, const uint8_t *src, int sw, int sh, int sstride,
                         int src_on_device, uint8_t *dst, int dw, int dh, int dstride,
                         int dst_on_device);
/* BGR -> gray, clifGrayscale (clif.cpp:241-271).  coefficients: OpenCV's fixed point
 * (R*4899 + G*9617 + B*1868 + 8192) >> 14, the CPU branch the clod path actually uses
 * (clod.cpp:366 -> clif.cpp:327-328). */
CLFD_API int clfd_bgr_to_gray(clfd_context *ctx, const uint8_t *bgr, int w, int h, int stride,
                              int channels, int src_on_device, uint8_t *gray, int gstride,
                              int dst_on_device);
/* clifGrayscaleIntegral (clif.cpp:318-381; clod.cpp:366 calls it for every frame): colour conversion and
 * integral images of one interleaved HOST image (1, 3 = BGR or 4 = BGRA channels) in one call.  The frame is
 * uploaded once and the gray plane never leaves the device (the reference's OpenCL branch downloads it and
 * uploads it again, clif.cpp:339-364); `gray` (host, gstride >= w) receives it if not NULL. */
CLFD_API int clfd_integral_image(clfd_context *ctx, const uint8_t *img, int w, int h, int stride, int channels,
                                 int32_t *sum, uint64_t *sqsum, int32_t *tilted, uint8_t *gray, int gstride);

/* ---- clod: multi-scale detection -----------------------------------------------------
 * Replaces clodInitBuffers / clodDetectObjects / clodReleaseBuffers (clod.cpp:102-170,
 * 1339-1500) with the semantics of the CV_HAAR_SCALE_IMAGE path the north star names
 * (tempcv.cpp:1257-1329, 1011-1103, 795-972): per level resize-from-original, integral,
 * every window on the ystep grid, raw (ungrouped) rects. */
typedef struct clfd_detector_config {
    int width, height;        /* frame shape (8-bit gray) */
    int max_batch;            /* frames per call */
    double scale_factor;      /* > 1 (reference hard-codes 1.1, clod.cpp:1349) */
    int min_w, min_h;         /* minimum window (0 = none) */
    int max_w, max_h;         /* maximum window (0 = image size, clod.cpp:394-397) */
    int want_codes;           /* keep per-window exit codes (parity tests) */
    int64_t max_rects;        /* device rect capacity per call (0 = default) */
    int mode;                 /* CLFD_MODE_SCALE_IMAGE (0, default) or CLFD_MODE_SCALE_CASCADE */
} clfd_detector_config;
/* CLFD_MODE_SCALE_IMAGE  : image pyramid, cascade at scale 1 -- the CV_HAAR_SCALE_IMAGE path the
 *                          north star names (tempcv.cpp:1257-1329).  Cascade windows up to 255 x 255:
 *                          the kernels keep corner offsets in bytes and the squared integral modulo
 *                          2^32, exact while (w-2)(h-2)*255^2 < 2^32.  clfd_detector_create returns
 *                          CLFD_ERR_INVALID for a cascade whose window is wider or taller than 255.
 * CLFD_MODE_SCALE_CASCADE: ONE integral image, features scaled per factor, window step
 *                          max(2, factor) and the skip-after-stage-0-reject rule -- what the
 *                          cvHaarDetectObjects call of main.cpp:145 (flags 0) computes
 *                          (tempcv.cpp:1330-1456, 1132-1175) and the formulation of clod's own
 *                          runStage (clod.cpp:1176-1336).  max_w / max_h are ignored (the
 *                          reference's scale loop has no upper limit but the image).  Any window
 *                          size (64-bit squared integral, int offsets).  Exit codes
 *                          additionally use -32768 (position skipped by the rule) and -32767
 *                          (window rejected by the bounds check).  clfd_level.ystep is 0: the step
 *                          is max(2, factor); window (ix, iy) sits at cvRound(ix*step), cvRound(iy*step). */
#define CLFD_MODE_SCALE_IMAGE 0
#define CLFD_MODE_SCALE_CASCADE 1

typedef struct clfd_rect {
    int32_t x, y, w, h;   /* CvRect of the accepted window (tempcv.cpp:1099-1100) */
    int32_t frame;        /* frame index within the call */
    int32_t cascade;      /* index into the detector's cascade list */
} clfd_rect;

typedef struct clfd_level {
    double factor;
    int img_w, img_h, win_w, win_h, ystep, nx, ny;
    int64_t win_base;     /* offset of this level in the exit-code array */
} clfd_level;

typedef struct clfd_run_stats {
    int64_t windows;          /* windows evaluated (all frames, all cascades) */
    int64_t rects;            /* accepted windows */
    int64_t deep_windows;     /* windows handed from the tile kernel to the generic kernels */
    int64_t kernel_launches;  /* kernels launched by the last enqueue */
    int64_t pyramid_pixels;   /* per frame */
    int64_t bytes_resize, bytes_integral, bytes_cascade; /* algorithmic bytes per frame (SURVEY 8-d); bytes_integral:
                                                            the upright pair, w*h + (w+1)(h+1)*12 per level */
    int64_t bytes_tilted;     /* tilted integral, w*h + (w+1)(h+1)*4 per level; 0 without tilted features */
    /* The tile kernel decides stumps and stage sums with FP32 filters and redoes a window's stage in the reference's
     * FP64 arithmetic whenever a decision could differ (DESIGN.md section 2).  Counted per (window, stage):
     *   exact_stage_evals     : stages redone in FP64
     *   near_threshold_events : of those, |stage_sum - threshold| <= 1e-5 * |threshold| (the tolerance the north star
     *                           allows for such windows; results are identical to the reference's anyway).  Every such
     *                           event takes the FP64 path, so the count is exact.  Image-pyramid mode.
     * Counted by detectors created with want_codes (a diagnostic instantiation of the tile kernel: the counting code
     * costs the production kernel 1.5-4.5 % even when no window takes the path); -1 otherwise. */
    int64_t exact_stage_evals, near_threshold_events;
} clfd_run_stats;

CLFD_API int clfd_detector_create(clfd_context *ctx, const clfd_cascade *const *cascades,
                                  int n_cascades, const clfd_detector_config *cfg,
                                  clfd_detector **out);
CLFD_API void clfd_detector_destroy(clfd_detector *det);
CLFD_API int clfd_detector_num_levels(const clfd_detector *det, int cascade);
CLFD_API int clfd_detector_get_levels(const clfd_detector *det, int cascade, clfd_level *levels,
                                      int max_levels);
CLFD_API int64_t clfd_detector_windows_per_frame(const clfd_detector *det, int cascade);

/* Device-resident input: enqueue every kernel of one batch on `cuda_stream` (a
 * cudaStream_t, NULL = the detector's own stream).  Does not synchronise. */
CLFD_API int clfd_detector_enqueue(clfd_detector *det, const uint8_t *frames_dev, int n_frames,
                                   size_t frame_stride, int row_stride, void *cuda_stream);
/* Copy the rects of the last enqueued batch to the host (synchronises the stream). */
CLFD_API int clfd_detector_fetch(clfd_detector *det, clfd_rect *rects, int64_t cap,
                                 int64_t *n_rects, void *cuda_stream);
/* Host input end to end: H2D (pinned staging) + enqueue + fetch. The call a clod user makes. */
CLFD_API int clfd_detect(clfd_detector *det, const uint8_t *frames_host, int n_frames,
                         size_t frame_stride, int row_stride, clfd_rect *rects, int64_t cap,
                         int64_t *n_rects);
/* One interleaved image (channels 1, or 3 / 4 = BGR / BGRA as in IplImage) from the host: the
 * colour conversion of clifGrayscale (clif.cpp:241-271) runs on the device and feeds the detector
 * directly.  This is the whole of clodDetectObjects' device work for one frame (its setupImage,
 * clod.cpp:360-369, converts every input from BGR).  It is clfd_detect_color with n_frames = 1 and
 * frame_stride = stride * height. */
CLFD_API int clfd_detect_image(clfd_detector *det, const uint8_t *img_host, int channels, int stride,
                               clfd_rect *rects, int64_t cap, int64_t *n_rects);
/* The same, split in two so that batches overlap: _submit copies batch i+1 (pinned host
 * memory, copy stream) while batch i still computes, _collect waits for the OLDEST submitted
 * batch and hands out its rects.  At most 2 batches in flight.  The reference has no such
 * call (clodDetectObjects blocks per stage, clod.cpp:1256-1302); this is the streaming form of
 * SURVEY 8-e ("pinned staging buffers, H2D / compute / D2H overlap"). */
CLFD_API int clfd_detect_submit(clfd_detector *det, const uint8_t *frames_host, int n_frames,
                                size_t frame_stride, int row_stride);
CLFD_API int clfd_detect_collect(clfd_detector *det, clfd_rect *rects, int64_t cap,
                                 int64_t *n_rects);
/* ---- colour batches ------------------------------------------------------------------
 * The batch forms of clfd_detect_image: n_frames interleaved 8-bit frames, channels 3 (BGR) or 4
 * (BGRA, alpha ignored), converted to gray on the device with the fixed point of clfd_bgr_to_gray
 * ((B*1868 + G*9617 + R*4899 + 8192) >> 14) and detected as that gray batch.  They replace
 * setupImage's per-frame cvCvtColor(BGR2GRAY) (clod.cpp:360-369) and clifGrayscale (clif.cpp:241-271)
 * for a whole batch; the rects are those of clfd_detect on the converted frames.
 *   Strides: row_stride >= width * channels bytes; frame i starts i * frame_stride bytes after the
 *   first one, any value (odd, smaller than height * row_stride, or 0 to repeat one frame).  Only the
 *   width * channels bytes of each row are read.  channels == 1 hands the call to the gray entry point
 *   unchanged; other channel counts, a short row stride or n_frames outside 1..max_batch return
 *   CLFD_ERR_INVALID.
 *   clfd_detect_submit_color: as clfd_detect_submit (pinned memory, two batches in flight; collect
 *   with clfd_detect_collect).  Each range of the batch is copied to a colour staging buffer of its
 *   slot (allocated at the first colour submit) and converted on the copy stream behind its copy.
 *   Colour and gray submits may alternate on one detector.
 *   clfd_detect_color: as clfd_detect (submit + collect).
 *   clfd_detector_enqueue_color: device-resident frames, converted on `cuda_stream` into the
 *   detector's own frame buffer, then enqueued as by clfd_detector_enqueue; collect with
 *   clfd_detector_fetch.  That buffer is also a submit slot's, so while submitted batches are in
 *   flight it returns CLFD_ERR_INVALID (clfd_detect_image has the same rule). */
CLFD_API int clfd_detector_enqueue_color(clfd_detector *det, const uint8_t *frames_dev, int n_frames,
                                         int channels, size_t frame_stride, int row_stride,
                                         void *cuda_stream);
CLFD_API int clfd_detect_submit_color(clfd_detector *det, const uint8_t *frames_host, int n_frames,
                                      int channels, size_t frame_stride, int row_stride);
CLFD_API int clfd_detect_color(clfd_detector *det, const uint8_t *frames_host, int n_frames,
                               int channels, size_t frame_stride, int row_stride, clfd_rect *rects,
                               int64_t cap, int64_t *n_rects);
/* Exit codes of the last batch (want_codes=1): int16 [n_frames][windows_per_frame(cascade)];
 * linear cascades: stages passed (n_stages = accepted); stage trees: 2*last_stage+accepted. */
CLFD_API int clfd_detector_get_codes(clfd_detector *det, int cascade, int16_t *codes,
                                     int64_t cap);
/* Pyramid level `level` (index into the union pyramid = cascade 0's level list when there
 * is one cascade) of frame `frame` from the last batch, dense layouts; NULLs skipped.
 * A pyramid-mode detector keeps its squared integral modulo 2^32 (all it ever needs are windows'
 * sums of squares, which are below 2^32): sqsum then returns those low words, widened.  It also stores the
 * int32 integral of the levels whose windows are 2 pixels apart column-de-interleaved (the tile kernel's
 * shared-memory order); `sum` is handed back in the natural order regardless.
 * A scale-cascade detector has one image, the frame itself: every level 0 .. num_levels-1 reads it
 * (pyr = the frame, the natural-order sum, the full 64-bit sqsum and, with tilted features, tilted).
 * sum and tilted are int32 like the reference's CV_32S integrals: on a frame whose pixels add up to
 * 2^31 or more they wrap modulo 2^32; the kernels only ever use differences of them (window sums). */
CLFD_API int clfd_detector_read_level(clfd_detector *det, int cascade, int level, int frame,
                                      uint8_t *pyr, int32_t *sum, uint64_t *sqsum,
                                      int32_t *tilted);
/* Reject-level / ROC output of the last batch (SURVEY 8-f row 4): what cvHaarDetectObjectsForROC
 * returns with outputRejectLevels = true on the image-pyramid path (tempcv.cpp:1084-1094): the
 * accepted windows (level = number of stages) AND the windows rejected by one of the last three
 * stages (level = index of that stage; a stage-tree cascade reports accepted windows only, its
 * evaluator returns 0 for every rejection), each with the stage sum of the last stage it
 * evaluated (double, the reference's summation order).  Needs want_codes = 1 and a completed
 * blocking clfd_detect / clfd_detect_image; candidates come back in the reference's scan order
 * (frame, level, y, x).  Not available in scale-cascade mode. */
CLFD_API int clfd_detector_reject_levels(clfd_detector *det, int cascade, clfd_rect *rects,
                                         int32_t *reject_levels, double *level_weights, int64_t cap,
                                         int64_t *n_out);
CLFD_API int clfd_detector_get_stats(clfd_detector *det, clfd_run_stats *stats);
/* Per-kernel device time (ms) of the last batch measured with CUDA events (read by
 * clfd_detector_fetch, and by clfd_detect_collect when it hands out the last submitted batch):
 * [0] resize+colsum [1] colscan [2] integral rows [3] tilted [4] cascade tile kernel
 * [5] cascade deep kernel [6] colour conversion (0 for a gray batch; with profiling on a colour
 * batch is submitted as one range, so [6] covers all its frames).  Enables event recording on
 * subsequent enqueues. */
CLFD_API int clfd_detector_set_profiling(clfd_detector *det, int enable);
CLFD_API int clfd_detector_get_kernel_ms(clfd_detector *det, float ms[8]);

/* ---- host-side rectangle grouping (stays on the host per the north star) --------------
 * AgroupRectangles(rects, weights, max(min_neighbors,1), 0.2) (tempcv.cpp:130-243,
 * call site 1462-1472).  rects in/out as x,y,w,h quadruples; returns new count in *n. */
CLFD_API int clfd_group_rectangles(int32_t *rects_xywh, int *n, int group_threshold, double eps,
                                   int32_t *weights);

/* The ROC variant (tempcv.cpp:255-258, used after outputRejectLevels detection): reject_levels /
 * level_weights per rect in; per kept class out: its highest level and the largest stage sum
 * seen at that level.  A class is kept when that LEVEL exceeds group_threshold (tempcv.cpp:210). */
CLFD_API int clfd_group_rectangles_roc(int32_t *rects_xywh, int *n, int group_threshold, double eps,
                                       int32_t *reject_levels, double *level_weights);

/* The same for the raw rects of a whole batch (as clfd_detect / clfd_detect_collect return
 * them): grouped per (frame, cascade) on n_threads host threads (0 = all).  Run it for batch i
 * while the GPU evaluates batch i+1 (clfd_detect_submit) and the O(N^2) grouping of
 * tempcv.cpp:1462-1472 leaves the critical path (SURVEY 8-f row 1).  Inside a (frame, cascade)
 * group the rects are first ordered by (w, y, x), so the result does not depend on the order in
 * which the device appended them.  out is sorted by (frame, cascade). */
CLFD_API int clfd_group_batch(const clfd_rect *rects, int64_t n, int group_threshold, double eps,
                              int n_threads, clfd_rect *out, int32_t *weights, int64_t cap,
                              int64_t *n_out);

#ifdef __cplusplus
}
#endif
#endif /* CLFD_B200_H */
