// kernels_clod.cu -- sliding-window Haar-cascade evaluation for sm_100a.  Replaces, from
// scratch, the reference's per-stage runStage kernel (clod.cl:32-93) and its host loop
// with a blocking round trip per stage per scale (clod.cpp:1270-1302, 789-818), with the
// window semantics of cvRunHaarClassifierCascadeSum (tempcv.cpp:795-972) on the pyramid
// grid of HaarDetectObjects_ScaleImage_Invoker (tempcv.cpp:1011-1103).
//
// One kernel (two launches: ystep-2 and ystep-1 levels) per cascade per batch, no host round trip:
//   k_cascade_tiles<ROWSTEP, TREE, NODES, TILE_H, COUNT> : one CTA per 64 x TILE_H-window tile of one level
//       of one frame.  The int32 integral tile (and, for cascades with tilted features, the tilted
//       integral tile behind it) is staged into shared memory (TMA bulk row copies, cp.async.bulk
//       + mbarrier, on ystep-1 levels), sigma is computed once per window in FP64, and the
//       cascade is evaluated in two phases: fixed geometry (thread per window column, no
//       compaction, stumps from the constant bank: the packed cascade is a __grid_constant__
//       kernel parameter, <= 32 KB) while most windows are alive, then warp-autonomous: a
//       warp carries its survivors through all remaining stages, re-dividing its lanes between
//       windows and stumps as windows die (stump records from global memory).
//       Every stock cascade is finished inside this kernel: stumps, tilted features, trees of
//       up to four nodes (NODES: per-window "node I am at" state over padded node records),
//       the alt_tree stage tree (TREE: stages in depth-first order, per-window target position).
//       The scale-cascade mode runs its step-2 scales through it as well (clfd_api.cu).
//   k_cascade_mid / k_cascade_deep : generic fallback for cascades the tile kernel cannot finish
//       (larger trees, a tile that does not fit shared memory): the survivors of the tile prefix
//       (or every window) are pooled in one global queue and evaluated one thread / one WARP per
//       window, lanes striding over the trees of a stage.  The stage sum is reduced with shuffles
//       when the packer proved the alpha sum exact in any order, otherwise accumulated in tree order.
//   k_roc_collect : reject-level output (tempcv.cpp:1084-1094) as a pass over the exit codes.
//
// Arithmetic is bit-identical to the reference's C expressions: integer rect sums; FP64
// variance with separately rounded mul/sub/sqrt; two_rects stages multiply in double
// (products of a <2^24 integer and a 24-bit float are exact, so one FMA equals mul+add);
// other stages multiply in FLOAT and accumulate in double (tempcv.cpp:782-786,907-910).
// Tensor cores are not used: this is gather + compare work, not a contraction.
#include <algorithm>
#include <cstdint>

#include "clfd_pack.h"
#include "kernels.h"

namespace clfd {

typedef unsigned long long ull;

// ------------------------------------------------------------------------------------
// small PTX helpers: mbarrier + TMA bulk copy (SASS: UBLKCP / SYNCS)
// ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------------------------
// shared pieces
// ------------------------------------------------------------------------------------
__device__ __forceinline__ double window_sigma(int s4, ull q4, double inv_area) {
    // tempcv.cpp:824-832, every operation rounded separately
    const double mean = __dmul_rn((double)s4, inv_area);
    const double v = __dsub_rn(__dmul_rn((double)q4, inv_area), __dmul_rn(mean, mean));
    return v >= 0. ? sqrt(v) : 1.;
}

// Sum of squares of a rectangle from the squared integral at element offset `at` (corner offsets g0..g3): 64-bit
// elements, or the integral modulo 2^32 (CascadeArgs::sq32; a window's sum of squares is below 2^32, so the low
// words' difference is the sum itself).
__device__ __forceinline__ ull sq_rect(const ull *sq, bool sq32, size_t at, int g0, int g1, int g2, int g3) {
    if (sq32) {
        const uint32_t *q = reinterpret_cast<const uint32_t *>(sq) + at;
        return (ull)(uint32_t)(__ldg(q + g0) - __ldg(q + g1) - __ldg(q + g2) + __ldg(q + g3));
    }
    const ull *q = sq + at;
    return __ldg(q + g0) - __ldg(q + g1) - __ldg(q + g2) + __ldg(q + g3);
}

__device__ __forceinline__ void emit_rect(const CascadeArgs &a, const CasLevel &CL, int frame, int px, int py) {
    if (!a.rects) return;   // scale-cascade mode: k_sc_rows makes the rects from the exit codes
    const ull slot = atomicAdd(a.counters + 0, 1ull);
    if (slot < a.rect_cap) {
        DevRect r;
        r.x = __double2int_rn(__dmul_rn((double)px, CL.factor));  // cvRound(x*factor), tempcv.cpp:1099
        r.y = __double2int_rn(__dmul_rn((double)py, CL.factor));
        r.w = CL.win_w; r.h = CL.win_h; r.frame = a.frame_base + frame; r.cascade = a.cascade_index;
        a.rects[slot] = r;
    } else {
        atomicAdd(a.counters + 2, 1ull);
    }
}

// ------------------------------------------------------------------------------------
// dense tile kernel
//
// One CTA (256 threads) per 64x32-window tile.  Shared memory:
//   tile    int32 [rows][S]   ystep-1 levels: natural layout, staged by TMA bulk row copies;
//                             ystep-2 levels: even columns in [0,S/2), odd columns in [S/2,S)
//                             of each row (LDG.128 + 2 x STS.64).  In both layouts a window's
//                             base word is ystep*wy*S + wx with ystep*S = 8 (mod 32), so its
//                             bank class is (wx + 8*wy) mod 32: the 32 lanes of a warp with
//                             consecutive wx never conflict, and neither do compacted rows
//                             whose windows have distinct classes.
//   sgf     float [2048]      per-window sigma rounded to FP32 for the phase-1 filter (the FP64
//                             value is recomputed where exact arithmetic needs it)
//   list    u16 [2048]        survivors (phase 1 output; per-warp segments compacted in place in phase 2)
//
// Phase 1, "fixed geometry" (stages 0 .. n_fixed-1, where most windows are still alive):
//   thread t owns the column of 8 windows (wx = t & 63, wy = (t >> 6) + 4k).  Their tile
//   addresses differ by a compile-time constant, so a corner address is computed ONCE per
//   stump and the 4 windows of a chunk are read with immediate offsets (LDS [R + k*ROWSTEP]):
//   no per-window address arithmetic, no compaction traffic, conflict-free banks.  Stumps
//   come from the constant bank (the packed cascade is a kernel parameter), a stage's two-rect
//   stumps with two common corners first, in their six-load form.  An FP32 filter
//   decides each stump; whenever |s32 - t32| is inside a guard band (2^-20 |t32| plus the
//   cancellation terms) the window's whole stage is redone by dense_stage_exact(), which
//   reproduces the reference's C expressions bit for bit.  Outside the band both agree by the
//   error analysis in DESIGN.md, so results are identical to the all-FP64 evaluation (tests
//   also run with force_exact = 1 and compare).
// Hand-over: the survivors are counting-sorted by bank class and dealt to the eight warps.
// Phase 2, warp-autonomous (all remaining stages the tile kernel knows; see the kernel body):
//   stump-based upright cascades are finished here; the others hand the survivors of their
//   eligible prefix to the queue of k_cascade_mid / k_cascade_deep.
// ------------------------------------------------------------------------------------
// Tile accesses use 32-bit shared-window addresses and explicit ld.shared (a generic pointer
// would make the compiler rebuild the shared window base inside every loop).
__device__ __forceinline__ int lds32(uint32_t addr) {
    int v;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
template <int IMM>
__device__ __forceinline__ int lds32i(uint32_t addr) {
    int v;
    asm volatile("ld.shared.s32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(IMM));
    return v;
}

struct DenseSmemPlan {
    size_t tile, sgf, list, ctl, bar, act, tgt, total;
};
// control block (ints): the tile's 32 per-class window counters
constexpr int kCtlInts = 32;
__host__ __device__ inline DenseSmemPlan dense_smem_plan(const DenseParams &P) {
    DenseSmemPlan p;
    const size_t rows = (size_t)(P.tile_h - 1) * P.ystep + P.win_h + 1, windows = (size_t)kTileW * P.tile_h;
    p.tile = 0;
    p.sgf = (rows * P.tile_stride * 4 + 127) & ~(size_t)127;
    if (P.tilted_tile) p.sgf *= 2;   // second tile: the tilted integral (same geometry)
    p.list = p.sgf + windows * sizeof(float);
    p.ctl = p.list + windows * sizeof(uint16_t);
    p.bar = p.ctl + kCtlInts * sizeof(int);
    p.act = p.tgt = p.total = p.bar + 16;
    if (P.exec_stages > P.tail_stages) {   // stage tree: the windows of the current stage, every window's target position
        p.tgt = p.act + windows * sizeof(uint16_t);
        p.total = p.tgt + windows;
    }
    return p;
}
#ifdef CLFD_TILES_COUNT_TU
constexpr bool kTilesCount = true;
#else
constexpr bool kTilesCount = false;
#endif

struct DenseCtx {
    uint32_t tile;    // shared-window address of the tile
    const ull *gsq;   // squared integral (frame base; 64-bit elements or, sq32, 32-bit ones)
    size_t sq_at;     // element offset of the tile origin
    bool sq32;
    int16_t *codes;   // this frame + level, or nullptr
    int sq_pitch;     // elements
    int row_mul;      // bytes between window rows in the tile
    int ystep, S, half;   // half: word offset of a row's odd columns (ystep-2 layout)
    int tx, wy_tile, nx;   // tile column; first window row of the tile
    int code_mul;
};

__device__ __forceinline__ uint32_t dense_base(const DenseCtx &c, int wid) {
    return c.tile + (uint32_t)((wid / kTileW) * c.row_mul + (wid & (kTileW - 1)) * 4);
}
__device__ __forceinline__ uint32_t dense_tile_off(const DenseCtx &c, int y, int x) {   // byte offset of integral (y, x) from a window base
    return 4u * (uint32_t)(c.ystep == 1 ? y * c.S + x : y * c.S + (x & 1) * c.half + (x >> 1));
}
__device__ __forceinline__ void dense_write_code(const DenseCtx &c, int wid, int code) {
    const int wx = wid & (kTileW - 1), wy = wid / kTileW;
    c.codes[(size_t)(c.wy_tile + wy) * c.nx + c.tx * kTileW + wx] = (int16_t)code;
}

// FP64 sigma of window `wid` (tempcv.cpp:824-832): int32 corners from the tile, uint64 from global
__device__ __forceinline__ double dense_sigma(const DenseParams &P, const DenseCtx &c, int wid) {
    const int wx = wid & (kTileW - 1), wy = wid / kTileW;
    const int ex = P.eq_x, ey = P.eq_y, eq_w = P.eq_w, eq_h = P.eq_h;
    const uint32_t base = dense_base(c, wid);
    const int s4 = lds32(base + dense_tile_off(c, ey, ex)) - lds32(base + dense_tile_off(c, ey, ex + eq_w)) -
                   lds32(base + dense_tile_off(c, ey + eq_h, ex)) + lds32(base + dense_tile_off(c, ey + eq_h, ex + eq_w));
    const int g0 = ey * c.sq_pitch + ex, g1 = g0 + eq_w, g2 = (ey + eq_h) * c.sq_pitch + ex, g3 = g2 + eq_w;
    const ull q4 = sq_rect(c.gsq, c.sq32, c.sq_at + (size_t)(wy * c.ystep) * c.sq_pitch + wx * c.ystep, g0, g1, g2, g3);
    return window_sigma(s4, q4, P.inv_area);
}
// the same, and whether the variance rectangle is FLAT (every pixel equal): Q A == S^2 exactly (Cauchy-Schwarz with equality)
__device__ __forceinline__ double dense_sigma_flat(const DenseParams &P, const DenseCtx &c, int wid, bool &eq_flat) {
    const int wx = wid & (kTileW - 1), wy = wid / kTileW;
    const int ex = P.eq_x, ey = P.eq_y, eq_w = P.eq_w, eq_h = P.eq_h;
    const uint32_t base = dense_base(c, wid);
    const int s4 = lds32(base + dense_tile_off(c, ey, ex)) - lds32(base + dense_tile_off(c, ey, ex + eq_w)) -
                   lds32(base + dense_tile_off(c, ey + eq_h, ex)) + lds32(base + dense_tile_off(c, ey + eq_h, ex + eq_w));
    const int g0 = ey * c.sq_pitch + ex, g1 = g0 + eq_w, g2 = (ey + eq_h) * c.sq_pitch + ex, g3 = g2 + eq_w;
    const ull q4 = sq_rect(c.gsq, c.sq32, c.sq_at + (size_t)(wy * c.ystep) * c.sq_pitch + wx * c.ystep, g0, g1, g2, g3);
    eq_flat = q4 * (ull)(eq_w * eq_h) == (ull)((long long)s4 * s4);
    return window_sigma(s4, q4, P.inv_area);
}

// Flat windows -- every pixel of the window equal: black bars, saturated or empty regions -- are the one systematic
// customer of the FP64 fallback: sigma is 0 or rounding noise and every feature sum cancels to (almost) nothing, so every
// stump lands inside its guard band and the window walks its stages one exact evaluation after the other (an all-black
// 1080p batch ran at 890 frames/s instead of 2300, frontalface_default at 306).  But a flat window's rect sums, its
// sigma and with them its whole path through the cascade depend on the pixel value alone, so its exit code comes from a
// table of 256 entries that the detector measured once with these same kernels (clfd_api.cu, build_flat_table).  The
// variance rectangle's flatness falls out of the sums sigma needs anyway; only then is the whole window tested (rare
// path, a function of its own).  Returns the window's exit code, or kNotFlat.
constexpr int kNotFlat = -0x8000;
static __device__ __noinline__ int flat_window_code(const DenseParams &P, const DenseCtx &c, int wid) {
    const uint32_t base = dense_base(c, wid);
    const int W = P.win_w, H = P.win_h;
    const uint32_t S4 = (uint32_t)(lds32(base + dense_tile_off(c, 0, 0)) - lds32(base + dense_tile_off(c, 0, W)) -
                                   lds32(base + dense_tile_off(c, H, 0)) + lds32(base + dense_tile_off(c, H, W)));   // <= 255 W H
    const ull Q4 = sq_rect(c.gsq, c.sq32, c.sq_at + (size_t)((wid / kTileW) * c.ystep) * c.sq_pitch + (wid & (kTileW - 1)) * c.ystep,
                           0, W, H * c.sq_pitch, H * c.sq_pitch + W);
    const uint32_t A = (uint32_t)(W * H);
    if (Q4 * (ull)A != (ull)S4 * (ull)S4) return kNotFlat;
    return (int)__ldg(P.flat_code + S4 / A);
}

// One stump in registers.
struct StumpRegs {
    uint32_t o[12];
    float w0, w1, w2, thr, a0, a1;
    uint32_t meta;
};
__device__ __forceinline__ StumpRegs stump_from_param(const DenseStump &q) {   // constant bank (LDC)
    StumpRegs r;
#pragma unroll
    for (int i = 0; i < 12; i++) r.o[i] = q.off[i];
    r.w0 = q.w[0]; r.w1 = q.w[1]; r.w2 = q.w[2]; r.thr = q.thr; r.a0 = q.a0; r.a1 = q.a1; r.meta = q.meta;
    return r;
}
// Global records of a stage are stored in blocks of 32 stumps, chunk-interleaved: the five 16-byte chunks of
// a record (offsets 0-3, 4-7, 8-11, weights + threshold, leaf values + meta) lie 512 bytes apart, chunk c of
// stump j at rec[(j / 32) * 160 + c * 32 + j % 32].  When the lanes of a warp are on different stumps (window x
// group mode: G consecutive stumps) one LDG.128 touches G/8 cache lines instead of the 0.6 G lines of
// 80-byte records -- 22 % of the kernel's L1 data-pipe wavefronts were record fetches (profiles/README.md) --
// and the chunks are still one pointer plus immediates.
__device__ __forceinline__ StumpRegs stump_from_global(const uint4 *__restrict__ rec, int j, bool any3) {   // 4-5 x LDG.128
    rec += (j >> 5) * 160 + (j & 31);
    const uint4 q0 = __ldg(rec), q1 = __ldg(rec + 32), q3 = __ldg(rec + 96), q4 = __ldg(rec + 128);
    uint4 q2 = make_uint4(0u, 0u, 0u, 0u);
    if (any3) q2 = __ldg(rec + 64);
    StumpRegs r;
    r.o[0] = q0.x; r.o[1] = q0.y; r.o[2] = q0.z; r.o[3] = q0.w;
    r.o[4] = q1.x; r.o[5] = q1.y; r.o[6] = q1.z; r.o[7] = q1.w;
    r.o[8] = q2.x; r.o[9] = q2.y; r.o[10] = q2.z; r.o[11] = q2.w;
    r.w0 = __uint_as_float(q3.x); r.w1 = __uint_as_float(q3.y); r.w2 = __uint_as_float(q3.z); r.thr = __uint_as_float(q3.w);
    r.a0 = __uint_as_float(q4.x); r.a1 = __uint_as_float(q4.y); r.meta = q4.z;
    return r;
}

// FP64 fallbacks / near-threshold stage sums of this CTA (clfd_run_stats): counted in shared memory -- a 32-bit
// address known at link time, so the rare path costs the hot kernel no register -- and added to
// CascadeArgs::counters[4], [5] by the last warp that leaves the CTA.
__shared__ unsigned int s_dense_exact, s_dense_near, s_dense_done;
#ifdef CLFD_TILE_TIMING   // diagnostic build (make EXTRA=-DCLFD_TILE_TIMING, tools/tile_timing.py): where a CTA's warp slots go
__shared__ unsigned int s_dense_t_busy, s_dense_t_p1;   // sum over warps: cycles until the warp left the kernel / entered phase 2
#endif

// Exact evaluation of one stage for one window: the reference's arithmetic, stumps in tree order.
template <bool NODES>
__device__ __noinline__ int dense_stage_exact(const DenseParams &P, const DenseCtx &c, uint32_t tail_first, int count, bool dbl,
                                               float sthr, int wid) {
    const uint32_t base = dense_base(c, wid);
    const double sigma = dense_sigma(P, c, wid);
    const uint4 *rec = reinterpret_cast<const uint4 *>(P.tail + tail_first);
    double S = 0.0;
    uint32_t at = 0;   // multi-node trees: the node this window is at (icvEvalHidHaarClassifier, tempcv.cpp:771-792)
    for (int j = 0; j < count; j++) {
        const StumpRegs q = stump_from_global(rec, j, true);
        if (NODES) {
            if ((q.meta & 255u) == 0u) at = 0;
            if ((q.meta & 255u) != at) continue;
        }
        const int r0 = lds32(base + q.o[0]) - lds32(base + q.o[1]) - lds32(base + q.o[2]) + lds32(base + q.o[3]);
        const int r1 = lds32(base + q.o[4]) - lds32(base + q.o[5]) - lds32(base + q.o[6]) + lds32(base + q.o[7]);
        const double t = __dmul_rn((double)q.thr, sigma);
        double sum;
        if (dbl) {  // tempcv.cpp:872-898; both products are exact in double, so fma == mul, mul, add
            sum = __fma_rn((double)r1, (double)q.w1, __dmul_rn((double)r0, (double)q.w0));
        } else {    // tempcv.cpp:899-930 / 782-786: float products, double accumulation
            sum = __dadd_rn((double)__fmul_rn(__int2float_rn(r0), q.w0), (double)__fmul_rn(__int2float_rn(r1), q.w1));
            if (q.o[11] != 0) {
                const int r2 = lds32(base + q.o[8]) - lds32(base + q.o[9]) - lds32(base + q.o[10]) + lds32(base + q.o[11]);
                sum = __dadd_rn(sum, (double)__fmul_rn(__int2float_rn(r2), q.w2));
            }
        }
        if (NODES) {
            at = ((sum >= t ? q.meta >> 16 : q.meta >> 8)) & 255u;
            if (at != kNodeLeaf) continue;   // on to a child node: nothing to add yet
        }
        S = __dadd_rn(S, (double)(sum >= t ? q.a1 : q.a0));
    }
    // counted and reported (north star): FP64 fallbacks, and stage sums within 1e-5 relative of the threshold --
    // the packer widens the FP32 band by that much, so every such event comes through here
    // bit 0: the verdict; bit 1: the stage sum lies within 1e-5 relative of the threshold (counted by the caller)
    const double thr = (double)sthr;
    return (S >= thr ? 1 : 0) | (fabs(__dsub_rn(S, thr)) <= __dmul_rn(1e-5, fabs(thr)) ? 2 : 0);
}

// FP32 filter: one stump for K windows of this thread.  The stump decision sign(s - t) is taken
// from FP32 arithmetic; near[k] records that |s32 - t32| fell inside the guard band (2^-20 |t32|
// plus the cancellation terms, DESIGN.md), S[k] adds the selected alpha in FP32.
//   FIXED = true : window k lives at base[0] + k*ROWSTEP (compile-time) -> immediate offsets
//   FIXED = false: window k lives at base[k]
//   NODES = true : multi-node trees; at[k] = the node window k is at, a record only counts for the
//                  windows that are at its node (the others still load its corners: uniform code)
//   TRACK = true : also Sa[k] += |selected alpha| (cascades with sentinel leaf values: the stage verdict then bounds the
//                  error of the FP32 sum by what was actually added, see stage_verdict)
template <int KK, int K, bool FIXED, int ROWSTEP, bool SHARED, bool NODES, bool TRACK>
__device__ __forceinline__ void stump_filter_window(const StumpRegs &q, bool dbl, bool three, float eps, const uint32_t (&c)[12],
                                                    const uint32_t (&base)[K], const float (&sg)[K], float (&S)[K], bool (&near)[K],
                                                    uint32_t (&at)[K], float (&Sa)[K]) {
    const float eps4 = eps * 0.25f;
    constexpr int IMM = KK * ROWSTEP;
    const uint32_t b = base[FIXED ? 0 : KK];
    int r0, r1;
    if (SHARED) {   // two rects with two common corners, six offsets (haar_pack.cpp)
        int e, f, g;
        if (FIXED) {
            e = lds32i<IMM>(c[0]) - lds32i<IMM>(c[1]); f = lds32i<IMM>(c[2]) - lds32i<IMM>(c[3]); g = lds32i<IMM>(c[4]) - lds32i<IMM>(c[5]);
        } else {
            e = lds32(b + q.o[0]) - lds32(b + q.o[1]); f = lds32(b + q.o[2]) - lds32(b + q.o[3]); g = lds32(b + q.o[4]) - lds32(b + q.o[5]);
        }
        r0 = e + f; r1 = e + g;
    } else if (FIXED) {   // LDS [corner of window 0 + immediate]
        r0 = lds32i<IMM>(c[0]) - lds32i<IMM>(c[1]) - lds32i<IMM>(c[2]) + lds32i<IMM>(c[3]);
        r1 = lds32i<IMM>(c[4]) - lds32i<IMM>(c[5]) - lds32i<IMM>(c[6]) + lds32i<IMM>(c[7]);
    } else {
        r0 = lds32(b + q.o[0]) - lds32(b + q.o[1]) - lds32(b + q.o[2]) + lds32(b + q.o[3]);
        r1 = lds32(b + q.o[4]) - lds32(b + q.o[5]) - lds32(b + q.o[6]) + lds32(b + q.o[7]);
    }
    // p0 is the reference's own float product; the second (and third) product goes into the sum unrounded (FFMA): that
    // is closer to the double-product stages' exact sum, and differs from a float-product stage's rounded product by at
    // most 2^-24 |r1 w1| <= 2^-24 (|p0| + |s32|).  Either way the band eps |t32| + eps/4 |p0| covers it (DESIGN.md).
    const float p0 = __fmul_rn(__int2float_rn(r0), q.w0);
    float s32 = __fmaf_rn(__int2float_rn(r1), q.w1, p0);
    // eps is a power of two: |thr| (sg eps) == |thr sg| eps, and sg eps does not depend on the stump (hoisted)
    float m = __fmaf_rn(fabsf(p0), eps4, __fmul_rn(fabsf(q.thr), __fmul_rn(sg[KK], eps)));
    if (!SHARED && three) {
        int r2;
        if (FIXED) r2 = lds32i<IMM>(c[8]) - lds32i<IMM>(c[9]) - lds32i<IMM>(c[10]) + lds32i<IMM>(c[11]);
        else r2 = lds32(b + q.o[8]) - lds32(b + q.o[9]) - lds32(b + q.o[10]) + lds32(b + q.o[11]);
        m = __fmaf_rn(fabsf(s32), eps4, m);   // rounding of the first sum, the third product unrounded
        s32 = __fmaf_rn(__int2float_rn(r2), q.w2, s32);
    }
    const float d = __fmaf_rn(-q.thr, sg[KK], s32);   // s32 - thr sigma, rounded once
    if (NODES) {
        const bool on = at[KK] == (q.meta & 255u);
        near[KK] = near[KK] || (on && fabsf(d) <= m);
        S[KK] = __fadd_rn(S[KK], on ? (d >= 0.f ? q.a1 : q.a0) : 0.f);   // a branch to another node carries 0
        at[KK] = on ? ((d >= 0.f ? q.meta >> 16 : q.meta >> 8) & 255u) : at[KK];
    } else {
        near[KK] = near[KK] || (fabsf(d) <= m);
        const float sel = d >= 0.f ? q.a1 : q.a0;
        S[KK] = __fadd_rn(S[KK], sel);
        if (TRACK) Sa[KK] = __fadd_rn(Sa[KK], fabsf(sel));
    }
}

template <int K, bool FIXED, int ROWSTEP, bool SHARED, bool NODES, bool TRACK>
__device__ __forceinline__ void stump_filter(const StumpRegs &q, bool dbl, bool any3, float eps, const uint32_t (&base)[K],
                                             const float (&sg)[K], float (&S)[K], bool (&near)[K], uint32_t (&at)[K], float (&Sa)[K]) {
    static_assert(K >= 1 && K <= 4, "1..4 windows per thread");
    const bool three = !SHARED && any3 && q.o[11] != 0u;   // warp-uniform per stump
    uint32_t c[12];
    if (FIXED) {   // corner addresses of window 0, shared by all K windows
#pragma unroll
        for (int i = 0; i < (SHARED ? 6 : 12); i++) c[i] = base[0] + q.o[i];
    }
    if (NODES && (q.meta & 255u) == 0u) {   // a tree's root: every window starts over
#pragma unroll
        for (int k = 0; k < K; k++) at[k] = 0u;
    }
    stump_filter_window<0, K, FIXED, ROWSTEP, SHARED, NODES, TRACK>(q, dbl, three, eps, c, base, sg, S, near, at, Sa);
    if (K > 1) stump_filter_window<(K > 1 ? 1 : 0), K, FIXED, ROWSTEP, SHARED, NODES, TRACK>(q, dbl, three, eps, c, base, sg, S, near, at, Sa);
    if (K > 2) stump_filter_window<(K > 2 ? 2 : 0), K, FIXED, ROWSTEP, SHARED, NODES, TRACK>(q, dbl, three, eps, c, base, sg, S, near, at, Sa);
    if (K > 3) stump_filter_window<(K > 3 ? 3 : 0), K, FIXED, ROWSTEP, SHARED, NODES, TRACK>(q, dbl, three, eps, c, base, sg, S, near, at, Sa);
}

// Stumps grp, grp + G, ... of stage st for K windows of this lane.  Stumps come from the
// constant bank when the stage is parameter resident (`resident`), else from global memory.
template <int K, bool FIXED, int ROWSTEP, bool NODES, bool TRACK>
__device__ __forceinline__ void stage_filter(const DenseParams &P, const DenseStage &st, bool resident, int grp, int G,
                                             const uint32_t (&base)[K], const float (&sg)[K], float (&S)[K], bool (&near)[K],
                                             float (&Sa)[K]) {
    uint32_t at[K];
#pragma unroll
    for (int k = 0; k < K; k++) at[k] = 0u;
    const int count = st.count;
    const uint32_t flags = st.flags;
    const bool dbl = flags & 1u, any3 = flags & 2u;
    const float eps = P.filter_eps;
    if (resident && G == 1) {   // all lanes on the same stump: constant bank (reordered copy: six-load stumps first)
        const int first = st.first, n6 = (int)st.n_shared;
#pragma unroll 1
        for (int j = 0; j < n6; j++) stump_filter<K, FIXED, ROWSTEP, true, false, TRACK>(stump_from_param(P.stump[first + j]), dbl, false, eps, base, sg, S, near, at, Sa);
#pragma unroll 1
        for (int j = n6; j < count; j++) stump_filter<K, FIXED, ROWSTEP, false, NODES, TRACK>(stump_from_param(P.stump[first + j]), dbl, any3, eps, base, sg, S, near, at, Sa);
    } else {
        const uint4 *__restrict__ rec = reinterpret_cast<const uint4 *>(P.tail + st.tail_first);
        if (NODES) {   // the groups split the stage by whole trees
            const int npt = P.npt;
#pragma unroll 1
            for (int j = grp * npt; j < count; j += G * npt)
#pragma unroll 1
                for (int i = 0; i < npt; i++)
                    stump_filter<K, FIXED, ROWSTEP, false, true, TRACK>(stump_from_global(rec, j + i, any3), dbl, any3, eps, base, sg, S, near, at, Sa);
        } else {
#pragma unroll 1
            for (int j = grp; j < count; j += G) stump_filter<K, FIXED, ROWSTEP, false, false, TRACK>(stump_from_global(rec, j, any3), dbl, any3, eps, base, sg, S, near, at, Sa);
        }
    }
}

// Stage verdict of one window from its FP32 stage sum.  |S32 - S| <= sum_eps for any summation
// order, so outside that band (and with no stump inside its own band) the FP32 verdict is the
// reference's; inside, the stage is redone exactly.
// TRACK (cascades with sentinel leaf values, DenseParams::track_abs): sum_eps is built from the LARGEST leaf of every
// stump; one leaf of 2e6 (haarcascade_mcs_upperbody, stage 2) makes it 24.5 and sends every window of the stage through
// the FP64 path.  There the bound is taken from what was actually added, n 2^-23 Sa with Sa = sum |selected alpha|
// (the same (n-1) 2^-24 sum|x| bound with 2x slack; Sa itself is an FP32 sum of non-negative terms, low by at most
// n 2^-24 relative), plus the same 1e-5 |thr| band: a window that picked the sentinel is far from the threshold, one
// that did not has a small Sa.
template <bool NODES, bool COUNT, bool TRACK>
__device__ __forceinline__ bool stage_verdict(const DenseParams &P, const DenseCtx &c, const DenseStage &st, float sthr, float seps,
                                              int wid, float S, bool near, float Sa) {
    if (TRACK && !P.force_exact)
        seps = __fadd_ru(__fmul_ru(__fmul_ru((float)st.count, 1.1920930e-7f), Sa), __fadd_ru(__fmul_ru(1.0001e-5f, fabsf(sthr)), 1.2e-38f));
    if (near || !(fabsf(__fadd_rn(S, -sthr)) > seps)) {
        const int r = dense_stage_exact<NODES>(P, c, st.tail_first, st.count, st.flags & 1u, st.thr, wid);
        if (COUNT) {   // diagnostic instantiation only: even these two lines cost the hot kernel 1.5-4.5 % (code growth at 8 sites)
            atomicAdd(&s_dense_exact, 1u);
            if (r & 2) atomicAdd(&s_dense_near, 1u);
        }
        return r & 1;
    }
    return S >= sthr;
}

// ROWSTEP_T: compile-time byte distance between a thread's consecutive windows in phase 1
// (= kDenseThreads / kTileW window rows), or 0 to use the runtime value (generic window sizes).
// TREE: the cascade is a stage tree the kernel walks itself (DenseParams::exec_stages > tail_stages).
// NODES: multi-node trees (DenseParams::npt > 1).
// TILE_H: window rows per tile (== DenseParams::tile_h).
template <int ROWSTEP_T, bool TREE, bool NODES, int TILE_H, bool COUNT, bool TRACK>
__device__ __forceinline__ void cascade_tiles_body(const DenseParams &P, const CascadeArgs &a, const int tile0, unsigned char *smem_raw) {
    const DenseSmemPlan plan = dense_smem_plan(P);
    unsigned char *tile = smem_raw + plan.tile;
    float *sgf = reinterpret_cast<float *>(smem_raw + plan.sgf);
    uint16_t *list = reinterpret_cast<uint16_t *>(smem_raw + plan.list);
    int *ctl = reinterpret_cast<int *>(smem_raw + plan.ctl);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw + plan.bar);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int frame = blockIdx.y;
    const int tile_id = tile0 + blockIdx.x;

    int cl = 0;   // which level does this tile belong to?
    {
        int lo = 0, hi = a.n_cas_levels - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (__ldg(&a.cas_levels[mid].tile_base) <= tile_id) lo = mid; else hi = mid - 1;
        }
        cl = lo;
    }
    const CasLevel CL = a.cas_levels[cl];
    const PyrLevel L = a.levels[CL.pyr_level];
    const int local = tile_id - CL.tile_base;
    const int tx = local % CL.tiles_x, ty = local / CL.tiles_x;
    const int ystep = P.ystep;   // == CL.ystep by construction of the launch
    constexpr int kTileWindows = kTileW * TILE_H, kDenseSlots = kTileWindows / kDenseThreads;   // (shadow the 32-row constants)
    constexpr int kDenseChunk = kDenseSlots % 4 == 0 ? 4 : 3;   // windows a thread carries through a fixed stage at once
    static_assert(kDenseSlots % kDenseChunk == 0 && kDenseSlots <= 8, "tile height: 12, 16, 24 or 32 window rows");
    const int px0 = tx * kTileW * ystep, py0 = ty * TILE_H * ystep;   // tile origin in the integral image
    const int n_wx = min(kTileW, CL.nx - tx * kTileW), n_wy = min(TILE_H, CL.ny - ty * TILE_H);
    const int rows = min((TILE_H - 1) * ystep + P.win_h + 1, L.h + 1 - py0);
    const int cols = ((kTileW - 1) * ystep + P.win_w + 1 + 3) & ~3;
    const int S = P.tile_stride;

    const size_t frame_off = (size_t)frame * a.sum_frame_stride + L.sum_off;
    const int32_t *__restrict__ gsum = a.sum + frame_off + (size_t)py0 * L.sum_pitch + px0;

    // ---- stage the integral tile ----
    for (int i = tid; i < kCtlInts; i += kDenseThreads) ctl[i] = 0;
    if (tid == 0) s_dense_exact = s_dense_near = s_dense_done = 0u;   // (a block barrier follows on either staging path)
#ifdef CLFD_TILE_TIMING
    const long long t_start = clock64();
    if (tid == 0) s_dense_t_busy = s_dense_t_p1 = 0u;
#endif
    const int n_tiles_smem = P.tilted_tile ? 2 : 1;
    const size_t tile2_off = ((size_t)((TILE_H - 1) * ystep + P.win_h + 1) * S * 4 + 127) & ~(size_t)127;
    const int32_t *__restrict__ gtil = a.tilted ? a.tilted + frame_off + (size_t)py0 * L.sum_pitch + px0 : gsum;
    if (ystep == 1) {   // natural layout: one TMA bulk copy per row
        if (tid == 0) mbar_init(bar, 1);
        __syncthreads();
        if (tid == 0) mbar_expect_tx(bar, (uint32_t)(rows * cols * 4 * n_tiles_smem));
        for (int r = tid; r < rows * n_tiles_smem; r += kDenseThreads) {
            const int t2 = r >= rows, rr = t2 ? r - rows : r;
            tma_bulk_g2s(tile + (t2 ? tile2_off : 0) + (size_t)rr * S * 4, (t2 ? gtil : gsum) + (size_t)rr * L.sum_pitch,
                         (uint32_t)(cols * 4), bar);
        }
        mbar_wait(bar, 0);
    } else {
        // ystep-2 layout: x -> (x&1)*half + (x>>1).  A level whose integral is stored de-interleaved (PyrLevel::di,
        // CascadeArgs::sum_di) is staged with two TMA bulk copies per row -- off the L1 data pipe this kernel is bound by;
        // anything else (the tilted integral's tile, detectors without di) with LDG.128 + 2 x STS.64
        const bool di = a.sum_di != 0;
        const int half = P.tile_half;
        if (di) {
            if (tid == 0) mbar_init(bar, 1);
            __syncthreads();
            const uint32_t hb = (uint32_t)half * 4u;   // bytes of one half row (>= cols / 2 elements, a 16-byte multiple)
            if (tid == 0) mbar_expect_tx(bar, (uint32_t)rows * 2u * hb);
            const int32_t *__restrict__ gdi = a.sum + frame_off + (size_t)py0 * L.sum_pitch + (px0 >> 1);
            for (int r = tid; r < rows * 2; r += kDenseThreads) {
                const int odd = r >= rows, rr = odd ? r - rows : r;
                tma_bulk_g2s(tile + (size_t)rr * S * 4 + (odd ? hb : 0u), gdi + (size_t)rr * L.sum_pitch + (odd ? (L.sum_pitch >> 1) : 0), hb, bar);
            }
        }
        const int c4 = cols >> 2, total = rows * c4;
        for (int i = (di ? total : 0) + tid; i < total * n_tiles_smem; i += kDenseThreads) {
            const int t2 = i >= total, ii = t2 ? i - total : i;
            const int r = ii / c4, cq = ii - r * c4;
            const int4 v = __ldg(reinterpret_cast<const int4 *>((t2 ? gtil : gsum) + (size_t)r * L.sum_pitch) + cq);
            int *row = reinterpret_cast<int *>(tile + (t2 ? tile2_off : 0)) + r * S;
            *reinterpret_cast<int2 *>(row + 2 * cq) = make_int2(v.x, v.z);
            *reinterpret_cast<int2 *>(row + half + 2 * cq) = make_int2(v.y, v.w);
        }
        __syncthreads();
        if (di) mbar_wait(bar, 0);
    }

    DenseCtx c;
    c.tile = smem_u32(tile); c.gsq = a.sq; c.sq_at = frame_off + (size_t)py0 * L.sum_pitch + px0; c.sq32 = a.sq32 != 0;
    c.codes = a.codes ? a.codes + (size_t)frame * a.windows_per_frame + CL.win_base : nullptr;
    c.sq_pitch = L.sum_pitch;
    c.row_mul = ystep * S * 4;
    c.ystep = ystep; c.S = S; c.half = P.tile_half;
    c.tx = tx; c.wy_tile = ty * TILE_H; c.nx = CL.nx;
    c.code_mul = P.is_tree ? 2 : 1;
    const float inf = __int_as_float(0x7f800000);

    // ---- phase 1: sigma, then the fixed-geometry stages ----
    constexpr int kRowsPerSlot = kDenseThreads / kTileW;   // window rows between a thread's slots (4)
    const int wx = tid & (kTileW - 1), wy0 = tid / kTileW;
    uint32_t alive = 0;   // bit k: window (wx, wy0 + 2k) still alive
#pragma unroll
    for (int k = 0; k < kDenseSlots; k++) {
        const int wy = wy0 + k * kRowsPerSlot;
        const int wid = wy * kTileW + wx;
        if (wx < n_wx && wy < n_wy) {
            bool eq_flat, live = true;
            sgf[wid] = (float)dense_sigma_flat(P, c, wid, eq_flat);
            if (!COUNT && eq_flat && P.flat_code) {   // (the diagnostic instantiation evaluates flat windows like any other)
                const int code = flat_window_code(P, c, wid);
                if (code != kNotFlat) {
                    live = false;
                    if (P.is_tree ? (code & 1) : (code == P.total_stages)) emit_rect(a, CL, frame, px0 + wx * ystep, py0 + wy * ystep);
                }
            }
            if (live) alive |= 1u << k;
        } else {
            sgf[wid] = 1.0f;
        }
    }
    // a thread reads back only sigmas it wrote itself: no barrier needed in phase 1
    int s = 0;
    for (; s < P.n_fixed; s++) {
        const float sthr = P.stage[s].thr, seps = P.force_exact ? inf : P.stage[s].sum_eps;
#pragma unroll 1
        for (int k0 = 0; k0 < kDenseSlots; k0 += kDenseChunk) {
            const uint32_t m4 = (alive >> k0) & ((1u << kDenseChunk) - 1u);
            if (!__any_sync(0xffffffffu, m4 != 0)) continue;   // whole 4 x 32 block is dead
            uint32_t base[kDenseChunk];
            float sg[kDenseChunk];
            float Ssum[kDenseChunk];
            bool near[kDenseChunk];
#pragma unroll
            for (int k = 0; k < kDenseChunk; k++) {
                const int wy = wy0 + (k0 + k) * kRowsPerSlot;
                base[k] = c.tile + (uint32_t)(wy * c.row_mul + wx * 4);   // == base[0] + k * rowstep
                sg[k] = sgf[wy * kTileW + wx];
                Ssum[k] = 0.f;
                near[k] = false;
            }
            float Sabs[kDenseChunk];
#pragma unroll
            for (int k = 0; k < kDenseChunk; k++) Sabs[k] = 0.f;
            if (ROWSTEP_T) stage_filter<kDenseChunk, true, ROWSTEP_T, NODES, TRACK>(P, P.stage[s], true, 0, 1, base, sg, Ssum, near, Sabs);
            else stage_filter<kDenseChunk, false, 0, NODES, TRACK>(P, P.stage[s], true, 0, 1, base, sg, Ssum, near, Sabs);
#pragma unroll
            for (int k = 0; k < kDenseChunk; k++) {
                if (!((m4 >> k) & 1u)) continue;
                const int wid = (wy0 + (k0 + k) * kRowsPerSlot) * kTileW + wx;
                if (!stage_verdict<NODES, COUNT, TRACK>(P, c, P.stage[s], sthr, seps, wid, Ssum[k], near[k], Sabs[k])) {
                    alive &= ~(1u << (k0 + k));
                    if (c.codes) dense_write_code(c, wid, s * c.code_mul);
                }
            }
        }
    }

    // ---- phase-1 survivors -> per-warp lists ----
    // A window's bank class is (wx + 8*wy) mod 32 (the skew of the tile rows): two windows of a
    // row conflict on every corner load iff their classes are equal, and a load costs as many
    // wavefronts as the row's most frequent class has members.  The survivors are dealt to the
    // warps in class-sorted order (rank i = windows of lower classes + position in the class:
    // warp i % 8, position p = i / 8, column-major over the warp's R rows: row p % R) -- windows of
    // one class end up in different warps / rows -- and every warp finishes its share on its own,
    // without block barriers.  One shared-memory atomic per thread reserves its windows' positions
    // in their class (a thread's windows share one: wy advances by 4 rows = 32 in 8*wy); every warp
    // derives the class prefix itself.
    constexpr int kSeg = kTileWindows / kDenseWarps;   // list segment of a warp (its share is at most this)
    const int na = __popc(alive), cq = (wx + 8 * wy0) & 31;
    int at = na ? atomicAdd(ctl + cq, na) : 0;
    __syncthreads();
    const int h = ctl[lane];
    int incl = h;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    const int n_alive = __shfl_sync(0xffffffffu, incl, 31);
    if (n_alive == 0) return;
    at += __shfl_sync(0xffffffffu, incl - h, cq);
#pragma unroll
    for (int k = 0; k < kDenseSlots; k++) {
        if ((alive >> k) & 1u) {
            const int i = at++;
            const int w = i % kDenseWarps, p = i / kDenseWarps;
            const int nw = (n_alive - w + kDenseWarps - 1) / kDenseWarps, Rw = (nw + 31) >> 5;
            const int col = p / Rw, row = p - col * Rw;
            list[w * kSeg + row * 32 + col] = (uint16_t)((wy0 + k * kRowsPerSlot) * kTileW + wx);
        }
    }
    __syncthreads();
    uint16_t *const cur = list + warp * kSeg;

    // ---- phase 2: every warp takes its share of the survivors through all remaining stages
    //      on its own: no block barrier, warp-local in-place re-compaction after every stage.
    //      More than 16 windows left: thread per window (rows of 32, two rows per pass so the
    //      stump loads are shared).  16 or fewer: the lanes are arranged as w window slots x G
    //      stump groups (w = smallest power of two >= windows, G = 32 / w): lane (slot, grp)
    //      evaluates stumps grp, grp + G, ... for window `slot`, and the G partial sums meet
    //      through xor-shuffles -- with one window left the warp does 32 stumps per pass. ----
#ifdef CLFD_TILE_TIMING
    if (lane == 0) atomicAdd(&s_dense_t_p1, (unsigned int)(clock64() - t_start));
#endif
    int n = (n_alive - warp + kDenseWarps - 1) / kDenseWarps;
    bool dealt = true;   // first compacted stage: balanced rows (row r holds (n - r + R - 1) / R entries)
    for (; s < P.tail_stages && n > 0; s++) {
        const float sthr = P.stage[s].thr, seps = P.force_exact ? inf : P.stage[s].sum_eps;
        int n_next = 0;
        // append the survivors among this pass's windows at cur[n_next..]: always at or below the
        // positions the pass has already read (in-place compaction)
        auto keep = [&](bool valid, int wid, float Ssum, bool near, float Sabs) {
            const bool pass = valid && stage_verdict<NODES, COUNT, TRACK>(P, c, P.stage[s], sthr, seps, wid, Ssum, near, Sabs);
            const unsigned m = __ballot_sync(0xffffffffu, pass);
            if (pass) cur[n_next + __popc(m & ((1u << lane) - 1u))] = (uint16_t)wid;
            n_next += __popc(m);
            if (valid && !pass && c.codes) dense_write_code(c, wid, s * c.code_mul);
        };
        if (n > P.g1_min) {
            const int R = (n + 31) >> 5;
            for (int r = 0; r < R; r += 2) {
                const int c0 = dealt ? (n - r + R - 1) / R : min(32, n - 32 * r);
                if (r + 1 < R) {   // two rows
                    const int c1 = dealt ? (n - r - 1 + R - 1) / R : min(32, n - 32 * (r + 1));
                    const bool v0 = lane < c0, v1 = lane < c1;
                    const int wid0 = cur[32 * r + (v0 ? lane : 0)], wid1 = cur[32 * r + 32 + (v1 ? lane : 0)];
                    __syncwarp();   // both rows are in registers before their slots are overwritten
                    const uint32_t base[2] = {dense_base(c, wid0), dense_base(c, wid1)};
                    const float sg[2] = {sgf[wid0], sgf[wid1]};
                    float Ssum[2] = {0.f, 0.f};
                    bool near[2] = {false, false};
                    float Sabs[2] = {0.f, 0.f};
                    stage_filter<2, false, 0, NODES, TRACK>(P, P.stage[s], s < P.n_stages, 0, 1, base, sg, Ssum, near, Sabs);
                    keep(v0, wid0, Ssum[0], near[0], Sabs[0]);
                    keep(v1, wid1, Ssum[1], near[1], Sabs[1]);
                } else {           // one row
                    const bool v0 = lane < c0;
                    const int wid0 = cur[32 * r + (v0 ? lane : 0)];
                    __syncwarp();
                    const uint32_t base[1] = {dense_base(c, wid0)};
                    const float sg[1] = {sgf[wid0]};
                    float Ssum[1] = {0.f};
                    bool near[1] = {false};
                    float Sabs[1] = {0.f};
                    stage_filter<1, false, 0, NODES, TRACK>(P, P.stage[s], s < P.n_stages, 0, 1, base, sg, Ssum, near, Sabs);
                    keep(v0, wid0, Ssum[0], near[0], Sabs[0]);
                }
            }
        } else {
            int lw = 4;
            while (lw > 0 && (1 << (lw - 1)) >= n) lw--;   // n <= 16 here
            const int slot = lane & ((1 << lw) - 1), grp = lane >> lw, G = 32 >> lw;
            const bool valid = slot < n;
            const int wid0 = cur[valid ? slot : 0];
            __syncwarp();
            const uint32_t base[1] = {dense_base(c, wid0)};
            const float sg[1] = {sgf[wid0]};
            float Ssum[1] = {0.f};
            bool near[1] = {false};
            float Sabs[1] = {0.f};
            if (valid) stage_filter<1, false, 0, NODES, TRACK>(P, P.stage[s], s < P.n_stages, grp, G, base, sg, Ssum, near, Sabs);
            float acc = Ssum[0], acc_abs = Sabs[0];
            unsigned nr = near[0];
            for (int d = 1 << lw; d < 32; d <<= 1) {
                acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, d));
                if (TRACK) acc_abs = __fadd_rn(acc_abs, __shfl_xor_sync(0xffffffffu, acc_abs, d));
                nr |= __shfl_xor_sync(0xffffffffu, nr, d);
            }
            keep(lane < n, wid0, acc, nr != 0, acc_abs);   // lane < n: slot == lane
        }
        __syncwarp();
        n = n_next;
        dealt = false;   // the compacted list is contiguous: rows of 32, the last one partial
    }
    if (TREE) {
        // ---- stage tree (tempcv.cpp:834-861): the remaining stages in execution order (depth-first
        //      preorder, haar_pack.cpp).  tgt[w] = the position window w waits for; at position e the
        //      warp splits its list into the windows whose turn it is (-> act) and the rest (stay in
        //      cur), evaluates act like a linear stage, and routes every window by the verdict:
        //      to a later position (back into cur), to a detection, or out. ----
        if (n == 0) return;
        uint16_t *act = reinterpret_cast<uint16_t *>(smem_raw + plan.act) + warp * kSeg;
        unsigned char *tgt = smem_raw + plan.tgt;
        const int e0 = s;
        for (int e = e0; e < P.exec_stages && n > 0; e++) {
            int n_wait = 0, n_act = 0;
            const int R = (n + 31) >> 5;
            for (int r = 0; r < R; r++) {
                const int c0 = dealt ? (n - r + R - 1) / R : min(32, n - 32 * r);
                const bool v = lane < c0;
                const int wid = cur[32 * r + (v ? lane : 0)];
                __syncwarp();
                const bool turn = v && (e == e0 || tgt[wid] == e);
                const unsigned mt = __ballot_sync(0xffffffffu, turn), mw = __ballot_sync(0xffffffffu, v && !turn);
                const unsigned below = (1u << lane) - 1u;
                if (turn) act[n_act + __popc(mt & below)] = (uint16_t)wid;
                else if (v) cur[n_wait + __popc(mw & below)] = (uint16_t)wid;
                n_act += __popc(mt);
                n_wait += __popc(mw);
            }
            __syncwarp();
            dealt = false;
            n = n_wait;
            if (n_act == 0) continue;
            const DenseStage st = P.stage_g[e];
            const float sthr = st.thr, seps = P.force_exact ? inf : st.sum_eps;
            const int orig = (st.flags >> 8) & 255;
            const uint32_t to_pass = (st.flags >> 16) & 255u, to_fail = st.flags >> 24;
            auto route = [&](bool valid, int wid, float Ssum, bool near, float Sabs) {
                uint32_t to = kRouteReject;
                bool pass = false;
                if (valid) {
                    pass = stage_verdict<NODES, COUNT, TRACK>(P, c, st, sthr, seps, wid, Ssum, near, Sabs);
                    to = pass ? to_pass : to_fail;
                }
                const bool on = valid && to < kRouteReject;
                const unsigned m = __ballot_sync(0xffffffffu, on);
                if (on) {
                    cur[n + __popc(m & ((1u << lane) - 1u))] = (uint16_t)wid;
                    tgt[wid] = (unsigned char)to;
                } else if (valid) {
                    if (to == kRouteAccept) emit_rect(a, CL, frame, px0 + (wid & (kTileW - 1)) * ystep, py0 + (wid / kTileW) * ystep);
                    if (c.codes) dense_write_code(c, wid, 2 * orig + (pass ? 1 : 0));
                }
                n += __popc(m);
            };
            if (n_act > P.g1_min) {
                const int Ra = (n_act + 31) >> 5;
                for (int r = 0; r < Ra; r += 2) {
                    const bool v0 = 32 * r + lane < n_act, v1 = 32 * r + 32 + lane < n_act;
                    const int wid0 = act[v0 ? 32 * r + lane : 0], wid1 = act[v1 ? 32 * r + 32 + lane : 0];
                    if (r + 1 < Ra) {
                        const uint32_t base[2] = {dense_base(c, wid0), dense_base(c, wid1)};
                        const float sg[2] = {sgf[wid0], sgf[wid1]};
                        float Ssum[2] = {0.f, 0.f};
                        bool near[2] = {false, false};
                        float Sabs[2] = {0.f, 0.f};
                        stage_filter<2, false, 0, NODES, TRACK>(P, st, false, 0, 1, base, sg, Ssum, near, Sabs);
                        route(v0, wid0, Ssum[0], near[0], Sabs[0]);
                        route(v1, wid1, Ssum[1], near[1], Sabs[1]);
                    } else {
                        const uint32_t base[1] = {dense_base(c, wid0)};
                        const float sg[1] = {sgf[wid0]};
                        float Ssum[1] = {0.f};
                        bool near[1] = {false};
                        float Sabs[1] = {0.f};
                        stage_filter<1, false, 0, NODES, TRACK>(P, st, false, 0, 1, base, sg, Ssum, near, Sabs);
                        route(v0, wid0, Ssum[0], near[0], Sabs[0]);
                    }
                }
            } else {
                int lw = 4;
                while (lw > 0 && (1 << (lw - 1)) >= n_act) lw--;
                const int slot = lane & ((1 << lw) - 1), grp = lane >> lw, G = 32 >> lw;
                const bool valid = slot < n_act;
                const int wid0 = act[valid ? slot : 0];
                const uint32_t base[1] = {dense_base(c, wid0)};
                const float sg[1] = {sgf[wid0]};
                float Ssum[1] = {0.f};
                bool near[1] = {false};
                float Sabs[1] = {0.f};
                if (valid) stage_filter<1, false, 0, NODES, TRACK>(P, st, false, grp, G, base, sg, Ssum, near, Sabs);
                float acc = Ssum[0], acc_abs = Sabs[0];
                unsigned nr = near[0];
                for (int d = 1 << lw; d < 32; d <<= 1) {
                    acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, d));
                    if (TRACK) acc_abs = __fadd_rn(acc_abs, __shfl_xor_sync(0xffffffffu, acc_abs, d));
                    nr |= __shfl_xor_sync(0xffffffffu, nr, d);
                }
                route(lane < n_act, wid0, acc, nr != 0, acc_abs);
            }
            __syncwarp();
        }
        return;
    }
    // ---- survivors: detections, or (cascades with a deep tail) queue items ----
    if (n == 0) return;
    ull qb = 0;
    if (s < P.total_stages) {
        if (lane == 0) qb = atomicAdd(a.counters + 1, (ull)n);
        qb = __shfl_sync(0xffffffffu, qb, 0);
    }
    const int Rn = (n + 31) >> 5;
    for (int idx = lane; idx < Rn * 32; idx += 32) {
        const int row = idx >> 5, col = idx & 31;
        if (col >= (dealt ? (n - row + Rn - 1) / Rn : min(32, n - 32 * row))) continue;
        const int i = dealt ? col * Rn + row : idx;   // rank of the entry, 0 .. n-1
        const int w = cur[idx];
        const int x = px0 + (w & (kTileW - 1)) * ystep, y = py0 + (w / kTileW) * ystep;
        if (s >= P.total_stages) {
            emit_rect(a, CL, frame, x, y);
            if (c.codes) dense_write_code(c, w, P.total_stages);
        } else if (qb + i < a.queue_cap) {
            QueueItem it;
            it.key = ((uint32_t)frame << 16) | ((uint32_t)cl << 8) | (uint32_t)s;
            it.xy = ((uint32_t)y << 16) | (uint32_t)x;
            a.queue[qb + i] = it;
        } else {
            atomicAdd(a.counters + 3, 1ull);
        }
    }
}

// COUNT: the diagnostic instantiation (detectors created with want_codes) that counts FP64 fallbacks and
// near-threshold stage sums; the production instantiation carries none of that code.
template <int ROWSTEP_T, bool TREE, bool NODES, int TILE_H, bool COUNT, bool TRACK = false>
__global__ void __launch_bounds__(kDenseThreads)   // (no min-blocks argument: "1" lets ptxas take 88 registers and costs a CTA per SM; "4" caps at 64 but was measured 2 % slower)
k_cascade_tiles(const __grid_constant__ DenseParams P, const __grid_constant__ CascadeArgs a, const int tile0) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
#ifdef CLFD_TILE_TIMING
    const long long t_cta = clock64();
#endif
    cascade_tiles_body<ROWSTEP_T, TREE, NODES, TILE_H, COUNT, TRACK>(P, a, tile0, smem_raw);
#ifdef CLFD_TILE_TIMING
    // counters[4] += sum over the CTA's warps of their busy cycles, [5] += 8 x the cycles of the CTA's last warp (the
    // warp slots the CTA held), [6] += sum of the warps' cycles up to the hand-over (phase 1 + staging)
    __syncwarp();
    if ((threadIdx.x & 31) == 0) {
        const unsigned int dt = (unsigned int)(clock64() - t_cta);
        atomicAdd(&s_dense_t_busy, dt);
        __threadfence_block();
        if (atomicAdd(&s_dense_done, 1u) == kDenseWarps - 1) {
            atomicAdd(a.counters + 4, (ull)s_dense_t_busy);
            atomicAdd(a.counters + 5, (ull)dt * kDenseWarps);
            atomicAdd(a.counters + 6, (ull)s_dense_t_p1);
        }
    }
    return;
#endif
    // every warp ends up here (the body's returns are warp uniform); the last one flushes the CTA's counters
    if (!COUNT) return;
    __syncwarp();
    if ((threadIdx.x & 31) == 0) {
        __threadfence_block();
        if (atomicAdd(&s_dense_done, 1u) == kDenseWarps - 1) {
            const unsigned int ne = s_dense_exact, nn = s_dense_near;
            if (ne) atomicAdd(a.counters + 4, (ull)ne);
            if (nn) atomicAdd(a.counters + 5, (ull)nn);
        }
    }
}

// row steps of the stock window sizes (bytes between a thread's consecutive phase-1 windows)
constexpr int dense_stride_ce(int win_w, int ystep) {   // == dense_tile_stride (haar_pack.cpp)
    int cols = ((kTileW - 1) * ystep + win_w + 1 + 3) & ~3;
    int s = ystep == 1 ? cols : 2 * ((cols / 2 + 3) & ~3);
    s = (s + 3) & ~3;
    while ((ystep * s) % 32 != 8) s += 4;
    return s;
}
constexpr int dense_rowstep_ce(int win_w, int ystep) { return (kDenseThreads / kTileW) * ystep * dense_stride_ce(win_w, ystep) * 4; }

template <int ROWSTEP_T, bool TREE, bool NODES, int TILE_H = kTileH>
static cudaError_t launch_tiles_tt(const DenseParams &P, const CascadeArgs &a, int tile0, int n_tiles, size_t smem, cudaStream_t stream) {
    // cascades with sentinel leaf values (DenseParams::track_abs; haarcascade_mcs_*: generic window sizes, stumps): the
    // instantiation whose stage verdicts bound the FP32 sum by the magnitudes actually added
    if constexpr (ROWSTEP_T == 0 && !TREE && !NODES) {
        if (P.track_abs) {
            static SmemLimitCache limit_track;
            if (cudaError_t e = limit_track.ensure(k_cascade_tiles<0, false, false, TILE_H, kTilesCount, true>, smem)) return e;
            k_cascade_tiles<0, false, false, TILE_H, kTilesCount, true><<<dim3(n_tiles, a.n_frames), kDenseThreads, smem, stream>>>(P, a, tile0);
            return cudaGetLastError();
        }
    }
    static SmemLimitCache limit;
    if (cudaError_t e = limit.ensure(k_cascade_tiles<ROWSTEP_T, TREE, NODES, TILE_H, kTilesCount>, smem)) return e;
    k_cascade_tiles<ROWSTEP_T, TREE, NODES, TILE_H, kTilesCount><<<dim3(n_tiles, a.n_frames), kDenseThreads, smem, stream>>>(P, a, tile0);
    return cudaGetLastError();
}
template <int ROWSTEP_T>
static cudaError_t launch_tiles_t(const DenseParams &P, const CascadeArgs &a, int tile0, int n_tiles, size_t smem, cudaStream_t stream) {
    // (20- and 24-pixel windows share their row steps on both kinds of level: one set of instantiations)
    constexpr int R = ROWSTEP_T;
    if (P.exec_stages > P.tail_stages) return launch_tiles_tt<R, true, false>(P, a, tile0, n_tiles, smem, stream);
    if (P.tile_h == kTileHSmall) {   // tilted cascades on ystep-2 levels
        if (P.npt > 1) return launch_tiles_tt<R, false, true, kTileHSmall>(P, a, tile0, n_tiles, smem, stream);
        return launch_tiles_tt<R, false, false, kTileHSmall>(P, a, tile0, n_tiles, smem, stream);
    }
    if (P.tile_h == 24) {   // plain stump cascades on ystep-2 levels (4 CTAs per SM)
        if (P.exec_stages > P.tail_stages || P.npt > 1) return cudaErrorInvalidValue;
        return launch_tiles_tt<ROWSTEP_T, false, false, 24>(P, a, tile0, n_tiles, smem, stream);
    }
    if (P.tile_h != kTileH) return cudaErrorInvalidValue;
    if (P.npt > 1) return launch_tiles_tt<R, false, true>(P, a, tile0, n_tiles, smem, stream);
    return launch_tiles_tt<ROWSTEP_T, false, false>(P, a, tile0, n_tiles, smem, stream);
}

// The tile kernel is compiled twice, in two translation units that build in parallel: this file as it is (the
// production instantiations) and through kernels_clod_count.cu (CLFD_TILES_COUNT_TU: the diagnostic instantiations
// that count FP64 fallbacks / near-threshold stage sums; only the tile kernel and this launcher are compiled there).
#ifdef CLFD_TILES_COUNT_TU
cudaError_t launch_cascade_tiles_count(const DenseParams &P, const CascadeArgs &a, int tile0, int n_tiles, cudaStream_t stream) {
#else
cudaError_t launch_cascade_tiles_count(const DenseParams &P, const CascadeArgs &a, int tile0, int n_tiles, cudaStream_t stream);
cudaError_t launch_cascade_tiles(const DenseParams &P, const CascadeArgs &a, int tile0, int n_tiles, cudaStream_t stream) {
    if (a.count_exact) return launch_cascade_tiles_count(P, a, tile0, n_tiles, stream);
#endif
    if (n_tiles <= 0 || a.n_frames == 0) return cudaSuccess;
    const size_t smem = dense_smem_plan(P).total;
    // byte distance between a thread's consecutive phase-1 windows: 2 window rows
    const int rowstep = (kDenseThreads / kTileW) * P.ystep * P.tile_stride * 4;
    // the common window widths (20 and 24 pixels) get immediate-offset code
    constexpr int r20_1 = dense_rowstep_ce(20, 1), r20_2 = dense_rowstep_ce(20, 2);
    constexpr int r24_1 = dense_rowstep_ce(24, 1), r24_2 = dense_rowstep_ce(24, 2);
    static_assert(r20_1 == r24_1 && r20_2 == r24_2 && r20_2 != r20_1, "row steps must be distinct switch labels");
    // sentinel-leaf cascades: only the generic row-step code has the TRACK instantiation (launch_tiles_tt)
    if (P.track_abs && P.exec_stages <= P.tail_stages && P.npt == 1) return launch_tiles_t<0>(P, a, tile0, n_tiles, smem, stream);
    switch (rowstep) {
        case r20_1: return launch_tiles_t<r20_1>(P, a, tile0, n_tiles, smem, stream);
        case r20_2: return launch_tiles_t<r20_2>(P, a, tile0, n_tiles, smem, stream);
        default:    return launch_tiles_t<0>(P, a, tile0, n_tiles, smem, stream);
    }
}

#ifndef CLFD_TILES_COUNT_TU
// ------------------------------------------------------------------------------------
// enqueue-all: cascades without a dense prefix start every window in the deep kernel
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_enqueue_all(const CascadeArgs a) {
    const long long w = (long long)blockIdx.x * 256 + threadIdx.x;
    const int frame = blockIdx.y;
    if (w == 0 && frame == 0) a.counters[1] = (ull)a.windows_per_frame * a.n_frames;
    if (w >= a.windows_per_frame) return;
    int lo = 0, hi = a.n_cas_levels - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(&a.cas_levels[mid].win_base) <= w) lo = mid; else hi = mid - 1;
    }
    const int nx = __ldg(&a.cas_levels[lo].nx), ystep = __ldg(&a.cas_levels[lo].ystep);
    const int local = (int)(w - __ldg(&a.cas_levels[lo].win_base));
    const int iy = local / nx, ix = local - iy * nx;
    QueueItem it;
    it.key = ((uint32_t)frame << 16) | ((uint32_t)lo << 8);
    it.xy = ((uint32_t)(iy * ystep) << 16) | (uint32_t)(ix * ystep);
    a.queue[(size_t)frame * a.windows_per_frame + w] = it;
}

cudaError_t launch_enqueue_all(const CascadeArgs &a, cudaStream_t stream) {
    if (a.windows_per_frame == 0 || a.n_frames == 0) return cudaSuccess;
    k_enqueue_all<<<dim3((unsigned)((a.windows_per_frame + 255) / 256), a.n_frames), 256, 0, stream>>>(a);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------
// deep kernel: one warp per queued window
// ------------------------------------------------------------------------------------
constexpr int kDeepThreads = 256;

// A window's view of an int32 integral in global memory: element (dy, dx) relative to the window origin.  Natural
// layout: sh = 0.  Column-de-interleaved level (PyrLevel::di; window origins have even x there): sh = 1, half =
// sum_pitch / 2, p = level + y * pitch + x / 2.
struct SumView {
    const int32_t *__restrict__ p;
    int pitch, half, sh;
    __device__ __forceinline__ int at(int dy, int dx) const { return __ldg(p + dy * pitch + (dx & sh) * half + (dx >> sh)); }
};
__device__ __forceinline__ SumView sum_view(const int32_t *__restrict__ plane, const PyrLevel &L, size_t frame_level_off, int y, int x, bool di) {
    SumView v;
    v.pitch = L.sum_pitch; v.half = L.sum_pitch >> 1; v.sh = di ? 1 : 0;
    v.p = plane + frame_level_off + (size_t)y * L.sum_pitch + (di ? x >> 1 : x);
    return v;
}
__device__ __forceinline__ int rect_sum_g(const SumView &v, uint32_t dxw, uint32_t dyw) {
    // dxw / dyw hold the 4 corner coordinates of one rectangle, one byte each
    return v.at((int)(dyw & 255u), (int)(dxw & 255u)) - v.at((int)((dyw >> 8) & 255u), (int)((dxw >> 8) & 255u)) -
           v.at((int)((dyw >> 16) & 255u), (int)((dxw >> 16) & 255u)) + v.at((int)(dyw >> 24), (int)(dxw >> 24));
}

// One tree of the generic cascade for one window: icvEvalHidHaarClassifier (tempcv.cpp:771-792) and
// the stump fast paths (tempcv.cpp:872-930).  Returns the leaf value.
__device__ __forceinline__ float deep_eval_tree(const DeepCascadeDev &D, int tree, const SumView &sum, const SumView &til,
                                                double sigma, bool dbl) {
    const int n0 = __ldg(D.tree_first_node + tree);
    int idx = 0;
    do {
        const uint4 *nd = reinterpret_cast<const uint4 *>(D.nodes + n0 + idx);
        const uint4 c0 = __ldg(nd), c1 = __ldg(nd + 1), c2 = __ldg(nd + 2);
        const int flags = __ldg(reinterpret_cast<const int *>(nd + 3));
        // c0 = dx[0..11], dy[0..3]; c1 = dy[4..11], w0, w1; c2 = w2, thr, left, right
        const SumView &base = (flags & 1) ? til : sum;
        const int r0 = rect_sum_g(base, c0.x, c0.w);
        const int r1 = rect_sum_g(base, c0.y, c1.x);
        const float w0 = __uint_as_float(c1.z), w1 = __uint_as_float(c1.w);
        const float thr = __uint_as_float(c2.y);
        const double t = __dmul_rn((double)thr, sigma);
        double sv;
        if (dbl) {
            sv = __fma_rn((double)r1, (double)w1, __dmul_rn((double)r0, (double)w0));
        } else {
            sv = __dadd_rn((double)__fmul_rn(__int2float_rn(r0), w0), (double)__fmul_rn(__int2float_rn(r1), w1));
            if ((flags >> 8) == 3) {
                const int r2 = rect_sum_g(base, c0.z, c1.y);
                sv = __dadd_rn(sv, (double)__fmul_rn(__int2float_rn(r2), __uint_as_float(c2.x)));
            }
        }
        idx = sv < t ? (int)c2.z : (int)c2.w;
    } while (idx > 0);
    return __ldg(D.alpha + n0 + tree - idx);
}

// ------------------------------------------------------------------------------------
// mid kernel: one THREAD per window for the stages [mid_begin, mid_end) of a linear cascade
// whose trees the tile kernel cannot evaluate (multi-node trees, tilted features).  Those
// stages have few trees (3, 9, 14, ... in frontalface_alt2), so a warp per window would idle
// most lanes, and they still see most windows.  Input: every grid window (cascades without a
// tile prefix) or the tile kernel's queue; survivors go to the second queue for the deep kernel.
// Lanes hold consecutive windows, so the corner loads of a warp fall into a few cache lines.
// Run in a few passes of two or three stages each, ping-ponging between the two queues, so
// the lanes are re-compacted while the survivor count still drops fast.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_cascade_mid(const __grid_constant__ CascadeArgs a) {
    const DeepCascadeDev &D = a.deep;
    const int lane = threadIdx.x & 31;
    const bool from_grid = a.mid_in == nullptr;
    ull n = from_grid ? (ull)a.windows_per_frame * a.n_frames : *a.mid_in_count;
    if (!from_grid && n > a.queue_cap) n = a.queue_cap;
    const ull stride = (ull)gridDim.x * 128;
    // whole warps iterate together (ballots below)
    for (ull base_item = ((ull)blockIdx.x * 128 + threadIdx.x) - lane; base_item < n; base_item += stride) {
        const ull item = base_item + lane;
        const bool valid = item < n;
        int frame = 0, cl = 0, x = 0, y = 0;
        if (valid) {
            if (from_grid) {
                frame = (int)(item / (ull)a.windows_per_frame);
                const long long w = (long long)(item - (ull)frame * a.windows_per_frame);
                int lo = 0, hi = a.n_cas_levels - 1;
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (__ldg(&a.cas_levels[mid].win_base) <= w) lo = mid; else hi = mid - 1;
                }
                cl = lo;
                const int nx = __ldg(&a.cas_levels[lo].nx), ystep = __ldg(&a.cas_levels[lo].ystep);
                const int local = (int)(w - __ldg(&a.cas_levels[lo].win_base));
                const int iy = local / nx;
                x = (local - iy * nx) * ystep; y = iy * ystep;
            } else {
                const QueueItem q = a.mid_in[item];
                frame = q.key >> 16; cl = (q.key >> 8) & 255;
                x = q.xy & 0xffff; y = q.xy >> 16;
            }
        }
        bool alive = valid;
        int stage = D.mid_begin;
        const CasLevel CL = a.cas_levels[cl];
        if (valid) {
            const PyrLevel L = a.levels[CL.pyr_level];
            const int pitch = L.sum_pitch;
            const size_t off = (size_t)frame * a.sum_frame_stride + L.sum_off + (size_t)y * pitch + x;
            const size_t lvl = (size_t)frame * a.sum_frame_stride + L.sum_off;
            const SumView sum = sum_view(a.sum, L, lvl, y, x, L.di != 0);
            const SumView til = a.tilted ? sum_view(a.tilted, L, lvl, y, x, false) : sum;
            const int eq_w = D.win_w - 2, eq_h = D.win_h - 2;
            const int g0 = pitch + 1, g1 = g0 + eq_w, g2 = (1 + eq_h) * pitch + 1, g3 = g2 + eq_w;
            const int s4 = sum.at(1, 1) - sum.at(1, 1 + eq_w) - sum.at(1 + eq_h, 1) + sum.at(1 + eq_h, 1 + eq_w);
            const ull q4 = sq_rect(a.sq, a.sq32 != 0, off, g0, g1, g2, g3);
            const double sigma = window_sigma(s4, q4, D.inv_area);
            for (; stage < D.mid_end; stage++) {
                const DeepStage st = D.stages[stage];
                const bool dbl = st.flags & 1;
                double S = 0.0;
                for (int j = 0; j < st.ntrees; j++)
                    S = __dadd_rn(S, (double)deep_eval_tree(D, st.first_tree + j, sum, til, sigma, dbl));
                if (S < (double)st.thr) { alive = false; break; }
            }
        }
        if (valid && !alive && a.codes)
            a.codes[(size_t)frame * a.windows_per_frame + CL.win_base + (size_t)(y / CL.ystep) * CL.nx + x / CL.ystep] = (int16_t)stage;
        const bool accepted = alive && D.mid_end >= D.n_stages;
        if (accepted) {
            emit_rect(a, CL, frame, x, y);
            if (a.codes)
                a.codes[(size_t)frame * a.windows_per_frame + CL.win_base + (size_t)(y / CL.ystep) * CL.nx + x / CL.ystep] = (int16_t)D.n_stages;
        }
        const bool pass_on = alive && !accepted;
        const unsigned m = __ballot_sync(0xffffffffu, pass_on);
        if (m) {
            ull qb = 0;
            if (lane == 0) qb = atomicAdd(a.mid_out_count, (ull)__popc(m));
            qb = __shfl_sync(0xffffffffu, qb, 0);
            if (pass_on) {
                const ull slot = qb + __popc(m & ((1u << lane) - 1u));
                if (slot < a.queue_cap) {
                    QueueItem it;
                    it.key = ((uint32_t)frame << 16) | ((uint32_t)cl << 8) | (uint32_t)D.mid_end;
                    it.xy = ((uint32_t)y << 16) | (uint32_t)x;
                    a.mid_out[slot] = it;
                } else {
                    atomicAdd(a.counters + 3, 1ull);
                }
            }
        }
    }
}

cudaError_t launch_cascade_mid(const CascadeArgs &a, int n_sms, cudaStream_t stream) {
    if (a.n_frames == 0) return cudaSuccess;
    k_cascade_mid<<<n_sms * 16, 128, 0, stream>>>(a);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(kDeepThreads) k_cascade_deep(const __grid_constant__ CascadeArgs a) {
    const int lane = threadIdx.x & 31;
    const ull warp0 = ((ull)blockIdx.x * kDeepThreads + threadIdx.x) >> 5;
    const ull nwarps = ((ull)gridDim.x * kDeepThreads) >> 5;
    ull n = *a.deep_count;
    if (n > a.queue_cap) n = a.queue_cap;
    const DeepCascadeDev &D = a.deep;

    for (ull item = warp0; item < n; item += nwarps) {
        const QueueItem q = a.deep_in[item];
        const int frame = q.key >> 16, cl = (q.key >> 8) & 255, stage0 = q.key & 255;
        const int x = q.xy & 0xffff, y = q.xy >> 16;
        const CasLevel CL = a.cas_levels[cl];
        const PyrLevel L = a.levels[CL.pyr_level];
        const int pitch = L.sum_pitch;
        const size_t off = (size_t)frame * a.sum_frame_stride + L.sum_off + (size_t)y * pitch + x;
        const size_t lvl = (size_t)frame * a.sum_frame_stride + L.sum_off;
        const SumView sum = sum_view(a.sum, L, lvl, y, x, L.di != 0);
        const SumView til = a.tilted ? sum_view(a.tilted, L, lvl, y, x, false) : sum;

        const int eq_w = D.win_w - 2, eq_h = D.win_h - 2;
        const int g0 = pitch + 1, g1 = g0 + eq_w, g2 = (1 + eq_h) * pitch + 1, g3 = g2 + eq_w;
        const int s4 = sum.at(1, 1) - sum.at(1, 1 + eq_w) - sum.at(1 + eq_h, 1) + sum.at(1 + eq_h, 1 + eq_w);
        const ull q4 = sq_rect(a.sq, a.sq32 != 0, off, g0, g1, g2, g3);
        const double sigma = window_sigma(s4, q4, D.inv_area);

        int ptr = stage0, last = stage0, accepted = 0;
        for (;;) {
            const DeepStage st = D.stages[ptr];
            last = ptr;
            const bool dbl = st.flags & 1, order_free = st.flags & 2;
            double S = 0.0, part = 0.0;
            for (int j0 = 0; j0 < st.ntrees; j0 += 32) {
                const int j = j0 + lane;
                float av = 0.f;
                if (j < st.ntrees) av = deep_eval_tree(D, st.first_tree + j, sum, til, sigma, dbl);
                if (order_free) {
                    part = __dadd_rn(part, (double)av);
                } else {
                    const int cnt = min(32, st.ntrees - j0);
                    for (int k = 0; k < cnt; k++) S = __dadd_rn(S, (double)__shfl_sync(0xffffffffu, av, k));
                }
            }
            if (order_free) {
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) part = __dadd_rn(part, __shfl_xor_sync(0xffffffffu, part, d));
                S = part;
            }
            const bool pass = S >= (double)st.thr;
            if (D.is_tree) {  // tempcv.cpp:849-859
                if (pass) {
                    ptr = st.child;
                    if (ptr < 0) { accepted = 1; break; }
                } else {
                    int p = ptr;
                    while (p >= 0 && __ldg(&D.stages[p].next) < 0) p = __ldg(&D.stages[p].parent);
                    if (p < 0) break;
                    ptr = __ldg(&D.stages[p].next);
                }
            } else {
                if (!pass) break;
                if (++ptr >= D.n_stages) { accepted = 1; break; }
            }
        }
        if (lane == 0) {
            if (accepted) emit_rect(a, CL, frame, x, y);
            if (a.codes) {
                const int code = D.is_tree ? 2 * last + accepted : (accepted ? D.n_stages : last);
                a.codes[(size_t)frame * a.windows_per_frame + CL.win_base + (size_t)(y / CL.ystep) * CL.nx + x / CL.ystep] = (int16_t)code;
            }
        }
    }
}

// ------------------------------------------------------------------------------------
// reject levels (cvHaarDetectObjectsForROC with outputRejectLevels, tempcv.cpp:1084-1094):
// a pass over the exit codes.  Thread per window; the rare candidates redo the last stage
// they evaluated with the generic node records, in the reference's order, to get its sum.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_roc_collect(const CascadeArgs a, RocItem *__restrict__ out, const ull cap, ull *counter) {
    const long long w = (long long)blockIdx.x * 256 + threadIdx.x;
    const int frame = blockIdx.y;
    if (w >= a.windows_per_frame) return;
    const DeepCascadeDev &D = a.deep;
    const int code = a.codes[(size_t)frame * a.windows_per_frame + w];
    int level, last;
    if (D.is_tree) {   // result 0 for every rejection: count + 0 < 4 never holds
        if (!(code & 1)) return;
        level = D.n_stages; last = code >> 1;
    } else {           // result -i for a rejection by stage i, -count when accepted
        if (D.n_stages - code >= 4) return;
        level = code; last = code == D.n_stages ? D.n_stages - 1 : code;
    }
    int lo = 0, hi = a.n_cas_levels - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(&a.cas_levels[mid].win_base) <= w) lo = mid; else hi = mid - 1;
    }
    const CasLevel CL = a.cas_levels[lo];
    const PyrLevel L = a.levels[CL.pyr_level];
    const int local = (int)(w - CL.win_base);
    const int iy = local / CL.nx, ix = local - iy * CL.nx;
    const int x = ix * CL.ystep, y = iy * CL.ystep;
    const int pitch = L.sum_pitch;
    const size_t off = (size_t)frame * a.sum_frame_stride + L.sum_off + (size_t)y * pitch + x;
    const size_t lvl = (size_t)frame * a.sum_frame_stride + L.sum_off;
    const SumView sum = sum_view(a.sum, L, lvl, y, x, L.di != 0);
    const SumView til = a.tilted ? sum_view(a.tilted, L, lvl, y, x, false) : sum;
    const int eq_w = D.win_w - 2, eq_h = D.win_h - 2;
    const int g0 = pitch + 1, g1 = g0 + eq_w, g2 = (1 + eq_h) * pitch + 1, g3 = g2 + eq_w;
    const int s4 = sum.at(1, 1) - sum.at(1, 1 + eq_w) - sum.at(1 + eq_h, 1) + sum.at(1 + eq_h, 1 + eq_w);
    const ull q4 = sq_rect(a.sq, a.sq32 != 0, off, g0, g1, g2, g3);
    const double sigma = window_sigma(s4, q4, D.inv_area);
    const DeepStage st = D.stages[last];
    double S = 0.0;
    for (int j = 0; j < st.ntrees; j++)
        S = __dadd_rn(S, (double)deep_eval_tree(D, st.first_tree + j, sum, til, sigma, st.flags & 1));
    const ull slot = atomicAdd(counter, 1ull);
    if (slot >= cap) return;
    RocItem it;
    it.r.x = __double2int_rn(__dmul_rn((double)x, CL.factor));
    it.r.y = __double2int_rn(__dmul_rn((double)y, CL.factor));
    it.r.w = CL.win_w; it.r.h = CL.win_h; it.r.frame = a.frame_base + frame; it.r.cascade = a.cascade_index;
    it.level = level; it.pad = 0; it.win = w; it.weight = S;
    out[slot] = it;
}

cudaError_t launch_roc_collect(const CascadeArgs &a, RocItem *out, unsigned long long cap, unsigned long long *counter, cudaStream_t stream) {
    if (a.windows_per_frame == 0 || a.n_frames == 0) return cudaSuccess;
    k_roc_collect<<<dim3((unsigned)((a.windows_per_frame + 255) / 256), a.n_frames), 256, 0, stream>>>(a, out, cap, counter);
    return cudaGetLastError();
}

cudaError_t launch_cascade_deep(const CascadeArgs &a, int n_sms, cudaStream_t stream) {
    if (a.n_frames == 0) return cudaSuccess;
    k_cascade_deep<<<n_sms * 8, kDeepThreads, 0, stream>>>(a);
    return cudaGetLastError();
}

#endif  // CLFD_TILES_COUNT_TU

}  // namespace clfd
