// kernels_clif.cu -- pyramid downscale + integral / squared-integral / tilted-integral
// images for sm_100a.  Replaces, from scratch, the reference's
//   * cvResize(img, level, CV_INTER_LINEAR) per pyramid level       (tempcv.cpp:1301)
//   * integralImageSumRows / integralImageSumCols                    (clif.cl:79-120)
//     and cvIntegral(sum, sqsum, tilted)                             (tempcv.cpp:1302)
//   * bgrToGrayscale                                                 (clif.cl:4-18), batched
//
// Design (HBM-bound byte work; no tensor cores):
//   K1 resize_colsum : all levels x frames x 32-row blocks in one launch.  Each thread makes
//                      4 adjacent level pixels per row (11-bit fixed-point bilinear, bit
//                      exact with OpenCV) and keeps their column sums / column square sums
//                      for the row block -> the vertical carries cost no extra pass.
//   K2 colscan       : exclusive prefix of those carries over row blocks (tiny).
//   K3 integral_rows : one CTA per (level, frame, 32-row block).  A thread owns 8 adjacent
//                      columns: running column sums in registers (seeded with the carry),
//                      thread-serial + warp-shuffle + cross-warp prefix along the row, and
//                      16-byte vector stores of int32 sums and uint64 square sums.  The image
//                      is read once (8 B loads) and every output byte is written once.
//   K4 tilted        : four launches, only for cascades with tilted features (fullbody & co): block-local
//                      diagonal sums, carries along the diagonals, column carries, then the rows -- warp
//                      tiles with halo columns, no barriers (see K4 below).
#include <cstdint>
#include <type_traits>
#include <cstdlib>

#include "kernels.h"

namespace clfd {

typedef unsigned long long ull;

// mbarrier + TMA bulk copy (cp.async.bulk, SASS: UBLKCP / SYNCS), as in kernels_clod.cu
__device__ __forceinline__ uint32_t clif_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void clif_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(clif_smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void clif_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(clif_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void clif_mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "CLIF_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra CLIF_DONE;\n"
        "bra CLIF_WAIT;\n"
        "CLIF_DONE:\n"
        "}" ::"r"(clif_smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void clif_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(clif_smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(clif_smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------------------------
// K1: pyramid level pixels + per-row-block column sums
// ------------------------------------------------------------------------------------
constexpr int kResizeThreads = 128;  // four warps, each with a work item of its own: (level, row block, 128-column chunk)
constexpr int kResizeCols = 32 * 4;  // columns per warp

// vertical pass of 4 pixels (OpenCV VResizeLinear, 8u: ((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2),
// r0s / r1s = the horizontal passes of the two source rows, already shifted right by 4.  The result is at most 255
// (b0 + b1 = 2048, r >> 4 <= 32640), so the four bytes pack without masks.
__device__ __forceinline__ uint32_t resize_vpass4(const int (&r0s)[4], const int (&r1s)[4], int b0, int b1, uint32_t (&cs)[4],
                                                  uint32_t (&cq)[4]) {
    uint32_t packed = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint32_t u = (uint32_t)((((b0 * r0s[i]) >> 16) + ((b1 * r1s[i]) >> 16) + 2) >> 2);
        packed |= u << (8 * i);
        cs[i] += u;
        cq[i] += u * u;
    }
    return packed;
}

// Word path of k_resize_colsum (source rows 4-byte aligned).  QUAD (factors < 2): the eight taps of the thread's
// four pixels lie within 8 bytes of the first one -> three aligned 32-bit loads per source row, two funnel shifts that
// put the first tap at byte 0, one PRMT + two IDP.2A per pixel pair.  !QUAD (factors up to 6): the same per pixel
// pair.  (The byte path spends 8 LDG.U8 and 16 address instructions on the same row.)
template <bool QUAD, bool GUARD>
__device__ __forceinline__ void resize_rows_words(const PyramidArgs &a, const PyrLevel &L, const uint8_t *__restrict__ src,
                                                  uint8_t *__restrict__ dst, int x0, int y0, int y1, const int (&sx0)[4],
                                                  const uint32_t (&coef)[4], uint32_t (&cs)[4], uint32_t (&cq)[4]) {
    const int last_word = (a.W - 1) & ~3;   // byte offset of the last source word that holds a pixel of the row
    int boff[2], sh[2];
    uint32_t sel[2];
    bool p1[2], p2[2];
#pragma unroll
    for (int j = 0; j < 2; j++) {
        const int first = QUAD ? sx0[0] : sx0[2 * j];
        boff[j] = first & ~3;
        sh[j] = (first & 3) * 8;
        const uint32_t o0 = (uint32_t)(sx0[2 * j] - first), o1 = (uint32_t)(sx0[2 * j + 1] - first);
        sel[j] = o0 | ((o0 + 1) << 4) | (o1 << 8) | ((o1 + 1) << 12);
        p1[j] = !GUARD || boff[j] + 4 <= last_word;
        p2[j] = !GUARD || boff[j] + 8 <= last_word;
    }
    // per-row table entries: lane k of every warp holds row y0 + k's clamped source rows and coefficients (<< 16, for
    // the multiply-high of the vertical pass); the row loop fetches them with shuffles instead of dependent loads
    const int lane = threadIdx.x & 31;
    const int ty = min(y0 + lane, L.h - 1);
    const int tsy = __ldg(a.yofs + L.ytab_off + ty);
    const short2 tb = __ldg(a.ybeta + L.ytab_off + ty);
    const uint32_t my_sy = (uint32_t)min(max(tsy, 0), a.H - 1) | ((uint32_t)min(max(tsy + 1, 0), a.H - 1) << 16);
    const uint32_t my_b0 = (uint32_t)tb.x << 16, my_b1 = (uint32_t)tb.y << 16;
    const uint8_t *__restrict__ srcA = src + boff[0];
    const uint8_t *__restrict__ srcB = src + boff[1];
    const uint32_t rstride = (uint32_t)a.row_stride;
    auto hrow = [&](uint32_t sy, uint32_t (&r)[4]) {
        const uint32_t *__restrict__ p = reinterpret_cast<const uint32_t *>(srcA + (size_t)sy * rstride);
        const uint32_t w0 = __ldg(p), w1 = p1[0] ? __ldg(p + 1) : 0u, w2 = p2[0] ? __ldg(p + 2) : 0u;
        uint32_t lo = __funnelshift_r(w0, w1, sh[0]), hi = __funnelshift_r(w1, w2, sh[0]);
        uint32_t P = __byte_perm(lo, hi, sel[0]);
        r[0] = __dp2a_lo(coef[0], P, 0u) >> 4;
        r[1] = __dp2a_hi(coef[1], P, 0u) >> 4;
        if (!QUAD) {
            const uint32_t *__restrict__ q = reinterpret_cast<const uint32_t *>(srcB + (size_t)sy * rstride);
            const uint32_t v0 = __ldg(q), v1 = p1[1] ? __ldg(q + 1) : 0u, v2 = p2[1] ? __ldg(q + 2) : 0u;
            lo = __funnelshift_r(v0, v1, sh[1]);
            hi = __funnelshift_r(v1, v2, sh[1]);
        }
        P = __byte_perm(lo, hi, sel[1]);
        r[2] = __dp2a_lo(coef[2], P, 0u) >> 4;
        r[3] = __dp2a_hi(coef[3], P, 0u) >> 4;
    };
    // OpenCV VResizeLinear, 8u: (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2; (b * s) >> 16 is the high
    // word of (b << 16) * s (b <= 2048, s <= 32640).  At most 255, so the bytes pack without masks.
    auto vrow = [&](const uint32_t (&r0)[4], const uint32_t (&r1)[4], uint32_t b0, uint32_t b1, uint8_t *__restrict__ out) {
        uint32_t u[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            u[i] = (__umulhi(b1, r1[i]) + (__umulhi(b0, r0[i]) + 2u)) >> 2;
            cs[i] += u[i];
            cq[i] += u[i] * u[i];
        }
        if (x0 < L.pyr_pitch)
            *reinterpret_cast<uint32_t *>(out) = __byte_perm(__byte_perm(u[0], u[1], 0x0040), __byte_perm(u[2], u[3], 0x0040), 0x5410);
    };
    uint32_t ra[4] = {0, 0, 0, 0}, rb[4];
    uint32_t prev_sy1 = 0xffffffffu;
    uint8_t *__restrict__ out = dst + (size_t)y0 * L.pyr_pitch + x0;
    // two output rows per iteration: the horizontal pass kept for the next row alternates between ra and rb
    for (int k = 0; k < y1 - y0; k += 2) {
        {
            const uint32_t sy = __shfl_sync(0xffffffffu, my_sy, k);
            const uint32_t b0 = __shfl_sync(0xffffffffu, my_b0, k), b1 = __shfl_sync(0xffffffffu, my_b1, k);
            // the horizontal pass of a source row is reused: at factors < 2 most rows' upper source row is the
            // previous row's lower one (block-uniform test, no divergence)
            if ((sy & 0xffffu) != prev_sy1) hrow(sy & 0xffffu, ra);
            hrow(sy >> 16, rb);
            prev_sy1 = sy >> 16;
            vrow(ra, rb, b0, b1, out);
            out += L.pyr_pitch;
        }
        if (k + 1 < y1 - y0) {
            const uint32_t sy = __shfl_sync(0xffffffffu, my_sy, k + 1);
            const uint32_t b0 = __shfl_sync(0xffffffffu, my_b0, k + 1), b1 = __shfl_sync(0xffffffffu, my_b1, k + 1);
            if ((sy & 0xffffu) != prev_sy1) hrow(sy & 0xffffu, rb);
            hrow(sy >> 16, ra);
            prev_sy1 = sy >> 16;
            vrow(rb, ra, b0, b1, out);
            out += L.pyr_pitch;
        }
    }
}

// (9 CTAs per SM: a cap of 56 registers costs 44 bytes of spills outside the row loop and buys 36 instead of 32 resident
//  warps for a kernel that waits on its own loads: 0.435 -> 0.426 ms; 10 CTAs = 48 registers spill in the loop: 0.452)
__global__ void __launch_bounds__(kResizeThreads, 9) k_resize_colsum(const PyramidArgs a) {
    // items are per WARP (the warps of a CTA never meet): a level's last 512 columns do not leave idle warps behind in
    // resident CTAs (14 % of the warp slots with 512-column items per CTA at 1080p, scale 1.2)
    const int4 it = a.resize_items[blockIdx.x * (kResizeThreads / 32) + (threadIdx.x >> 5)];
    if (it.x < 0) return;                                          // padding of the item list
    const PyrLevel L = a.levels[it.x];
    const int frame = blockIdx.y;
    const int x0 = it.z * kResizeCols + (threadIdx.x & 31) * 4;
    const int xw = it.z * kResizeCols;                             // first column of this warp (128 columns)
    if (xw >= max(L.pyr_pitch, L.sum_pitch)) return;               // whole warps only: the word path shuffles

    const uint8_t *__restrict__ src = a.frames + (size_t)frame * a.frame_stride;
    uint8_t *__restrict__ dst = a.pyr + (size_t)frame * a.pyr_frame_stride + L.pyr_off;

    int sx0[4];
    uint32_t coef[4];   // (a0, a1) as two u16: the table's short2
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int x = x0 + i;
        sx0[i] = x < L.w ? __ldg(a.xofs + L.xtab_off + x) : (i ? sx0[i > 0 ? i - 1 : 0] : 0);
        coef[i] = x < L.w ? __ldg(reinterpret_cast<const uint32_t *>(a.xalpha + L.xtab_off + x)) : 0u;
    }
    uint32_t cs[4] = {0, 0, 0, 0}, cq[4] = {0, 0, 0, 0};
    const bool aligned = (a.row_stride & 3) == 0 && (a.frame_stride & 3) == 0 && (reinterpret_cast<uintptr_t>(a.frames) & 3) == 0;
    // whole groups of 4 pixels of an unscaled level with 4-byte aligned source rows
    const bool copy4 = L.w == a.W && L.h == a.H && xw + 128 <= L.w && aligned;   // (warp uniform)
    const int mode = aligned ? L.resize_mode : kResizeBytes;
    const int y0 = it.y * kRowBlock, y1 = min(y0 + kRowBlock, L.h);

    if (copy4) {   // the level of factor 1: the resize is the identity (coefficients 2048 / 0), 4 pixels per load
        for (int y = y0; y < y1; y++) {
            const uint32_t packed = __ldg(reinterpret_cast<const uint32_t *>(src + (size_t)y * a.row_stride + x0));
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const uint32_t u = (packed >> (8 * i)) & 255u;
                cs[i] += u;
                cq[i] += u * u;
            }
            *reinterpret_cast<uint32_t *>(dst + (size_t)y * L.pyr_pitch + x0) = packed;
        }
    } else if (mode == kResizeQuad || mode == kResizePair) {
        // GUARD: the words behind a row's last pixel are not loaded.  Only the CTAs that read the last source row of
        // the batch's last frame need that (everywhere else the bytes behind a row belong to the next row or frame);
        // output row h - 2 reads it too when the factor is 1
        const bool guard = frame == a.n_frames - 1 && y1 + 1 >= L.h;
        if (mode == kResizeQuad) {
            if (guard) resize_rows_words<true, true>(a, L, src, dst, x0, y0, y1, sx0, coef, cs, cq);
            else resize_rows_words<true, false>(a, L, src, dst, x0, y0, y1, sx0, coef, cs, cq);
        } else {
            if (guard) resize_rows_words<false, true>(a, L, src, dst, x0, y0, y1, sx0, coef, cs, cq);
            else resize_rows_words<false, false>(a, L, src, dst, x0, y0, y1, sx0, coef, cs, cq);
        }
    } else {
        // byte path: any factor, any alignment
        int sx1[4], a0[4], a1[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            sx1[i] = min(sx0[i] + 1, a.W - 1);
            a0[i] = (int)(coef[i] & 0xffffu); a1[i] = (int)(coef[i] >> 16);
        }
        int prev[4] = {0, 0, 0, 0}, prev_sy1 = -1;
        for (int y = y0; y < y1; y++) {
            const int sy = __ldg(a.yofs + L.ytab_off + y);
            const short2 b = __ldg(a.ybeta + L.ytab_off + y);
            const int sy0 = min(max(sy, 0), a.H - 1), sy1 = min(max(sy + 1, 0), a.H - 1);
            const uint8_t *__restrict__ S0 = src + (size_t)sy0 * a.row_stride;
            const uint8_t *__restrict__ S1 = src + (size_t)sy1 * a.row_stride;
            const bool reuse = sy0 == prev_sy1;
            prev_sy1 = sy1;
            int r0[4], r1[4];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                r0[i] = reuse ? prev[i] : ((int)__ldg(S0 + sx0[i]) * a0[i] + (int)__ldg(S0 + sx1[i]) * a1[i]) >> 4;
                r1[i] = ((int)__ldg(S1 + sx0[i]) * a0[i] + (int)__ldg(S1 + sx1[i]) * a1[i]) >> 4;
                prev[i] = r1[i];
            }
            const uint32_t packed = resize_vpass4(r0, r1, b.x, b.y, cs, cq);
            if (x0 < L.pyr_pitch) *reinterpret_cast<uint32_t *>(dst + (size_t)y * L.pyr_pitch + x0) = packed;
        }
    }
    if (x0 < L.sum_pitch) {
        uint32_t *c0 = a.col + (size_t)frame * a.col_frame_stride + L.col_off + (size_t)it.y * L.sum_pitch + x0;
        *reinterpret_cast<uint4 *>(c0) = make_uint4(cs[0], cs[1], cs[2], cs[3]);
        *reinterpret_cast<uint4 *>(c0 + a.col_plane_stride) = make_uint4(cq[0], cq[1], cq[2], cq[3]);
    }
}

cudaError_t launch_resize_colsum(const PyramidArgs &a, cudaStream_t stream) {
    if (a.n_resize_items == 0 || a.n_frames == 0) return cudaSuccess;
    k_resize_colsum<<<dim3(a.n_resize_items / (kResizeThreads / 32), a.n_frames), kResizeThreads, 0, stream>>>(a);   // (the list is padded to whole CTAs)
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------
// K2: exclusive prefix over row blocks of the column sums (in place)
// ------------------------------------------------------------------------------------
constexpr int kColscanThreads = 128;

__global__ void __launch_bounds__(kColscanThreads) k_colscan(const PyramidArgs a) {
    const int4 it = a.colscan_items[blockIdx.x];
    const PyrLevel L = a.levels[it.x];
    const int X = (it.y * kColscanThreads + threadIdx.x) * 4;
    if (X >= L.sum_pitch) return;
#pragma unroll
    for (int plane = 0; plane < 2; plane++) {
        uint32_t *p = a.col + (size_t)blockIdx.y * a.col_frame_stride + plane * a.col_plane_stride + L.col_off + X;
        uint4 acc = make_uint4(0, 0, 0, 0);
        // eight row blocks per step: all loads first (independent, in flight together), then the stores --
        // a load behind a store to the same array is otherwise serialised, one DRAM latency per row block
        constexpr int kAhead = 8;
        for (int rb0 = 0; rb0 < L.nrb; rb0 += kAhead) {
            uint4 v[kAhead];
#pragma unroll
            for (int k = 0; k < kAhead; k++)
                if (rb0 + k < L.nrb) v[k] = *reinterpret_cast<const uint4 *>(p + (size_t)(rb0 + k) * L.sum_pitch);
#pragma unroll
            for (int k = 0; k < kAhead; k++) {
                if (rb0 + k < L.nrb) {
                    *reinterpret_cast<uint4 *>(p + (size_t)(rb0 + k) * L.sum_pitch) = acc;
                    acc.x += v[k].x; acc.y += v[k].y; acc.z += v[k].z; acc.w += v[k].w;
                }
            }
        }
    }
}

cudaError_t launch_colscan(const PyramidArgs &a, cudaStream_t stream) {
    if (a.n_colscan_items == 0 || a.n_frames == 0) return cudaSuccess;
    k_colscan<<<dim3(a.n_colscan_items, a.n_frames), kColscanThreads, 0, stream>>>(a);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------
// K3: integral rows.  sum[Y][X] = sum_{y<Y, x<X} I, written for Y in the row block.
// ------------------------------------------------------------------------------------
// SQ32: the squared integral modulo 2^32 (PyramidArgs::sq32): 32-bit scans and half the bytes written.
template <int NT, bool SQ32>
__global__ void __launch_bounds__(NT) k_integral_rows(const PyramidArgs a, const int4 *__restrict__ items) {
    typedef typename std::conditional<SQ32, uint32_t, ull>::type sq_t;
    constexpr int NW = NT / 32;
    __shared__ uint32_t wtot_s[2][NW];
    __shared__ sq_t wtot_q[2][NW];

    const int4 it = items[blockIdx.x];
    const PyrLevel L = a.levels[it.x];
    const int rb = it.y, frame = blockIdx.y;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int X0 = t * 8;
    const bool in_sum = X0 < L.sum_pitch;
    const bool in_pyr = X0 < L.pyr_pitch;

    const uint8_t *__restrict__ pyr = a.pyr + (size_t)frame * a.pyr_frame_stride + L.pyr_off;
    int32_t *__restrict__ sum = a.sum + (size_t)frame * a.sum_frame_stride + L.sum_off;
    sq_t *__restrict__ sq = reinterpret_cast<sq_t *>(a.sq) + (size_t)frame * a.sum_frame_stride + L.sum_off;

    uint32_t ca[8], cq[8];
    if (in_sum) {
        const uint32_t *c0 = a.col + (size_t)frame * a.col_frame_stride + L.col_off + (size_t)rb * L.sum_pitch + X0;
        const uint4 s0 = *reinterpret_cast<const uint4 *>(c0), s1 = *reinterpret_cast<const uint4 *>(c0 + 4);
        const uint4 q0 = *reinterpret_cast<const uint4 *>(c0 + a.col_plane_stride);
        const uint4 q1 = *reinterpret_cast<const uint4 *>(c0 + a.col_plane_stride + 4);
        ca[0] = s0.x; ca[1] = s0.y; ca[2] = s0.z; ca[3] = s0.w; ca[4] = s1.x; ca[5] = s1.y; ca[6] = s1.z; ca[7] = s1.w;
        cq[0] = q0.x; cq[1] = q0.y; cq[2] = q0.z; cq[3] = q0.w; cq[4] = q1.x; cq[5] = q1.y; cq[6] = q1.z; cq[7] = q1.w;
    } else {
#pragma unroll
        for (int i = 0; i < 8; i++) ca[i] = cq[i] = 0;
    }

    const int y0 = rb * kRowBlock, y1 = min(y0 + kRowBlock, L.h);
    if (rb == 0 && in_sum) {  // row 0 of every integral image is zero
        int4 *s = reinterpret_cast<int4 *>(sum + X0);
        s[0] = make_int4(0, 0, 0, 0); s[1] = make_int4(0, 0, 0, 0);
        if (SQ32) {
            uint4 *q = reinterpret_cast<uint4 *>(sq + X0);
            q[0] = q[1] = make_uint4(0, 0, 0, 0);
        } else {
            ulonglong2 *q = reinterpret_cast<ulonglong2 *>(sq + X0);
            q[0] = q[1] = q[2] = q[3] = make_ulonglong2(0, 0);
        }
    }

    // cross-warp exclusive prefix of per-warp totals (lane 31 holds the warp's inclusive total)
    auto left_of_warp = [&](int buf, uint32_t tot_s, sq_t tot_q, uint32_t &os, sq_t &oq) {
        os = 0; oq = 0;
        if (NW > 1) {
            if (lane == 31) { wtot_s[buf][warp] = tot_s; wtot_q[buf][warp] = tot_q; }
            __syncthreads();
            if (NW <= 8) {
                for (int w = 0; w < warp; w++) { os += wtot_s[buf][w]; oq += wtot_q[buf][w]; }
            } else {
                uint32_t ws = lane < warp ? wtot_s[buf][lane] : 0u;
                sq_t wq = lane < warp ? wtot_q[buf][lane] : (sq_t)0;
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) {
                    ws += __shfl_xor_sync(0xffffffffu, ws, d);
                    wq += __shfl_xor_sync(0xffffffffu, wq, d);
                }
                os = ws; oq = wq;
            }
        }
    };

    // Integral row y0 of this thread's 8 columns = exclusive horizontal prefix of the column carries
    // (64-bit scan, ONCE per row block).  After that every row only adds its own exclusive pixel
    // prefix -- out[y+1][x] = out[y][x] + sum_{x' < x} p[y][x'] -- whose scans fit 32 bits: a row of
    // 8-bit pixels sums to < 2^21 and its squares to < 2^30 up to 16384 columns.
    uint32_t Is[8];
    sq_t Iq[8];
    {
        uint32_t ts = 0;
        sq_t tq = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) { ts += ca[i]; tq += cq[i]; }
        uint32_t is = ts;
        sq_t iq = tq;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t vs = __shfl_up_sync(0xffffffffu, is, d);
            const sq_t vq = __shfl_up_sync(0xffffffffu, iq, d);
            if (lane >= d) { is += vs; iq += vq; }
        }
        uint32_t os; sq_t oq;
        left_of_warp(0, is, iq, os, oq);
        uint32_t es = os + is - ts;
        sq_t eq = oq + iq - tq;
#pragma unroll
        for (int i = 0; i < 8; i++) { Is[i] = es; Iq[i] = eq; es += ca[i]; eq += cq[i]; }
    }

    uint2 nxt = make_uint2(0, 0);
    if (in_pyr) nxt = __ldg(reinterpret_cast<const uint2 *>(pyr + (size_t)y0 * L.pyr_pitch + X0));
    int buf = 1;
    for (int y = y0; y < y1; y++) {
        const uint2 cur = nxt;
        if (in_pyr && y + 1 < y1) nxt = __ldg(reinterpret_cast<const uint2 *>(pyr + (size_t)(y + 1) * L.pyr_pitch + X0));
        uint32_t p[8], ts = 0, tq = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const uint32_t word = i < 4 ? cur.x : cur.y;
            p[i] = (word >> (8 * (i & 3))) & 255u;
            ts += p[i];
            tq += p[i] * p[i];
        }
        uint32_t is = ts, iq = tq;  // warp inclusive scan of the thread totals, 32 bits each
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t vs = __shfl_up_sync(0xffffffffu, is, d);
            const uint32_t vq = __shfl_up_sync(0xffffffffu, iq, d);
            if (lane >= d) { is += vs; iq += vq; }
        }
        uint32_t os; sq_t oq;
        left_of_warp(buf, is, (sq_t)iq, os, oq);
        buf ^= 1;
        if (in_sum) {
            uint32_t rs = os + is - ts;              // exclusive pixel prefix of this row at column X0
            uint32_t rq = (uint32_t)oq + iq - tq;
#pragma unroll
            for (int i = 0; i < 8; i++) { Is[i] += rs; Iq[i] += rq; rs += p[i]; rq += p[i] * p[i]; }
            if (L.di) {   // column-de-interleaved row: even columns in the first half, odd columns in the second
                int32_t *row = sum + (size_t)(y + 1) * L.sum_pitch + (X0 >> 1);
                *reinterpret_cast<int4 *>(row) = make_int4((int)Is[0], (int)Is[2], (int)Is[4], (int)Is[6]);
                *reinterpret_cast<int4 *>(row + (L.sum_pitch >> 1)) = make_int4((int)Is[1], (int)Is[3], (int)Is[5], (int)Is[7]);
            } else {
                int4 *s = reinterpret_cast<int4 *>(sum + (size_t)(y + 1) * L.sum_pitch + X0);
                s[0] = make_int4((int)Is[0], (int)Is[1], (int)Is[2], (int)Is[3]);
                s[1] = make_int4((int)Is[4], (int)Is[5], (int)Is[6], (int)Is[7]);
            }
            if (SQ32) {
                uint4 *q = reinterpret_cast<uint4 *>(sq + (size_t)(y + 1) * L.sum_pitch + X0);
                q[0] = make_uint4((uint32_t)Iq[0], (uint32_t)Iq[1], (uint32_t)Iq[2], (uint32_t)Iq[3]);
                q[1] = make_uint4((uint32_t)Iq[4], (uint32_t)Iq[5], (uint32_t)Iq[6], (uint32_t)Iq[7]);
            } else {
                ulonglong2 *q = reinterpret_cast<ulonglong2 *>(sq + (size_t)(y + 1) * L.sum_pitch + X0);
                q[0] = make_ulonglong2(Iq[0], Iq[1]); q[1] = make_ulonglong2(Iq[2], Iq[3]);
                q[2] = make_ulonglong2(Iq[4], Iq[5]); q[3] = make_ulonglong2(Iq[6], Iq[7]);
            }
        }
    }
}

cudaError_t launch_integral_rows(const PyramidArgs &a, cudaStream_t stream, int *n_launches) {
    int n = 0;
#define CLFD_LAUNCH_INT(K, NT)                                                                          \
    if (a.n_integral_items[K] > 0 && a.n_frames > 0) {                                                  \
        if (a.sq32) k_integral_rows<NT, true><<<dim3(a.n_integral_items[K], a.n_frames), NT, 0, stream>>>(a, a.integral_items[K]); \
        else k_integral_rows<NT, false><<<dim3(a.n_integral_items[K], a.n_frames), NT, 0, stream>>>(a, a.integral_items[K]); \
        n++;                                                                                            \
    }
    CLFD_LAUNCH_INT(0, 32)
    CLFD_LAUNCH_INT(1, 64)
    CLFD_LAUNCH_INT(2, 128)
    CLFD_LAUNCH_INT(3, 256)
    CLFD_LAUNCH_INT(4, 512)
    CLFD_LAUNCH_INT(5, 1024)
#undef CLFD_LAUNCH_INT
    if (n_launches) *n_launches = n;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------
// K4: tilted integral.  tilted[Y][X] = sum_{y<Y, |x-(X-1)| <= (Y-1)-y} I[y][x]   (cvIntegral's third output,
//     tempcv.cpp:1302; the cone above pixel (Y-1, X-1)).
//
//     With A(y,x) = I(y,x) + A(y-1,x-1) and B(y,x) = I(y,x) + B(y-1,x+1) (the up-left / up-right diagonal
//     prefix sums, zero outside the image, one virtual zero column x = -1 that B runs into) the cone grows
//     from row to row by its two edges:  T(Y,X) = T(Y-1,X) + A(Y-1,X-1) + B(Y-1,X-1) - I(Y-1,X-1),  i.e.
//     T is the COLUMN prefix sum of G = A + B - I, and A, B are prefix sums along diagonals.  That makes it a
//     bandwidth problem with the same carry structure as the upright integral, only sheared:
//
//     k_tilt_tiles<false>  per (level, 32-row block, 192-column tile) one WARP: the block's own diagonal sums
//                          at its last row (LA, LB) and its column sums of G (LG), all from zero carries
//     k_tilt_diag          A / B carries at the top of every row block: a prefix over row blocks ALONG the
//                          diagonal (column shifts by 32 per block), one thread per diagonal
//     k_tilt_tcarry        T carries: prefix over row blocks of LG + the 32-wide window sums of the A / B
//                          carries that flow through the block (warp scans), one thread per column
//     k_tilt_tiles<true>   the same row loop seeded with the carries; writes T
//
//     The row loop is barrier free: a lane owns 8 columns, the diagonal shift is one shuffle per array and
//     row, and instead of exchanging diagonals between warps a tile carries 32 halo columns on either side
//     (inside a 32-row block a diagonal moves at most 31 columns), recomputing A / B there.  The pixel tile of
//     a warp is staged in shared memory by TMA bulk row copies; T is written 32 bytes per lane and row.
// ------------------------------------------------------------------------------------
constexpr int kTiltCols = 8;                        // columns per lane (16 was measured too: 84-106 registers, 16-20
                                                    // warps per SM, latency bound; 8 columns halve the register need)
constexpr int kTiltWords = kTiltCols / 4;           // 32-bit words of pixels / int4 vectors of sums per lane and row
constexpr int kTiltHalo = 32;                       // halo columns on either side
constexpr int kTiltHaloLanes = kTiltHalo / kTiltCols;
constexpr int kTiltInterior = 32 * kTiltCols - 2 * kTiltHalo;   // output columns per warp tile
constexpr int kTiltWarps = 4;                       // warp tiles per CTA
constexpr int kTiltRowBytes = 32 * kTiltCols;       // pixel bytes of one tile row
constexpr int kTiltSmemLocal = kRowBlock * kTiltRowBytes + 16;   // the warp's pixel tile + its mbarrier
static_assert(kTiltHalo >= kRowBlock && kTiltHalo % kTiltCols == 0, "a diagonal crosses < kRowBlock columns inside a block");
static_assert(kTiltCols == 8 || kTiltCols == 16, "pixel vectors of 8 or 16 bytes");

// planes of the carry buffer (each laid out like one plane of the column-sum buffer: [row block][X], pitch sum_pitch)
enum { kTcLA = 0, kTcLB, kTcLG, kTcAC, kTcBC, kTcTC, kTcPlanes };

struct TiltPix { uint32_t w[kTiltWords]; };
__device__ __forceinline__ TiltPix tilt_load_pix(const void *p) {
    TiltPix r;
    if (kTiltWords == 2) { const uint2 v = *reinterpret_cast<const uint2 *>(p); r.w[0] = v.x; r.w[1] = v.y; }
    else { const uint4 v = *reinterpret_cast<const uint4 *>(p); r.w[0] = v.x; r.w[1] = v.y; r.w[kTiltWords - 2] = v.z; r.w[kTiltWords - 1] = v.w; }
    return r;
}

template <bool FINAL>
__global__ void __launch_bounds__(32 * kTiltWarps) k_tilt_tiles(const PyramidArgs a) {
    extern __shared__ __align__(128) unsigned char tilt_smem[];
    const int lane = threadIdx.x & 31;
    const int item = blockIdx.x * kTiltWarps + (threadIdx.x >> 5);
    if (item >= a.n_tilt_tile_items) return;
    const int4 it = a.tilt_tile_items[item];   // (level, row block, column tile, -)
    const PyrLevel L = a.levels[it.x];
    const int frame = blockIdx.y, rb = it.y;
    // output columns X = x + 1 of this lane: [X0, X0 + kTiltCols); its pixel columns x = X0 - 1 + i
    const int X0 = it.z * kTiltInterior - kTiltHalo + lane * kTiltCols;
    const bool interior = lane >= kTiltHaloLanes && lane < 32 - kTiltHaloLanes && X0 < L.sum_pitch;
    const uint8_t *__restrict__ pyr = a.pyr + (size_t)frame * a.pyr_frame_stride + L.pyr_off;
    int32_t *__restrict__ til = a.tilted + (size_t)frame * a.sum_frame_stride + L.sum_off;
    int32_t *__restrict__ car = a.tcar + (size_t)frame * a.tcar_frame_stride + L.col_off + (size_t)rb * L.sum_pitch;
    const bool in_car = X0 >= 0 && X0 < L.sum_pitch;   // (sum_pitch and X0 are multiples of 8: whole int4 pairs)
    const bool in_pix = X0 >= 0 && X0 < L.pyr_pitch;   // aligned pixel vectors; padding bytes are zero

    int A[kTiltCols], B[kTiltCols], T[kTiltCols];
#pragma unroll
    for (int i = 0; i < kTiltCols; i++) A[i] = B[i] = T[i] = 0;
    const int n_vec = in_car ? min(kTiltCols, L.sum_pitch - X0) / 4 : 0;   // int4 vectors of this lane inside the row
    if (FINAL) {
#pragma unroll
        for (int v = 0; v < kTiltWords; v++) {
            if (v < n_vec) {
                const int4 va = *reinterpret_cast<const int4 *>(car + kTcAC * a.col_plane_stride + X0 + 4 * v);
                const int4 vb = *reinterpret_cast<const int4 *>(car + kTcBC * a.col_plane_stride + X0 + 4 * v);
                const int4 vt = *reinterpret_cast<const int4 *>(car + kTcTC * a.col_plane_stride + X0 + 4 * v);
                A[4 * v] = va.x; A[4 * v + 1] = va.y; A[4 * v + 2] = va.z; A[4 * v + 3] = va.w;
                B[4 * v] = vb.x; B[4 * v + 1] = vb.y; B[4 * v + 2] = vb.z; B[4 * v + 3] = vb.w;
                T[4 * v] = vt.x; T[4 * v + 1] = vt.y; T[4 * v + 2] = vt.z; T[4 * v + 3] = vt.w;
            }
        }
    }
    const int y0 = rb * kRowBlock, y1 = min(y0 + kRowBlock, L.h);
    if (FINAL && rb == 0 && interior) {   // row 0 of the tilted integral is zero
        for (int v = 0; v < n_vec; v++) *reinterpret_cast<int4 *>(til + X0 + 4 * v) = make_int4(0, 0, 0, 0);
    }
    // The warp's whole pixel tile (32 rows) is staged with one TMA bulk copy per row, all in flight at once: a warp
    // walks its rows one after the other, and register prefetching of a row or four ahead left it latency bound
    // (one DRAM round trip per row).  Lane r copies row y0 + r; columns outside [0, pyr_pitch) are not copied
    // (those lanes use zeros).
    unsigned char *wsm = tilt_smem + (size_t)(threadIdx.x >> 5) * kTiltSmemLocal;
    {
        uint64_t *bar = reinterpret_cast<uint64_t *>(wsm + kRowBlock * kTiltRowBytes);
        const int Xs = it.z * kTiltInterior - kTiltHalo;   // pixel column of the tile's first byte
        const int cs = max(Xs, 0), ce = min(Xs + kTiltRowBytes, L.pyr_pitch);
        const int nrows = y1 - y0;
        if (lane == 0) clif_mbar_init(bar, 1);
        __syncwarp();
        if (ce > cs) {
            if (lane == 0) clif_mbar_expect_tx(bar, (uint32_t)(nrows * (ce - cs)));
            __syncwarp();
            if (lane < nrows)
                clif_bulk_g2s(wsm + lane * kTiltRowBytes + (cs - Xs), pyr + (size_t)(y0 + lane) * L.pyr_pitch + cs, (uint32_t)(ce - cs), bar);
            clif_mbar_wait(bar, 0);
        }
    }
    for (int y = y0; y < y1; y++) {
        TiltPix cur;
#pragma unroll
        for (int k = 0; k < kTiltWords; k++) cur.w[k] = 0u;
        if (in_pix) cur = tilt_load_pix(wsm + (y - y0) * kTiltRowBytes + lane * kTiltCols);
        // p[i] = I(y, X0 - 1 + i): the left neighbour's last byte, then my first kTiltCols - 1
        int p[kTiltCols];
        p[0] = (int)(__shfl_up_sync(0xffffffffu, cur.w[kTiltWords - 1], 1) >> 24);
        if (lane == 0) p[0] = 0;
#pragma unroll
        for (int i = 1; i < kTiltCols; i++) p[i] = (int)((cur.w[(i - 1) >> 2] >> (8 * ((i - 1) & 3))) & 255u);
        int a_in = __shfl_up_sync(0xffffffffu, A[kTiltCols - 1], 1);     // A(y-1, x-1) for my first column
        int b_in = __shfl_down_sync(0xffffffffu, B[0], 1);              // B(y-1, x+1) for my last column
        if (lane == 0) a_in = 0;
        if (lane == 31) b_in = 0;
        // B(y,x) = I + B(y-1,x+1): ascending, in place
#pragma unroll
        for (int i = 0; i < kTiltCols; i++) B[i] = p[i] + (i + 1 < kTiltCols ? B[i + 1] : b_in);
        // A(y,x) = I + A(y-1,x-1): descending, in place;  G = A + B - I = A(y-1,x-1) + B(y,x)
#pragma unroll
        for (int i = kTiltCols - 1; i >= 0; i--) {
            const int up_left = i ? A[i - 1] : a_in;
            T[i] += up_left + B[i];
            A[i] = p[i] + up_left;
        }
        if (FINAL && interior) {
            int32_t *out = til + (size_t)(y + 1) * L.sum_pitch + X0;
#pragma unroll
            for (int v = 0; v < kTiltWords; v++)
                if (v < n_vec) *reinterpret_cast<int4 *>(out + 4 * v) = make_int4(T[4 * v], T[4 * v + 1], T[4 * v + 2], T[4 * v + 3]);
        }
    }
    if (!FINAL && interior) {
        // block-local diagonal sums at the last row and column sums of G; columns beyond the image hold zeros
#pragma unroll
        for (int i = 0; i < kTiltCols; i++)
            if (X0 + i > L.w) A[i] = B[i] = T[i] = 0;
#pragma unroll
        for (int v = 0; v < kTiltWords; v++) {
            if (v < n_vec) {
                *reinterpret_cast<int4 *>(car + kTcLA * a.col_plane_stride + X0 + 4 * v) = make_int4(A[4 * v], A[4 * v + 1], A[4 * v + 2], A[4 * v + 3]);
                *reinterpret_cast<int4 *>(car + kTcLB * a.col_plane_stride + X0 + 4 * v) = make_int4(B[4 * v], B[4 * v + 1], B[4 * v + 2], B[4 * v + 3]);
                *reinterpret_cast<int4 *>(car + kTcLG * a.col_plane_stride + X0 + 4 * v) = make_int4(T[4 * v], T[4 * v + 1], T[4 * v + 2], T[4 * v + 3]);
            }
        }
    }
}

// A / B carries.  AC_b(X) = A(32 b - 1, X - 1) = AC_{b-1}(X - 32) + LA_{b-1}(X): a prefix over row blocks along
// the diagonal X - 32 b = const; BC_b(X) = BC_{b-1}(X + 32) + LB_{b-1}(X) along X + 32 b = const.  blockIdx.z
// selects A or B; one thread per diagonal (all row blocks but the last are 32 rows high, and nobody needs the
// carries below the last one).
__global__ void __launch_bounds__(256) k_tilt_diag(const PyramidArgs a) {
    const int4 it = a.tilt_diag_items[blockIdx.x];   // (level, chunk of 256 diagonals, -, -)
    const PyrLevel L = a.levels[it.x];
    const int frame = blockIdx.y;
    const bool is_b = blockIdx.z != 0;
    const int span = (L.nrb - 1) * kRowBlock;         // diagonals start up to this far outside the image
    const int d = it.y * 256 + threadIdx.x;           // 0 .. w + span
    if (d > L.w + span) return;
    int32_t *__restrict__ car = a.tcar + (size_t)frame * a.tcar_frame_stride + L.col_off;
    const int32_t *__restrict__ loc = car + (is_b ? kTcLB : kTcLA) * a.col_plane_stride;
    int32_t *__restrict__ out = car + (is_b ? kTcBC : kTcAC) * a.col_plane_stride;
    // A: X_b = d - span + 32 b (enters from the left);  B: X_b = d - 32 b (enters from the right)
    // AC_b(X_b) = AC_{b-1}(X_{b-1}) + LA_{b-1}(X_b) while the diagonal is inside the image (the block's local sum
    // belongs to the column the diagonal LEAVES the block at), zero where it enters
    const int step = is_b ? -kRowBlock : kRowBlock;
    const int X0 = is_b ? d : d - span;
    int b_lo, b_hi;   // row blocks whose X_b = X0 + step * b lies in [0, w]
    if (is_b) { b_lo = X0 > L.w ? (X0 - L.w + kRowBlock - 1) / kRowBlock : 0; b_hi = X0 / kRowBlock; }
    else { b_lo = X0 < 0 ? (-X0 + kRowBlock - 1) / kRowBlock : 0; b_hi = (L.w - X0) / kRowBlock; }
    b_hi = min(b_hi, L.nrb - 1);
    int acc = 0;
    constexpr int kBatch = 8;    // loads in flight per thread, then the dependent adds and the stores (a 1080p level has 34 steps)
    for (int b0 = b_lo; b0 <= b_hi; b0 += kBatch) {
        int v[kBatch];
#pragma unroll
        for (int k = 0; k < kBatch; k++) {
            const int b = b0 + k;
            v[k] = (b <= b_hi && b > 0) ? __ldg(loc + (size_t)(b - 1) * L.sum_pitch + X0 + step * b) : 0;
        }
#pragma unroll
        for (int k = 0; k < kBatch; k++) {
            const int b = b0 + k;
            if (b <= b_hi) { acc += v[k]; out[(size_t)b * L.sum_pitch + X0 + step * b] = acc; }
        }
    }
}

// T carries.  TC_b(X) = T(32 b, X) = sum over the row blocks above of their column sums of G, where a block's
// G column sum = LG (its own pixels) + what the carries contribute while they cross the block:
// sum_{j=1..32} AC(X - j) + sum_{j=1..32} BC(X + j).  One warp per 32 columns, eight neighbouring groups per CTA:
// every warp scans its own group's AC and BC once and the neighbours meet through shared memory (the first warp also
// scans the group to its left, the last one the group to its right), one block barrier per row block on two buffers.
__global__ void __launch_bounds__(256) k_tilt_tcarry(const PyramidArgs a) {
    __shared__ int s_exa[2][9][32], s_tota[2][9], s_inb[2][9][32];   // [buffer][group -1 .. 7 (A) / 0 .. 8 (B)][lane]
    const int4 it = a.tilt_tc_items[blockIdx.x];     // (level, chunk of 8 column groups, -, -)
    const PyrLevel L = a.levels[it.x];
    const int frame = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int X = (it.y * 8 + w) * 32 + lane;
    int32_t *__restrict__ car = a.tcar + (size_t)frame * a.tcar_frame_stride + L.col_off;
    const size_t ps = a.col_plane_stride;
    auto at = [&](int plane, int b, int x) -> int {   // zero outside [0, w]
        return (x >= 0 && x <= L.w) ? car[plane * ps + (size_t)b * L.sum_pitch + x] : 0;
    };
    auto incl_scan = [&](int v) {
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, v, d);
            if (lane >= d) v += u;
        }
        return v;
    };
    int acc = 0;
    constexpr int kSteps = 4;   // row blocks whose loads are in flight together (8 measured slower: registers)
    for (int b0 = 0; b0 + 1 < L.nrb; b0 += kSteps) {
        int a_cur[kSteps], b_cur[kSteps], edge[kSteps], lg[kSteps];
#pragma unroll
        for (int k = 0; k < kSteps; k++) {
            const int b = min(b0 + k, L.nrb - 1);
            a_cur[k] = at(kTcAC, b, X); b_cur[k] = at(kTcBC, b, X);
            lg[k] = at(kTcLG, b, X);
            edge[k] = w == 0 ? at(kTcAC, b, X - 32) : w == 7 ? at(kTcBC, b, X + 32) : 0;   // (warp uniform)
        }
#pragma unroll
        for (int k = 0; k < kSteps; k++) {
            const int b = b0 + k;
            if (b + 1 >= L.nrb) break;   // (uniform over the CTA: one level)
            const int buf = b & 1;
            if (X <= L.w) car[kTcTC * ps + (size_t)b * L.sum_pitch + X] = acc;
            const int sa = incl_scan(a_cur[k]), sb = incl_scan(b_cur[k]);
            s_exa[buf][w + 1][lane] = sa - a_cur[k];
            s_inb[buf][w][lane] = sb;
            if (lane == 31) s_tota[buf][w + 1] = sa;
            if (w == 0) {
                const int se = incl_scan(edge[k]);
                s_exa[buf][0][lane] = se - edge[k];
                if (lane == 31) s_tota[buf][0] = se;
            } else if (w == 7) {
                s_inb[buf][8][lane] = incl_scan(edge[k]);
            }
            __syncthreads();
            // columns X-32 .. X-1: the previous group's lanes >= mine, this group's lanes < mine
            const int wa = (s_tota[buf][w] - s_exa[buf][w][lane]) + (sa - a_cur[k]);
            // columns X+1 .. X+32: this group's lanes > mine, the next group's lanes <= mine
            const int wb = (__shfl_sync(0xffffffffu, sb, 31) - sb) + s_inb[buf][w + 1][lane];
            acc += lg[k] + wa + wb;
        }
    }
    if (X <= L.w) car[kTcTC * ps + (size_t)(L.nrb - 1) * L.sum_pitch + X] = acc;
}

cudaError_t launch_tilted(const PyramidArgs &a, cudaStream_t stream, int *n_launches) {
    *n_launches = 0;
    if (a.n_tilt_tile_items == 0 || a.n_frames == 0 || !a.tilted) return cudaSuccess;
    *n_launches = 4;
    const dim3 tiles((a.n_tilt_tile_items + kTiltWarps - 1) / kTiltWarps, a.n_frames);
    const size_t smem = (size_t)kTiltWarps * kTiltSmemLocal;
    static SmemLimitCache lim_local, lim_final;
    if (cudaError_t e = lim_local.ensure(k_tilt_tiles<false>, smem)) return e;
    if (cudaError_t e = lim_final.ensure(k_tilt_tiles<true>, smem)) return e;
    k_tilt_tiles<false><<<tiles, 32 * kTiltWarps, smem, stream>>>(a);
    k_tilt_diag<<<dim3(a.n_tilt_diag_items, a.n_frames, 2), 256, 0, stream>>>(a);
    k_tilt_tcarry<<<dim3(a.n_tilt_tc_items, a.n_frames), 256, 0, stream>>>(a);
    k_tilt_tiles<true><<<tiles, 32 * kTiltWarps, smem, stream>>>(a);
    return cudaGetLastError();
}
int tilt_tile_interior() { return kTiltInterior; }

// ------------------------------------------------------------------------------------
// BGR(A) -> gray, OpenCV fixed point: (B*1868 + G*9617 + R*4899 + 8192) >> 14, a batch of interleaved frames per launch
// ------------------------------------------------------------------------------------
// A thread makes 16 gray pixels of one row and writes them with one 16-byte store (the gray pitch is a multiple of 16).
// Its source bytes are the 16 pixels' 16 * C bytes: read as C words of 16 bytes when the row starts 16-byte aligned, as
// 4 * C words of 4 bytes when it starts 4-byte aligned (a BGR group of 4 pixels is three words), and byte by byte
// otherwise (odd strides or base pointer) and for a row's last, partial group.  No byte behind a row's W * C bytes is
// read: the caller's buffer may end there (a frame stride below H * row_stride, or 0).
__device__ __forceinline__ uint32_t gray_of(uint32_t b, uint32_t g, uint32_t r) {
    return (b * 1868u + g * 9617u + r * 4899u + 8192u) >> 14;
}

template <int C>
__device__ __forceinline__ uint4 gray16_words(const uint8_t *__restrict__ p, bool a16) {
    constexpr int NW = 4 * C;   // 32-bit words of the group
    uint32_t w[NW];
    if (a16) {
#pragma unroll
        for (int k = 0; k < C; k++) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p) + k);
            w[4 * k] = v.x; w[4 * k + 1] = v.y; w[4 * k + 2] = v.z; w[4 * k + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int k = 0; k < NW; k++) w[k] = __ldg(reinterpret_cast<const uint32_t *>(p) + k);
    }
    uint32_t out[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const int j = i * C;   // byte offset of pixel i
        const uint32_t b = (w[j >> 2] >> (8 * (j & 3))) & 255u;
        const uint32_t g = (w[(j + 1) >> 2] >> (8 * ((j + 1) & 3))) & 255u;
        const uint32_t r = (w[(j + 2) >> 2] >> (8 * ((j + 2) & 3))) & 255u;
        out[i >> 2] |= gray_of(b, g, r) << (8 * (i & 3));
    }
    return make_uint4(out[0], out[1], out[2], out[3]);
}

// grid: (ceil(H * groups per row / 256), n_frames); one item = (row, group of 16 pixels)
template <int C>
__global__ void __launch_bounds__(256) k_color_to_gray(const ColorArgs a) {
    const int groups = (a.W + 15) >> 4;
    const int item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= a.H * groups) return;
    const int y = item / groups, x0 = (item - y * groups) * 16;
    const uint8_t *__restrict__ row = a.src + (size_t)blockIdx.y * a.frame_stride + (size_t)y * a.row_stride;
    const uint8_t *__restrict__ p = row + (size_t)x0 * C;
    uint4 v;
    if (x0 + 16 <= a.W && (reinterpret_cast<uintptr_t>(row) & 3) == 0) {
        v = gray16_words<C>(p, (reinterpret_cast<uintptr_t>(row) & 15) == 0);
    } else {
        uint32_t out[4] = {0u, 0u, 0u, 0u};   // pixels behind the row's end: zero padding of the gray row
        const int n = min(16, a.W - x0);
        for (int i = 0; i < n; i++)
            out[i >> 2] |= gray_of(__ldg(p + i * C), __ldg(p + i * C + 1), __ldg(p + i * C + 2)) << (8 * (i & 3));
        v = make_uint4(out[0], out[1], out[2], out[3]);
    }
    *reinterpret_cast<uint4 *>(a.dst + (size_t)blockIdx.y * a.dst_frame_stride + (size_t)y * a.dst_pitch + x0) = v;
}

cudaError_t launch_color_to_gray(const ColorArgs &a, cudaStream_t stream) {
    if (a.W <= 0 || a.H <= 0 || a.n_frames <= 0) return cudaSuccess;
    const long long items = (long long)a.H * ((a.W + 15) >> 4);
    const dim3 grid((unsigned)((items + 255) / 256), a.n_frames);
    if (a.channels == 4) k_color_to_gray<4><<<grid, 256, 0, stream>>>(a);
    else k_color_to_gray<3><<<grid, 256, 0, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace clfd
