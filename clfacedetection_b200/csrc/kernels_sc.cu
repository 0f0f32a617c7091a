// kernels_sc.cu -- scale-cascade mode (REF-SC) for sm_100a: the semantics of the
// cvHaarDetectObjects call of main.cpp:145 (flags = 0), i.e. tempcv.cpp:1330-1456 +
// HaarDetectObjects_ScaleCascade_Invoker (tempcv.cpp:1132-1175) + cvRunHaarClassifierCascadeSum
// (tempcv.cpp:795-972) on ONE full-frame integral image with the features scaled per factor.
// It is also the formulation clod itself uses (clod.cpp:1176-1336 / clod.cl:32-93: scaled
// features, one integral), so this is what replaces runStage when the caller asks for the
// demo's other column.
//
// The windows are evaluated by the tile kernel (scales of window step 2) and by the generic kernels
// (kernels_clod.cu, ScaleWindow): one thread per grid position (scale, iy, ix), lanes = consecutive ix,
// so the 32 corner loads of a warp are 32 * ystep * 4 bytes apart at most (a few cache lines); the
// integral image of a frame (8-25 MB) lives in L2.  Linear cascades run in a few passes over growing
// stage ranges with the survivors re-compacted through a queue in between, and the large late stages
// (>= 50 trees) one warp per survivor, lanes over trees.  Every position is evaluated -- the
// reference's skip rule makes the set of evaluated windows depend on the RESULTS of their left
// neighbours, so it is applied afterwards:
//   k_sc_rows : one thread per grid row walks its exit codes left to right with the invoker's
//       rule "ixstep = result != 0 ? 1 : 2" (tempcv.cpp:1161), marks the positions the
//       reference never evaluates and appends a rect for every evaluated, accepted window.
#include <cstdint>

#include "kernels.h"

namespace clfd {

typedef unsigned long long ull;

__global__ void __launch_bounds__(128) k_sc_rows(const __grid_constant__ ScArgs a) {
    const int row = blockIdx.x * 128 + threadIdx.x;
    const int frame = blockIdx.y;
    if (row >= a.rows_per_frame) return;
    int lo = 0, hi = a.n_scales - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(&a.scales[mid].row_base) <= row) lo = mid; else hi = mid - 1;
    }
    const ScLevel L = a.scales[lo];
    const int iy = row - L.row_base;
    int16_t *codes = a.codes + (size_t)frame * a.windows_per_frame + L.win_base + (size_t)iy * L.nx;
    const DeepCascadeDev &D = a.deep;
    const int y = __double2int_rn(__dmul_rn((double)iy, L.ystep));
    bool evaluate = true;   // tempcv.cpp:1141-1161: ixstep = result != 0 ? 1 : 2
    for (int ix = 0; ix < L.nx; ix++) {
        if (!evaluate) {
            codes[ix] = (int16_t)kScCodeSkipped;
            evaluate = true;
            continue;
        }
        const int code = codes[ix];
        int result;   // what cvRunHaarClassifierCascade returned
        if (code == kScCodeOutside) result = -1;
        else if (D.is_tree) result = code & 1;
        else result = code == D.n_stages ? 1 : -code;
        if (result > 0) {
            const ull slot = atomicAdd(a.counters + 0, 1ull);
            if (slot < a.rect_cap) {
                DevRect r;
                r.x = __double2int_rn(__dmul_rn((double)ix, L.ystep)); r.y = y;
                r.w = L.win_w; r.h = L.win_h; r.frame = a.frame_base + frame; r.cascade = a.cascade_index;
                a.rects[slot] = r;
            } else {
                atomicAdd(a.counters + 2, 1ull);
            }
        }
        evaluate = result != 0;
    }
}

cudaError_t launch_sc_rows(const ScArgs &a, cudaStream_t stream) {
    if (a.windows_per_frame == 0 || a.n_frames == 0) return cudaSuccess;
    k_sc_rows<<<dim3((unsigned)((a.rows_per_frame + 127) / 128), a.n_frames), 128, 0, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace clfd
