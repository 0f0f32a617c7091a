// clfd_pack.h -- host-side packed cascade (device-ready arrays) and helpers.
#pragma once
#include "clfd_internal.h"

namespace clfd {

struct PackedCascade {
    DenseParams dense[2];              // kernel-parameter blobs of the smem-tile kernel: [ystep-1]
    int dense_stumps = 0;              // stumps in the stages the tile kernel evaluates
    std::vector<TailStump> tail[2];    // stumps of the tile-evaluated stages in tile-offset form, [ystep-1]
    std::vector<DenseStage> stage_tab[2];   // stage trees the tile kernel walks: all stages in execution order
    std::vector<DeepStage> deep_stages;  // global-memory blob of the deep kernel
    std::vector<DeepNode> deep_nodes;
    std::vector<int> tree_first_node;
    std::vector<float> alpha;
};

void pack_cascade(const HostCascade &c, PackedCascade &out);
// cvSetImagesForHaarClassifierCascade(scale) (tempcv.cpp:549-768) for one factor of the scale-cascade
// mode: fills L.inv_area / L.eq_off and n_nodes() ScNodes at `out` (pitch = elements per integral row)
void pack_sc_level(const HostCascade &c, double factor, int pitch, ScLevel &L, ScNode *out);
// scale-cascade mode, scales with window step 2: this scale as a ystep-2 blob of the tile kernel; false if
// the tile kernel cannot finish the cascade at this scale (the detector then keeps the generic kernels for it)
bool pack_sc_dense(const HostCascade &c, double scale, DenseParams &P, std::vector<TailStump> &tail,
                   std::vector<DenseStage> &stage_tab);
const char *get_error();

int dense_tile_stride(int win_w, int ystep);  // ints per smem tile row (ystep * stride = 8 mod 32)
int dense_tile_half(int win_w, int ystep);    // ystep 2: word offset of a row's odd columns inside a tile row (multiple of 4)
int dense_tile_rows(int win_h, int ystep, int tile_h);    // integral rows a tile needs
int dense_tile_cols(int win_w, int ystep);    // integral columns a tile needs (multiple of 4)

}  // namespace clfd
