// score_rows_masked_cc.cu -- 32- and 64-group-tile instantiations of score_rows_kernel with masks (see score_rows_masked.cu)
#include "score_rows.cuh"

namespace distb200 {

template <>
int launch_crosscat_tile<32, false, true>(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s,
                                          const MaskList *masks) {
    return launch_modes<32, -1, 256, true>(ctx, feats, a, s, masks);
}

template <>
int launch_crosscat_tile<64, false, true>(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s,
                                          const MaskList *masks) {
    return launch_modes<64, -1, 256, true>(ctx, feats, a, s, masks);
}

}  // namespace distb200
