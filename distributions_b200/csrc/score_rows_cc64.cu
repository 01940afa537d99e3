// score_rows_cc64.cu -- feature-list (cross-cat) instantiations of score_rows_kernel: 64-group tiles (see score_rows.cuh;
// split from score_rows.cu for compile time)
#include "score_rows.cuh"

namespace distb200 {

template <>
int launch_crosscat_tile<64, false, false>(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s,
                                           const MaskList *) {
    return launch_modes<64, -1, 256>(ctx, feats, a, s);
}

}  // namespace distb200
