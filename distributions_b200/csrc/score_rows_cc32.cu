// score_rows_cc32.cu -- feature-list (cross-cat) instantiations of score_rows_kernel: 32-group tiles and the kSub streaming
// kernel (see score_rows.cuh; split from score_rows.cu for compile time)
#include "score_rows.cuh"

namespace distb200 {

template <>
int launch_crosscat_tile<32, false, false>(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s,
                                           const MaskList *) {
    return launch_modes<32, -1, 256>(ctx, feats, a, s);
}

template <>
int launch_crosscat_tile<128, true, false>(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s,
                                           const MaskList *) {
    return launch_variant<128, -1, true, false, 128, true>(ctx, feats, a, s);
}

}  // namespace distb200
