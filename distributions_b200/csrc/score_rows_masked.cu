// score_rows_masked.cu -- feature-list instantiations of score_rows_kernel with masks (missing cells): 128-group tiles and
// the kSub streaming kernel.  The 32- and 64-group tiles live in score_rows_masked_cc.cu (compile time).
#include "score_rows.cuh"

namespace distb200 {

template <>
int launch_crosscat_tile<128, false, true>(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s,
                                           const MaskList *masks) {
    return launch_modes<128, -1, 128, true>(ctx, feats, a, s, masks);
}

template <>
int launch_crosscat_tile<128, true, true>(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s,
                                          const MaskList *masks) {
    return launch_variant<128, -1, true, false, 128, true, true>(ctx, feats, a, s, masks);
}

}  // namespace distb200
