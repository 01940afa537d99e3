// score_rows_masked_cc.cu -- 32- and 64-group-tile instantiations of score_rows_kernel with masks (see score_rows_masked.cu)
#include "score_rows.cuh"

namespace distb200 {

template <int CHUNK>
static int masked_modes(dist_b200_ctx *ctx, const FeatList &feats, const MaskList &masks, const RowsArgs &a, cudaStream_t s) {
    if (a.logp) return launch_variant<CHUNK, -1, false, false, 256, false, true>(ctx, feats, a, s, &masks);
    if (a.assign && a.scores) return launch_variant<CHUNK, -1, true, true, 256, false, true>(ctx, feats, a, s, &masks);
    if (a.assign) return launch_variant<CHUNK, -1, true, false, 256, false, true>(ctx, feats, a, s, &masks);
    return launch_variant<CHUNK, -1, false, true, 256, false, true>(ctx, feats, a, s, &masks);
}

int launch_masked_tile32(dist_b200_ctx *ctx, const FeatList &feats, const MaskList &masks, const RowsArgs &a, cudaStream_t s) {
    return masked_modes<32>(ctx, feats, masks, a, s);
}

int launch_masked_tile64(dist_b200_ctx *ctx, const FeatList &feats, const MaskList &masks, const RowsArgs &a, cudaStream_t s) {
    return masked_modes<64>(ctx, feats, masks, a, s);
}

}  // namespace distb200
