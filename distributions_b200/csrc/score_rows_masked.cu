// score_rows_masked.cu -- feature lists with missing cells: dispatch of score_rows_kernel with masks (score_rows.cuh) and its
// 128-group-tile and kSub instantiations.  The 32- and 64-group tiles live in score_rows_masked_cc.cu (compile time).
// The tiers are those of the unmasked feature-list kernel (launch_tiers<-1>); the A/B options are not consulted.
#include "score_rows.cuh"

namespace distb200 {

int launch_masked_tile32(dist_b200_ctx *ctx, const FeatList &feats, const MaskList &masks, const RowsArgs &a, cudaStream_t s);
int launch_masked_tile64(dist_b200_ctx *ctx, const FeatList &feats, const MaskList &masks, const RowsArgs &a, cudaStream_t s);

int launch_score_rows_masked(dist_b200_ctx *ctx, const FeatList &feats, const MaskList &masks, int G, size_t N,
                             const float *prior, const float *u, int32_t *assign, float *scores, int accumulate,
                             float *logp, cudaStream_t s) {
    if (N == 0 || G == 0) return DIST_B200_OK;
    if (!assign && !scores && !logp) return fail(ctx, DIST_B200_ERR_INVALID, "score_rows: nothing to produce");
    RowsArgs a{};
    a.G = G;
    a.N = N;
    a.prior = prior;
    a.u = u;
    a.assign = assign;
    a.scores = scores;
    a.accumulate = accumulate;
    a.t = ctx->tables;
    a.logp = logp;
    if (G <= 32) return launch_masked_tile32(ctx, feats, masks, a, s);
    if (G <= 64) return launch_masked_tile64(ctx, feats, masks, a, s);
    if (G <= 128) {
        if (logp) return launch_masked_tile64(ctx, feats, masks, a, s);  // (a 128-group logp tile does not fit in registers)
        if (assign && scores) return launch_variant<128, -1, true, true, 128, false, true>(ctx, feats, a, s, &masks);
        if (assign) return launch_variant<128, -1, true, false, 128, false, true>(ctx, feats, a, s, &masks);
        return launch_variant<128, -1, false, true, 128, false, true>(ctx, feats, a, s, &masks);
    }
    if (assign && !scores && ksub_wanted(feats, G)) {
        FeatList local;
        if (int rc = ksub_list(ctx, feats, G, local, s)) return rc;
        const int rc = launch_variant<128, -1, true, false, 128, true, true>(ctx, local, a, s, &masks);
        if (rc != DIST_B200_ERR_UNSUPPORTED) return rc;
    }
    if (scores) return launch_masked_tile64(ctx, feats, masks, a, s);
    return launch_masked_tile32(ctx, feats, masks, a, s);
}

}  // namespace distb200
