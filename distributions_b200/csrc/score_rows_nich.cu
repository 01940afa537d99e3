// score_rows_nich.cu -- single-feature instantiations of score_rows_kernel for one model (see score_rows.cuh)
#include "score_rows.cuh"

namespace distb200 {

int launch_nich_rows(dist_b200_ctx *ctx, const float4 *params, const void *column, int G, size_t N, const float *prior,
                     const float *u, int32_t *assign, cudaStream_t s);  // nich_rows.cu
int launch_nich_logp(dist_b200_ctx *ctx, const float4 *params, const void *column, int G, size_t N, const float *prior,
                     float *logp, cudaStream_t s);  // nich_rows.cu

int launch_single_nich(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s) {
    // DIST_B200_OPT_NICH_PACKED (A/B runs): 0 = default, 1 = scalar loop (round 1), 2 = packed fp32x2 loop, one row per thread
    const int v = ctx->opt[DIST_B200_OPT_NICH_PACKED];
    if (v == 1) return launch_tiers<DIST_B200_NICH>(ctx, feats, a, s);
    if (v == 0 && a.G > 128 && a.logp) {  // logp: the static-reference kernel without slots (nich_rows.cu)
        const int rc = launch_nich_logp(ctx, static_cast<const float4 *>(feats.f[0].params), feats.f[0].column, a.G, a.N, a.prior,
                                        a.logp, s);
        if (rc != DIST_B200_ERR_UNSUPPORTED) return rc;
    }
    if ((v == 0 || v == 3) && a.G > 128 && a.assign && !a.scores && !a.accumulate && !a.n_push) {  // sampling only: nich_rows.cu
        const int rc = launch_nich_rows(ctx, static_cast<const float4 *>(feats.f[0].params), feats.f[0].column, a.G, a.N, a.prior,
                                        a.u, a.assign, s);
        if (rc != DIST_B200_ERR_UNSUPPORTED) return rc;
    }
    return launch_tiers<kKindNichPacked>(ctx, feats, a, s);
}

}  // namespace distb200
