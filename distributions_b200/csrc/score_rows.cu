// score_rows.cu -- dispatch of the row-mapped fused score(+prior)(+sample) kernel (score_rows.cuh), the cross-cat
// instantiations (KIND = -1: any feature list) and the GammaPoisson value-table builder.  The single-feature
// instantiations live in score_rows_{nich,gp,bnb,bb,dd}.cu.
#include "score_rows.cuh"

namespace distb200 {

// table[g][x] = GammaPoisson term of value x for group g, x < kGpTableX: built with gp_term itself (this
// translation unit, same flags) so the tabulated and the direct path agree bit for bit
__global__ void gp_table_kernel(const GpTableBatch b, NumericTables t) {
    __shared__ __align__(16) float coeff[33 * kLgammaRowStride];
    __shared__ float logfact[64];
    for (int i = threadIdx.x; i < 33 * kLgammaRowStride; i += blockDim.x) coeff[i] = t.lgamma5[i];
    if (threadIdx.x < 64) logfact[threadIdx.x] = t.log_factorial[threadIdx.x];
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= b.n_groups[blockIdx.y] * kGpTableX) return;
    const int g = i / kGpTableX, x = i % kGpTableX;
    const float v = gp_term(b.params[blockIdx.y][g], static_cast<uint32_t>(x), coeff, logfact);
    b.table[blockIdx.y][i] = v;
    // transposed copy [x][capacity] behind the table: the kSub re-score reads 16 consecutive groups of one value
    const int cap = b.n_groups[blockIdx.y];
    b.table[blockIdx.y][static_cast<size_t>(kGpTableX + x) * cap + g] = v;
}

int launch_gp_table_batch(dist_b200_ctx *ctx, const GpTableBatch &b, cudaStream_t s) {
    int most = 0;
    for (int i = 0; i < b.n; ++i) most = b.n_groups[i] > most ? b.n_groups[i] : most;
    if (b.n <= 0 || most <= 0) return DIST_B200_OK;
    const int n = most * kGpTableX;
    gp_table_kernel<<<dim3((n + 255) / 256, b.n), 256, 0, s>>>(b, ctx->tables);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("gp_table launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

template <>
int launch_crosscat_tile<128, false, false>(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s,
                                            const MaskList *) {
    return launch_modes<128, -1, 128>(ctx, feats, a, s);
}

int launch_score_rows(dist_b200_ctx *ctx, const FeatList &feats, int G, size_t N, const float *prior,
                      const float *u, int32_t *assign, float *scores, int accumulate, cudaStream_t s,
                      const PushTargets *push, float *logp, const MaskList *masks) {
    if (N == 0 || G == 0) return DIST_B200_OK;
    RowsArgs a{};
    if (push) {
        a.n_push = push->n;
        a.row0 = push->row0;
        a.block_rows = push->block_rows;
        for (int i = 0; i < push->n; ++i) a.push[i] = push->ptr[i];
        scores = push->ptr[0];  // selects the score-materialising kernel variants
    }
    a.G = G;
    a.N = N;
    a.prior = prior;
    a.u = u;
    a.assign = assign;
    a.scores = scores;
    a.accumulate = accumulate;
    a.t = ctx->tables;
    a.logp = logp;
    if (!assign && !scores && !logp) return fail(ctx, DIST_B200_ERR_INVALID, "score_rows: nothing to produce");
    if (feats.n == 1 && !masks) {  // a masked list of one runs the feature-list kernel
        int rc = DIST_B200_ERR_UNSUPPORTED;
        switch (feats.f[0].kind) {
            case DIST_B200_NICH: rc = launch_single_nich(ctx, feats, a, s); break;
            case DIST_B200_GP: rc = launch_single_gp(ctx, feats, a, s); break;
            case DIST_B200_BNB: rc = launch_single_bnb(ctx, feats, a, s); break;
            case DIST_B200_BB: rc = launch_single_bb(ctx, feats, a, s); break;
            case DIST_B200_DD: rc = launch_single_dd(ctx, feats, a, s); break;
        }
        if (rc != DIST_B200_ERR_UNSUPPORTED) return rc;
    }
    return launch_tiers<-1>(ctx, feats, a, s, masks);
}

}  // namespace distb200
