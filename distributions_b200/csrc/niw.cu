// niw.cu -- NormalInverseWishart<d>: batched form of looping Group::score_value over groups.
//
// The reference has no NIW Mixture; a value is scored by Scorer::eval (models/niw.hpp:343-361):
//   post  = Shared::plus_group(group)                                  (niw.hpp:82-103)
//   dof   = post.nu - d + 1;  sigma = post.psi * (post.kappa + 1) / (post.kappa * dof)
//   score = score_mv_student_t(value, dof, post.mu, sigma)             (random.hpp:160-185)
// and score_mv_student_t re-derives sigma.inverse() and sigma.determinant() on EVERY call.
//
// Here the per-group work is hoisted into niw_prep_kernel (once per batch, double precision):
// posterior, Cholesky sigma = L L^T, whitening matrix W = L^-1, determinant, Student-t constants.
// Then  diff^T sigma^-1 diff = |W (x - mu')|^2, a sum of squares (non-negative, no cancellation in the
// final sum), and
//   score[n][g] = C_g - 0.5 (dof_g + d) * fast_log(1 + |W_g (x_n - mu'_g)|^2 / dof_g).
//
// niw_score_kernel (this file, FP32 CUDA-core form): rows on lanes, two rows per thread held in
// registers, group tiles (mu', W, constants) streamed through shared memory with cp.async double
// buffering and read as broadcast LDS.128; scores leave through a padded per-warp tile so that global
// stores are coalesced.  The sampler then runs over the materialised scores (gather_rows.cu).
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "posterior.cuh"

namespace distb200 {

// per-group record: mu'[DP] | W[DP][DP] row-major lower triangular (zero above the diagonal) |
// {C_g, -0.5 (dof + d) ln 2, 1 / dof, 0}
__host__ __device__ constexpr int niw_group_floats(int dp) { return dp + dp * dp + 4; }

// one block per group; d <= 32
__global__ void niw_prep_kernel(int d, int dp, const float *__restrict__ mu, float kappa,
                                const float *__restrict__ psi, float nu, const int32_t *__restrict__ count,
                                const float *__restrict__ sum_x, const float *__restrict__ sum_xxT,
                                float *__restrict__ out, NumericTables t) {
    __shared__ double S[32][33];  // sigma, then its Cholesky factor L (lower)
    __shared__ double Winv[32][33];
    __shared__ double xbar[32], diff[32];
    const int g = blockIdx.x, tid = threadIdx.x;
    const double dof = niw_posterior_cholesky(d, mu, kappa, psi, nu, count[g], sum_x + static_cast<size_t>(g) * d,
                                              sum_xxT + static_cast<size_t>(g) * d * d, S, xbar, diff);
    // W = L^-1 by forward substitution, one column per thread
    if (tid < d) {
        const int c = tid;
        for (int i = 0; i < d; ++i) {
            double s = (i == c) ? 1.0 : 0.0;
            for (int k = c; k < i; ++k) s -= S[i][k] * Winv[k][c];
            Winv[i][c] = (i >= c) ? s / S[i][i] : 0.0;
        }
    }
    __syncthreads();
    float *rec = out + static_cast<size_t>(g) * niw_group_floats(dp);
    for (int i = tid; i < dp; i += blockDim.x)
        rec[i] = i < d ? static_cast<float>(niw_post_mu(kappa, count[g], mu[i], xbar[i])) : 0.f;
    for (int e = tid; e < dp * dp; e += blockDim.x) {
        const int i = e / dp, j = e % dp;
        rec[dp + e] = (i < d && j <= i) ? static_cast<float>(Winv[i][j]) : 0.f;
    }
    if (tid == 0) {
        double det = 1.0, logdet = 0.0;
        for (int i = 0; i < d; ++i) {
            det *= S[i][i] * S[i][i];
            logdet += 2.0 * log(S[i][i]);
        }
        // score_mv_student_t's constant terms, with its float/double mix (random.hpp:166-178)
        const float dof_f = static_cast<float>(dof);
        const float log_pi = 1.1447298858494002f;
        const float term1 = fast_lgamma_exact(static_cast<float>(dof_f / 2. + static_cast<float>(d) / 2.), t.lgamma5) -
                            fast_lgamma_exact(static_cast<float>(dof_f / 2.), t.lgamma5);
        const float term2 = static_cast<float>(-0.5 * niw_log_det(det, logdet, t.log2_table) -
                                               static_cast<float>(d) / 2. * (fast_log_table(dof_f, t.log2_table) + log_pi));
        float *k4 = rec + dp + dp * dp;
        k4[0] = term1 + term2;
        k4[1] = static_cast<float>(-0.5 * (dof_f + static_cast<float>(d))) * kLn2;
        k4[2] = 1.f / dof_f;
        k4[3] = 0.f;
    }
}

// 32 < d <= 128: the same record at DP = 64 / 128, except that its first DP floats hold b = W (mu' - mu0) (mu0 = Shared.mu)
// instead of mu' -- the tensor-core route scores x - mu0 against it (niw_tc_wide.cu).  One block of kNiwWideThreads per
// group; a double [128][129] matrix is 132 KB, so W = L^-1 overwrites L in place (dynamic shared memory).
constexpr int kNiwWideThreads = 256;
constexpr int kNiwWideLd = 129;
constexpr size_t kNiwWidePrepSmem = sizeof(double) * (128 * kNiwWideLd + 4 * 128);

__global__ void __launch_bounds__(kNiwWideThreads) niw_prep_wide_kernel(int d, int dp, const float *__restrict__ mu, float kappa,
                                                                        const float *__restrict__ psi, float nu,
                                                                        const int32_t *__restrict__ count, const float *__restrict__ sum_x,
                                                                        const float *__restrict__ sum_xxT, float *__restrict__ out,
                                                                        NumericTables t) {
    extern __shared__ double wsm[];
    double(*S)[kNiwWideLd] = reinterpret_cast<double(*)[kNiwWideLd]>(wsm);  // sigma, then L (lower), then W = L^-1 (lower)
    double *xbar = wsm + 128 * kNiwWideLd, *diff = xbar + 128, *col = diff + 128, *dm = col + 128;
    __shared__ double det_s[2];
    const int g = blockIdx.x, tid = threadIdx.x;
    const double dof = niw_posterior_cholesky<kNiwWideLd>(d, mu, kappa, psi, nu, count[g], sum_x + static_cast<size_t>(g) * d,
                                                          sum_xxT + static_cast<size_t>(g) * d * d, S, xbar, diff);
    if (tid == 0) {
        double det = 1.0, logdet = 0.0;
        for (int i = 0; i < d; ++i) {
            det *= S[i][i] * S[i][i];
            logdet += 2.0 * log(S[i][i]);
        }
        det_s[0] = det;
        det_s[1] = logdet;
    }
    if (tid < d) dm[tid] = niw_post_mu(kappa, count[g], mu[tid], xbar[tid]) - static_cast<double>(mu[tid]);
    // in-place inverse, right to left: with L = [l 0; c L2], W = [1/l 0; -L2^-1 c / l  L2^-1], so column j of W needs
    // column j of L (saved first) and the columns right of j, which already hold W
    for (int j = d - 1; j >= 0; --j) {
        __syncthreads();
        if (tid > j && tid < d) col[tid] = S[tid][j];
        __syncthreads();
        const double ljj = S[j][j];
        __syncthreads();
        if (tid > j && tid < d) {
            double s = 0.0;
            for (int k = j + 1; k <= tid; ++k) s += S[tid][k] * col[k];
            S[tid][j] = -s / ljj;
        }
        if (tid == j) S[j][j] = 1.0 / ljj;
    }
    __syncthreads();
    float *rec = out + static_cast<size_t>(g) * niw_group_floats(dp);
    for (int i = tid; i < dp; i += blockDim.x) {
        double b = 0.0;
        if (i < d)
            for (int k = 0; k <= i; ++k) b += S[i][k] * dm[k];
        rec[i] = static_cast<float>(b);
    }
    for (int e = tid; e < dp * dp; e += blockDim.x) {
        const int i = e / dp, j = e % dp;
        rec[dp + e] = (i < d && j <= i) ? static_cast<float>(S[i][j]) : 0.f;
    }
    if (tid == 0) {  // as niw_prep_kernel
        const float dof_f = static_cast<float>(dof);
        const float log_pi = 1.1447298858494002f;
        const float term1 = fast_lgamma_exact(static_cast<float>(dof_f / 2. + static_cast<float>(d) / 2.), t.lgamma5) -
                            fast_lgamma_exact(static_cast<float>(dof_f / 2.), t.lgamma5);
        const float term2 = static_cast<float>(-0.5 * niw_log_det(det_s[0], det_s[1], t.log2_table) -
                                               static_cast<float>(d) / 2. * (fast_log_table(dof_f, t.log2_table) + log_pi));
        float *k4 = rec + dp + dp * dp;
        k4[0] = term1 + term2;
        k4[1] = static_cast<float>(-0.5 * (dof_f + static_cast<float>(d))) * kLn2;
        k4[2] = 1.f / dof_f;
        k4[3] = 0.f;
    }
}

int niw_padded_dim(int d);

constexpr int kNiwThreads = 128;
constexpr int kNiwRows = 2;  // rows per thread

__device__ __forceinline__ void niw_cp_async16(void *smem_dst, const void *gmem_src) {
    const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}

struct NiwArgs {
    int G, d, accumulate;
    size_t N;
    const float *recs;    // [G] group records
    const float *values;  // [N][d]
    const float *prior;   // [G] or nullptr
    float *scores;        // [N][G]
};

// DP: padded dimension (4, 8, 16, 32); GT: groups per staging tile
template <int DP, int GT>
__global__ void __launch_bounds__(kNiwThreads) niw_score_kernel(const NiwArgs a) {
    constexpr int REC = niw_group_floats(DP);
    extern __shared__ __align__(16) float smem[];
    float *stage = smem;                              // [2][GT * REC]
    float *tile = smem + 2 * GT * REC;                // [warps][rows per thread][32][33]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = a.G, d = a.d;
    const int ntile_g = (G + GT - 1) / GT;
    const size_t rows_per_block = static_cast<size_t>(kNiwThreads) * kNiwRows;
    const size_t nblk = (a.N + rows_per_block - 1) / rows_per_block;

    for (size_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const size_t base = blk * rows_per_block;
        float x[kNiwRows][DP];
#pragma unroll
        for (int r = 0; r < kNiwRows; ++r) {
            size_t row = base + static_cast<size_t>(r) * kNiwThreads + tid;
            if (row >= a.N) row = a.N - 1;
            const float *src = a.values + row * d;
#pragma unroll
            for (int k = 0; k < DP; ++k) x[r][k] = k < d ? src[k] : 0.f;
        }
        __syncthreads();  // staging buffers free
        {   // stage group tile 0
            const float *src = a.recs;
            const int n = min(GT, G) * REC;
            for (int i = tid * 4; i < n; i += kNiwThreads * 4) niw_cp_async16(stage + i, src + i);
            asm volatile("cp.async.commit_group;\n" ::);
        }
        for (int gt = 0; gt < ntile_g; ++gt) {
            if (gt + 1 < ntile_g) {
                const float *src = a.recs + static_cast<size_t>(gt + 1) * GT * REC;
                const int n = min(GT, G - (gt + 1) * GT) * REC;
                float *dst = stage + ((gt + 1) & 1) * GT * REC;
                for (int i = tid * 4; i < n; i += kNiwThreads * 4) niw_cp_async16(dst + i, src + i);
                asm volatile("cp.async.commit_group;\n" ::);
                asm volatile("cp.async.wait_group 1;\n" ::);
            } else {
                asm volatile("cp.async.wait_group 0;\n" ::);
            }
            __syncthreads();
            const float *buf = stage + (gt & 1) * GT * REC;
            const int ng = min(GT, G - gt * GT);
            for (int j = 0; j < ng; ++j) {
                const float *rec = buf + j * REC;
                float z[kNiwRows][DP];
#pragma unroll
                for (int k = 0; k < DP; k += 4) {
                    const float4 m = *reinterpret_cast<const float4 *>(rec + k);
#pragma unroll
                    for (int r = 0; r < kNiwRows; ++r) {
                        z[r][k] = x[r][k] - m.x;
                        z[r][k + 1] = x[r][k + 1] - m.y;
                        z[r][k + 2] = x[r][k + 2] - m.z;
                        z[r][k + 3] = x[r][k + 3] - m.w;
                    }
                }
                float q[kNiwRows];
#pragma unroll
                for (int r = 0; r < kNiwRows; ++r) q[r] = 0.f;
                const float *W = rec + DP;
#pragma unroll
                for (int i = 0; i < DP; ++i) {
                    float y[kNiwRows];
#pragma unroll
                    for (int r = 0; r < kNiwRows; ++r) y[r] = 0.f;
#pragma unroll
                    for (int k = 0; k <= i; k += 4) {
                        const float4 w = *reinterpret_cast<const float4 *>(W + i * DP + k);
#pragma unroll
                        for (int r = 0; r < kNiwRows; ++r) {
                            y[r] = fmaf(w.x, z[r][k], y[r]);
                            if (k + 1 <= i) y[r] = fmaf(w.y, z[r][k + 1], y[r]);
                            if (k + 2 <= i) y[r] = fmaf(w.z, z[r][k + 2], y[r]);
                            if (k + 3 <= i) y[r] = fmaf(w.w, z[r][k + 3], y[r]);
                        }
                    }
#pragma unroll
                    for (int r = 0; r < kNiwRows; ++r) q[r] = fmaf(y[r], y[r], q[r]);
                }
                const float4 c = *reinterpret_cast<const float4 *>(rec + DP + DP * DP);
                const int g = gt * GT + j;
                const float pr = (a.prior && !a.accumulate) ? a.prior[g] : 0.f;
#pragma unroll
                for (int r = 0; r < kNiwRows; ++r) {
                    // C_g - 0.5 (dof + d) * fast_log(1 + q / dof)
                    const float arg = __fadd_rn(1.f, __fmul_rn(c.z, q[r]));
                    const float s = fmaf(c.y, fast_log2_cell(arg), c.x) + pr;
                    // park in the per-warp tile: column (g & 31), flushed every 32 groups
                    float *tw = tile + (warp * kNiwRows + r) * 32 * 33;
                    tw[lane * 33 + (g & 31)] = s;
                    if (((g & 31) == 31 || g == G - 1)) {
                        __syncwarp();
                        const int g0 = g & ~31;
                        const int gl = g0 + lane;
                        const size_t wrow0 = base + static_cast<size_t>(r) * kNiwThreads + warp * 32;
                        if (gl <= g) {
                            for (int i = 0; i < 32; ++i) {
                                const size_t rr = wrow0 + i;
                                if (rr >= a.N) break;
                                float *dst = a.scores + rr * G + gl;
                                const float v = tw[i * 33 + lane];
                                *dst = a.accumulate ? *dst + v : v;
                            }
                        }
                        __syncwarp();
                    }
                }
            }
            __syncthreads();  // buffer (gt & 1) is refilled two tiles from now
        }
    }
}

template <int DP>
static int launch_niw_dp(dist_b200_ctx *ctx, const NiwArgs &a, cudaStream_t s) {
    constexpr int GT = DP >= 32 ? 8 : (DP >= 16 ? 16 : 32);
    const size_t smem = sizeof(float) * (2 * GT * niw_group_floats(DP) + (kNiwThreads / 32) * kNiwRows * 32 * 33);
    auto kern = niw_score_kernel<DP, GT>;
    DISTB200_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    int per_sm = 0;
    DISTB200_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kNiwThreads, smem));
    if (per_sm < 1) per_sm = 1;
    const size_t rows_per_block = static_cast<size_t>(kNiwThreads) * kNiwRows;
    const size_t nblk = (a.N + rows_per_block - 1) / rows_per_block;
    const size_t cap = static_cast<size_t>(ctx->sm_count) * per_sm;
    kern<<<static_cast<unsigned>(nblk < cap ? nblk : cap), kNiwThreads, smem, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("niw launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

// ------------------------------------------------------------------------------------------------
// niw_rows_kernel -- d <= 8, sampling only: scores, clustering prior and sample_from_scores fused, nothing materialised
// (the generic route above writes [N][G] scores and runs the stand-alone sampler: at d = 3 the sampler alone costs as
// much as the scoring, and the scoring runs 8 warps per SM on broadcast LDS.128s amortised over two rows).
// Same plan as nich_rows2_kernel (nich_rows.cu): rows on lanes, R rows per thread, the group records resident in shared
// memory, weights formed directly against a STATIC reference
//   score_g(x) = C_g + prior_g - 0.5 (dof + d) ln(1 + q / dof) <= C_g + prior_g,   M* = max_g (C_g + prior_g),
//   e_g = 2^(co_g lg2(1 + q / dof) + (C_g + prior_g - M*) log2 e),
// summed per slot of 16 groups; the slot holding u * total is re-evaluated and walked.  For small d the bound is close
// (own-cluster q ~ d); rows whose total comes out below 2^-40 are re-evaluated with their own maximum.  The quadratic form
// is accumulated exactly as niw_score_kernel does (same fmaf order), so both routes see the same fast_log argument.
constexpr int kNiwSmallThreads = 256;
constexpr int kNiwSlotGroups = 16;
constexpr float kNiwRedo = 9.094947e-13f;  // 2^-40

struct NiwRowsArgs {
    int G, d;
    size_t N;
    const float *recs;
    const float *values;
    const float *prior;
    const float *u;
    int32_t *assign;
};

// exponents of one PAIR of groups: the block's records are interleaved element-wise per pair, {-mu', W, co, sc', 1 / dof, -}
// of groups (a, b) as (e_a, e_b) pairs, so an LDS.128 yields two packed fp32x2 operands and every FADD / FFMA of the
// quadratic form serves both groups (fma.rn.f32x2: each element rounded as the scalar fmaf of niw_score_kernel)
template <int DP>
__device__ __forceinline__ uint64_t niw_small_arg2(const float *__restrict__ rec2, const uint64_t (&x2)[DP]) {
    uint64_t z2[DP];
#pragma unroll
    for (int k = 0; k < DP; k += 2) {
        const float4 m = *reinterpret_cast<const float4 *>(rec2 + 2 * k);
        z2[k] = f2_add(x2[k], f2_pack(m.x, m.y));
        z2[k + 1] = f2_add(x2[k + 1], f2_pack(m.z, m.w));
    }
    uint64_t q2 = f2_pack(0.f, 0.f);
    const float *W2 = rec2 + 2 * DP;
#pragma unroll
    for (int i = 0; i < DP; ++i) {
        uint64_t y2 = f2_pack(0.f, 0.f);
#pragma unroll
        for (int k = 0; k <= i; k += 2) {
            const float4 w = *reinterpret_cast<const float4 *>(W2 + 2 * (i * DP + k));
            y2 = f2_fma(f2_pack(w.x, w.y), z2[k], y2);
            if (k + 1 <= i) y2 = f2_fma(f2_pack(w.z, w.w), z2[k + 1], y2);
        }
        q2 = f2_fma(y2, y2, q2);
    }
    const float4 c0 = *reinterpret_cast<const float4 *>(rec2 + 2 * (DP + DP * DP));      // co a, co b, sc' a, sc' b
    const float4 c1 = *reinterpret_cast<const float4 *>(rec2 + 2 * (DP + DP * DP) + 4);  // 1 / dof a, 1 / dof b
    const uint64_t one2 = f2_pack(1.f, 1.f);
    float aa, ab;
    f2_unpack(f2_fma(f2_mul(f2_pack(c1.x, c1.y), q2), one2, one2), aa, ab);  // unfused 1 + q / dof
    return f2_fma(f2_pack(c0.x, c0.y), f2_pack(fast_log2_cell(aa), fast_log2_cell(ab)), f2_pack(c0.z, c0.w));
}

// scores_to_likelihoods + sample_from_likelihoods with the row's own maximum (random.cc:94-106, random.hpp:315-333)
template <int DP>
__device__ __noinline__ int niw_small_row_exact(const float *__restrict__ recs_s, int G, const float (&x)[DP], float u) {
    constexpr int REC = niw_group_floats(DP);
    uint64_t x2[DP];
#pragma unroll
    for (int k = 0; k < DP; ++k) x2[k] = f2_pack(x[k], x[k]);
    const int npairs = (G + 1) / 2;
    float m = -INFINITY;
    for (int p = 0; p < npairs; ++p) {
        float a0, a1;
        f2_unpack(niw_small_arg2<DP>(recs_s + p * 2 * REC, x2), a0, a1);
        m = fmaxf(m, fmaxf(a0, a1));  // the padding half of an odd last pair is -inf
    }
    float total = 0.f;
    for (int p = 0; p < npairs; ++p) {
        float a0, a1;
        f2_unpack(niw_small_arg2<DP>(recs_s + p * 2 * REC, x2), a0, a1);
        total += mufu_ex2(a0 - m);
        total += mufu_ex2(a1 - m);
    }
    float t = total * u;
    int count = 0;
    for (int p = 0; p < npairs; ++p) {
        float a0, a1;
        f2_unpack(niw_small_arg2<DP>(recs_s + p * 2 * REC, x2), a0, a1);
        t -= mufu_ex2(a0 - m);
        count += 1 - static_cast<int>(__float_as_uint(t) >> 31);
        t -= mufu_ex2(a1 - m);
        count += 1 - static_cast<int>(__float_as_uint(t) >> 31);
    }
    return min(count, G - 1);
}

template <int DP, int R>
__global__ void __launch_bounds__(kNiwSmallThreads) niw_rows_kernel(const NiwRowsArgs a) {
    constexpr int REC = niw_group_floats(DP);
    extern __shared__ __align__(16) float smem[];
    __shared__ float red[kNiwSmallThreads / 32];
    const int G = a.G, d = a.d, tid = threadIdx.x;
    const int nslots = (G + kNiwSlotGroups - 1) / kNiwSlotGroups;
    const int npairs = (G + 1) / 2;
    float *recs_s = smem;                                            // [npairs][REC] pairs
    float *slots = smem + static_cast<size_t>(npairs) * 2 * REC;     // [R][nslots][threads]

    // M* = max_g (C_g + prior_g); then the block-private pair records with {co, sc', 1 / dof} as constants and -mu'
    float m = -INFINITY;
    for (int g = tid; g < G; g += kNiwSmallThreads)
        m = fmaxf(m, a.recs[static_cast<size_t>(g) * REC + DP + DP * DP] + (a.prior ? a.prior[g] : 0.f));
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((tid & 31) == 0) red[tid >> 5] = m;
    __syncthreads();
    m = red[0];
#pragma unroll
    for (int w = 1; w < kNiwSmallThreads / 32; ++w) m = fmaxf(m, red[w]);
    for (int i = tid; i < npairs * 2 * REC; i += kNiwSmallThreads) {
        const int g = i / REC, e = i - g * REC;
        float v = g < G ? a.recs[i] : 0.f;  // the padding half of an odd last pair: zero record, sc' = -inf
        int at = e;
        if (e < DP) v = -v;
        if (e == DP + DP * DP) {  // C_g -> sc' (second constant)
            v = g < G ? (v + (a.prior ? a.prior[g] : 0.f) - m) * kLog2e : -INFINITY;
            at = e + 1;
        } else if (e == DP + DP * DP + 1) {  // -0.5 (dof + d) ln 2 -> co = -0.5 (dof + d) (first constant)
            v = static_cast<float>(static_cast<double>(v) * 1.4426950408889634);
            at = e - 1;
        }
        recs_s[(g >> 1) * 2 * REC + 2 * at + (g & 1)] = v;
    }
    __syncthreads();

    const size_t tile_rows = static_cast<size_t>(kNiwSmallThreads) * R;
    const size_t ntiles = (a.N + tile_rows - 1) / tile_rows;
    for (size_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        float x[R][DP], urow[R];
        uint64_t x2[R][DP];
        size_t row[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            row[r] = tile * tile_rows + static_cast<size_t>(r) * kNiwSmallThreads + tid;
            const size_t rr = row[r] < a.N ? row[r] : a.N - 1;
            const float *src = a.values + rr * d;
#pragma unroll
            for (int k = 0; k < DP; ++k) {
                x[r][k] = k < d ? __ldg(src + k) : 0.f;
                x2[r][k] = f2_pack(x[r][k], x[r][k]);
            }
            urow[r] = __ldg(a.u + rr);
        }
        for (int sl = 0; sl < nslots; ++sl) {
            float sum[R];
#pragma unroll
            for (int r = 0; r < R; ++r) sum[r] = 0.f;
            const int p1 = min(npairs, (sl + 1) * (kNiwSlotGroups / 2));
#pragma unroll 2
            for (int p = sl * (kNiwSlotGroups / 2); p < p1; ++p) {
                const float *rec2 = recs_s + p * 2 * REC;
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    float a0, a1;
                    f2_unpack(niw_small_arg2<DP>(rec2, x2[r]), a0, a1);
                    sum[r] += mufu_ex2(a0);
                    sum[r] += mufu_ex2(a1);
                }
            }
#pragma unroll
            for (int r = 0; r < R; ++r) slots[(r * nslots + sl) * kNiwSmallThreads + tid] = sum[r];
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float *sp = slots + (r * nslots) * kNiwSmallThreads + tid;
            float total = 0.f;
            for (int k = 0; k < nslots; ++k) total += sp[k * kNiwSmallThreads];
            int result;
            if (!(total >= kNiwRedo)) {
                result = niw_small_row_exact<DP>(recs_s, G, x[r], urow[r]);
            } else {
                float t = total * urow[r];
                int sel = nslots - 1;
                for (int k = 0; k < nslots; ++k) {
                    const float w = sp[k * kNiwSmallThreads];
                    if (t <= w) {
                        sel = k;
                        break;
                    }
                    if (k + 1 < nslots) t -= w;
                }
                int count = 0;
                const int p1 = min(npairs, (sel + 1) * (kNiwSlotGroups / 2));
                for (int p = sel * (kNiwSlotGroups / 2); p < p1; ++p) {
                    float a0, a1;
                    f2_unpack(niw_small_arg2<DP>(recs_s + p * 2 * REC, x2[r]), a0, a1);
                    t -= mufu_ex2(a0);
                    count += 1 - static_cast<int>(__float_as_uint(t) >> 31);  // t >= +0 continues (an exact 0: a near-tie)
                    t -= mufu_ex2(a1);
                    count += 1 - static_cast<int>(__float_as_uint(t) >> 31);
                }
                result = min(sel * kNiwSlotGroups + count, G - 1);
            }
            if (row[r] < a.N) a.assign[row[r]] = result;
        }
    }
}

template <int DP, int R>
static int launch_niw_rows_t(dist_b200_ctx *ctx, const NiwRowsArgs &a, cudaStream_t s) {
    const int nslots = (a.G + kNiwSlotGroups - 1) / kNiwSlotGroups;
    const size_t smem = sizeof(float) * (static_cast<size_t>((a.G + 1) / 2) * 2 * niw_group_floats(DP) + static_cast<size_t>(R) * nslots * kNiwSmallThreads);
    if (smem > 200 * 1024) return DIST_B200_ERR_UNSUPPORTED;
    auto kern = niw_rows_kernel<DP, R>;
    DISTB200_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    int per_sm = 0;
    DISTB200_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kNiwSmallThreads, smem));
    if (per_sm < 1) per_sm = 1;
    const size_t tile_rows = static_cast<size_t>(kNiwSmallThreads) * R;
    const size_t ntiles = (a.N + tile_rows - 1) / tile_rows;
    const size_t cap = static_cast<size_t>(ctx->sm_count) * per_sm;
    kern<<<static_cast<unsigned>(ntiles < cap ? ntiles : cap), kNiwSmallThreads, smem, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("niw_rows launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

// one niw feature with d <= 8, sampling only; DIST_B200_ERR_UNSUPPORTED -> the caller takes the materialising route
int launch_niw_rows_small(dist_b200_ctx *ctx, const dist_b200_feature *f, const void *values, size_t N, const float *prior,
                          const float *u, int32_t *assign, cudaStream_t s) {
    if (N == 0 || f->G == 0) return DIST_B200_OK;
    if (f->dim > 8 || !u || !assign) return DIST_B200_ERR_UNSUPPORTED;
    NiwRowsArgs a{};
    a.G = f->G;
    a.d = f->dim;
    a.N = N;
    a.recs = f->niw_buf;
    a.values = static_cast<const float *>(values);
    a.prior = prior;
    a.u = u;
    a.assign = assign;
    // rows per thread: a group's record is read with broadcast LDS.128s (four wavefronts each) -- the more rows share them the better
    // rows per thread: 8 / 4 measured slower than 4 / 2 (d = 3: 0.205 -> 0.228 ms, d = 8: 0.856 -> 0.944: registers, not the
    // broadcast LDS.128s, are what the extra rows cost)
    if (niw_padded_dim(f->dim) == 4) return launch_niw_rows_t<4, 4>(ctx, a, s);
    return launch_niw_rows_t<8, 2>(ctx, a, s);
}

int niw_padded_dim(int d) { return d <= 4 ? 4 : (d <= 8 ? 8 : (d <= 16 ? 16 : (d <= 32 ? 32 : (d <= 64 ? 64 : 128)))); }

int launch_niw_prep(dist_b200_ctx *ctx, int d, const float *mu, float kappa, const float *psi, float nu, int G,
                    const int32_t *count, const float *sum_x, const float *sum_xxT, float *recs, cudaStream_t s) {
    if (G <= 0) return DIST_B200_OK;
    if (d <= 32) {
        niw_prep_kernel<<<G, 64, 0, s>>>(d, niw_padded_dim(d), mu, kappa, psi, nu, count, sum_x, sum_xxT, recs, ctx->tables);
    } else {
        DISTB200_CUDA(ctx, cudaFuncSetAttribute(niw_prep_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                static_cast<int>(kNiwWidePrepSmem)));
        niw_prep_wide_kernel<<<G, kNiwWideThreads, kNiwWidePrepSmem, s>>>(d, niw_padded_dim(d), mu, kappa, psi, nu, count, sum_x,
                                                                           sum_xxT, recs, ctx->tables);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("niw prep launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

int launch_niw_scores(dist_b200_ctx *ctx, const dist_b200_feature *f, const void *values, size_t N,
                      const float *prior, float *scores, int accumulate, cudaStream_t s) {
    if (N == 0 || f->G == 0) return DIST_B200_OK;
    // 32 < d <= 128: tcgen05 on x - mu0, the only route there
    if (f->dim > 32) return launch_niw_tc_wide(ctx, f->G, f->dim, f->niw_tc, f->alphas_dev, values, N, prior, scores, accumulate, s);
    // d = 32: tcgen05 with split fp16 operands; DIST_B200_OPT_NIW_PATH = 1 keeps the FP32 CUDA-core kernel for A/B runs
    if (f->dim == 32 && f->niw_tc && ctx->opt[DIST_B200_OPT_NIW_PATH] == 0) {
        const int rc = launch_niw_tc(ctx, f->G, f->niw_tc, values, N, prior, scores, accumulate, nullptr, nullptr, s);
        if (rc != DIST_B200_ERR_UNSUPPORTED) return rc;
    }
    NiwArgs a{};
    a.G = f->G;
    a.d = f->dim;
    a.accumulate = accumulate;
    a.N = N;
    a.recs = f->niw_buf;
    a.values = static_cast<const float *>(values);
    a.prior = prior;
    a.scores = scores;
    switch (niw_padded_dim(f->dim)) {
        case 4: return launch_niw_dp<4>(ctx, a, s);
        case 8: return launch_niw_dp<8>(ctx, a, s);
        case 16: return launch_niw_dp<16>(ctx, a, s);
        default: return launch_niw_dp<32>(ctx, a, s);
    }
}

}  // namespace distb200
