// niw_stats.cu -- NormalInverseWishart group statistics on the device (SURVEY.md 8f ranks 1 and 2):
//   * batched Group::add_value / remove_value (niw.hpp:247-276): count += 1, sum_x += x, sum_xxT += x x^T for every
//     (row, assigned group) pair of a block of rows -- a per-group SYRK;
//   * Group::score_data (niw.hpp:296-308) over all groups and a grid of Shareds (mixture.hpp:427-438).
//
// add_rows.  Rows are bucketed by group first (histogram -> exclusive scan -> scatter of row ids), so that a block
// accumulates ONE group's outer products in registers (double, 4 of the d x d entries per thread) over up to 256 of its
// rows, staged through shared memory 32 rows at a time, and touches global memory once per (group, slice) with double
// atomics.  The atomics land in a [G][1 + d + d^2] double block {count, sum_x, sum_xxT}, which is also the row-shard
// exchange block of this model.  A second kernel folds the block into the resident float statistics:
// stat = float(double(stat) +- acc).  The reference adds row by row in float; the sums here are the correctly rounded
// ones, the difference is the reference's own accumulation error (tests compare at 1e-5 relative to sum |x x^T|).
#include "common.cuh"

namespace distb200 {

constexpr int kNsThreads = 256;
constexpr int kNsSlice = 256;  // rows of one group per work unit

struct NiwScanArgs {
    int G;
    const int32_t *hist;  // [G]
    int32_t *offsets;     // [G + 1] first position of the group in perm
    int32_t *cursor;      // [G] scatter cursors (= offsets)
    int32_t *unit_off;    // [G + 1] first work unit of the group
};

// one block: exclusive scans of the histogram (row offsets) and of ceil(hist / slice) (work units)
__global__ void __launch_bounds__(1024) niw_scan_kernel(const NiwScanArgs a) {
    __shared__ int32_t part_rows[1024], part_units[1024];
    const int tid = threadIdx.x;
    const int per = (a.G + 1023) / 1024;
    const int g0 = tid * per, g1 = min(g0 + per, a.G);
    int32_t rows = 0, units = 0;
    for (int g = g0; g < g1; ++g) {
        rows += a.hist[g];
        units += (a.hist[g] + kNsSlice - 1) / kNsSlice;
    }
    part_rows[tid] = rows;
    part_units[tid] = units;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {  // Hillis-Steele inclusive scan
        const int32_t r = tid >= o ? part_rows[tid - o] : 0, u = tid >= o ? part_units[tid - o] : 0;
        __syncthreads();
        part_rows[tid] += r;
        part_units[tid] += u;
        __syncthreads();
    }
    int32_t ro = part_rows[tid] - rows, uo = part_units[tid] - units;
    for (int g = g0; g < g1; ++g) {
        a.offsets[g] = ro;
        a.cursor[g] = ro;
        a.unit_off[g] = uo;
        ro += a.hist[g];
        uo += (a.hist[g] + kNsSlice - 1) / kNsSlice;
    }
    if (tid == 1023) {
        a.offsets[a.G] = part_rows[1023];
        a.unit_off[a.G] = part_units[1023];
    }
}

__global__ void __launch_bounds__(256) niw_scatter_kernel(const int32_t *__restrict__ assign, size_t N, int G, int32_t *__restrict__ cursor,
                                                          int32_t *__restrict__ perm) {
    for (size_t n = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; n < N; n += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int g = assign[n];
        if (g >= 0 && g < G) perm[atomicAdd(&cursor[g], 1)] = static_cast<int32_t>(n);
    }
}

struct NiwAccArgs {
    int G, d;
    const float *values;  // [N][d]
    const int32_t *offsets, *unit_off, *perm;
    double *acc;          // [G][1 + d + d * d]
};

__global__ void __launch_bounds__(kNsThreads) niw_accumulate_kernel(const NiwAccArgs a) {
    __shared__ float xs[32][33];
    const int tid = threadIdx.x, d = a.d, dd = d * d;
    const int total_units = a.unit_off[a.G];
    // this thread's entries of the d x d matrix: e = tid + 256 k
    int ei[4], ej[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int e = tid + kNsThreads * k;
        ei[k] = e < dd ? e / d : -1;
        ej[k] = e < dd ? e % d : 0;
    }
    for (int u = blockIdx.x; u < total_units; u += gridDim.x) {
        int lo = 0, hi = a.G;  // the group whose unit range holds u: last g with unit_off[g] <= u
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (a.unit_off[mid] <= u) lo = mid;
            else hi = mid;
        }
        const int g = lo;
        const int first = a.offsets[g] + (u - a.unit_off[g]) * kNsSlice;
        const int last = min(first + kNsSlice, a.offsets[g + 1]);
        double m[4] = {0.0, 0.0, 0.0, 0.0}, sx = 0.0;
        for (int r0 = first; r0 < last; r0 += 32) {
            const int nr = min(32, last - r0);
            __syncthreads();
            for (int e = tid; e < 32 * d; e += kNsThreads) {  // a warp reads one row's d floats: coalesced
                const int r = e / d, k = e - r * d;
                xs[r][k] = r < nr ? a.values[static_cast<size_t>(a.perm[r0 + r]) * d + k] : 0.f;
            }
            __syncthreads();
            for (int r = 0; r < nr; ++r) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (ei[k] >= 0) m[k] = fma(static_cast<double>(xs[r][ei[k]]), static_cast<double>(xs[r][ej[k]]), m[k]);
                if (tid < d) sx += static_cast<double>(xs[r][tid]);
            }
        }
        double *out = a.acc + static_cast<size_t>(g) * (1 + d + dd);
        if (tid == 0) atomicAdd(out, static_cast<double>(last - first));
        if (tid < d) atomicAdd(out + 1 + tid, sx);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (ei[k] >= 0) atomicAdd(out + 1 + d + tid + kNsThreads * k, m[k]);
    }
}

// resident float statistics += sign * accumulated block; a group the batch empties is reset to exact zeros (what
// Group::init gives the next value that joins it; the reference's float subtraction leaves rounding residue there)
__global__ void niw_apply_kernel(int G, int d, int sign, const double *__restrict__ acc, int32_t *__restrict__ count,
                                 float *__restrict__ sum_x, float *__restrict__ sum_xxT) {
    const int per = 1 + d + d * d;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < static_cast<size_t>(G) * per;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int g = static_cast<int>(i / per), e = static_cast<int>(i - static_cast<size_t>(g) * per);
        const double delta = acc[i];
        const long long dn = llrint(acc[static_cast<size_t>(g) * per]);
        const int new_count = count[g] + static_cast<int>(sign > 0 ? dn : -dn);  // every thread of the group reads the OLD count:
        if (e == 0) continue;                                                     // it is written by the second pass below
        float *dst = e <= d ? sum_x + static_cast<size_t>(g) * d + (e - 1) : sum_xxT + static_cast<size_t>(g) * d * d + (e - 1 - d);
        *dst = new_count == 0 ? 0.f : static_cast<float>(static_cast<double>(*dst) + (sign > 0 ? delta : -delta));
    }
}
__global__ void niw_apply_count_kernel(int G, int d, int sign, const double *__restrict__ acc, int32_t *__restrict__ count) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    const long long dn = llrint(acc[static_cast<size_t>(g) * (1 + d + d * d)]);
    count[g] += static_cast<int>(sign > 0 ? dn : -dn);
}

size_t niw_add_rows_bytes(int G, int d, size_t N) {
    return round_up(sizeof(double) * static_cast<size_t>(G) * (1 + d + d * d), 256) + 4 * round_up(sizeof(int32_t) * (static_cast<size_t>(G) + 1), 256) +
           round_up(sizeof(int32_t) * N, 256);
}

// accumulate the rows' {count, sum_x, sum_xxT} per group into acc (zeroed here); work = niw_add_rows_bytes() scratch
int launch_niw_accumulate(dist_b200_ctx *ctx, int G, int d, const void *values, const int32_t *assign, size_t N, double *acc,
                          void *work, cudaStream_t s) {
    if (G <= 0) return DIST_B200_OK;
    if (N > 0x7FFFFFFFull) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "niw add_rows: more than 2^31 rows in one batch");
    DISTB200_CUDA(ctx, cudaMemsetAsync(acc, 0, sizeof(double) * static_cast<size_t>(G) * (1 + d + d * d), s));
    if (N == 0) return DIST_B200_OK;
    char *p = static_cast<char *>(work);
    const size_t gi = round_up(sizeof(int32_t) * (static_cast<size_t>(G) + 1), 256);
    int32_t *hist = reinterpret_cast<int32_t *>(p), *offsets = reinterpret_cast<int32_t *>(p + gi), *cursor = reinterpret_cast<int32_t *>(p + 2 * gi),
            *unit_off = reinterpret_cast<int32_t *>(p + 3 * gi), *perm = reinterpret_cast<int32_t *>(p + 4 * gi);
    int rc = launch_count_assignments(ctx, assign, N, G, hist, 0, s);
    if (rc) return rc;
    niw_scan_kernel<<<1, 1024, 0, s>>>(NiwScanArgs{G, hist, offsets, cursor, unit_off});
    const size_t want = (N + 255) / 256, cap = static_cast<size_t>(ctx->sm_count) * 8;
    niw_scatter_kernel<<<static_cast<unsigned>(want < cap ? want : cap), 256, 0, s>>>(assign, N, G, cursor, perm);
    NiwAccArgs a{G, d, static_cast<const float *>(values), offsets, unit_off, perm, acc};
    const size_t units_bound = N / kNsSlice + G + 1;
    niw_accumulate_kernel<<<static_cast<unsigned>(units_bound < cap ? units_bound : cap), kNsThreads, 0, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("niw add_rows launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

int launch_niw_apply(dist_b200_ctx *ctx, int G, int d, int sign, const double *acc, int32_t *count, float *sum_x, float *sum_xxT,
                     cudaStream_t s) {
    if (G <= 0) return DIST_B200_OK;
    const size_t n = static_cast<size_t>(G) * (1 + d + d * d), want = (n + 255) / 256, cap = static_cast<size_t>(ctx->sm_count) * 8;
    niw_apply_kernel<<<static_cast<unsigned>(want < cap ? want : cap), 256, 0, s>>>(G, d, sign, acc, count, sum_x, sum_xxT);
    niw_apply_count_kernel<<<(G + 255) / 256, 256, 0, s>>>(G, d, sign, acc, count);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("niw apply launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

// ---------------------------------------------------------------------------------------------
// score_data: out[i] += sum over groups of Group::score_data(shared_i) (niw.hpp:296-308):
//   lmultigamma(d, post.nu / 2) + nu / 2 fast_log(det psi) - count d / 2 log_pi - lmultigamma(d, nu / 2)
//   - post.nu / 2 fast_log(det post.psi) + d / 2 fast_log(kappa / post.kappa)
// with post = Shared::plus_group (niw.hpp:82-103).  One block per (group, grid point); the determinants come from
// Cholesky factorisations in double (the reference: Eigen's float LU), then the reference's float expression.
// Packed Shared i at shareds + i * stride: kappa, nu, mu[d], psi[d][d].
// returns log det; *det_out = det (may overflow to inf, underflow to 0)
__device__ double chol_logdet_free(double (*S)[33], int d, int tid, int nthreads, double *det_out) {
    for (int k = 0; k < d; ++k) {
        if (tid == 0) S[k][k] = sqrt(S[k][k]);
        __syncthreads();
        if (tid > k && tid < d) S[tid][k] /= S[k][k];
        __syncthreads();
        for (int e = tid; e < d * d; e += nthreads) {
            const int i = e / d, j = e % d;
            if (j > k && i >= j) S[i][j] -= S[i][k] * S[j][k];
        }
        __syncthreads();
    }
    if (tid == 0) {
        double det = 1.0, logdet = 0.0;
        for (int i = 0; i < d; ++i) {
            det *= S[i][i] * S[i][i];
            logdet += 2.0 * log(S[i][i]);
        }
        det_out[0] = det;
        det_out[1] = logdet;
    }
    __syncthreads();
    return det_out[1];
}

__device__ float lmultigamma_dev(int d, float a, const NumericTables &t) {  // special.hpp:278-286
    const float log_pi = 1.1447298858494002f;
    const float term1 = static_cast<float>(0.25 * static_cast<float>(d * (d - 1))) * log_pi;
    float term2 = 0.f;
    for (int j = 1; j <= d; ++j) term2 += fast_lgamma_exact(static_cast<float>(a + 0.5 * static_cast<float>(1 - j)), t.lgamma5);
    return term1 + term2;
}

struct NiwScoreDataArgs {
    int G, d;
    size_t stride;
    const float *shareds;
    const int32_t *count;
    const float *sum_x, *sum_xxT;
    double *acc;
};

__global__ void __launch_bounds__(64) niw_score_data_kernel(const NiwScoreDataArgs a, NumericTables t) {
    __shared__ double S[32][33], P[32][33];
    __shared__ double xbar[32], diff[32];
    __shared__ double det_prior[2], det_post[2];  // {det, log det}
    const int g = blockIdx.x, tid = threadIdx.x, d = a.d;
    const float *sh = a.shareds + blockIdx.y * a.stride;
    const float kappa = sh[0], nu = sh[1];
    const float *mu = sh + 2, *psi = sh + 2 + d;
    const float *sx = a.sum_x + static_cast<size_t>(g) * d, *sxx = a.sum_xxT + static_cast<size_t>(g) * d * d;
    const int cnt = a.count[g];
    const double n = cnt, kap = kappa;
    if (tid < d) {
        xbar[tid] = cnt ? static_cast<double>(sx[tid]) / n : 0.0;
        diff[tid] = xbar[tid] - static_cast<double>(mu[tid]);
    }
    __syncthreads();
    for (int e = tid; e < d * d; e += blockDim.x) {
        const int i = e / d, j = e % d;
        const double c_n = static_cast<double>(sxx[e]) - static_cast<double>(sx[i]) * xbar[j] - xbar[i] * static_cast<double>(sx[j]) + n * xbar[i] * xbar[j];
        P[i][j] = static_cast<double>(psi[e]);
        S[i][j] = static_cast<double>(psi[e]) + c_n + kap * n / (kap + n) * diff[i] * diff[j];
    }
    __syncthreads();
    chol_logdet_free(P, d, tid, blockDim.x, det_prior);
    chol_logdet_free(S, d, tid, blockDim.x, det_post);
    if (tid == 0) {
        const float log_pi = 1.1447298858494002f;
        const float post_nu = nu + static_cast<float>(cnt), post_kappa = kappa + static_cast<float>(cnt);
        const float score = lmultigamma_dev(d, static_cast<float>(post_nu * 0.5), t) +
                            static_cast<float>(nu * 0.5) * niw_log_det(det_prior[0], det_prior[1], t.log2_table) -
                            static_cast<float>(static_cast<float>(cnt * d) * 0.5) * log_pi - lmultigamma_dev(d, static_cast<float>(nu * 0.5), t) -
                            static_cast<float>(post_nu * 0.5) * niw_log_det(det_post[0], det_post[1], t.log2_table) +
                            static_cast<float>(static_cast<float>(d) * 0.5) * fast_log_table(kappa / post_kappa, t.log2_table);
        atomicAdd(a.acc + blockIdx.y, static_cast<double>(score));
    }
}

int launch_niw_score_data(dist_b200_ctx *ctx, int G, int d, const int32_t *count, const float *sum_x, const float *sum_xxT,
                          const float *shareds_dev, size_t n_grid, size_t stride, double *acc, cudaStream_t s) {
    if (n_grid == 0 || G <= 0) return DIST_B200_OK;
    NiwScoreDataArgs a{G, d, stride, shareds_dev, count, sum_x, sum_xxT, acc};
    for (size_t i0 = 0; i0 < n_grid; i0 += 65535) {  // grid.y limit
        NiwScoreDataArgs b = a;
        const size_t n = n_grid - i0 < 65535 ? n_grid - i0 : 65535;
        b.shareds = shareds_dev + i0 * stride;
        b.acc = acc + i0;
        niw_score_data_kernel<<<dim3(static_cast<unsigned>(G), static_cast<unsigned>(n)), 64, 0, s>>>(b, ctx->tables);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("niw score_data launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

}  // namespace distb200
