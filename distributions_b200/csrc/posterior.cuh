// posterior.cuh -- Shared::plus_group of the conjugate models: the posterior hyper-parameters of one group.
// The cache rebuilds (prep.cu, niw.cu) and the posterior-predictive sampler (sample_values.cu) share these, so
// a draw and a score always see the same posterior.  Expressions keep the reference's operation order (prep.cu
// and sample_values.cu are compiled without FMA contraction).
#pragma once
#include <stdint.h>

namespace distb200 {

// NormalInverseChiSq: Shared::plus_group (nich.hpp:58-69)
struct NichPost {
    float mu, kappa, sigmasq, nu;
};
__device__ __forceinline__ NichPost nich_plus_group(float mu, float kappa, float sigmasq, float nu, int32_t count, float mean,
                                                    float ctv) {
    const float cnt = static_cast<float>(count);
    const float mu_1 = mu - mean;
    NichPost p;
    p.kappa = kappa + cnt;
    p.mu = (kappa * mu + mean * cnt) / p.kappa;
    p.nu = nu + cnt;
    p.sigmasq = 1.f / p.nu * (nu * sigmasq + ctv + (cnt * kappa * mu_1 * mu_1) / p.kappa);
    return p;
}

// GammaPoisson: plus_group (gp.hpp:56-61) -> {post alpha (shape), post inv_beta (rate)}
__device__ __forceinline__ float2 gp_plus_group(float alpha, float inv_beta, uint32_t count, uint32_t sum) {
    return make_float2(alpha + static_cast<float>(sum), inv_beta + static_cast<float>(count));
}

// BetaNegativeBinomial: plus_group (bnb.hpp:57-63) -> {post alpha, post beta}
__device__ __forceinline__ float2 bnb_plus_group(float alpha, float beta, float r, uint32_t count, uint32_t sum) {
    return make_float2(alpha + r * static_cast<float>(count), beta + static_cast<float>(sum));
}

// BetaBernoulli (bb.hpp:276-292) -> {alpha + heads, beta + tails}
__device__ __forceinline__ float2 bb_plus_group(float alpha, float beta, int32_t heads, int32_t tails) {
    return make_float2(alpha + static_cast<float>(heads), beta + static_cast<float>(tails));
}

// NormalInverseWishart: Shared::plus_group (niw.hpp:82-103) for one group's statistics (count, sum_x[d], sum_xxT[d][d])
// and the Cholesky factor of the Student-t scale of Scorer::eval (niw.hpp:343-361),
//   sigma = psi' (kappa' + 1) / (kappa' dof),  dof = nu' - d + 1,
// in double.  Block-cooperative: every thread of the block calls it (d <= LD - 1 and d <= blockDim.x).  On return S[i][j],
// j <= i, holds L with sigma = L L^T (the upper triangle is scratch), xbar the group mean; the return value is dof.
template <int LD>
__device__ __forceinline__ double niw_posterior_cholesky(int d, const float *mu, float kappa, const float *psi, float nu,
                                                         int32_t count, const float *sx, const float *sxx, double (*S)[LD],
                                                         double *xbar, double *diff) {
    const int tid = threadIdx.x;
    const double n = static_cast<double>(count);
    const double kap = kappa, post_kappa = kap + n, post_nu = static_cast<double>(nu) + n;
    const double dof = post_nu - static_cast<double>(d) + 1.0;
    if (tid < d) {
        xbar[tid] = count ? static_cast<double>(sx[tid]) / n : 0.0;
        diff[tid] = xbar[tid] - static_cast<double>(mu[tid]);
    }
    __syncthreads();
    for (int e = tid; e < d * d; e += blockDim.x) {
        const int i = e / d, j = e % d;
        const double c_n = static_cast<double>(sxx[e]) - static_cast<double>(sx[i]) * xbar[j] -
                           xbar[i] * static_cast<double>(sx[j]) + n * xbar[i] * xbar[j];
        const double post_psi = static_cast<double>(psi[e]) + c_n + kap * n / (kap + n) * diff[i] * diff[j];
        S[i][j] = post_psi * (post_kappa + 1.0) / (post_kappa * dof);
    }
    __syncthreads();
    // Cholesky (right-looking), lower triangle in place
    for (int k = 0; k < d; ++k) {
        if (tid == 0) S[k][k] = sqrt(S[k][k]);
        __syncthreads();
        if (tid > k && tid < d) S[tid][k] /= S[k][k];
        __syncthreads();
        for (int e = tid; e < d * d; e += blockDim.x) {
            const int i = e / d, j = e % d;
            if (j > k && i >= j) S[i][j] -= S[i][k] * S[j][k];
        }
        __syncthreads();
    }
    return dof;
}

// coordinate i of the posterior mean mu' = (kappa mu + n xbar) / (kappa + n) (niw.hpp:82-103)
__device__ __forceinline__ double niw_post_mu(float kappa, int32_t count, float mu_i, double xbar_i) {
    const double kap = kappa, n = static_cast<double>(count);
    return kap / (kap + n) * static_cast<double>(mu_i) + n / (kap + n) * xbar_i;
}

}  // namespace distb200
