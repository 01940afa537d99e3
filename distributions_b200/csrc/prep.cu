// prep.cu -- cache rebuild kernels: raw group statistics -> the per-group caches the score kernels
// read (MixtureValueScorer::update_all / update_group of every model), the Pitman-Yor prior vector,
// and the numerics probe.  O(G * dim) work, once per batch: not the hot path.  This translation
// unit is compiled with --fmad=false so that every expression keeps the reference's operation
// order and rounding (the reference builds for SSE4.1, which has no FMA).
#include <algorithm>

#include "common.cuh"
#include "posterior.cuh"

namespace distb200 {

// ---------------------------------------------------------------------------------------------
// NormalInverseChiSq: Shared::plus_group (nich.hpp:58-69) + Scorer::init (nich.hpp:239-250)
// packed as float4 {mean, precision, log_coeff * ln 2, score}: the hot loop multiplies the coefficient
// with MUFU.LG2's base-2 logarithm directly.  The unscaled log_coeff_ is kept in `aux` for read-back.
__device__ __forceinline__ void nich_prep_one(float mu, float kappa, float sigmasq, float nu, int32_t count, float mean,
                                              float ctv, float4 *params, float *aux, const NumericTables &t) {
    const NichPost post = nich_plus_group(mu, kappa, sigmasq, nu, count, mean, ctv);
    const float post_kappa = post.kappa, post_mu = post.mu, post_nu = post.nu, post_sigmasq = post.sigmasq;
    const float lambda = post_kappa / ((post_kappa + 1.f) * post_sigmasq);
    const float score = fast_lgamma_nu(post_nu, t.lgamma_nu3) +
                        0.5f * fast_log_table(lambda / (3.14159265358979f * post_nu), t.log2_table);
    const float log_coeff = -0.5f * post_nu - 0.5f;
    const float precision = lambda / post_nu;
    *params = make_float4(post_mu, precision, log_coeff * kLn2, score);
    *aux = log_coeff;
}

__global__ void nich_prep_kernel(float mu, float kappa, float sigmasq, float nu, int g0, int n,
                                 const int32_t *__restrict__ count, const float *__restrict__ mean,
                                 const float *__restrict__ ctv, float4 *__restrict__ params,
                                 float *__restrict__ aux, NumericTables t) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    nich_prep_one(mu, kappa, sigmasq, nu, count[i], mean[i], ctv[i], params + g0 + i, aux + g0 + i, t);
}

// GammaPoisson: plus_group (gp.hpp:56-61) + Scorer::init (gp.hpp:198-207); {post_alpha, score_coeff, score, 0}
__device__ __forceinline__ float4 gp_prep_one(float alpha, float inv_beta, uint32_t count, uint32_t sum, const NumericTables &t) {
    const float2 post = gp_plus_group(alpha, inv_beta, count, sum);
    const float post_alpha = post.x, post_inv_beta = post.y;
    const float score_coeff = -fast_log_table(1.f + post_inv_beta, t.log2_table);
    const float score = -fast_lgamma_exact(post_alpha, t.lgamma5) +
                        post_alpha * (fast_log_table(post_inv_beta, t.log2_table) + score_coeff);
    return make_float4(post_alpha, score_coeff, score, 0.f);
}

__global__ void gp_prep_kernel(float alpha, float inv_beta, int g0, int n, const uint32_t *__restrict__ count,
                               const uint32_t *__restrict__ sum, float4 *__restrict__ params, NumericTables t) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    params[g0 + i] = gp_prep_one(alpha, inv_beta, count[i], sum[i], t);
}

// BetaNegativeBinomial: plus_group (bnb.hpp:57-63) + Scorer::init (bnb.hpp:200-211); {post_beta, alpha, score, 0}
__device__ __forceinline__ float4 bnb_prep_one(float alpha, float beta, float r, uint32_t count, uint32_t sum,
                                               const NumericTables &t) {
    const float2 post = bnb_plus_group(alpha, beta, r, count, sum);
    const float post_alpha = post.x, post_beta = post.y;
    const float a = post_alpha + r;
    const float score = fast_lgamma_exact(post_alpha + post_beta, t.lgamma5) - fast_lgamma_exact(post_alpha, t.lgamma5) -
                        fast_lgamma_exact(post_beta, t.lgamma5) + fast_lgamma_exact(a, t.lgamma5);
    return make_float4(post_beta, a, score, 0.f);
}

__global__ void bnb_prep_kernel(float alpha, float beta, float r, int g0, int n, const uint32_t *__restrict__ count,
                                const uint32_t *__restrict__ sum, float4 *__restrict__ params, NumericTables t) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    params[g0 + i] = bnb_prep_one(alpha, beta, r, count[i], sum[i], t);
}

// BetaBernoulli: update_all (bb.hpp:276-292); {heads_score, tails_score, 0, 0}
__device__ __forceinline__ float4 bb_prep_one(float alpha, float beta, int32_t heads, int32_t tails, const NumericTables &t) {
    const float2 post = bb_plus_group(alpha, beta, heads, tails);
    const float h = post.x, tl = post.y;
    return make_float4(fast_log_table(h / (h + tl), t.log2_table), fast_log_table(tl / (h + tl), t.log2_table), 0.f, 0.f);
}

__global__ void bb_prep_kernel(float alpha, float beta, int g0, int n, const int32_t *__restrict__ heads,
                               const int32_t *__restrict__ tails, float4 *__restrict__ params, NumericTables t) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    params[g0 + i] = bb_prep_one(alpha, beta, heads[i], tails[i], t);
}

// Batched add_value, second half: fold the per-feature batch accumulators (stats.cu) into the stored
// statistics and rebuild that group's cache entry, for every pooled feature of the launch.
//   nich: (m, sum x, sum x^2) in double -> (m, mean_b, ctv_b), merged by the pairwise formula of Group::merge
//         (nich.hpp:167-179) in double;  gp: count += m, sum += sum x (uint32 wrap-around, as gp.hpp:109-116);
//   bb: heads / tails += counts (bb.hpp:102-107).  b.sign = -1 is the batched remove_value (nich.hpp:146-165,
//   gp.hpp:128-135, bb.hpp:117-122): the same accumulators subtracted, nich by inverting the merge.
__global__ void merge_prep_batch_kernel(const AddBatch b, NumericTables t) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= b.G) return;
    const AddDesc &d = b.d[blockIdx.y];
    const char *acc = b.acc + b.acc_stride * blockIdx.y;
    const size_t ci = (static_cast<size_t>(b.G) * 4 + 255) / 256 * 256, di = (static_cast<size_t>(b.G) * 8 + 255) / 256 * 256;
    // accumulators of this (feature, group): the launch's own, or the all-reduced exchange buffer
    // ([feature][4][G] doubles: integers are exact in a double, gp's wrapped uint32 partial sums add mod 2^32)
    int acc_a, acc_b;
    double acc_x, acc_xx;
    if (b.xchg) {
        const double *x = b.xchg + static_cast<size_t>(b.xchg_first + blockIdx.y) * 4 * b.G;
        acc_a = static_cast<int>(static_cast<long long>(x[g]));
        acc_b = static_cast<int>(static_cast<unsigned int>(static_cast<unsigned long long>(x[b.G + g])));
        acc_x = x[2 * b.G + g];
        acc_xx = x[3 * b.G + g];
    } else {
        acc_a = reinterpret_cast<const int *>(acc)[g];
        acc_b = reinterpret_cast<const int *>(acc + ci)[g];
        acc_x = reinterpret_cast<const double *>(acc + 2 * ci)[g];
        acc_xx = reinterpret_cast<const double *>(acc + 2 * ci + di)[g];
    }
    if (d.model == DIST_B200_NICH) {
        int32_t *count = reinterpret_cast<int32_t *>(d.st0);
        float *mean = reinterpret_cast<float *>(d.st1), *ctv = reinterpret_cast<float *>(d.st2);
        const int m = acc_a;
        if (m != 0) {
            const double mean_b = acc_x / m;
            const double ctv_b = fmax(acc_xx - m * mean_b * mean_b, 0.0);
            if (b.sign > 0) {
                const double n = count[g], tot = n + m;
                const double delta = mean_b - static_cast<double>(mean[g]);
                const double source_part = static_cast<double>(m) / tot;
                const double cross_part = n * source_part;
                count[g] = static_cast<int32_t>(tot);
                mean[g] = static_cast<float>(static_cast<double>(mean[g]) + source_part * delta);
                ctv[g] = static_cast<float>(static_cast<double>(ctv[g]) + ctv_b + cross_part * delta * delta);
            } else {
                // the inverse of the merge: (count, mean, ctv) = merge(rest, batch) solved for `rest`; a group
                // emptied by the batch is reset like Group::remove_value does (nich.hpp:146-165)
                const double tot = count[g], n = tot - m;
                if (n <= 0) {
                    count[g] = 0;
                    mean[g] = 0.f;
                    ctv[g] = 0.f;
                } else {
                    const double mean_r = (tot * static_cast<double>(mean[g]) - m * mean_b) / n;
                    const double delta = mean_b - mean_r;
                    count[g] = static_cast<int32_t>(n);
                    // one value left: its variance term is exactly 0, as Group::remove_value forces it
                    // (nich.hpp:146-165); otherwise rounding may not push the remainder below 0
                    ctv[g] = n <= 1 ? 0.f
                                    : static_cast<float>(fmax(static_cast<double>(ctv[g]) - ctv_b - (n * m / tot) * delta * delta, 0.0));
                    mean[g] = static_cast<float>(mean_r);
                }
            }
        }
        nich_prep_one(d.shared[0], d.shared[1], d.shared[2], d.shared[3], count[g], mean[g], ctv[g], d.params + g, d.aux + g, t);
    } else if (d.model == DIST_B200_GP || d.model == DIST_B200_BNB) {
        const uint32_t c = d.st0[g] + static_cast<uint32_t>(b.sign * acc_a);
        const uint32_t sm = d.st1[g] + static_cast<uint32_t>(b.sign) * static_cast<uint32_t>(acc_b);
        d.st0[g] = c;
        d.st1[g] = sm;
        d.params[g] = d.model == DIST_B200_GP ? gp_prep_one(d.shared[0], d.shared[1], c, sm, t)
                                              : bnb_prep_one(d.shared[0], d.shared[1], d.shared[2], c, sm, t);
    } else {  // bb
        int32_t *heads = reinterpret_cast<int32_t *>(d.st0), *tails = reinterpret_cast<int32_t *>(d.st1);
        const int32_t h = heads[g] + b.sign * acc_a, tl = tails[g] + b.sign * acc_b;
        heads[g] = h;
        tails[g] = tl;
        d.params[g] = bb_prep_one(d.shared[0], d.shared[1], h, tl, t);
    }
}

// DirichletDiscrete: update_all (dd.hpp:399-421) folded with score_value's subtraction
// (dd.hpp:433-445 -> vector_math.cc:160-168): table[g][v] (stride_g, stride_v) =
// fast_log(alphas[v] + counts[g][v]) - fast_log(alpha_sum + count_sum[g])
__global__ void dd_prep_kernel(int dim, const float *__restrict__ alphas, float alpha_sum, int g0, int n,
                               const int32_t *__restrict__ counts, float *__restrict__ table, size_t stride_g,
                               size_t stride_v, NumericTables t) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t *c = counts + static_cast<size_t>(i) * dim;
    int32_t count_sum = 0;
    for (int v = 0; v < dim; ++v) count_sum += c[v];
    const float shift = fast_log_table(alpha_sum + static_cast<float>(count_sum), t.log2_table);
    float *out = table + static_cast<size_t>(g0 + i) * stride_g;
    for (int v = 0; v < dim; ++v) {
        out[v * stride_v] = fast_log_table(alphas[v] + static_cast<float>(c[v]), t.log2_table) - shift;
    }
}

// DirichletProcessDiscrete: update_all (dpd.hpp:471-497) folded with score_value (dpd.hpp:517-543):
// value-major table[(V+1)][G]; row V is the OTHER / unseen row fast_log(alpha*beta0) - shift[g].
__global__ void dpd_shift_kernel(float alpha, int V, int G, const int32_t *__restrict__ counts,
                                 float *__restrict__ shift, NumericTables t) {
    // one warp per group: total count over the V known values
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= G) return;
    long long total = 0;
    for (int v = lane; v < V; v += 32) total += counts[static_cast<size_t>(g) * V + v];
    for (int o = 16; o; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
    if (lane == 0) shift[g] = fast_log_table(alpha + static_cast<float>(total), t.log2_table);
}

__global__ void dpd_table_kernel(float alpha, float beta0, int V, const float *__restrict__ betas, int G,
                                 const int32_t *__restrict__ counts, const float *__restrict__ shift,
                                 float *__restrict__ table, NumericTables t) {
    // 32x32 tile transpose: counts are [G][V] (read along v), table is [V+1][G] (written along g)
    __shared__ int32_t tile[32][33];
    const int v0 = blockIdx.x * 32, g0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int g = g0 + r, v = v0 + threadIdx.x;
        tile[r][threadIdx.x] = (g < G && v < V) ? counts[static_cast<size_t>(g) * V + v] : 0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int v = v0 + r, g = g0 + threadIdx.x;
        if (g >= G || v > V) continue;
        float s;
        if (v < V) {
            s = fast_log_table(alpha * betas[v] + static_cast<float>(tile[threadIdx.x][r]), t.log2_table);
        } else {
            s = fast_log_table(alpha * beta0, t.log2_table);
        }
        table[static_cast<size_t>(v) * G + g] = s - shift[g];
    }
}

// Pitman-Yor prior vector: CachedMixture::init + score_value (clustering.hpp:151-161,195-230)
// every block reduces all G sizes itself (G is small) and writes its own slice of the vector
__global__ void prior_prep_kernel(float alpha, float d, int G, const int32_t *__restrict__ sizes,
                                  float *__restrict__ prior, NumericTables t) {
    __shared__ long long s_total;
    __shared__ int s_empty;
    if (threadIdx.x == 0) {
        s_total = 0;
        s_empty = 0;
    }
    __syncthreads();
    long long total = 0;
    int empty = 0;
    for (int g = threadIdx.x; g < G; g += blockDim.x) {
        total += sizes[g];
        empty += (sizes[g] == 0);
    }
    for (int o = 16; o; o >>= 1) {
        total += __shfl_xor_sync(0xffffffffu, total, o);
        empty += __shfl_xor_sync(0xffffffffu, empty, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(reinterpret_cast<unsigned long long *>(&s_total), static_cast<unsigned long long>(total));
        atomicAdd(&s_empty, empty);
    }
    __syncthreads();
    const int nonempty = G - s_empty;
    const float numer = alpha + d * static_cast<float>(nonempty);
    const float denom = static_cast<float>(s_empty);
    const float empty_score = fast_log_table(numer / denom, t.log2_table);
    const float shift = -fast_log_table(static_cast<float>(s_total) + alpha, t.log2_table);
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < G; g += gridDim.x * blockDim.x) {
        const float shifted =
            sizes[g] ? fast_log_table(static_cast<float>(sizes[g]) - d, t.log2_table) : empty_score;
        prior[g] = shifted + shift;
    }
}

// LowEntropy clustering prior: LowEntropy::score_add_value (clustering.hpp:265-293, :318-327) for every
// group, as the uncached MixtureDriver::score_value evaluates it (mixture.hpp:123-141); overwrites prior[G].
__global__ void low_entropy_prep_kernel(int dataset_size, int G, const int32_t *__restrict__ sizes,
                                        float *__restrict__ prior, NumericTables t) {
    __shared__ int s_total, s_empty;
    if (threadIdx.x == 0) {
        s_total = 0;
        s_empty = 0;
    }
    __syncthreads();
    int total = 0, empty = 0;
    for (int g = threadIdx.x; g < G; g += blockDim.x) {
        total += sizes[g];
        empty += (sizes[g] == 0);
    }
    for (int o = 16; o; o >>= 1) {
        total += __shfl_xor_sync(0xffffffffu, total, o);
        empty += __shfl_xor_sync(0xffffffffu, empty, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&s_total, total);
        atomicAdd(&s_empty, empty);
    }
    __syncthreads();
    const int sample_size = s_total;
    float empty_score = -fast_log_table(static_cast<float>(s_empty), t.log2_table);
    if (sample_size + 1 < dataset_size) {
        const float n = static_cast<float>(sample_size + 1);
        const float exponent = 0.45f - 0.1f / n - 0.1f / dataset_size;
        const float scale = dataset_size / n;
        empty_score += fast_log_table(scale, t.log2_table) * exponent;
    }
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < G; g += gridDim.x * blockDim.x) {
        const int group_size = sizes[g];
        float score;
        if (group_size == 0) {
            score = empty_score;
        } else {
            const float bigger = 1.f + group_size;
            if (group_size > 10000) score = 1.f + fast_log_table(bigger, t.log2_table);
            else score = fast_log_table(bigger / group_size, t.log2_table) * group_size + fast_log_table(bigger, t.log2_table);
        }
        prior[g] = score;
    }
}

// ---------------------------------------------------------------------------------------------
// score_data_grid (SURVEY.md 8f rank 2): MixtureSlave::score_data_grid (mixture.hpp:427-438) -- the log
// marginal likelihood of ALL groups under each of n_grid hyper-parameter settings, from the device-resident
// group statistics.  Terms are the reference's fp32 expressions operation by operation (this translation
// unit is built without FMA contraction; fast_lgamma / fast_log through the reference's tables); only the
// accumulation differs: the reference adds them in group order in fp32, here every term goes into a double
// block reduction, one atomicAdd(double) per block.  grid = (blocks over cells, n_grid).
struct ScoreDataArgs {
    int model, G, dim;            // dim: dd dim / dpd V
    size_t n_grid, stride;        // packed Shareds: n_grid x stride floats
    const float *shareds;
    const uint32_t *st0, *st1, *st2;   // statistics arrays (see dist_b200_feature::stats)
    const float *betas;           // dpd
    const float *log_prod;        // gp
    float r;                      // bnb
    double *acc;                  // [n_grid], zeroed
};

__device__ __forceinline__ double block_sum(double v) {
    __shared__ double warp_part[32];
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) warp_part[warp] = v;
    __syncthreads();
    v = (threadIdx.x < (blockDim.x >> 5)) ? warp_part[threadIdx.x] : 0.0;
    if (warp == 0)
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;  // valid in thread 0
}

__global__ void __launch_bounds__(256) score_data_kernel(const ScoreDataArgs a, NumericTables t) {
    const float *sh = a.shareds + blockIdx.y * a.stride;
    const int G = a.G;
    double part = 0.0;
    if (a.model == DIST_B200_NICH) {  // nich.hpp:262-288
        const float mu = sh[0], kappa = sh[1], sigmasq = sh[2], nu = sh[3];
        const float nu_part = fast_lgamma_exact(0.5f * nu, t.lgamma5);
        const float kappa_part = 0.5f * fast_log_table(kappa, t.log2_table);
        const float sigmasq_part = 0.5f * nu * fast_log_table(nu * sigmasq, t.log2_table);
        const float log_pi = 1.1447298858493991f;
        const int32_t *count = reinterpret_cast<const int32_t *>(a.st0);
        const float *mean = reinterpret_cast<const float *>(a.st1), *ctv = reinterpret_cast<const float *>(a.st2);
        for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < G; g += gridDim.x * blockDim.x) {
            if (!count[g]) continue;
            const float n = static_cast<float>(count[g]);
            const float mu_1 = mu - mean[g];
            const float post_kappa = kappa + n;
            const float post_nu = nu + n;
            const float post_sigmasq = 1.f / post_nu * (nu * sigmasq + ctv[g] + (n * kappa * mu_1 * mu_1) / post_kappa);
            part += static_cast<double>(fast_lgamma_exact(0.5f * post_nu, t.lgamma5) - nu_part);
            part += static_cast<double>(kappa_part - 0.5f * fast_log_table(post_kappa, t.log2_table));
            part += static_cast<double>(sigmasq_part - 0.5f * post_nu * fast_log_table(post_nu * post_sigmasq, t.log2_table));
            part += static_cast<double>(-0.5f * log_pi * count[g]);
        }
    } else if (a.model == DIST_B200_GP) {  // gp.hpp:220-241
        const float alpha = sh[0], inv_beta = sh[1];
        const float alpha_part = fast_lgamma_exact(alpha, t.lgamma5);
        const float beta_part = alpha * fast_log_table(inv_beta, t.log2_table);
        for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < G; g += gridDim.x * blockDim.x) {
            if (!a.st0[g]) continue;
            const float post_alpha = alpha + static_cast<float>(a.st1[g]);
            const float post_inv_beta = inv_beta + static_cast<float>(a.st0[g]);
            part += static_cast<double>(fast_lgamma_exact(post_alpha, t.lgamma5) - alpha_part);
            part += static_cast<double>(beta_part - post_alpha * fast_log_table(post_inv_beta, t.log2_table));
            part += static_cast<double>(-a.log_prod[g]);
        }
    } else if (a.model == DIST_B200_BNB) {  // bnb.hpp:221-243; packed (alpha, beta), r = a.r
        const float alpha = sh[0], beta = sh[1];
        const float shared_part = fast_lgamma_exact(alpha + beta, t.lgamma5) - fast_lgamma_exact(alpha, t.lgamma5) -
                                  fast_lgamma_exact(beta, t.lgamma5);
        for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < G; g += gridDim.x * blockDim.x) {
            if (!a.st0[g]) continue;
            const float post_alpha = alpha + a.r * static_cast<float>(a.st0[g]);
            const float post_beta = beta + static_cast<float>(a.st1[g]);
            part += static_cast<double>(fast_lgamma_exact(post_alpha, t.lgamma5) + fast_lgamma_exact(post_beta, t.lgamma5) -
                                        fast_lgamma_exact(post_alpha + post_beta, t.lgamma5));
            part += static_cast<double>(shared_part);
        }
    } else if (a.model == DIST_B200_BB) {  // bb.hpp:207-229
        const float alpha0 = sh[0], beta0 = sh[1];
        const float shared_part = fast_lgamma_exact(alpha0 + beta0, t.lgamma5) - fast_lgamma_exact(alpha0, t.lgamma5) -
                                  fast_lgamma_exact(beta0, t.lgamma5);
        const int32_t *heads = reinterpret_cast<const int32_t *>(a.st0), *tails = reinterpret_cast<const int32_t *>(a.st1);
        for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < G; g += gridDim.x * blockDim.x) {
            const float alpha = alpha0 + heads[g];
            const float beta = beta0 + tails[g];
            const float group_part = fast_lgamma_exact(alpha, t.lgamma5) + fast_lgamma_exact(beta, t.lgamma5) -
                                     fast_lgamma_exact(alpha + beta, t.lgamma5);
            part += static_cast<double>(shared_part + group_part);
        }
    } else if (a.model == DIST_B200_DD) {  // dd.hpp:291-324; one thread per (group, value) cell
        const int dim = a.dim;
        const int32_t *counts = reinterpret_cast<const int32_t *>(a.st0);
        float alpha_sum = 0;  // dd.hpp:297-302, sequential
        for (int v = 0; v < dim; ++v) alpha_sum += sh[v];
        const float total_part = fast_lgamma_exact(alpha_sum, t.lgamma5);
        const size_t cells = static_cast<size_t>(G) * dim;
        for (size_t c = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; c < cells;
             c += static_cast<size_t>(gridDim.x) * blockDim.x) {
            const int g = static_cast<int>(c / dim), v = static_cast<int>(c % dim);
            const int32_t *row = counts + static_cast<size_t>(g) * dim;
            int32_t count_sum = 0;
            for (int k = 0; k < dim; ++k) count_sum += row[k];
            if (!count_sum) continue;
            const float alpha = sh[v];
            part += static_cast<double>(fast_lgamma_exact(alpha + row[v], t.lgamma5) - fast_lgamma_exact(alpha, t.lgamma5));
            if (v == 0) part += static_cast<double>(total_part - fast_lgamma_exact(alpha_sum + count_sum, t.lgamma5));
        }
    } else {  // dpd: dpd.hpp:344-374; one warp per group, lanes over the V known values
        const int V = a.dim;
        const float alpha = sh[0];
        const int32_t *counts = reinterpret_cast<const int32_t *>(a.st0);
        const float shared_total = fast_lgamma_exact(alpha, t.lgamma5);
        const int lane = threadIdx.x & 31;
        const int warps = (gridDim.x * blockDim.x) >> 5;
        for (int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; g < G; g += warps) {
            const int32_t *row = counts + static_cast<size_t>(g) * V;
            long long total = 0;
            for (int v = lane; v < V; v += 32) {
                const int32_t c = row[v];
                total += c;
                if (!c) continue;
                const float prior_i = a.betas[v] * alpha;
                part += static_cast<double>(fast_lgamma_exact(prior_i + c, t.lgamma5) - fast_lgamma_exact(alpha * a.betas[v], t.lgamma5));
            }
            for (int o = 16; o; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
            if (lane == 0 && total) part += static_cast<double>(shared_total - fast_lgamma_exact(alpha + static_cast<float>(total), t.lgamma5));
        }
    }
    const double sum = block_sum(part);
    if (threadIdx.x == 0 && sum != 0.0) atomicAdd(&a.acc[blockIdx.y], sum);
}

__global__ void score_data_finish_kernel(size_t n, const double *__restrict__ acc, float *__restrict__ out) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) out[i] = static_cast<float>(acc[i]);
}

// numerics probe (dist_b200_numerics_probe)
__global__ void numerics_probe_kernel(int fn, size_t n, const float *__restrict__ in, float *__restrict__ out,
                                      NumericTables t) {
    __shared__ __align__(16) float coeff[33 * kLgammaRowStride];
    for (int i = threadIdx.x; i < 33 * kLgammaRowStride; i += blockDim.x) coeff[i] = t.lgamma5[i];
    __syncthreads();
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float x = in[i];
    float y = 0.f;
    switch (fn) {
        case 0: y = fast_log_table(x, t.log2_table); break;
        case 1: y = fast_exp_neg(x); break;
        case 2: y = fast_lgamma_cell(x, coeff); break;
        case 3: y = fast_lgamma_nu(x, t.lgamma_nu3); break;
        case 4: y = fast_log_factorial(__float_as_uint(x), t.log_factorial, t.lgamma5); break;
        case 5: y = fast_log_cell(x); break;
        case 6: y = fast_lgamma_exact(x, t.lgamma5); break;
    }
    out[i] = y;
}

// hot layout -> the reference's struct-of-arrays cache layout (dist_b200_feature_download_caches)
__global__ void unpack_float4_kernel(int model, int G, const float4 *__restrict__ params,
                                     const float *__restrict__ aux, float *__restrict__ out) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    const float4 p = params[g];
    if (model == DIST_B200_NICH) {  // score_, log_coeff_, precision_, mean_
        out[0 * G + g] = p.w;
        out[1 * G + g] = aux[g];
        out[2 * G + g] = p.y;
        out[3 * G + g] = p.x;
    } else if (model == DIST_B200_GP || model == DIST_B200_BNB) {  // gp: score_, post_alpha_, score_coeff_; bnb: score_, post_beta_, alpha_
        out[0 * G + g] = p.z;
        out[1 * G + g] = p.x;
        out[2 * G + g] = p.y;
    } else {  // bb: heads_scores_, tails_scores_
        out[0 * G + g] = p.x;
        out[1 * G + g] = p.y;
    }
}

__global__ void transpose_table_kernel(int G, int dim, const float *__restrict__ table_gv, float *__restrict__ out_vg) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    for (int v = 0; v < dim; ++v) out_vg[static_cast<size_t>(v) * G + g] = table_gv[static_cast<size_t>(g) * dim + v];
}

// ---------------------------------------------------------------------------------------------
static inline int blocks_for(size_t n, int threads) { return static_cast<int>((n + threads - 1) / threads); }

#define LAUNCH_CHECK(ctx)                                                                     \
    do {                                                                                      \
        cudaError_t e__ = cudaGetLastError();                                                 \
        if (e__ != cudaSuccess)                                                               \
            return fail((ctx), DIST_B200_ERR_CUDA, std::string("launch: ") + cudaGetErrorString(e__)); \
    } while (0)

int launch_nich_prep(dist_b200_ctx *ctx, const float sh[4], int G, int g0, int n, const int32_t *count,
                     const float *mean, const float *ctv, float4 *params, float *aux, cudaStream_t s) {
    (void)G;
    if (n <= 0) return DIST_B200_OK;
    nich_prep_kernel<<<blocks_for(n, 128), 128, 0, s>>>(sh[0], sh[1], sh[2], sh[3], g0, n, count, mean, ctv,
                                                        params, aux, ctx->tables);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_gp_prep(dist_b200_ctx *ctx, const float sh[2], int g0, int n, const uint32_t *count,
                   const uint32_t *sum, float4 *params, cudaStream_t s) {
    if (n <= 0) return DIST_B200_OK;
    gp_prep_kernel<<<blocks_for(n, 128), 128, 0, s>>>(sh[0], sh[1], g0, n, count, sum, params, ctx->tables);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_bnb_prep(dist_b200_ctx *ctx, const float sh[3], int g0, int n, const uint32_t *count,
                    const uint32_t *sum, float4 *params, cudaStream_t s) {
    if (n <= 0) return DIST_B200_OK;
    bnb_prep_kernel<<<blocks_for(n, 128), 128, 0, s>>>(sh[0], sh[1], sh[2], g0, n, count, sum, params, ctx->tables);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_bb_prep(dist_b200_ctx *ctx, const float sh[2], int g0, int n, const int32_t *heads,
                   const int32_t *tails, float4 *params, cudaStream_t s) {
    if (n <= 0) return DIST_B200_OK;
    bb_prep_kernel<<<blocks_for(n, 128), 128, 0, s>>>(sh[0], sh[1], g0, n, heads, tails, params, ctx->tables);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

// accumulators of one launch -> the exchange layout [feature][4][G] doubles (what an all-reduce can sum)
__global__ void pack_accumulators_kernel(const AddBatch b, double *__restrict__ xchg) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= b.G) return;
    const char *acc = b.acc + b.acc_stride * blockIdx.y;
    const size_t ci = (static_cast<size_t>(b.G) * 4 + 255) / 256 * 256, di = (static_cast<size_t>(b.G) * 8 + 255) / 256 * 256;
    double *x = xchg + static_cast<size_t>(b.xchg_first + blockIdx.y) * 4 * b.G;
    const int model = b.d[blockIdx.y].model;
    x[g] = static_cast<double>(reinterpret_cast<const int *>(acc)[g]);
    const int cb = reinterpret_cast<const int *>(acc + ci)[g];
    // gp / bnb: the sum accumulator is a wrapped uint32; bb: a plain count
    x[b.G + g] = (model == DIST_B200_GP || model == DIST_B200_BNB) ? static_cast<double>(static_cast<unsigned int>(cb)) : static_cast<double>(cb);
    x[2 * b.G + g] = reinterpret_cast<const double *>(acc + 2 * ci)[g];
    x[3 * b.G + g] = reinterpret_cast<const double *>(acc + 2 * ci + di)[g];
}

int launch_pack_accumulators(dist_b200_ctx *ctx, const AddBatch &b, double *xchg, cudaStream_t s) {
    if (b.n <= 0 || b.G <= 0) return DIST_B200_OK;
    pack_accumulators_kernel<<<dim3(blocks_for(b.G, 128), b.n), 128, 0, s>>>(b, xchg);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_merge_prep_batch(dist_b200_ctx *ctx, const AddBatch &b, cudaStream_t s) {
    if (b.n <= 0 || b.G <= 0) return DIST_B200_OK;
    merge_prep_batch_kernel<<<dim3(blocks_for(b.G, 128), b.n), 128, 0, s>>>(b, ctx->tables);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_dd_prep(dist_b200_ctx *ctx, int dim, const float *alphas, float alpha_sum, int g0, int n,
                   const int32_t *counts, float *table, cudaStream_t s) {
    if (n <= 0) return DIST_B200_OK;
    dd_prep_kernel<<<blocks_for(n, 128), 128, 0, s>>>(dim, alphas, alpha_sum, g0, n, counts, table,
                                                      static_cast<size_t>(dim), 1, ctx->tables);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_dpd_prep(dist_b200_ctx *ctx, float alpha, float beta0, int V, const float *betas, int G,
                    const int32_t *counts, float *table, cudaStream_t s) {
    if (G <= 0) return DIST_B200_OK;
    // shift lives in the tail of the table allocation: rows [0, V] are the table, row V+1 is shift
    float *shift = table + static_cast<size_t>(V + 1) * G;
    dpd_shift_kernel<<<blocks_for(static_cast<size_t>(G) * 32, 256), 256, 0, s>>>(alpha, V, G, counts, shift,
                                                                                 ctx->tables);
    LAUNCH_CHECK(ctx);
    dim3 grid((V + 1 + 31) / 32, (G + 31) / 32), block(32, 8);
    dpd_table_kernel<<<grid, block, 0, s>>>(alpha, beta0, V, betas, G, counts, shift, table, ctx->tables);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

// MixtureValueScorer::update_group for dpd (dpd.hpp:430-469 rebuild one group's entries): column g of the table
// and shift[g], from that group's dense counts row.  One block.
__global__ void dpd_update_group_kernel(float alpha, float beta0, int V, const float *__restrict__ betas, int G, int g,
                                        const int32_t *__restrict__ counts_row, float *__restrict__ table, NumericTables t) {
    __shared__ long long part[8];
    __shared__ float s_shift;
    long long total = 0;
    for (int v = threadIdx.x; v < V; v += blockDim.x) total += counts_row[v];
    for (int o = 16; o; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = total;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long all = 0;
        for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) all += part[w];
        s_shift = fast_log_table(alpha + static_cast<float>(all), t.log2_table);
        table[static_cast<size_t>(V + 1) * G + g] = s_shift;
    }
    __syncthreads();
    const float shift = s_shift;
    for (int v = threadIdx.x; v <= V; v += blockDim.x) {
        const float sc = v < V ? fast_log_table(alpha * betas[v] + static_cast<float>(counts_row[v]), t.log2_table)
                               : fast_log_table(alpha * beta0, t.log2_table);
        table[static_cast<size_t>(v) * G + g] = sc - shift;
    }
}

int launch_dpd_update_group(dist_b200_ctx *ctx, float alpha, float beta0, int V, const float *betas, int G, int g,
                            const int32_t *counts_row, float *table, cudaStream_t s) {
    dpd_update_group_kernel<<<1, 256, 0, s>>>(alpha, beta0, V, betas, G, g, counts_row, table, ctx->tables);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_prior_prep(dist_b200_ctx *ctx, float alpha, float d, int G, const int32_t *sizes, float *prior,
                      cudaStream_t s) {
    const int blocks = G <= 256 ? 1 : (G + 255) / 256 < 64 ? (G + 255) / 256 : 64;
    prior_prep_kernel<<<blocks, 256, 0, s>>>(alpha, d, G, sizes, prior, ctx->tables);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_score_data(dist_b200_ctx *ctx, const dist_b200_feature *f, const uint32_t *st0, const uint32_t *st1,
                      const uint32_t *st2, const float *betas, const float *log_prod, const float *shareds_dev,
                      size_t n_grid, size_t stride, double *acc, float *out_dev, cudaStream_t s) {
    if (n_grid == 0) return DIST_B200_OK;
    ScoreDataArgs a{};
    a.model = f->model;
    a.G = f->G;
    a.dim = f->dim;
    a.n_grid = n_grid;
    a.stride = stride;
    a.shareds = shareds_dev;
    a.st0 = st0;
    a.st1 = st1;
    a.st2 = st2;
    a.betas = betas;
    a.log_prod = log_prod;
    a.r = f->shared[2];
    a.acc = acc;
    cudaError_t e = cudaMemsetAsync(acc, 0, sizeof(double) * n_grid, s);
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, cudaGetErrorString(e));
    size_t work = static_cast<size_t>(f->G);
    if (f->model == DIST_B200_DD) work *= f->dim;
    if (f->model == DIST_B200_DPD) work *= 32;  // one warp per group
    size_t blocks = (work + 255) / 256;
    const size_t cap = std::max<size_t>(1, static_cast<size_t>(ctx->sm_count) * 8 / std::min<size_t>(n_grid, 8));
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    for (size_t i0 = 0; i0 < n_grid; i0 += 65535) {  // grid.y limit
        ScoreDataArgs b = a;
        const size_t n = std::min<size_t>(65535, n_grid - i0);
        b.shareds = shareds_dev + i0 * stride;
        b.acc = acc + i0;
        score_data_kernel<<<dim3(static_cast<unsigned>(blocks), static_cast<unsigned>(n)), 256, 0, s>>>(b, ctx->tables);
        LAUNCH_CHECK(ctx);
    }
    score_data_finish_kernel<<<blocks_for(n_grid, 256), 256, 0, s>>>(n_grid, acc, out_dev);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_score_data_finish(dist_b200_ctx *ctx, size_t n_grid, const double *acc, float *out_dev, cudaStream_t s) {
    if (n_grid == 0) return DIST_B200_OK;
    score_data_finish_kernel<<<blocks_for(n_grid, 256), 256, 0, s>>>(n_grid, acc, out_dev);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_low_entropy_prep(dist_b200_ctx *ctx, int dataset_size, int G, const int32_t *sizes, float *prior, cudaStream_t s) {
    const int blocks = G <= 256 ? 1 : (G + 255) / 256 < 64 ? (G + 255) / 256 : 64;
    low_entropy_prep_kernel<<<blocks, 256, 0, s>>>(dataset_size, G, sizes, prior, ctx->tables);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_numerics_probe(dist_b200_ctx *ctx, int fn, size_t n, const float *in, float *out, cudaStream_t s) {
    if (n == 0) return DIST_B200_OK;
    numerics_probe_kernel<<<blocks_for(n, 256), 256, 0, s>>>(fn, n, in, out, ctx->tables);
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

int launch_unpack_caches(dist_b200_ctx *ctx, const dist_b200_feature *f, float *out, cudaStream_t s) {
    const int G = f->G;
    if (G <= 0) return DIST_B200_OK;
    switch (f->model) {
        case DIST_B200_NICH:
        case DIST_B200_GP:
        case DIST_B200_BB:
        case DIST_B200_BNB:
            unpack_float4_kernel<<<blocks_for(G, 128), 128, 0, s>>>(f->model, G,
                                                                    static_cast<const float4 *>(f->params), f->aux, out);
            break;
        case DIST_B200_DD:
            transpose_table_kernel<<<blocks_for(G, 128), 128, 0, s>>>(G, f->dim, static_cast<const float *>(f->params),
                                                                      out);
            break;
        case DIST_B200_DPD: {
            cudaError_t e = cudaMemcpyAsync(out, f->params, sizeof(float) * static_cast<size_t>(f->dim + 1) * G,
                                            cudaMemcpyDeviceToDevice, s);
            if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, cudaGetErrorString(e));
        } break;
        default:
            return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "download_caches: model has no flat cache layout");
    }
    LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

}  // namespace distb200
