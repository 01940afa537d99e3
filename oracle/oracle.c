/* oracle/oracle.c -- plain-C restatement of the reference's mixture-scoring hot path.
 * TEST INFRASTRUCTURE ONLY (see oracle.h for the rules and the parity status).
 * Citations are file:line under /root/reference. */
#include "oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "oracle_tables.h"

/* ------------------------------------------------------------------------------------------ */
/* tables                                                                                      */

#define LOG_BITS 14
static float g_log2_table[1 << LOG_BITS]; /* special.cc:35-44 */
static unsigned int g_exp_table[1024];    /* vendor/fmath.hpp:157-162 */
static float g_exp_a, g_exp_b;            /* vendor/fmath.hpp:146-150 */
static int g_ready = 0;
static pthread_once_t g_once = PTHREAD_ONCE_INIT;

static float bits_to_float(unsigned int b) {
    float f;
    memcpy(&f, &b, 4);
    return f;
}
static unsigned int float_to_bits(float f) {
    unsigned int b;
    memcpy(&b, &f, 4);
    return b;
}

static void build_tables(void) {
    for (int i = 0; i < (1 << LOG_BITS); ++i) {
        /* float v = 1.0 + float(float(i) * 2^(23-N)) / 2^23;  table = log2(v) on a float argument,
         * i.e. the float overload (v is exact in float either way).  NOTE: the gcc -O3 -ffast-math
         * build of the reference vectorises this loop through libmvec's _ZGVbN4v_log2f (<= 4 ulp),
         * so oracle/_ref's table differs from this one by a few ulp in ~1/4 of its entries;
         * tests/test_oracle_vs_reference.py states that envelope. */
        float scaled = (float)i * (float)(1 << (23 - LOG_BITS));
        float v = (float)(1.0 + (double)(scaled / (float)(1 << 23)));
        g_log2_table[i] = log2f(v);
    }
    float log_2 = logf(2.0f);
    g_exp_a = 1024.0f / log_2;
    g_exp_b = log_2 / 1024.0f;
    for (int i = 0; i < 1024; ++i) {
        float y = powf(2.0f, (float)i / 1024.0f);
        g_exp_table[i] = float_to_bits(y) & 0x7fffffu;
    }
    g_ready = 1;
}

void orc_init(void) { pthread_once(&g_once, build_tables); }

/* ------------------------------------------------------------------------------------------ */
/* numerics                                                                                    */

/* special.hpp:57-67: sign bit ignored, exponent + table[top 14 mantissa bits], times ln 2 */
float orc_fast_log(float x) {
    if (!g_ready) orc_init();
    int intx = (int)float_to_bits(x);
    int e = ((intx >> 23) & 255) - 127;
    int man = (intx & 0x7FFFFF) >> (23 - LOG_BITS);
    return ((float)e + g_log2_table[man]) * 0.69314718055994529f;
}

/* vendor/fmath.hpp:438-459 (the SSE branch that is compiled in) */
float orc_fast_exp(float x) {
    if (!g_ready) orc_init();
    /* _mm_cvtss_si32 = round-to-nearest-even conversion; out-of-range gives 0x80000000 */
    float x1 = x;
    long c0 = (x1 != x1 || x1 >= 2147483648.0f || x1 < -2147483648.0f) ? (long)0x80000000u
                                                                        : lrintf(x1);
    int limit = (int)((unsigned int)c0 & 0x7fffffffu);
    if (limit > 0x42b00000) {
        x1 = x1 < 88.0f ? x1 : 88.0f;  /* _mm_min_ss then _mm_max_ss */
        x1 = x1 > -88.0f ? x1 : -88.0f;
    }
    float xa = x1 * g_exp_a;
    int r = (xa != xa || xa >= 2147483648.0f || xa < -2147483648.0f) ? (int)0x80000000u
                                                                     : (int)lrintf(xa);
    unsigned int v = (unsigned int)r & 1023u;
    float rb = (float)r * g_exp_b;
    float t = x1 - rb;
    int u = r >> 10;
    unsigned int fi = ((unsigned int)(u + 127) << 23) | g_exp_table[v];
    return (1.0f + t) * bits_to_float(fi);
}

/* floor(log2(v)) of a positive float from its exponent field, subnormals via the byte table
 * walk of special.hpp:131-146 (LogTable256[t] = floor(log2 t)) */
static int exponent_of(float v) {
    int x = (int)float_to_bits(v);
    int c = x >> 23;
    if (c) return c - 127;
    unsigned int t = (unsigned int)x;
    int lg = -1;
    while (t) {
        ++lg;
        t >>= 1;
    }
    return lg - 149; /* x >> 16 ? lg(x>>16) + 16 - 149 : ... all equal floor(log2 x) - 149 */
}

/* special.hpp:114-171 */
float orc_fast_lgamma(float y) {
    if (y < 2.5f || 4294967295.0f <= y) {
        return lgammaf(y);
    }
    int pos = exponent_of(y) * 6;
    float a5 = bits_to_float(kLgammaCoeff5Bits[pos]);
    float a4 = bits_to_float(kLgammaCoeff5Bits[pos + 1]);
    float a3 = bits_to_float(kLgammaCoeff5Bits[pos + 2]);
    float a2 = bits_to_float(kLgammaCoeff5Bits[pos + 3]);
    float a1 = bits_to_float(kLgammaCoeff5Bits[pos + 4]);
    float a0 = bits_to_float(kLgammaCoeff5Bits[pos + 5]);
    double yprod = y;
    double sum = a0;
    sum += a1 * yprod;
    yprod *= y;
    sum += a2 * yprod;
    yprod *= y;
    sum += a3 * yprod;
    yprod *= y;
    sum += a4 * yprod;
    yprod *= y;
    sum += a5 * yprod;
    return (float)sum;
}

/* special.hpp:208-214 */
float orc_fast_log_factorial(uint32_t n) {
    if (n < 64) return bits_to_float(kLogFactorialBits[n]);
    return orc_fast_lgamma((float)(uint32_t)(n + 1u)); /* fast_lgamma(n + 1): uint32 arithmetic, then -> float */
}

/* special.hpp:224-235,239-273 */
float orc_fast_lgamma_nu(float nu) {
    if (nu < 0.0625f || 4294967295.0f <= nu) {
        return lgammaf(nu * 0.5f + 0.5f) - lgammaf(nu * 0.5f);
    }
    int c = exponent_of(nu);
    int pos = ((c + 4) / 2) * 4;
    float a3 = bits_to_float(kLgammaNuCoeff3Bits[pos]);
    float a2 = bits_to_float(kLgammaNuCoeff3Bits[pos + 1]);
    float a1 = bits_to_float(kLgammaNuCoeff3Bits[pos + 2]);
    float a0 = bits_to_float(kLgammaNuCoeff3Bits[pos + 3]);
    return a0 + nu * a1 + nu * nu * a2 + nu * nu * nu * a3;
}

void orc_vec(int fn, size_t n, const float *in, float *out) {
    for (size_t i = 0; i < n; ++i) {
        switch (fn) {
            case 0: out[i] = orc_fast_log(in[i]); break;
            case 1: out[i] = orc_fast_exp(in[i]); break;
            case 2: out[i] = orc_fast_lgamma(in[i]); break;
            case 3: out[i] = orc_fast_lgamma_nu(in[i]); break;
            case 4: out[i] = orc_fast_log_factorial(float_to_bits(in[i])); break;
            default: out[i] = 0.f;
        }
    }
}

/* ------------------------------------------------------------------------------------------ */
/* clustering prior                                                                            */

/* clustering.hpp:81-104 */
float orc_py_score_add_value(float alpha, float d, int32_t group_size, int32_t nonempty,
                             int32_t sample_size, int32_t empty_count) {
    if (group_size == 0) {
        float numer = alpha + d * (float)nonempty;
        float denom = ((float)sample_size + alpha) * (float)empty_count;
        return orc_fast_log(numer / denom);
    }
    return orc_fast_log(((float)group_size - d) / ((float)sample_size + alpha));
}

/* clustering.hpp:151-161 (init), :215-230 (shifted scores), :195-208 (score_value, overwrite) */
void orc_py_prior(float alpha, float d, size_t G, const int32_t *sizes, float *out) {
    size_t empty = 0;
    long total = 0;
    for (size_t g = 0; g < G; ++g) {
        total += sizes[g];
        empty += (sizes[g] == 0);
    }
    size_t nonempty = G - empty;
    float numer = alpha + d * (float)nonempty;
    float denom = (float)empty;
    float empty_score = orc_fast_log(numer / denom);
    float shift = -orc_fast_log((float)total + alpha);
    for (size_t g = 0; g < G; ++g) {
        float shifted = sizes[g] ? orc_fast_log((float)sizes[g] - d) : empty_score;
        out[g] = shifted + shift;
    }
}

/* LowEntropy clustering prior: score_add_value (clustering.hpp:265-293, _approximate_postpred_correction
 * :318-327) evaluated for every group by the uncached MixtureDriver::score_value (mixture.hpp:123-141):
 * an OVERWRITE of the [G] vector, like the Pitman-Yor one. */
static float le_postpred_correction(int32_t dataset_size, float sample_size) {
    float exponent = 0.45f - 0.1f / sample_size - 0.1f / dataset_size;
    float scale = dataset_size / sample_size;
    return orc_fast_log(scale) * exponent;
}

float orc_low_entropy_score_add_value(int32_t dataset_size, int32_t group_size, int32_t sample_size,
                                      int32_t empty_group_count) {
    if (group_size == 0) {
        float score = -orc_fast_log((float)empty_group_count);
        if (sample_size + 1 < dataset_size) score += le_postpred_correction(dataset_size, (float)(sample_size + 1));
        return score;
    }
    const int32_t very_large = 10000;
    float bigger = 1.f + group_size;
    if (group_size > very_large) return 1.f + orc_fast_log(bigger);
    return orc_fast_log(bigger / group_size) * group_size + orc_fast_log(bigger);
}

void orc_low_entropy_prior(int32_t dataset_size, size_t G, const int32_t *sizes, float *out) {
    int32_t empty = 0, total = 0;
    for (size_t g = 0; g < G; ++g) {
        total += sizes[g];
        empty += (sizes[g] == 0);
    }
    for (size_t g = 0; g < G; ++g) out[g] = orc_low_entropy_score_add_value(dataset_size, sizes[g], total, empty);
}

/* ------------------------------------------------------------------------------------------ */
/* score_data: MixtureDataScorer::score_data of every model (SURVEY.md 8f rank 2) -- the log marginal  */
/* likelihood of all groups under one Shared, fp32, accumulated in group order like the reference.    */
/* `abs_sum` (optional) receives sum |term|: the scale the fp32 accumulation error is relative to.    */

/* abs_sum[0] += |term| (the scale of the accumulation error), abs_sum[1] += term (the same fp32 terms
 * accumulated in double: what the device computes) */
static float acc_term(float score, float term, double *abs_sum) {
    if (abs_sum) {
        abs_sum[0] += fabs((double)term);
        abs_sum[1] += (double)term;
    }
    return score + term;
}

/* nich.hpp:262-288 (Shared::plus_group nich.hpp:58-69) */
float orc_nich_score_data(const float sh[4], size_t G, const int32_t *count, const float *mean,
                          const float *ctv, double *abs_sum) {
    const float mu = sh[0], kappa = sh[1], sigmasq = sh[2], nu = sh[3];
    const float nu_part = orc_fast_lgamma(0.5f * nu);
    const float kappa_part = 0.5f * orc_fast_log(kappa);
    const float sigmasq_part = 0.5f * nu * orc_fast_log(nu * sigmasq);
    const float log_pi = 1.1447298858493991f;
    float score = 0;
    if (abs_sum) abs_sum[0] = abs_sum[1] = 0;
    for (size_t g = 0; g < G; ++g) {
        if (!count[g]) continue;
        float n = (float)count[g];
        float mu_1 = mu - mean[g];
        float post_kappa = kappa + n;
        float post_nu = nu + n;
        float post_sigmasq =
            1.f / post_nu * (nu * sigmasq + ctv[g] + (n * kappa * mu_1 * mu_1) / post_kappa);
        score = acc_term(score, orc_fast_lgamma(0.5f * post_nu) - nu_part, abs_sum);
        score = acc_term(score, kappa_part - 0.5f * orc_fast_log(post_kappa), abs_sum);
        score = acc_term(score, sigmasq_part - 0.5f * post_nu * orc_fast_log(post_nu * post_sigmasq), abs_sum);
        score = acc_term(score, -0.5f * log_pi * count[g], abs_sum);
    }
    return score;
}

/* gp.hpp:220-241 (plus_group gp.hpp:56-61) */
float orc_gp_score_data(const float sh[2], size_t G, const uint32_t *count, const uint32_t *sum,
                        const float *log_prod, double *abs_sum) {
    const float alpha_part = orc_fast_lgamma(sh[0]);
    const float beta_part = sh[0] * orc_fast_log(sh[1]);
    float score = 0;
    if (abs_sum) abs_sum[0] = abs_sum[1] = 0;
    for (size_t g = 0; g < G; ++g) {
        if (!count[g]) continue;
        float post_alpha = sh[0] + (float)sum[g];
        float post_inv_beta = sh[1] + (float)count[g];
        score = acc_term(score, orc_fast_lgamma(post_alpha) - alpha_part, abs_sum);
        score = acc_term(score, beta_part - post_alpha * orc_fast_log(post_inv_beta), abs_sum);
        score = acc_term(score, -log_prod[g], abs_sum);
    }
    return score;
}

/* bb.hpp:207-229 */
float orc_bb_score_data(const float sh[2], size_t G, const int32_t *heads, const int32_t *tails, double *abs_sum) {
    const float shared_part = orc_fast_lgamma(sh[0] + sh[1]) - orc_fast_lgamma(sh[0]) - orc_fast_lgamma(sh[1]);
    float score = 0;
    if (abs_sum) abs_sum[0] = abs_sum[1] = 0;
    for (size_t g = 0; g < G; ++g) {
        float alpha = sh[0] + heads[g];
        float beta = sh[1] + tails[g];
        float group_part = orc_fast_lgamma(alpha) + orc_fast_lgamma(beta) - orc_fast_lgamma(alpha + beta);
        score = acc_term(score, shared_part + group_part, abs_sum);
    }
    return score;
}

/* bnb.hpp:221-243 */
float orc_bnb_score_data(float alpha, float beta, uint32_t r, size_t G, const uint32_t *count, const uint32_t *sum,
                         double *abs_sum) {
    const float shared_part = orc_fast_lgamma(alpha + beta) - orc_fast_lgamma(alpha) - orc_fast_lgamma(beta);
    float score = 0;
    if (abs_sum) abs_sum[0] = abs_sum[1] = 0;
    for (size_t g = 0; g < G; ++g) {
        if (!count[g]) continue;
        float post_alpha = alpha + (float)r * count[g];
        float post_beta = beta + sum[g];
        score = acc_term(score, orc_fast_lgamma(post_alpha) + orc_fast_lgamma(post_beta) - orc_fast_lgamma(post_alpha + post_beta), abs_sum);
        score = acc_term(score, shared_part, abs_sum);
    }
    return score;
}

/* dd.hpp:250-256 = _init (291-320) + _eval (322-324): per-value partial sums over the groups, then the
 * (dim + 1)-vector is summed (vector_math.cc:85-93) */
float orc_dd_score_data(int dim, const float *alphas, size_t G, const int32_t *counts, double *abs_sum) {
    float shared_part[257], scores[257];
    float alpha_sum = 0;
    for (int i = 0; i < dim; ++i) {
        alpha_sum += alphas[i];
        shared_part[i] = orc_fast_lgamma(alphas[i]);
        scores[i] = 0;
    }
    shared_part[dim] = orc_fast_lgamma(alpha_sum);
    scores[dim] = 0;
    if (abs_sum) abs_sum[0] = abs_sum[1] = 0;
    for (size_t g = 0; g < G; ++g) {
        const int32_t *c = counts + g * dim;
        int32_t count_sum = 0;
        for (int i = 0; i < dim; ++i) count_sum += c[i];
        if (!count_sum) continue;
        for (int i = 0; i < dim; ++i)
            scores[i] = acc_term(scores[i], orc_fast_lgamma(alphas[i] + c[i]) - shared_part[i], abs_sum);
        scores[dim] = acc_term(scores[dim], shared_part[dim] - orc_fast_lgamma(alpha_sum + count_sum), abs_sum);
    }
    float total = 0;
    for (int i = 0; i <= dim; ++i) total += scores[i];
    return total;
}

/* dpd.hpp:344-374; counts dense [G][V] (the sparse counters hold exactly the non-zero entries; the
 * reference iterates them in hash-map order, this restatement in value order) */
float orc_dpd_score_data(float alpha, size_t V, const float *betas, size_t G, const int32_t *counts, double *abs_sum) {
    const float shared_total = orc_fast_lgamma(alpha);
    float score = 0;
    if (abs_sum) abs_sum[0] = abs_sum[1] = 0;
    for (size_t g = 0; g < G; ++g) {
        const int32_t *c = counts + g * V;
        long total = 0;
        for (size_t v = 0; v < V; ++v) total += c[v];
        if (!total) continue;
        for (size_t v = 0; v < V; ++v) {
            if (!c[v]) continue;
            float prior_i = betas[v] * alpha;
            score = acc_term(score, orc_fast_lgamma(prior_i + c[v]) - orc_fast_lgamma(alpha * betas[v]), abs_sum);
        }
        score = acc_term(score, shared_total - orc_fast_lgamma(alpha + total), abs_sum);
    }
    return score;
}

/* ------------------------------------------------------------------------------------------ */
/* cache rebuilds                                                                              */

void orc_nich_caches(const float sh[4], size_t G, const int32_t *count, const float *mean,
                     const float *ctv, float *cache) {
    const float mu = sh[0], kappa = sh[1], sigmasq = sh[2], nu = sh[3];
    for (size_t g = 0; g < G; ++g) {
        /* Shared::plus_group, nich.hpp:58-69 */
        float n = (float)count[g];
        float mu_1 = mu - mean[g];
        float post_kappa = kappa + n;
        float post_mu = (kappa * mu + mean[g] * n) / post_kappa;
        float post_nu = nu + n;
        float post_sigmasq =
            1.f / post_nu * (nu * sigmasq + ctv[g] + (n * kappa * mu_1 * mu_1) / post_kappa);
        /* Scorer::init, nich.hpp:239-250 */
        float lambda = post_kappa / ((post_kappa + 1.f) * post_sigmasq);
        cache[0 * G + g] =
            orc_fast_lgamma_nu(post_nu) + 0.5f * orc_fast_log(lambda / (3.14159265358979f * post_nu));
        cache[1 * G + g] = -0.5f * post_nu - 0.5f;
        cache[2 * G + g] = lambda / post_nu;
        cache[3 * G + g] = post_mu;
    }
}

void orc_gp_caches(const float sh[2], size_t G, const uint32_t *count, const uint32_t *sum,
                   float *cache) {
    for (size_t g = 0; g < G; ++g) {
        float post_alpha = sh[0] + (float)sum[g];      /* gp.hpp:56-61 */
        float post_inv_beta = sh[1] + (float)count[g];
        float coeff = -orc_fast_log(1.f + post_inv_beta); /* gp.hpp:198-207 */
        cache[0 * G + g] = -orc_fast_lgamma(post_alpha) + post_alpha * (orc_fast_log(post_inv_beta) + coeff);
        cache[1 * G + g] = post_alpha;
        cache[2 * G + g] = coeff;
    }
}

/* BetaNegativeBinomial: plus_group bnb.hpp:57-63, Scorer::init bnb.hpp:200-211; cache[3][G] = score, post_beta, alpha */
void orc_bnb_caches(float alpha, float beta, uint32_t r, size_t G, const uint32_t *count, const uint32_t *sum,
                    float *cache) {
    for (size_t g = 0; g < G; ++g) {
        float post_alpha = alpha + (float)r * count[g];
        float post_beta = beta + sum[g];
        float a = post_alpha + r;
        cache[0 * G + g] = orc_fast_lgamma(post_alpha + post_beta) - orc_fast_lgamma(post_alpha) -
                           orc_fast_lgamma(post_beta) + orc_fast_lgamma(a);
        cache[1 * G + g] = post_beta;
        cache[2 * G + g] = a;
    }
}

void orc_bb_caches(const float sh[2], size_t G, const int32_t *heads, const int32_t *tails,
                   float *cache) {
    for (size_t g = 0; g < G; ++g) { /* bb.hpp:276-292 */
        float h = sh[0] + (float)heads[g];
        float t = sh[1] + (float)tails[g];
        cache[0 * G + g] = orc_fast_log(h / (h + t));
        cache[1 * G + g] = orc_fast_log(t / (h + t));
    }
}

void orc_dd_caches(int dim, const float *alphas, size_t G, const int32_t *counts, float *cache) {
    float alpha_sum = 0; /* dd.hpp:399-421 */
    for (int v = 0; v < dim; ++v) alpha_sum += alphas[v];
    for (size_t g = 0; g < G; ++g) {
        int32_t count_sum = 0;
        for (int v = 0; v < dim; ++v) {
            int32_t c = counts[g * (size_t)dim + v];
            count_sum += c;
            cache[(size_t)v * G + g] = orc_fast_log(alphas[v] + (float)c);
        }
        cache[(size_t)dim * G + g] = orc_fast_log(alpha_sum + (float)count_sum);
    }
}

void orc_dpd_caches(float alpha, float beta0, size_t V, const float *betas, size_t G,
                    const int32_t *counts, float *cache) {
    for (size_t g = 0; g < G; ++g) { /* dpd.hpp:471-497 */
        long total = 0;
        for (size_t v = 0; v < V; ++v) {
            int32_t c = counts[g * V + v];
            total += c;
            cache[v * G + g] = orc_fast_log(alpha * betas[v] + (float)c);
        }
        cache[V * G + g] = orc_fast_log(alpha * beta0); /* dpd.hpp:533-537, OTHER / unseen */
        cache[(V + 1) * G + g] = orc_fast_log(alpha + (float)total);
    }
}

/* ------------------------------------------------------------------------------------------ */
/* score_value over rows (accumulate)                                                          */

void orc_nich_score_rows(size_t G, const float *cache, size_t n, const float *values, float *scores) {
    const float *score = cache, *log_coeff = cache + G, *precision = cache + 2 * G,
                *mean = cache + 3 * G;
    for (size_t i = 0; i < n; ++i) { /* src/models/nich.cc:59-65 */
        float v = values[i];
        float *acc = scores + i * G;
        for (size_t g = 0; g < G; ++g) {
            float d = v - mean[g];
            float temp = 1.f + precision[g] * (d * d);
            acc[g] += score[g] + log_coeff[g] * orc_fast_log(temp);
        }
    }
}

void orc_gp_score_rows(size_t G, const float *cache, size_t n, const uint32_t *values, float *scores) {
    const float *score = cache, *post_alpha = cache + G, *coeff = cache + 2 * G;
    for (size_t i = 0; i < n; ++i) { /* src/models/gp.cc:56-66 */
        float v = (float)values[i];
        float lf = orc_fast_log_factorial(values[i]);
        float *acc = scores + i * G;
        for (size_t g = 0; g < G; ++g) {
            float temp = orc_fast_lgamma(post_alpha[g] + v);
            acc[g] += score[g] + temp - lf + coeff[g] * v;
        }
    }
}

void orc_bnb_score_rows(size_t G, const float *cache, size_t n, const uint32_t *values, float *scores) {
    const float *score = cache, *post_beta = cache + G, *alpha = cache + 2 * G;
    for (size_t i = 0; i < n; ++i) { /* bnb.hpp:308-319 */
        float *acc = scores + i * G;
        for (size_t g = 0; g < G; ++g) {
            float beta = post_beta[g] + values[i];
            acc[g] += score[g] + orc_fast_lgamma(beta) - orc_fast_lgamma(beta + alpha[g]);
        }
    }
}

void orc_bb_score_rows(size_t G, const float *cache, size_t n, const uint8_t *values, float *scores) {
    for (size_t i = 0; i < n; ++i) { /* bb.hpp:303-313 */
        const float *row = values[i] ? cache : cache + G;
        float *acc = scores + i * G;
        for (size_t g = 0; g < G; ++g) acc[g] += row[g];
    }
}

void orc_dd_score_rows(int dim, size_t G, const float *cache, size_t n, const int32_t *values,
                       float *scores) {
    const float *shift = cache + (size_t)dim * G;
    for (size_t i = 0; i < n; ++i) { /* dd.hpp:433-445 -> vector_math.cc:160-168 */
        const float *row = cache + (size_t)values[i] * G;
        float *acc = scores + i * G;
        for (size_t g = 0; g < G; ++g) acc[g] += row[g] - shift[g];
    }
}

void orc_dpd_score_rows(size_t V, size_t G, const float *cache, size_t n, const uint32_t *rows,
                        float *scores) {
    const float *shift = cache + (V + 1) * G;
    for (size_t i = 0; i < n; ++i) { /* dpd.hpp:517-543 -> vector_math.cc:160-178 */
        size_t r = rows[i] < V ? rows[i] : V;
        const float *row = cache + r * G;
        float *acc = scores + i * G;
        for (size_t g = 0; g < G; ++g) acc[g] += row[g] - shift[g];
    }
}

/* ------------------------------------------------------------------------------------------ */
/* NIW                                                                                         */

/* inverse and determinant of an SPD-ish d x d matrix by Gauss-Jordan with partial pivoting in
 * double (the reference calls Eigen's float inverse()/determinant(), random.hpp:171-172; Eigen
 * is absent here, hence "parity unpinned" for this step). a is destroyed. */
static double g_logabsdet; /* sum of log |pivot| of the last invert() call: the determinant's log when det overflows a float */
static double invert(int d, double *a, double *inv) {
    double det = 1.0;
    g_logabsdet = 0.0;
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j) inv[i * d + j] = (i == j);
    for (int c = 0; c < d; ++c) {
        int p = c;
        for (int r = c + 1; r < d; ++r)
            if (fabs(a[r * d + c]) > fabs(a[p * d + c])) p = r;
        if (p != c) {
            for (int j = 0; j < d; ++j) {
                double t = a[c * d + j]; a[c * d + j] = a[p * d + j]; a[p * d + j] = t;
                t = inv[c * d + j]; inv[c * d + j] = inv[p * d + j]; inv[p * d + j] = t;
            }
            det = -det;
        }
        double piv = a[c * d + c];
        det *= piv;
        g_logabsdet += log(fabs(piv));
        for (int j = 0; j < d; ++j) {
            a[c * d + j] /= piv;
            inv[c * d + j] /= piv;
        }
        for (int r = 0; r < d; ++r) {
            if (r == c) continue;
            double f = a[r * d + c];
            if (f == 0.0) continue;
            for (int j = 0; j < d; ++j) {
                a[r * d + j] -= f * a[c * d + j];
                inv[r * d + j] -= f * inv[c * d + j];
            }
        }
    }
    return det;
}

/* fast_log(det) as the reference writes it, while det is a normal float; beyond that (the reference's float determinant()
 * has overflowed to inf or flushed to 0, and its score is meaningless) the log of the
 * determinant itself, as the reference's exact-math Python flavour computes it (dbg/models/niw.py:213,216) */
static float log_det(double det, double logabsdet) {
    const float f = (float)det;
    if (isfinite(f) && f >= 1.17549435e-38f) return orc_fast_log(f);
    return (float)logabsdet;
}

void orc_niw_score_rows(int d, const float *mu, float kappa, const float *psi, float nu, size_t G,
                        const int32_t *count, const float *sum_x, const float *sum_xxT, size_t n,
                        const float *values, float *scores) {
    const size_t dd = (size_t)d * d;
    float *post_mu = (float *)malloc(sizeof(float) * G * d);
    float *sig_inv = (float *)malloc(sizeof(float) * G * dd);
    float *konst = (float *)malloc(sizeof(float) * G * 3); /* term1+term2, coeff3, 1/dof */
    double *a = (double *)malloc(sizeof(double) * dd), *inv = (double *)malloc(sizeof(double) * dd);
    float *xbar = (float *)malloc(sizeof(float) * d), *diff = (float *)malloc(sizeof(float) * d);
    const float log_pi = 1.1447298858494002f;
    for (size_t g = 0; g < G; ++g) {
        /* Shared::plus_group, niw.hpp:82-103 */
        const float cnt = (float)count[g];
        const float *sx = sum_x + g * d, *sxx = sum_xxT + g * dd;
        for (int i = 0; i < d; ++i) xbar[i] = count[g] ? sx[i] / cnt : 0.f;
        for (int i = 0; i < d; ++i)
            post_mu[g * d + i] = kappa / (kappa + cnt) * mu[i] + cnt / (kappa + cnt) * xbar[i];
        float post_kappa = kappa + cnt, post_nu = nu + cnt;
        for (int i = 0; i < d; ++i) diff[i] = xbar[i] - mu[i];
        /* Scorer::eval, niw.hpp:353-360 */
        float dof = post_nu - (float)d + 1.f;
        for (int i = 0; i < d; ++i)
            for (int j = 0; j < d; ++j) {
                float c_n = sxx[i * d + j] - sx[i] * xbar[j] - xbar[i] * sx[j] + cnt * xbar[i] * xbar[j];
                float post_psi = psi[i * d + j] + c_n + kappa * cnt / (kappa + cnt) * (diff[i] * diff[j]);
                float sigma = post_psi * (post_kappa + 1.f) / (post_kappa * dof);
                a[i * d + j] = sigma;
            }
        double det = invert(d, a, inv);
        for (size_t k = 0; k < dd; ++k) sig_inv[g * dd + k] = (float)inv[k];
        /* score_mv_student_t, random.hpp:160-185 (mixed float/double arithmetic as written) */
        float term1 = orc_fast_lgamma((float)(dof / 2. + (float)d / 2.)) - orc_fast_lgamma((float)(dof / 2.));
        float term2 = (float)(-0.5 * log_det(det, g_logabsdet) - (float)d / 2. * (orc_fast_log(dof) + log_pi));
        konst[g * 3 + 0] = term1 + term2;
        konst[g * 3 + 1] = (float)(-0.5 * (dof + (float)d));
        konst[g * 3 + 2] = dof;
    }
    for (size_t r = 0; r < n; ++r) {
        const float *x = values + r * d;
        for (size_t g = 0; g < G; ++g) {
            for (int i = 0; i < d; ++i) diff[i] = x[i] - post_mu[g * d + i];
            float q = 0.f;
            for (int i = 0; i < d; ++i) {
                float row = 0.f;
                for (int j = 0; j < d; ++j) row += sig_inv[g * dd + i * d + j] * diff[j];
                q += diff[i] * row;
            }
            float dof = konst[g * 3 + 2];
            float term3 = (float)((double)konst[g * 3 + 1] * orc_fast_log((float)(1. + 1. / dof * q)));
            scores[r * G + g] += konst[g * 3 + 0] + term3;
        }
    }
    free(post_mu); free(sig_inv); free(konst); free(a); free(inv); free(xbar); free(diff);
}

/* Group::score_data (niw.hpp:296-308) summed over the groups, as SmallMixtureSlave's data scorer does for a model
 * without a FastMixture (mixture.hpp:300-319); lmultigamma is special.hpp:278-286.  The determinants are taken by
 * the Gauss-Jordan above in double (the reference: Eigen's float determinant(); Eigen is absent here). */
static float orc_lmultigamma(int d, float a) {
    const float log_pi = 1.1447298858494002f;
    const float term1 = (float)(0.25 * (float)(d * (d - 1))) * log_pi;
    float term2 = 0.f;
    for (int j = 1; j <= d; ++j) term2 += orc_fast_lgamma((float)(a + 0.5 * (float)(1 - j)));
    return term1 + term2;
}

float orc_niw_score_data(int d, const float *mu, float kappa, const float *psi, float nu, size_t G, const int32_t *count,
                         const float *sum_x, const float *sum_xxT) {
    const size_t dd = (size_t)d * d;
    double *a = (double *)malloc(sizeof(double) * dd), *inv = (double *)malloc(sizeof(double) * dd);
    float *xbar = (float *)malloc(sizeof(float) * d), *diff = (float *)malloc(sizeof(float) * d);
    const float log_pi = 1.1447298858494002f;
    for (size_t k = 0; k < dd; ++k) a[k] = psi[k];
    const double det_prior_d = invert(d, a, inv);
    const float log_det_prior = log_det(det_prior_d, g_logabsdet);
    float total = 0.f;
    for (size_t g = 0; g < G; ++g) {
        const float cnt = (float)count[g];
        const float *sx = sum_x + g * d, *sxx = sum_xxT + g * dd;
        for (int i = 0; i < d; ++i) xbar[i] = count[g] ? sx[i] / cnt : 0.f;
        for (int i = 0; i < d; ++i) diff[i] = xbar[i] - mu[i];
        const float post_kappa = kappa + cnt, post_nu = nu + cnt;
        for (int i = 0; i < d; ++i)
            for (int j = 0; j < d; ++j) {
                float c_n = sxx[i * d + j] - sx[i] * xbar[j] - xbar[i] * sx[j] + cnt * xbar[i] * xbar[j];
                a[i * d + j] = psi[i * d + j] + c_n + kappa * cnt / (kappa + cnt) * (diff[i] * diff[j]);
            }
        const double det_post_d = invert(d, a, inv);
        const float log_det_post = log_det(det_post_d, g_logabsdet);
        total += orc_lmultigamma(d, (float)(post_nu * 0.5)) + (float)(nu * 0.5) * log_det_prior -
                 (float)((float)(count[g] * d) * 0.5) * log_pi - orc_lmultigamma(d, (float)(nu * 0.5)) -
                 (float)(post_nu * 0.5) * log_det_post + (float)((float)d * 0.5) * orc_fast_log(kappa / post_kappa);
    }
    free(a); free(inv); free(xbar); free(diff);
    return total;
}

/* Group::add_value / remove_value (niw.hpp:247-276), one value at a time in float as the reference's Eigen expressions */
void orc_niw_group_update(int sign, int d, int32_t *count, float *sum_x, float *sum_xxT, size_t n, const float *values) {
    for (size_t r = 0; r < n; ++r) {
        const float *x = values + r * d;
        *count += sign;
        for (int i = 0; i < d; ++i) sum_x[i] += sign > 0 ? x[i] : -x[i];
        for (int i = 0; i < d; ++i)
            for (int j = 0; j < d; ++j) sum_xxT[i * d + j] += sign > 0 ? x[i] * x[j] : -(x[i] * x[j]);
    }
}

/* ------------------------------------------------------------------------------------------ */
/* sampler                                                                                     */

float orc_scores_to_likelihoods(size_t G, float *s) { /* random.cc:94-106, vector_math.cc:74-83 */
    float m = s[0];
    for (size_t i = 0; i < G; ++i) m = s[i] > m ? s[i] : m;
    float total = 0;
    for (size_t i = 0; i < G; ++i) {
        s[i] = orc_fast_exp(s[i] - m);
        total += s[i];
    }
    return total;
}

int32_t orc_sample_from_likelihoods(size_t G, const float *lik, float total, float u) {
    float t = total * u; /* random.hpp:315-333 */
    for (size_t i = 0; i < G; ++i) {
        t -= lik[i];
        if (t <= 0) return (int32_t)i;
    }
    return (int32_t)G - 1;
}

void orc_sample_rows(size_t n, size_t G, float *scores, const float *u, int32_t *assign) {
    for (size_t i = 0; i < n; ++i) { /* random.hpp:360-366 */
        float total = orc_scores_to_likelihoods(G, scores + i * G);
        assign[i] = orc_sample_from_likelihoods(G, scores + i * G, total, u[i]);
    }
}

/* ------------------------------------------------------------------------------------------ */
/* Group bookkeeping                                                                           */

void orc_nich_group_update(int op, int32_t *count, float *mean, float *ctv, const float *values, size_t n) {
    for (size_t i = 0; i < n; ++i) {
        float value = values[i];
        if (op > 0) { /* nich.hpp:125-133 */
            ++*count;
            float delta = value - *mean;
            *mean += delta / (float)*count;
            *ctv += delta * (value - *mean);
        } else { /* nich.hpp:146-165 */
            float total = *mean * (float)*count;
            float delta = value - *mean;
            --*count;
            *mean = (*count == 0) ? 0.f : (total - value) / (float)*count;
            if (*count <= 1) *ctv = 0.f;
            else *ctv -= delta * (value - *mean);
        }
    }
}

void orc_gp_group_update(int op, uint32_t *count, uint32_t *sum, float *log_prod, const uint32_t *values,
                         size_t n) {
    for (size_t i = 0; i < n; ++i) { /* gp.hpp:109-135 */
        if (op > 0) {
            ++*count; *sum += values[i]; *log_prod += orc_fast_log_factorial(values[i]);
        } else {
            --*count; *sum -= values[i]; *log_prod -= orc_fast_log_factorial(values[i]);
        }
    }
}

/* ------------------------------------------------------------------------------------------ */
/* timing helper                                                                               */

typedef struct {
    size_t G, lo, hi;
    const float *cache, *prior, *values, *u;
    int32_t *assign;
} bench_arg;

static void *bench_worker(void *p) {
    bench_arg *a = (bench_arg *)p;
    float *buf = (float *)malloc(sizeof(float) * a->G);
    for (size_t i = a->lo; i < a->hi; ++i) {
        memcpy(buf, a->prior, sizeof(float) * a->G);
        orc_nich_score_rows(a->G, a->cache, 1, a->values + i, buf);
        float total = orc_scores_to_likelihoods(a->G, buf);
        a->assign[i] = orc_sample_from_likelihoods(a->G, buf, total, a->u[i]);
    }
    free(buf);
    return NULL;
}

double orc_bench_nich(size_t G, const float *cache, const float *prior, size_t n, const float *values,
                      const float *u, int32_t *assign, int n_threads) {
    orc_init();
    if (n_threads < 1) n_threads = 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * n_threads);
    bench_arg *args = (bench_arg *)malloc(sizeof(bench_arg) * n_threads);
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (int t = 0; t < n_threads; ++t) {
        bench_arg a = {G, n * t / n_threads, n * (t + 1) / n_threads, cache, prior, values, u, assign};
        args[t] = a;
        pthread_create(&th[t], NULL, bench_worker, &args[t]);
    }
    for (int t = 0; t < n_threads; ++t) pthread_join(th[t], NULL);
    clock_gettime(CLOCK_MONOTONIC, &t1);
    free(th);
    free(args);
    return (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
}
