// sample_values.cu -- batched Group::sample_value: one draw from the posterior predictive of each row's group
// (dist_b200_sample_values_batch).  The reference draws a value as Sampler::init from the posterior followed by one
// Sampler::eval (nich.hpp, gp.hpp, bnb.hpp, bb.hpp, dd.hpp, dpd.hpp, niw.hpp); with fresh parameters per value that is
// exactly one draw from the posterior predictive, which is what the row kernels below draw directly:
//   nich  Student-t(nu', mu', sigmasq' (kappa' + 1) / kappa')     mu' + scale z sqrt((nu'/2) / Gamma(nu'/2))
//   gp    Poisson(lambda), lambda ~ Gamma(alpha', rate inv_beta')
//   bnb   NegBin(r, p), p ~ Beta(alpha', beta')                   Poisson(Gamma(r) Gamma(beta') / Gamma(alpha'))
//   bb    Bernoulli(alpha' / (alpha' + beta'))
//   dd    categorical over v < dim, weights alphas[v] + counts[g][v]
//   dpd   categorical over the known values, weights alpha betas[v] + counts[g][v], and OTHER with alpha beta0
//   niw   multivariate t(dof = nu' - d + 1, mu', psi' (kappa' + 1) / (kappa' dof))     mu' + L z sqrt((dof/2) / Gamma(dof/2))
// The posteriors come from posterior.cuh, the code the cache rebuilds use.
//
// Two passes per feature.  A prep pass, O(G dim), turns the device-resident statistics into per-group records: the
// predictive's parameters (scalar models), a CDF with prefix sums in double plus a guide table (dd / dpd), the
// Cholesky factor L of the scale matrix (niw).  A row kernel then draws one value per row: rows on threads (niw: a
// sub-warp of the next power of two >= d lanes per row, lanes over coordinates), coalesced assign loads and stores.
//
// Random numbers: Philox4x32-10 keyed by the seed, counter (global row, feature position, block index within the
// value).  A draw is a pure function of (seed, row0 + n, position, the group's statistics): launch geometry, n_rows
// and chunking do not enter, so row shards that pass their own row0 reproduce one call over all rows bit for bit.
//
// This translation unit is compiled with --fmad=false so that the posteriors round as in prep.cu.
#include <curand_philox4x32_x.h>

#include "common.cuh"
#include "posterior.cuh"

namespace distb200 {
namespace {

// Counter-based random stream of one value: block b of (seed; row, feature, first + b)
struct ValueRng {
    uint4 ctr;
    uint2 key;
    uint4 buf;
    int left;
    __device__ ValueRng(uint64_t seed, uint64_t row, uint32_t feature, uint32_t first)
        : ctr(make_uint4(static_cast<uint32_t>(row), static_cast<uint32_t>(row >> 32), feature, first)),
          key(make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32))), buf(make_uint4(0, 0, 0, 0)), left(0) {}
    __device__ __forceinline__ uint32_t next() {
        if (left == 0) {
            buf = curand_Philox4x32_10(ctr, key);
            ++ctr.w;
            left = 4;
        }
        const uint32_t r = buf.x;  // shift instead of indexing: the words stay in registers
        buf.x = buf.y;
        buf.y = buf.z;
        buf.z = buf.w;
        --left;
        return r;
    }
    // (0, 1) on a 2^-32 grid, never 0 or 1: safe under log
    __device__ __forceinline__ double open01() { return (static_cast<double>(next()) + 0.5) * 2.3283064365386963e-10; }
    // [0, 1) with 53 random bits (CDF walks)
    __device__ __forceinline__ double unit53() {
        const uint32_t hi = next() >> 5, lo = next() >> 6;
        return (static_cast<double>(hi) * 67108864.0 + static_cast<double>(lo)) * 1.1102230246251565e-16;
    }
    // standard normal (Box-Muller, cosine branch)
    __device__ __forceinline__ double normal() {
        const double u = open01(), v = open01();
        return sqrt(-2.0 * log(u)) * cospi(2.0 * v);
    }
};

// log of a Gamma(a, 1) draw, a > 0 (Marsaglia & Tsang 2000).  Shapes below 1 take the boost
// Gamma(a) = Gamma(a + 1) U^(1/a), kept in log space so that it cannot underflow.  The acceptance test
// log u < z^2/2 + d (1 - v + log v) runs in double with 1 - v + log v = 3 log1p(w) - w (3 + w (3 + w)), v = (1 + w)^3:
// at the shapes of large groups (10^6 and more) the fp32 form loses every digit to cancellation.
__device__ double log_gamma_draw(ValueRng &r, double a) {
    double boost = 0.0;
    if (a < 1.0) {
        boost = log(r.open01()) / a;
        a += 1.0;
    }
    const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    for (;;) {
        double z, w;
        do {
            z = r.normal();
            w = c * z;
        } while (w <= -1.0);
        const double u = r.open01(), z2 = z * z;
        const double v = (1.0 + w) * (1.0 + w) * (1.0 + w);
        if (u < 1.0 - 0.0331 * z2 * z2 || log(u) < 0.5 * z2 + d * (3.0 * log1p(w) - w * (3.0 + w * (3.0 + w))))
            return log(d * v) + boost;
    }
}

// Poisson(lam), exact at every mean: inversion below 10, PTRS (Hoermann 1993, transformed rejection with squeeze)
// above, its acceptance test with the double-precision lgamma (accurate log k! at any k).
__device__ uint32_t poisson_draw(ValueRng &r, double lam) {
    if (!(lam > 0.0)) return 0;
    if (lam < 10.0) {
        const double u = r.open01();
        double p = exp(-lam), s = p;
        uint32_t k = 0;
        while (u > s && k < 256) {
            ++k;
            p *= lam / k;
            s += p;
        }
        return k;
    }
    const double slam = sqrt(lam), loglam = log(lam);
    const double b = 0.931 + 2.53 * slam, a = -0.059 + 0.02483 * b;
    const double inv_alpha = 1.1239 + 1.1328 / (b - 3.4), vr = 0.9277 - 3.6224 / (b - 2.0);
    for (;;) {
        const double U = r.open01() - 0.5, V = r.open01();
        const double us = 0.5 - fabs(U);
        const double k = floor((2.0 * a / us + b) * U + lam + 0.43);
        if (us >= 0.07 && V <= vr) return k >= 4294967295.0 ? 0xFFFFFFFFu : static_cast<uint32_t>(k);
        if (k < 0.0 || (us < 0.013 && V > us)) continue;
        if (log(V) + log(inv_alpha) - log(a / (us * us) + b) <= -lam + k * loglam - lgamma(k + 1.0))
            return k >= 4294967295.0 ? 0xFFFFFFFFu : static_cast<uint32_t>(k);
    }
}

struct Rec {  // per-group record of the scalar models
    double a, b, c, pad;
};

struct SampleArgs {
    int G, K, V;         // K: categories (dd dim, dpd V + 1)
    int d, W;            // niw: dimension, lanes per row (power of two >= d)
    size_t N;
    const int32_t *assign;
    void *out;
    uint64_t seed, row0;
    uint32_t feature;
    const Rec *rec;
    const double *cdf;   // [G][K]
    const int *guide;    // [G][K]
    const uint32_t *colkey;  // dpd: key of each counts column
    const float *niw;    // [G][niw_sample_floats]
    int niw_stride;
};

__host__ __device__ constexpr int niw_lanes(int d) { return d <= 1 ? 1 : d <= 2 ? 2 : d <= 4 ? 4 : d <= 8 ? 8 : d <= 16 ? 16 : 32; }
// niw record: mu'[W] | Lt[d][W] (Lt[k][i] = L[i][k], zero above the diagonal of L) | dof / 2
__host__ __device__ constexpr int niw_sample_floats(int d) { return niw_lanes(d) * (d + 1) + 1; }

// ---- prep ----------------------------------------------------------------------------------------------------------
__global__ void scalar_prep_kernel(const SampleSrc src, Rec *__restrict__ rec) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= src.G) return;
    const float *sh = src.shared;
    Rec r{0, 0, 0, 0};
    switch (src.model) {
        case DIST_B200_NICH: {
            const NichPost p = nich_plus_group(sh[0], sh[1], sh[2], sh[3], static_cast<int32_t>(src.st0[g]),
                                               __uint_as_float(src.st1[g]), __uint_as_float(src.st2[g]));
            r.a = p.mu;
            r.b = sqrt(static_cast<double>(p.sigmasq) * (static_cast<double>(p.kappa) + 1.0) / static_cast<double>(p.kappa));
            r.c = 0.5 * static_cast<double>(p.nu);
        } break;
        case DIST_B200_GP: {
            const float2 p = gp_plus_group(sh[0], sh[1], src.st0[g], src.st1[g]);
            r.a = p.x;  // shape
            r.b = p.y;  // rate
        } break;
        case DIST_B200_BNB: {
            const float2 p = bnb_plus_group(sh[0], sh[1], sh[2], src.st0[g], src.st1[g]);
            r.a = p.x;
            r.b = p.y;
            r.c = sh[2];
        } break;
        default: {  // bb
            const float2 p = bb_plus_group(sh[0], sh[1], static_cast<int32_t>(src.st0[g]), static_cast<int32_t>(src.st1[g]));
            r.a = static_cast<double>(p.x) / (static_cast<double>(p.x) + static_cast<double>(p.y));
        }
    }
    rec[g] = r;
}

__device__ __forceinline__ double cat_weight(const SampleSrc &src, int g, int k) {
    if (src.model == DIST_B200_DD)
        return static_cast<double>(src.alphas[k]) + static_cast<double>(reinterpret_cast<const int32_t *>(src.st0)[static_cast<size_t>(g) * src.dim + k]);
    if (k < src.dim)
        return static_cast<double>(src.shared[0]) * src.alphas[k] +
               static_cast<double>(reinterpret_cast<const int32_t *>(src.st0)[static_cast<size_t>(g) * src.dim + k]);
    return static_cast<double>(src.shared[0]) * src.shared[1];  // OTHER: alpha beta0
}

// one warp per group: cdf[k] = P(X <= k) from prefix sums in double (2.0 from the last category of non-zero weight on,
// so that the walk always stops there), guide[j] = the smallest k with cdf[k] > j / K
__global__ void cdf_prep_kernel(const SampleSrc src, int K, double *__restrict__ cdf, int *__restrict__ guide) {
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (g >= src.G) return;
    double total = 0.0;
    int last = 0;
    for (int k = lane; k < K; k += 32) {
        const double w = cat_weight(src, g, k);
        total += w;
        if (w > 0.0) last = k;
    }
    for (int o = 16; o; o >>= 1) {
        total += __shfl_xor_sync(0xffffffffu, total, o);
        last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
    }
    double *c = cdf + static_cast<size_t>(g) * K;
    double carry = 0.0;
    for (int k0 = 0; k0 < K; k0 += 32) {
        const int k = k0 + lane;
        double s = k < K ? cat_weight(src, g, k) : 0.0;
        for (int o = 1; o < 32; o <<= 1) {
            const double t = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += t;
        }
        if (k < K) c[k] = k >= last ? 2.0 : (carry + s) / total;
        carry += __shfl_sync(0xffffffffu, s, 31);
    }
    __syncwarp();
    int *gd = guide + static_cast<size_t>(g) * K;
    for (int j = lane; j < K; j += 32) {
        const double x = static_cast<double>(j) / K;
        int lo = 0, hi = last;  // cdf[last] = 2 > x
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (c[mid] > x) hi = mid;
            else lo = mid + 1;
        }
        gd[j] = lo;
    }
}

// dpd: the key of each counts column (keys_dev is sorted, key_rows_dev[i] the column of sorted key i)
__global__ void colkey_kernel(int V, const uint32_t *__restrict__ sorted, const int *__restrict__ rows, uint32_t *__restrict__ colkey) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < V) colkey[rows[i]] = sorted[i];
}

// one block per group (d <= 32): the posterior and L from the code niw_prep_kernel runs
__global__ void niw_sample_prep_kernel(const SampleSrc src, float *__restrict__ out) {
    __shared__ double S[32][33];
    __shared__ double xbar[32], diff[32];
    const int g = blockIdx.x, tid = threadIdx.x, d = src.dim, W = niw_lanes(d);
    const float *mu = src.alphas, *psi = src.alphas + d;
    const int32_t count = reinterpret_cast<const int32_t *>(src.st0)[g];
    const float *sx = reinterpret_cast<const float *>(src.st1) + static_cast<size_t>(g) * d;
    const float *sxx = reinterpret_cast<const float *>(src.st2) + static_cast<size_t>(g) * d * d;
    const double dof = niw_posterior_cholesky(d, mu, src.shared[0], psi, src.shared[1], count, sx, sxx, S, xbar, diff);
    float *rec = out + static_cast<size_t>(g) * niw_sample_floats(d);
    for (int i = tid; i < W; i += blockDim.x) rec[i] = i < d ? static_cast<float>(niw_post_mu(src.shared[0], count, mu[i], xbar[i])) : 0.f;
    for (int e = tid; e < d * W; e += blockDim.x) {
        const int k = e / W, i = e % W;
        rec[W + e] = (i < d && i >= k) ? static_cast<float>(S[i][k]) : 0.f;
    }
    if (tid == 0) rec[W + d * W] = static_cast<float>(0.5 * dof);
}

// 32 < d <= 128: the same record with niw_wide_cols(d) columns per Lt row; a double [128][129] matrix (dynamic shared memory)
__host__ __device__ constexpr int niw_wide_cols(int d) { return (d + 31) / 32 * 32; }
__host__ __device__ constexpr int niw_wide_sample_floats(int d) { return niw_wide_cols(d) * (d + 1) + 1; }
constexpr int kNiwWideLd = 129;
constexpr size_t kNiwWideSampleSmem = sizeof(double) * (128 * kNiwWideLd + 2 * 128);

__global__ void __launch_bounds__(256) niw_sample_prep_wide_kernel(const SampleSrc src, float *__restrict__ out) {
    extern __shared__ double ssm[];
    double(*S)[kNiwWideLd] = reinterpret_cast<double(*)[kNiwWideLd]>(ssm);
    double *xbar = ssm + 128 * kNiwWideLd, *diff = xbar + 128;
    const int g = blockIdx.x, tid = threadIdx.x, d = src.dim, W = niw_wide_cols(d);
    const float *mu = src.alphas, *psi = src.alphas + d;
    const int32_t count = reinterpret_cast<const int32_t *>(src.st0)[g];
    const float *sx = reinterpret_cast<const float *>(src.st1) + static_cast<size_t>(g) * d;
    const float *sxx = reinterpret_cast<const float *>(src.st2) + static_cast<size_t>(g) * d * d;
    const double dof = niw_posterior_cholesky<kNiwWideLd>(d, mu, src.shared[0], psi, src.shared[1], count, sx, sxx, S, xbar, diff);
    float *rec = out + static_cast<size_t>(g) * niw_wide_sample_floats(d);
    for (int i = tid; i < W; i += blockDim.x) rec[i] = i < d ? static_cast<float>(niw_post_mu(src.shared[0], count, mu[i], xbar[i])) : 0.f;
    for (int e = tid; e < d * W; e += blockDim.x) {
        const int k = e / W, i = e % W;
        rec[W + e] = (i < d && i >= k) ? static_cast<float>(S[i][k]) : 0.f;
    }
    if (tid == 0) rec[W + d * W] = static_cast<float>(0.5 * dof);
}

// ---- rows ----------------------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(256) sample_rows_kernel(const SampleArgs a) {
    const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
    for (size_t n = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; n < a.N; n += stride) {
        const int g = a.assign[n];
        if (g < 0 || g >= a.G) continue;
        ValueRng r(a.seed, a.row0 + n, a.feature, 0);
        if (MODEL == DIST_B200_DD || MODEL == DIST_B200_DPD) {
            const double u = r.unit53();
            const double *c = a.cdf + static_cast<size_t>(g) * a.K;
            int k = a.guide[static_cast<size_t>(g) * a.K + min(static_cast<int>(u * a.K), a.K - 1)];
            while (k > 0 && c[k - 1] > u) --k;
            while (u >= c[k]) ++k;
            if (MODEL == DIST_B200_DD) static_cast<int32_t *>(a.out)[n] = k;
            else static_cast<uint32_t *>(a.out)[n] = k < a.V ? a.colkey[k] : 0xFFFFFFFFu;
        } else {
            const Rec p = a.rec[g];
            if (MODEL == DIST_B200_BB) {
                static_cast<uint8_t *>(a.out)[n] = r.open01() < p.a ? 1 : 0;
            } else if (MODEL == DIST_B200_NICH) {
                const double z = r.normal();
                const double t = z * exp(0.5 * (log(p.c) - log_gamma_draw(r, p.c)));
                static_cast<float *>(a.out)[n] = static_cast<float>(p.a + p.b * t);
            } else if (MODEL == DIST_B200_GP) {
                static_cast<uint32_t *>(a.out)[n] = poisson_draw(r, exp(log_gamma_draw(r, p.a)) / p.b);
            } else {  // bnb: p ~ Beta(alpha', beta') = X / (X + Y); NegBin(r, p) = Poisson(Gamma(r) (1 - p) / p), (1 - p) / p = Y / X
                const double lx = log_gamma_draw(r, p.a), ly = log_gamma_draw(r, p.b), lr = log_gamma_draw(r, p.c);
                static_cast<uint32_t *>(a.out)[n] = poisson_draw(r, exp(lr + ly - lx));
            }
        }
    }
}

// niw: W lanes per row (W = power of two >= d), lane c owns coordinate c: z_c from block c of the row's stream, the
// chi-square from block 32 on (lane 0), x_c = mu'_c + s sum_{k <= c} L[c][k] z_k with z_k shuffled within the row's lanes
__global__ void __launch_bounds__(256) niw_sample_rows_kernel(const SampleArgs a) {
    const int lane = threadIdx.x & 31, W = a.W, d = a.d;
    const int sub = lane / W, c = lane & (W - 1), rows_per_warp = 32 / W;
    const unsigned mask = W == 32 ? 0xffffffffu : ((1u << W) - 1) << (sub * W);
    const size_t warp = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const size_t warps = (static_cast<size_t>(gridDim.x) * blockDim.x) >> 5;
    for (size_t base = warp * rows_per_warp; base < a.N; base += warps * rows_per_warp) {
        const size_t n = base + sub;
        if (n >= a.N) continue;
        const int g = a.assign[n];
        if (g < 0 || g >= a.G) continue;
        const float *rec = a.niw + static_cast<size_t>(g) * a.niw_stride;
        float z = 0.f, s = 0.f;
        if (c < d) {
            ValueRng r(a.seed, a.row0 + n, a.feature, c);
            z = static_cast<float>(r.normal());
        }
        if (c == 0) {
            const double h = rec[W + d * W];
            ValueRng r(a.seed, a.row0 + n, a.feature, 32);
            s = static_cast<float>(exp(0.5 * (log(h) - log_gamma_draw(r, h))));
        }
        s = __shfl_sync(mask, s, 0, W);
        float acc = 0.f;
        for (int k = 0; k < d; ++k) {
            const float zk = __shfl_sync(mask, z, k, W);
            acc = fmaf(rec[W + k * W + c], zk, acc);  // zero above L's diagonal and in the padding lanes
        }
        if (c < d) static_cast<float *>(a.out)[n * d + c] = fmaf(s, acc, rec[c]);
    }
}

// 32 < d <= 128: one warp per row, lane c owns coordinates c, c + 32, ...: z_c from block c of the row's stream, the
// chi-square from block max(32, d) on (lane 0), so no block serves two quantities
__global__ void __launch_bounds__(256) niw_sample_rows_wide_kernel(const SampleArgs a) {
    const int lane = threadIdx.x & 31, d = a.d, W = a.W;
    const size_t warp = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const size_t warps = (static_cast<size_t>(gridDim.x) * blockDim.x) >> 5;
    for (size_t n = warp; n < a.N; n += warps) {
        const int g = a.assign[n];
        if (g < 0 || g >= a.G) continue;
        const float *rec = a.niw + static_cast<size_t>(g) * a.niw_stride;
        float z[4] = {0.f, 0.f, 0.f, 0.f}, s = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = lane + 32 * j;
            if (c < d) {
                ValueRng r(a.seed, a.row0 + n, a.feature, c);
                z[j] = static_cast<float>(r.normal());
            }
        }
        if (lane == 0) {
            const double h = rec[W + d * W];
            ValueRng r(a.seed, a.row0 + n, a.feature, d > 32 ? d : 32);
            s = static_cast<float>(exp(0.5 * (log(h) - log_gamma_draw(r, h))));
        }
        s = __shfl_sync(0xffffffffu, s, 0);
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int jk = 0; jk < 4; ++jk) {
            if (32 * jk >= d) break;
            for (int kk = 0; kk < 32; ++kk) {
                const int k = 32 * jk + kk;
                const float zk = __shfl_sync(0xffffffffu, z[jk], kk);
                if (k >= d) continue;
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (32 * j < W) acc[j] = fmaf(rec[W + k * W + lane + 32 * j], zk, acc[j]);  // zero above L's diagonal
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = lane + 32 * j;
            if (c < d) static_cast<float *>(a.out)[n * d + c] = fmaf(s, acc[j], rec[c]);
        }
    }
}

}  // namespace

#define SAMPLE_LAUNCH_CHECK(ctx)                                                                               \
    do {                                                                                                       \
        cudaError_t e__ = cudaGetLastError();                                                                  \
        if (e__ != cudaSuccess)                                                                                \
            return fail((ctx), DIST_B200_ERR_CUDA, std::string("sample_values launch: ") + cudaGetErrorString(e__)); \
    } while (0)

static size_t sample_buf_bytes(const SampleSrc &src) {
    const size_t G = static_cast<size_t>(src.G);
    switch (src.model) {
        case DIST_B200_DD: return round_up(G * src.dim * 8, 256) + round_up(G * src.dim * 4, 256);
        case DIST_B200_DPD: return round_up(G * (src.dim + 1) * 8, 256) + round_up(G * (src.dim + 1) * 4, 256) + round_up(4 * static_cast<size_t>(src.dim), 256);
        case DIST_B200_NIW: return G * (src.dim > 32 ? niw_wide_sample_floats(src.dim) : niw_sample_floats(src.dim)) * 4;
        default: return G * sizeof(Rec);
    }
}

int launch_sample_values(dist_b200_ctx *ctx, dist_b200_feature *f, const SampleSrc &src, uint32_t position, const int32_t *assign,
                         size_t N, uint64_t seed, uint64_t row0, void *out, cudaStream_t s) {
    if (N == 0 || src.G <= 0) return DIST_B200_OK;
    if (int rc = grow(ctx, f->sample_buf, f->sample_bytes, sample_buf_bytes(src))) return rc;
    char *buf = static_cast<char *>(f->sample_buf);
    SampleArgs a{};
    a.G = src.G;
    a.N = N;
    a.assign = assign;
    a.out = out;
    a.seed = seed;
    a.row0 = row0;
    a.feature = position;
    const int threads = 256;
    const size_t row_blocks = std::min<size_t>((N + threads - 1) / threads, static_cast<size_t>(ctx->sm_count) * 32);
    const unsigned blocks = static_cast<unsigned>(std::max<size_t>(row_blocks, 1));
    switch (src.model) {
        case DIST_B200_DD:
        case DIST_B200_DPD: {
            a.K = src.model == DIST_B200_DD ? src.dim : src.dim + 1;
            a.V = src.dim;
            double *cdf = reinterpret_cast<double *>(buf);
            int *guide = reinterpret_cast<int *>(buf + round_up(static_cast<size_t>(src.G) * a.K * 8, 256));
            cdf_prep_kernel<<<(src.G * 32 + threads - 1) / threads, threads, 0, s>>>(src, a.K, cdf, guide);
            SAMPLE_LAUNCH_CHECK(ctx);
            a.cdf = cdf;
            a.guide = guide;
            if (src.model == DIST_B200_DPD) {
                uint32_t *colkey = reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(guide) + round_up(static_cast<size_t>(src.G) * a.K * 4, 256));
                colkey_kernel<<<(src.dim + 255) / 256, 256, 0, s>>>(src.dim, src.keys_sorted, src.key_rows, colkey);
                SAMPLE_LAUNCH_CHECK(ctx);
                a.colkey = colkey;
                sample_rows_kernel<DIST_B200_DPD><<<blocks, threads, 0, s>>>(a);
            } else {
                sample_rows_kernel<DIST_B200_DD><<<blocks, threads, 0, s>>>(a);
            }
        } break;
        case DIST_B200_NIW: {
            float *recs = reinterpret_cast<float *>(buf);
            if (src.dim > 32) {
                DISTB200_CUDA(ctx, cudaFuncSetAttribute(niw_sample_prep_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                        static_cast<int>(kNiwWideSampleSmem)));
                niw_sample_prep_wide_kernel<<<src.G, 256, kNiwWideSampleSmem, s>>>(src, recs);
                SAMPLE_LAUNCH_CHECK(ctx);
                a.d = src.dim;
                a.W = niw_wide_cols(src.dim);
                a.niw = recs;
                a.niw_stride = niw_wide_sample_floats(src.dim);
                const unsigned nb = static_cast<unsigned>(std::max<size_t>(1, std::min<size_t>((N * 32 + threads - 1) / threads,
                                                                                               static_cast<size_t>(ctx->sm_count) * 32)));
                niw_sample_rows_wide_kernel<<<nb, threads, 0, s>>>(a);
                break;
            }
            niw_sample_prep_kernel<<<src.G, 64, 0, s>>>(src, recs);
            SAMPLE_LAUNCH_CHECK(ctx);
            a.d = src.dim;
            a.W = niw_lanes(src.dim);
            a.niw = recs;
            a.niw_stride = niw_sample_floats(src.dim);
            const size_t warps = (N + 32 / a.W - 1) / (32 / a.W);
            const unsigned nb = static_cast<unsigned>(std::max<size_t>(1, std::min<size_t>((warps * 32 + threads - 1) / threads,
                                                                                           static_cast<size_t>(ctx->sm_count) * 32)));
            niw_sample_rows_kernel<<<nb, threads, 0, s>>>(a);
        } break;
        default: {
            Rec *rec = reinterpret_cast<Rec *>(buf);
            scalar_prep_kernel<<<(src.G + 127) / 128, 128, 0, s>>>(src, rec);
            SAMPLE_LAUNCH_CHECK(ctx);
            a.rec = rec;
            switch (src.model) {
                case DIST_B200_NICH: sample_rows_kernel<DIST_B200_NICH><<<blocks, threads, 0, s>>>(a); break;
                case DIST_B200_GP: sample_rows_kernel<DIST_B200_GP><<<blocks, threads, 0, s>>>(a); break;
                case DIST_B200_BNB: sample_rows_kernel<DIST_B200_BNB><<<blocks, threads, 0, s>>>(a); break;
                case DIST_B200_BB: sample_rows_kernel<DIST_B200_BB><<<blocks, threads, 0, s>>>(a); break;
                default: return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "sample_values: unsupported model");
            }
        }
    }
    SAMPLE_LAUNCH_CHECK(ctx);
    return DIST_B200_OK;
}

}  // namespace distb200
