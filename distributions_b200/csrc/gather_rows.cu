// gather_rows.cu -- warp-per-row kernels: groups mapped to lanes.
//
//  (1) value-major cache tables too large for shared memory -- DirichletProcessDiscrete
//      (dpd.hpp:517-543: scores_[value][g] - scores_shift_[g], or the OTHER row) -- where a row's
//      whole score vector is one contiguous table row: each warp gathers the row of its value with
//      coalesced loads (the table lives in L2: (V+1)*G*4 B = 8.4 MB at V=4096, G=512), adds the prior
//      vector and samples.
//  (2) sample_from_scores over materialised [N][G] scores (random.hpp:386-392), e.g. after the
//      feature-shard reduction: same code with the score row read from HBM.
//
// Sampler (scores_to_likelihoods + sample_from_likelihoods, random.cc:94-106, random.hpp:315-333):
// lanes hold the row striped (g = 32k + lane) for coalescing; max and total by warp butterflies; the
// likelihoods are parked in a skew-padded shared-memory row so that each lane can then own a
// CONTIGUOUS segment of groups: lane sums -> warp prefix -> the lane whose segment holds u*total
// walks it with the reference's `t -= l[i]; t <= 0` loop.
#include "common.cuh"

namespace distb200 {

constexpr int kGatherThreadsMax = 256;

__device__ __forceinline__ int skew(int g) { return g + (g >> 5); }

struct GatherArgs {
    int G;
    int V;                   // table mode: number of known values (row V = OTHER)
    int keys_dense;          // table mode: value == row index
    int accumulate;
    size_t N;
    const float *table;      // [(V+1)][G] or nullptr (scores mode)
    const uint32_t *values;  // table mode: the value column
    const uint32_t *keys;    // sorted keys (when !keys_dense)
    const int *key_rows;     // table row of sorted key i
    const float *prior;      // [G] or nullptr
    const float *scores_in;  // scores mode: [N][G]
    int n_slots;             // scores mode: the row is the sum of n_slots partial rows ...
    size_t slot_stride;      // ... slot_stride floats apart (feature-shard slots, summed in slot order)
    const float *u;
    int32_t *assign;         // nullable
    float *scores_out;       // nullable ([N][G])
};

__device__ __forceinline__ int table_row(const GatherArgs &a, uint32_t value) {
    if (a.keys_dense) return value < static_cast<uint32_t>(a.V) ? static_cast<int>(value) : a.V;
    int lo = 0, hi = a.V;  // lower_bound over sorted keys
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a.keys[mid] < value) lo = mid + 1;
        else hi = mid;
    }
    return (lo < a.V && a.keys[lo] == value) ? a.key_rows[lo] : a.V;
}

__global__ void __launch_bounds__(kGatherThreadsMax) gather_rows_kernel(const GatherArgs a, int seg) {
    extern __shared__ float lik_all[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    const int G = a.G;
    const int row_floats = skew(32 * seg) + 1;  // seg = ceil(G / 32) groups per lane
    float *lik = lik_all + static_cast<size_t>(warp) * row_floats;
    const bool sample = a.assign != nullptr;

    for (size_t n = static_cast<size_t>(blockIdx.x) * warps + warp; n < a.N;
         n += static_cast<size_t>(gridDim.x) * warps) {
        const float *src = a.table ? a.table + static_cast<size_t>(table_row(a, a.values[n])) * G
                                   : a.scores_in + n * G;
        float *out = a.scores_out ? a.scores_out + n * G : nullptr;
        // pass 1: scores (striped, coalesced), row maximum (vector_max, vector_math.cc:74-83)
        float m = -INFINITY;
        for (int g = lane; g < G; g += 32) {
            float s = src[g];
            for (int k = 1; k < a.n_slots; ++k) s += src[k * a.slot_stride + g];
            if (a.table) {
                if (a.accumulate) s += out[g];          // slave semantic: accumulate onto the buffer
                else if (a.prior) s = a.prior[g] + s;   // clustering overwrite, then the slave adds
            }
            if (out) out[g] = s;
            if (sample) {
                lik[skew(g)] = s;
                m = fmaxf(m, s);
            }
        }
        if (!sample) continue;
#pragma unroll
        for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        __syncwarp();
        // pass 2: each lane owns groups [lane*seg, lane*seg+seg): likelihoods and their sum
        const int gbeg = lane * seg, gend = min(G, gbeg + seg);
        float part = 0.f;
        for (int g = gbeg; g < gend; ++g) {
            const float l = fast_exp_neg(lik[skew(g)] - m);
            lik[skew(g)] = l;
            part += l;
        }
        // inclusive prefix over lanes = the reference's left-to-right total at segment granularity
        float incl = part;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const float total = __shfl_sync(0xffffffffu, incl, 31);
        const float t0 = total * a.u[n];
        // first lane whose inclusive prefix reaches t0 (fallthrough: last lane), then walk its segment
        const unsigned hit = __ballot_sync(0xffffffffu, incl >= t0 && gbeg < G);
        const int owner = hit ? __ffs(hit) - 1 : min(31, (G - 1) / seg);
        if (lane == owner) {
            float t = t0 - (incl - part);
            int idx = gend - 1;
            for (int g = gbeg; g < gend; ++g) {
                t -= lik[skew(g)];
                if (t <= 0.f) {
                    idx = g;
                    break;
                }
            }
            if (!hit) idx = G - 1;
            a.assign[n] = idx;
        }
        __syncwarp();
    }
}

// Register-tiled form for G <= 32 * K (K = 1..32 cells per lane, compile time): the row is held striped
// in registers (g = 32 k + lane) through max / exp / sum with fully unrolled loops; only the likelihoods
// cross shared memory once (skewed, conflict-free both ways) so that each lane can sum a CONTIGUOUS
// segment; the segment holding u * total is then resolved by a K-lane prefix scan instead of a serial
// walk.  Sampling only (the materialising variants stay on the generic kernel above).
constexpr int kFastWarps = 8;

template <int K>
__global__ void __launch_bounds__(kFastWarps * 32) gather_rows_fast_kernel(const GatherArgs a) {
    __shared__ float lik_all[kFastWarps][33 * K + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int G = a.G;
    float *lik = lik_all[warp];
    float prior[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int g = 32 * k + lane;
        prior[k] = (a.table && a.prior && g < G) ? a.prior[g] : 0.f;
    }
    // this lane's contiguous segment [lane*K, lane*K + K) in skewed coordinates: K divides 32, so the
    // segment never crosses a 32-boundary and skew(lane*K + kk) = seg0 + kk
    const int seg0 = lane * K + ((lane * K) >> 5);
    const unsigned full = 0xffffffffu;
    for (size_t n = static_cast<size_t>(blockIdx.x) * kFastWarps + warp; n < a.N;
         n += static_cast<size_t>(gridDim.x) * kFastWarps) {
        const float *src = a.table ? a.table + static_cast<size_t>(table_row(a, a.values[n])) * G
                                   : a.scores_in + n * G;
        float s[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {  // K independent loads in flight
            const int g = 32 * k + lane;
            s[k] = g < G ? src[g] + prior[k] : -INFINITY;  // prior + (scores_[v][g] - shift[g])
        }
        for (int sl = 1; sl < a.n_slots; ++sl) {  // feature-shard slots, summed in fixed slot order
            const float *ss = src + sl * a.slot_stride;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int g = 32 * k + lane;
                if (g < G) s[k] += ss[g];
            }
        }
        float m = s[0];
#pragma unroll
        for (int k = 1; k < K; ++k) m = fmaxf(m, s[k]);
#pragma unroll
        for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(full, m, o));
        const float nm = -m * kLog2e;
        __syncwarp();
#pragma unroll
        for (int k = 0; k < K; ++k) lik[33 * k + lane] = mufu_ex2(fmaf(s[k], kLog2e, nm));  // skew(32k + lane)
        __syncwarp();
        float part = 0.f;
#pragma unroll
        for (int kk = 0; kk < K; ++kk) part += lik[seg0 + kk];
        float incl = part;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float v = __shfl_up_sync(full, incl, o);
            if (lane >= o) incl += v;
        }
        const float total = __shfl_sync(full, incl, 31);
        const float t0 = total * a.u[n];
        const unsigned hit = __ballot_sync(full, incl >= t0 && lane * K < G);
        int idx = G - 1;
        if (hit) {
            const int owner = __ffs(hit) - 1;
            const float resid = t0 - __shfl_sync(full, incl - part, owner);  // draw left inside the segment
            // K-lane inclusive scan over the owner's segment: first element reaching the residual
            const int i = owner * K + (lane < K ? lane : K - 1);
            float c = (lane < K && i < G) ? lik[i + (i >> 5)] : 0.f;
#pragma unroll
            for (int o = 1; o < K; o <<= 1) {
                const float v = __shfl_up_sync(full, c, o);
                if (lane >= o) c += v;
            }
            const unsigned h2 = __ballot_sync(full, lane < K && c >= resid);
            const int last = min(G, owner * K + K) - 1;
            idx = h2 ? min(owner * K + __ffs(h2) - 1, last) : last;
        }
        if (lane == 0) a.assign[n] = idx;
    }
}

template <int K>
static int launch_gather_fast(dist_b200_ctx *ctx, const GatherArgs &a, cudaStream_t s) {
    auto kern = gather_rows_fast_kernel<K>;
    int per_sm = 0;
    DISTB200_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kFastWarps * 32, 0));
    if (per_sm < 1) per_sm = 1;
    const size_t want = (a.N + kFastWarps - 1) / kFastWarps;
    const size_t cap = static_cast<size_t>(ctx->sm_count) * per_sm;
    kern<<<static_cast<unsigned>(want < cap ? want : cap), kFastWarps * 32, 0, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("gather_rows_fast launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

static int launch_gather(dist_b200_ctx *ctx, const GatherArgs &a, cudaStream_t s) {
    if (a.N == 0 || a.G == 0) return DIST_B200_OK;
    if (a.assign && !a.scores_out && !a.accumulate && a.G <= 1024) {
        const int k = (a.G + 31) / 32;
        if (k <= 1) return launch_gather_fast<1>(ctx, a, s);
        if (k <= 2) return launch_gather_fast<2>(ctx, a, s);
        if (k <= 4) return launch_gather_fast<4>(ctx, a, s);
        if (k <= 8) return launch_gather_fast<8>(ctx, a, s);
        if (k <= 16) return launch_gather_fast<16>(ctx, a, s);
        return launch_gather_fast<32>(ctx, a, s);
    }
    const int seg = (a.G + 31) / 32;
    const size_t row_bytes = sizeof(float) * (static_cast<size_t>(32 * seg) + seg + 1);
    int threads = kGatherThreadsMax;
    while (threads > 32 && row_bytes * (threads / 32) > 200 * 1024) threads >>= 1;
    const size_t smem = a.assign ? row_bytes * (threads / 32) : 0;
    if (smem > 227 * 1024) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "gather_rows: G too large for one warp's row buffer");
    DISTB200_CUDA(ctx, cudaFuncSetAttribute(gather_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            static_cast<int>(smem > 48 * 1024 ? smem : 48 * 1024)));
    int per_sm = 0;
    DISTB200_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gather_rows_kernel, threads, smem));
    if (per_sm < 1) per_sm = 1;
    const size_t warps = threads / 32;
    const size_t want = (a.N + warps - 1) / warps;
    const size_t cap = static_cast<size_t>(ctx->sm_count) * per_sm;
    const unsigned grid = static_cast<unsigned>(want < cap ? want : cap);
    gather_rows_kernel<<<grid, threads, smem, s>>>(a, seg);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("gather_rows launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

int launch_gather_rows(dist_b200_ctx *ctx, const dist_b200_feature *f, const void *column, size_t N,
                       const float *prior, const float *u, int32_t *assign, float *scores, int accumulate,
                       cudaStream_t s) {
    GatherArgs a{};
    a.G = f->G;
    a.V = f->dim;
    a.keys_dense = f->keys_dense ? 1 : 0;
    a.accumulate = accumulate;
    a.N = N;
    a.table = static_cast<const float *>(f->params);
    a.values = static_cast<const uint32_t *>(column);
    a.keys = f->keys_dev;
    a.key_rows = f->key_rows_dev;
    a.prior = prior;
    a.u = u;
    a.assign = assign;
    a.scores_out = scores;
    a.n_slots = 1;
    return launch_gather(ctx, a, s);
}

int launch_sample_scores(dist_b200_ctx *ctx, const float *scores, size_t N, int G, const float *u,
                         int32_t *assign, cudaStream_t s, int n_slots, size_t slot_stride) {
    GatherArgs a{};
    a.G = G;
    a.N = N;
    a.scores_in = scores;
    a.n_slots = n_slots;
    a.slot_stride = slot_stride;
    a.u = u;
    a.assign = assign;
    return launch_gather(ctx, a, s);
}

// logp[n] = log sum_g exp(scores[n][g]): one warp per row, coalesced reads, the row maximum then the sum of exp
constexpr int kLogpWarps = 8;
__global__ void __launch_bounds__(kLogpWarps * 32) logp_scores_kernel(const float *__restrict__ scores, size_t N, int G,
                                                                       float *__restrict__ logp) {
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const size_t step = static_cast<size_t>(gridDim.x) * kLogpWarps;
    for (size_t n = static_cast<size_t>(blockIdx.x) * kLogpWarps + (threadIdx.x >> 5); n < N; n += step) {
        const float *row = scores + n * static_cast<size_t>(G);
        float m = -INFINITY;
        for (int g = lane; g < G; g += 32) m = fmaxf(m, __ldg(row + g));
#pragma unroll
        for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(full, m, o));
        const float nm = fminf(-m * kLog2e, 3.0e38f);  // finite when the whole row is -inf: the sum is then 0
        float sum = 0.f;
        for (int g = lane; g < G; g += 32) sum += mufu_ex2(fmaf(__ldg(row + g), kLog2e, nm));
#pragma unroll
        for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(full, sum, o);
        if (lane == 0) logp[n] = logp_finish(nm, sum);
    }
}

int launch_logp_scores(dist_b200_ctx *ctx, const float *scores, size_t N, int G, float *logp, cudaStream_t s) {
    if (N == 0) return DIST_B200_OK;
    const size_t want = (N + kLogpWarps - 1) / kLogpWarps, cap = static_cast<size_t>(ctx->sm_count) * 16;
    logp_scores_kernel<<<static_cast<unsigned>(want < cap ? want : cap), kLogpWarps * 32, 0, s>>>(scores, N, G, logp);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("logp_scores launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

}  // namespace distb200
