// stats.cu -- batched Group::add_value on the device (SURVEY.md §8f, first "next" row).
//
// The reference adds one value to one group at a time (nich.hpp:125-133, gp.hpp:109-116, bb.hpp:102-107,
// dd.hpp:123-130, dpd.hpp:188-196) and refreshes that group's cache entries (update_group).  After a
// batched score + sample, the N sampled assignments are folded into the device-resident group statistics
// with one segmented reduction (shared-memory accumulators per block, then global atomics), merged into
// the stored statistics, and the caches are rebuilt by the same prep code update_all uses -- the
// score -> sample -> update loop never returns to the host.  All pooled features (nich / gp / bb) of one
// kind go through ONE accumulate launch (grid.y = feature) and ONE merge + cache-rebuild launch (prep.cu).
//
//   nich : per group (m, sum x, sum x^2) in double -> (m, mean_b, ctv_b) -> merged with the stored
//          (count, mean, count_times_variance) by the pairwise formula of Group::merge (nich.hpp:167-179).
//          The reference's one-at-a-time Welford updates round differently: statistics agree to ~1e-6
//          relative, counts exactly.
//   gp   : count += m, sum += sum x (uint32, wraps like the reference's)   bb : heads / tails += counts (exact)
//   dd   : counts[g][x] += 1 (exact)                            dpd: counts[g][row(x)] += 1 (exact; OTHER skipped)
#include "common.cuh"

namespace distb200 {

constexpr int kAddThreads = 256;
constexpr int kAddSmemGroups = 2048;   // groups whose accumulators fit in shared memory (24 B / group)
constexpr int kCountSmemBins = 12288;  // int bins of a shared-memory histogram (48 KB)
constexpr int kPeelRounds = 4;         // popular groups combined in registers per warp row

size_t add_rows_acc_bytes(int G) {
    // cnt_a | cnt_b | sum_x | sum_xx, each G entries, 256-byte aligned regions
    const size_t g = static_cast<size_t>(G);
    return 2 * ((g * 4 + 255) / 256 * 256) + 2 * ((g * 8 + 255) / 256 * 256);
}

// ---------------------------------------------------------------------------------------------
// Row streaming shared by the kernels below: every thread takes groups of four consecutive rows with
// 16-byte (assign, 4-byte columns) / 4-byte (uint8 columns) loads, two groups in flight before the first
// atomic, so the loop is bound by the atomics and not by two dependent DRAM latencies per row.  kVec
// needs 16-byte aligned assign / column pointers (the launcher checks); the scalar form takes anything.
template <typename T>
__device__ __forceinline__ void load4(const T *p, size_t q, T (&v)[4]) {
    if constexpr (sizeof(T) == 4) {
        const uint4 r = __ldg(reinterpret_cast<const uint4 *>(p) + q);
        v[0] = reinterpret_cast<const T &>(r.x);
        v[1] = reinterpret_cast<const T &>(r.y);
        v[2] = reinterpret_cast<const T &>(r.z);
        v[3] = reinterpret_cast<const T &>(r.w);
    } else {
        static_assert(sizeof(T) == 1, "4- or 1-byte columns");
        const uint32_t r = __ldg(reinterpret_cast<const uint32_t *>(p) + q);
        v[0] = static_cast<T>(r & 0xff);
        v[1] = static_cast<T>((r >> 8) & 0xff);
        v[2] = static_cast<T>((r >> 16) & 0xff);
        v[3] = static_cast<T>(r >> 24);
    }
}

// kMask: `observed` (NULL = every row) holds one bit per row (dist_b200.h, missing cells); a row whose bit is 0 reaches `fn`
// with group -1, which every caller skips -- so the row's cell is left out of this feature only.  Four consecutive rows
// from a multiple of 4 share one mask word.
__device__ __forceinline__ int32_t observed_or_skip(const uint32_t *observed, size_t n, int32_t g) {
    return !observed || ((__ldg(observed + (n >> 5)) >> (n & 31)) & 1u) ? g : -1;
}
__device__ __forceinline__ void mask4(const uint32_t *observed, size_t q, int32_t (&g)[4]) {
    if (!observed) return;
    const uint32_t bits = __ldg(observed + ((4 * q) >> 5)) >> ((4 * q) & 31);
#pragma unroll
    for (int k = 0; k < 4; ++k) g[k] = (bits >> k) & 1u ? g[k] : -1;
}

template <bool kVec, bool kMask = false, typename T, typename Fn>
__device__ __forceinline__ void for_each_row(const int32_t *__restrict__ assign, const T *__restrict__ col, size_t N, int threads,
                                             Fn &&fn, const uint32_t *__restrict__ observed = nullptr) {
    const size_t stride = static_cast<size_t>(gridDim.x) * threads;
    const size_t first = static_cast<size_t>(blockIdx.x) * threads + threadIdx.x;
    if constexpr (kVec) {
        const size_t n4 = N / 4;
        size_t q = first;
        for (; q + stride < n4; q += 2 * stride) {
            int32_t g0[4], g1[4];
            T x0[4], x1[4];
            load4(assign, q, g0);
            load4(assign, q + stride, g1);
            load4(col, q, x0);
            load4(col, q + stride, x1);
            if constexpr (kMask) {
                mask4(observed, q, g0);
                mask4(observed, q + stride, g1);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) fn(g0[k], x0[k]);
#pragma unroll
            for (int k = 0; k < 4; ++k) fn(g1[k], x1[k]);
        }
        if (q < n4) {
            int32_t g0[4];
            T x0[4];
            load4(assign, q, g0);
            load4(col, q, x0);
            if constexpr (kMask) mask4(observed, q, g0);
#pragma unroll
            for (int k = 0; k < 4; ++k) fn(g0[k], x0[k]);
        }
        const size_t n = 4 * n4 + first;  // the last N % 4 rows
        if constexpr (kMask) {
            if (n < N) fn(observed_or_skip(observed, n, assign[n]), col[n]);
        } else {
            if (n < N) fn(assign[n], col[n]);
        }
    } else {
        if constexpr (kMask) {
            for (size_t n = first; n < N; n += stride) fn(observed_or_skip(observed, n, assign[n]), col[n]);
        } else {
            for (size_t n = first; n < N; n += stride) fn(assign[n], col[n]);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// pooled models: grid (row tiles, features)
// kMask: `observed` (NULL = fully observed) is the mask of feature d[blockIdx.y]
template <bool kSmem, bool kVec, bool kMask>
__device__ __forceinline__ void add_rows_pooled(const AddBatch &b, const uint32_t *observed) {
    extern __shared__ __align__(8) unsigned char add_smem[];
    const int G = b.G;
    const AddDesc &d = b.d[blockIdx.y];
    char *acc = b.acc + b.acc_stride * blockIdx.y;
    const size_t ci = (static_cast<size_t>(G) * 4 + 255) / 256 * 256, di = (static_cast<size_t>(G) * 8 + 255) / 256 * 256;
    int *g_ca = reinterpret_cast<int *>(acc);
    int *g_cb = reinterpret_cast<int *>(acc + ci);
    double *g_x = reinterpret_cast<double *>(acc + 2 * ci);
    double *g_xx = reinterpret_cast<double *>(acc + 2 * ci + di);
    double *s_x = reinterpret_cast<double *>(add_smem);
    double *s_xx = s_x + G;
    int *s_ca = reinterpret_cast<int *>(s_xx + G);
    int *s_cb = s_ca + G;
    const int model = d.model;
    if (kSmem) {
        for (int g = threadIdx.x; g < G; g += kAddThreads) {
            s_x[g] = 0.0;
            s_xx[g] = 0.0;
            s_ca[g] = 0;
            s_cb[g] = 0;
        }
        __syncthreads();
    }
    int *ca = kSmem ? s_ca : g_ca, *cb = kSmem ? s_cb : g_cb;
    double *ax = kSmem ? s_x : g_x, *axx = kSmem ? s_xx : g_xx;
    // Assignments under a CRP prior are skewed: many lanes of a warp hit the same group.  Integer
    // shared-memory atomics take that well (measured, profiles/experiments/add_rows_modes.txt: 1.1x for a
    // Zipf assignment, 2x with 85% of the rows in two groups; match.any or ballot-based combining costs more
    // than it saves), but the double sums are CAS loops that degrade 9-14x.  For nich the lanes of the
    // warp's popular groups are therefore combined in registers first (masked butterfly, one atomic per
    // peeled group); lanes of unpopular groups go direct.
    if (model == DIST_B200_NICH) {
        for_each_row<kVec, kMask>(b.assign, static_cast<const float *>(d.column), b.N, kAddThreads, [&](int g, float xf) {
            const unsigned active = __activemask();
            const int lane = threadIdx.x & 31;
            bool pending = g >= 0 && g < G;
            const double x = static_cast<double>(xf), xx = x * x;
            if (active == 0xffffffffu) {
#pragma unroll 1
                for (int round = 0; round < kPeelRounds; ++round) {
                    const unsigned todo = __ballot_sync(active, pending);
                    if (!todo) break;
                    const int leader = __ffs(todo) - 1;
                    const int gl = __shfl_sync(active, g, leader);
                    const bool mine = pending && g == gl;
                    const unsigned grp = __ballot_sync(active, mine);
                    if (__popc(grp) < 4) break;  // the double butterfly costs ~20 shuffles: only for heavy groups
                    double sx = mine ? x : 0.0, sxx = mine ? xx : 0.0;
#pragma unroll
                    for (int o = 16; o; o >>= 1) {
                        sx += __shfl_xor_sync(active, sx, o);
                        sxx += __shfl_xor_sync(active, sxx, o);
                    }
                    if (lane == leader) {
                        atomicAdd(&ca[gl], __popc(grp));
                        atomicAdd(&ax[gl], sx);
                        atomicAdd(&axx[gl], sxx);
                    }
                    if (mine) pending = false;
                }
            }
            if (pending) {
                atomicAdd(&ca[g], 1);
                atomicAdd(&ax[g], x);
                atomicAdd(&axx[g], xx);
            }
        }, observed);
    } else if (model == DIST_B200_GP || model == DIST_B200_BNB) {
        for_each_row<kVec, kMask>(b.assign, static_cast<const uint32_t *>(d.column), b.N, kAddThreads, [&](int g, uint32_t x) {
            if (g < 0 || g >= G) return;
            atomicAdd(&ca[g], 1);
            atomicAdd(reinterpret_cast<unsigned int *>(&cb[g]), x);
        }, observed);
    } else {  // bb
        for_each_row<kVec, kMask>(b.assign, static_cast<const uint8_t *>(d.column), b.N, kAddThreads, [&](int g, uint8_t x) {
            if (g < 0 || g >= G) return;
            atomicAdd(x != 0 ? &ca[g] : &cb[g], 1);
        }, observed);
    }
    if (kSmem) {
        __syncthreads();
        for (int g = threadIdx.x; g < G; g += kAddThreads) {
            if (s_ca[g]) atomicAdd(&g_ca[g], s_ca[g]);
            if (s_cb[g]) atomicAdd(&g_cb[g], s_cb[g]);
            if (model == DIST_B200_NICH && s_ca[g]) {
                atomicAdd(&g_x[g], s_x[g]);
                atomicAdd(&g_xx[g], s_xx[g]);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------

template <bool kSmem, bool kVec>
__global__ void __launch_bounds__(kAddThreads) add_rows_pooled_kernel(const AddBatch b) {
    add_rows_pooled<kSmem, kVec, false>(b, nullptr);
}

// the same with per-feature observed masks (masks.m[f] for feature d[f])
template <bool kSmem, bool kVec>
__global__ void __launch_bounds__(kAddThreads) add_rows_pooled_masked_kernel(const AddBatch b, const AddMasks masks) {
    add_rows_pooled<kSmem, kVec, true>(b, masks.m[blockIdx.y]);
}

// ---------------------------------------------------------------------------------------------
// dd / dpd: counts[g][row] += 1 in place; a shared-memory histogram when the whole table fits
struct CountArgs {
    int model, G, dim, keys_dense, sign;
    size_t N;
    const void *column;
    const int32_t *assign;
    int32_t *counts;
    const uint32_t *keys;
    const int *key_rows;
};

__device__ __forceinline__ int dpd_row(const CountArgs &a, uint32_t value) {
    if (a.keys_dense) return value < static_cast<uint32_t>(a.dim) ? static_cast<int>(value) : -1;
    int lo = 0, hi = a.dim;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a.keys[mid] < value) lo = mid + 1;
        else hi = mid;
    }
    return (lo < a.dim && a.keys[lo] == value) ? a.key_rows[lo] : -1;
}

template <bool kSmem, bool kVec, bool kMask>
__device__ __forceinline__ void add_rows_counts(const CountArgs &a, const uint32_t *observed) {
    extern __shared__ int32_t bins[];
    const int cells = a.G * a.dim;
    if (kSmem) {
        for (int i = threadIdx.x; i < cells; i += kAddThreads) bins[i] = 0;
        __syncthreads();
    }
    int32_t *dst = kSmem ? bins : a.counts;
    // dd values are int32 ids, dpd values uint32 keys: both stream as uint32
    for_each_row<kVec, kMask>(a.assign, static_cast<const uint32_t *>(a.column), a.N, kAddThreads, [&](int g, uint32_t x) {
        int cell = -1;
        if (g >= 0 && g < a.G) {
            if (a.model == DIST_B200_DD) {
                if (x < static_cast<uint32_t>(a.dim)) cell = g * a.dim + static_cast<int>(x);
            } else {
                const int r = dpd_row(a, x);
                if (r >= 0) cell = g * a.dim + r;
            }
        }
        if (cell < 0) return;
        if (a.sign > 0) atomicAdd(&dst[cell], 1);
        else atomicAdd(&dst[cell], -1);
    }, observed);
    if (kSmem) {
        __syncthreads();
        for (int i = threadIdx.x; i < cells; i += kAddThreads)
            if (bins[i]) atomicAdd(&a.counts[i], bins[i]);
    }
}

template <bool kSmem, bool kVec>
__global__ void __launch_bounds__(kAddThreads) add_rows_counts_kernel(const CountArgs a) {
    add_rows_counts<kSmem, kVec, false>(a, nullptr);
}

template <bool kSmem, bool kVec>
__global__ void __launch_bounds__(kAddThreads) add_rows_counts_masked_kernel(const CountArgs a, const uint32_t *observed) {
    add_rows_counts<kSmem, kVec, true>(a, observed);
}

// kMask: rows whose bit in `observed` is 0 are not counted (the niw histogram of a feature with missing cells)
template <bool kSmem, bool kVec, bool kMask>
__device__ __forceinline__ void count_assignments(const int32_t *__restrict__ assign, size_t N, int G, int32_t *__restrict__ counts,
                                                  const uint32_t *observed) {
    extern __shared__ int32_t bins[];
    if (kSmem) {
        for (int i = threadIdx.x; i < G; i += kAddThreads) bins[i] = 0;
        __syncthreads();
    }
    int32_t *dst = kSmem ? bins : counts;
    for_each_row<kVec, kMask>(assign, assign, N, kAddThreads, [&](int g, int) {
        if (g >= 0 && g < G) atomicAdd(&dst[g], 1);
    }, observed);
    if (kSmem) {
        __syncthreads();
        for (int i = threadIdx.x; i < G; i += kAddThreads)
            if (bins[i]) atomicAdd(&counts[i], bins[i]);
    }
}

template <bool kSmem, bool kVec>
__global__ void __launch_bounds__(kAddThreads) count_assignments_kernel(const int32_t *__restrict__ assign, size_t N, int G,
                                                                        int32_t *__restrict__ counts) {
    count_assignments<kSmem, kVec, false>(assign, N, G, counts, nullptr);
}

template <bool kSmem, bool kVec>
__global__ void __launch_bounds__(kAddThreads) count_observed_kernel(const int32_t *__restrict__ assign, size_t N, int G,
                                                                     int32_t *__restrict__ counts, const uint32_t *observed) {
    count_assignments<kSmem, kVec, true>(assign, N, G, counts, observed);
}

// ---------------------------------------------------------------------------------------------
static bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static unsigned row_tiles(const dist_b200_ctx *ctx, size_t N, int per_sm, int split) {
    // enough blocks to fill the machine, few enough that the per-block flush stays negligible
    const size_t want = (N + kAddThreads - 1) / kAddThreads;
    size_t cap = static_cast<size_t>(ctx->sm_count) * per_sm / (split > 0 ? split : 1);
    if (cap < 1) cap = 1;
    return static_cast<unsigned>(want < cap ? want : cap);
}

// masks (may be NULL): the batch's observed masks; a batch whose masks are all NULL takes the unmasked kernel
int launch_add_rows_pooled(dist_b200_ctx *ctx, const AddBatch &b_in, cudaStream_t s, const AddMasks *masks) {
    if (b_in.G == 0 || b_in.n == 0) return DIST_B200_OK;
    const AddBatch &b = b_in;
    // zeroed BEFORE the empty-batch early-out: the merge / pack that follows an empty batch (a rank whose row
    // shard is empty) must see zeros, not the previous batch's sums
    DISTB200_CUDA(ctx, cudaMemsetAsync(b.acc, 0, b.acc_stride * b.n, s));
    if (b.N == 0) return DIST_B200_OK;
    const dim3 grid(row_tiles(ctx, (b.N + 3) / 4, 8, b.n), b.n);
    bool vec = aligned16(b.assign);
    for (int i = 0; i < b.n; ++i) vec = vec && aligned16(b.d[i].column);
    const bool smem = b.G <= kAddSmemGroups;
    const size_t sb = smem ? static_cast<size_t>(b.G) * 24 : 0;
    bool masked = false;
    for (int i = 0; masks && i < b.n; ++i) masked = masked || masks->m[i];
    if (masked) {
        if (smem && vec) add_rows_pooled_masked_kernel<true, true><<<grid, kAddThreads, sb, s>>>(b, *masks);
        else if (smem) add_rows_pooled_masked_kernel<true, false><<<grid, kAddThreads, sb, s>>>(b, *masks);
        else if (vec) add_rows_pooled_masked_kernel<false, true><<<grid, kAddThreads, 0, s>>>(b, *masks);
        else add_rows_pooled_masked_kernel<false, false><<<grid, kAddThreads, 0, s>>>(b, *masks);
    } else if (smem && vec) add_rows_pooled_kernel<true, true><<<grid, kAddThreads, sb, s>>>(b);
    else if (smem) add_rows_pooled_kernel<true, false><<<grid, kAddThreads, sb, s>>>(b);
    else if (vec) add_rows_pooled_kernel<false, true><<<grid, kAddThreads, 0, s>>>(b);
    else add_rows_pooled_kernel<false, false><<<grid, kAddThreads, 0, s>>>(b);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("add_rows launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

// dst: the count table to update (nullptr = the feature's own statistics); observed: the feature's mask, or NULL
int launch_add_rows_counts(dist_b200_ctx *ctx, dist_b200_feature *f, const void *column, const int32_t *assign, size_t N,
                           int sign, cudaStream_t s, int32_t *dst, const uint32_t *observed) {
    if (N == 0 || f->G == 0) return DIST_B200_OK;
    CountArgs a{};
    a.model = f->model;
    a.G = f->G;
    a.dim = f->dim;
    a.keys_dense = f->keys_dense ? 1 : 0;
    a.sign = sign;
    a.N = N;
    a.column = column;
    a.assign = assign;
    a.counts = dst ? dst : reinterpret_cast<int32_t *>(f->stats[0]);  // dd: counts[G][dim]; dpd: counts[G][V]
    a.keys = f->keys_dev;
    a.key_rows = f->key_rows_dev;
    const size_t cells = static_cast<size_t>(f->G) * f->dim;
    const bool vec = aligned16(assign) && aligned16(column);
    if (observed) {
        const bool smem = cells <= kCountSmemBins;
        const unsigned grid = row_tiles(ctx, (N + 3) / 4, smem ? 4 : 8, 1);
        const size_t sb = smem ? cells * 4 : 0;
        if (smem && vec) add_rows_counts_masked_kernel<true, true><<<grid, kAddThreads, sb, s>>>(a, observed);
        else if (smem) add_rows_counts_masked_kernel<true, false><<<grid, kAddThreads, sb, s>>>(a, observed);
        else if (vec) add_rows_counts_masked_kernel<false, true><<<grid, kAddThreads, 0, s>>>(a, observed);
        else add_rows_counts_masked_kernel<false, false><<<grid, kAddThreads, 0, s>>>(a, observed);
    } else if (cells <= kCountSmemBins) {
        const unsigned grid = row_tiles(ctx, (N + 3) / 4, 4, 1);
        if (vec) add_rows_counts_kernel<true, true><<<grid, kAddThreads, cells * 4, s>>>(a);
        else add_rows_counts_kernel<true, false><<<grid, kAddThreads, cells * 4, s>>>(a);
    } else {
        const unsigned grid = row_tiles(ctx, (N + 3) / 4, 8, 1);
        if (vec) add_rows_counts_kernel<false, true><<<grid, kAddThreads, 0, s>>>(a);
        else add_rows_counts_kernel<false, false><<<grid, kAddThreads, 0, s>>>(a);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("add_rows launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

// Row-shard exchange of a count table (dd / dpd): the rank's delta counts travel as doubles (integers are exact in
// them), so that one float64 all-reduce carries the pooled accumulators and the tables alike.
__global__ void counts_to_doubles_kernel(const int32_t *__restrict__ src, double *__restrict__ dst, size_t n) {
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x)
        dst[i] = static_cast<double>(src[i]);
}
__global__ void merge_counts_kernel(int32_t *__restrict__ counts, const double *__restrict__ delta, size_t n, int sign) {
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const long long d = llrint(delta[i]);
        if (d) counts[i] += static_cast<int32_t>(sign > 0 ? d : -d);
    }
}

int launch_counts_to_doubles(dist_b200_ctx *ctx, const int32_t *src, double *dst, size_t n, cudaStream_t s) {
    if (n == 0) return DIST_B200_OK;
    const size_t want = (n + 255) / 256, cap = static_cast<size_t>(ctx->sm_count) * 8;
    counts_to_doubles_kernel<<<static_cast<unsigned>(want < cap ? want : cap), 256, 0, s>>>(src, dst, n);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("counts_to_doubles launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

int launch_merge_counts(dist_b200_ctx *ctx, int32_t *counts, const double *delta, size_t n, int sign, cudaStream_t s) {
    if (n == 0) return DIST_B200_OK;
    const size_t want = (n + 255) / 256, cap = static_cast<size_t>(ctx->sm_count) * 8;
    merge_counts_kernel<<<static_cast<unsigned>(want < cap ? want : cap), 256, 0, s>>>(counts, delta, n, sign);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("merge_counts launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

int launch_count_assignments(dist_b200_ctx *ctx, const int32_t *assign, size_t N, int G, int32_t *counts, int accumulate,
                             cudaStream_t s, const uint32_t *observed) {
    if (!accumulate) DISTB200_CUDA(ctx, cudaMemsetAsync(counts, 0, sizeof(int32_t) * G, s));
    if (N == 0) return DIST_B200_OK;
    const unsigned grid = row_tiles(ctx, (N + 3) / 4, 4, 1);
    const bool vec = aligned16(assign), smem = G <= kCountSmemBins;
    const size_t sb = smem ? static_cast<size_t>(G) * 4 : 0;
    if (observed) {
        if (smem && vec) count_observed_kernel<true, true><<<grid, kAddThreads, sb, s>>>(assign, N, G, counts, observed);
        else if (smem) count_observed_kernel<true, false><<<grid, kAddThreads, sb, s>>>(assign, N, G, counts, observed);
        else if (vec) count_observed_kernel<false, true><<<grid, kAddThreads, 0, s>>>(assign, N, G, counts, observed);
        else count_observed_kernel<false, false><<<grid, kAddThreads, 0, s>>>(assign, N, G, counts, observed);
    } else if (smem && vec) count_assignments_kernel<true, true><<<grid, kAddThreads, sb, s>>>(assign, N, G, counts);
    else if (smem) count_assignments_kernel<true, false><<<grid, kAddThreads, sb, s>>>(assign, N, G, counts);
    else if (vec) count_assignments_kernel<false, true><<<grid, kAddThreads, 0, s>>>(assign, N, G, counts);
    else count_assignments_kernel<false, false><<<grid, kAddThreads, 0, s>>>(assign, N, G, counts);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("count_assignments launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

}  // namespace distb200
