// regroup.cu -- group births and deaths in one batch (dist_b200_regroup_batch): the survivors' ids, the relabelled
// assignments and the compacted per-group arrays of many features, with launch counts that do not depend on how
// many groups die or are born.
#include <algorithm>

#include "common.cuh"

namespace distb200 {

namespace {

constexpr int kRemapThreads = 1024;

// One block scans counts[G] in chunks of kRemapThreads groups: a group is alive iff counts[g] > 0, and the survivors
// keep their order.  remap[g] = new id or -1; inv[new] = old id for new < K+, -1 for the n_empty fresh groups;
// counts_out (nullable) = the compacted counts followed by n_empty zeros; *k_out = K+.
__global__ void __launch_bounds__(kRemapThreads) regroup_remap_kernel(const int32_t *__restrict__ counts, int G, int n_empty,
                                                                      int32_t *__restrict__ remap, int32_t *__restrict__ inv,
                                                                      int32_t *__restrict__ counts_out, int32_t *__restrict__ k_out) {
    __shared__ int warp_sum[kRemapThreads / 32];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    int base = 0;  // survivors before this chunk
    for (int g0 = 0; g0 < G; g0 += kRemapThreads) {
        const int g = g0 + t;
        const int c = g < G ? counts[g] : 0;
        const bool alive = c > 0;
        const unsigned ballot = __ballot_sync(0xffffffffu, alive);
        if (lane == 0) warp_sum[warp] = __popc(ballot);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < kRemapThreads / 32; ++w) {
            const int v = warp_sum[w];
            before += w < warp ? v : 0;
            total += v;
        }
        const int id = base + before + __popc(ballot & ((1u << lane) - 1u));
        if (g < G) remap[g] = alive ? id : -1;
        if (alive) {
            inv[id] = g;
            if (counts_out) counts_out[id] = c;
        }
        base += total;
        __syncthreads();  // warp_sum is rewritten by the next chunk
    }
    for (int i = t; i < n_empty; i += kRemapThreads) {
        inv[base + i] = -1;
        if (counts_out) counts_out[base + i] = 0;
    }
    if (t == 0) *k_out = base;
}

// assign[n] <- remap[assign[n]]; negative ids stay, ids >= G become -1.  remap is staged in shared memory when it fits.
template <bool kSmem>
__global__ void regroup_relabel_kernel(int32_t *__restrict__ assign, size_t N, const int32_t *__restrict__ remap, int G) {
    extern __shared__ int32_t s_remap[];
    const int32_t *map = remap;
    if (kSmem) {
        for (int g = threadIdx.x; g < G; g += blockDim.x) s_remap[g] = remap[g];
        __syncthreads();
        map = s_remap;
    }
    for (size_t n = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; n < N; n += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int32_t a = assign[n];
        if (a < 0) continue;
        assign[n] = a < G ? map[a] : -1;
    }
}

// Per-group arrays of many features, `rows` groups each.  Gather (b.inv != NULL): dst row r is src row inv[r] for
// r < K+ and zeros from K+ on.  Copy (b.inv == NULL): dst row r is src row r.  Never in place.
__global__ void regroup_arrays_kernel(const RegroupBatch b) {
    const RegroupArray &a = b.a[blockIdx.y];
    const size_t w = a.words, total = static_cast<size_t>(b.rows) * w;
    const int K = b.inv ? *b.k : b.rows;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t r = i / w, e = i - r * w;
        uint32_t v = 0;
        if (static_cast<int>(r) < K) v = a.src[(b.inv ? static_cast<size_t>(b.inv[r]) : r) * w + e];
        a.dst[i] = v;
    }
}

}  // namespace

int launch_regroup_remap(dist_b200_ctx *ctx, const int32_t *counts, int G, int n_empty, int32_t *remap, int32_t *inv,
                         int32_t *counts_out, int32_t *k_out, cudaStream_t s) {
    regroup_remap_kernel<<<1, kRemapThreads, 0, s>>>(counts, G, n_empty, remap, inv, counts_out, k_out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("regroup remap launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

int launch_regroup_relabel(dist_b200_ctx *ctx, int32_t *assign, size_t N, const int32_t *remap, int G, cudaStream_t s) {
    if (N == 0) return DIST_B200_OK;
    constexpr int kThreads = 256;
    const size_t want = (N + kThreads - 1) / kThreads;
    const unsigned grid = static_cast<unsigned>(std::min<size_t>(want, static_cast<size_t>(ctx->sm_count) * 8));
    const size_t sb = sizeof(int32_t) * static_cast<size_t>(G);
    if (sb <= 48 * 1024) regroup_relabel_kernel<true><<<grid, kThreads, sb, s>>>(assign, N, remap, G);
    else regroup_relabel_kernel<false><<<grid, kThreads, 0, s>>>(assign, N, remap, G);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("regroup relabel launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

int launch_regroup_arrays(dist_b200_ctx *ctx, const RegroupBatch &b, cudaStream_t s) {
    if (b.n == 0 || b.rows == 0) return DIST_B200_OK;
    constexpr int kThreads = 256;
    size_t most = 0;
    for (int i = 0; i < b.n; ++i) most = std::max(most, static_cast<size_t>(b.rows) * b.a[i].words);
    // enough blocks per array to cover the largest one, bounded so that a long list does not queue a huge grid
    const size_t cap = std::max<size_t>(1, static_cast<size_t>(ctx->sm_count) * 16 / b.n);
    const unsigned gx = static_cast<unsigned>(std::min((most + kThreads - 1) / kThreads, cap));
    regroup_arrays_kernel<<<dim3(gx, b.n), kThreads, 0, s>>>(b);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("regroup arrays launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

}  // namespace distb200
