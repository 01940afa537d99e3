// table_rows.cu -- single-feature kernels for the models whose score is a TABLE LOOKUP:
//   DirichletProcessDiscrete  scores_[value][g] - scores_shift_[g], OTHER row for unseen values (dpd.hpp:517-543)
//   DirichletDiscrete         scores_[value][g] - scores_shift_[g]                             (dd.hpp:433-445)
//   BetaBernoulli             value ? heads_scores_[g] : tails_scores_[g]                      (bb.hpp:303-313)
// followed by sample_from_scores_overwrite (random.hpp:360-366, random.cc:94-106).
//
// (1) table_rows_kernel -- the full per-row evaluation, one WARP per row, everything in registers.
//     Per call the dpd table is re-laid out (table_hot_fold_kernel, O(V G): a few us at c4) into a "hot" copy
//       hot[v][p(g)] = (prior[g] + scores_[v][g] - shift[g] - m_v) * log2(e),   m_v = max_g of that row,
//     i.e. with the clustering prior folded in (as score_rows folds it into its block-private caches) and the row
//     maximum that scores_to_likelihoods subtracts (random.cc:94-106) already taken, so a cell is ONE MUFU.EX2.
//     The physical order p(g) makes a coalesced LDG.128 hand every lane a CONTIGUOUS segment of logical groups
//     (lane L owns groups [L*seg, (L+1)*seg)), so the reference's left-to-right walk needs no shared-memory
//     transpose: per row 4 x LDG.128 per lane (G = 512), 16 MUFU.EX2, one 5-step inclusive scan over the lane
//     sums, one vote, and the owning lane's walk over its registers.  The 32 rows of a warp iteration load their
//     values / uniforms with one coalesced load and store their indices with one coalesced store.
//     Bound: 1 MUFU.EX2 + 4 B of L2 gather per cell (the 8.4 MB table of c4 is L2-resident).
//
// (2) value_cdf_* -- SURVEY.md 8(d) "algorithmic shortcut": with frozen statistics and ONE table feature the
//     whole likelihood vector of a row depends only on its value, so it is evaluated once per distinct value
//     (V+1 rows), stored as inclusive prefix sums in an 8-ary search tree (one 32-byte sector per node), and
//     each data row costs three sector reads.  value-group scores/s of this path are reported WITH that flag and
//     beside (1) (bench.py; DIST_B200_OPT_VALUE_CDF = 0 disables it).
#include "common.cuh"

namespace distb200 {

// ------------------------------------------------------------------------------------------------
// value -> table row (OTHER / unseen values -> row V), shared by both kernels
struct KeyMap {
    int V, dense;
    const uint32_t *keys;   // sorted (when !dense)
    const int *key_rows;    // table row of sorted key i
};
__device__ __forceinline__ int key_row(const KeyMap &k, uint32_t value) {
    if (k.dense) return value < static_cast<uint32_t>(k.V) ? static_cast<int>(value) : k.V;
    int lo = 0, hi = k.V;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (k.keys[mid] < value) lo = mid + 1;
        else hi = mid;
    }
    return (lo < k.V && k.keys[lo] == value) ? k.key_rows[lo] : k.V;
}

// ------------------------------------------------------------------------------------------------
// hot layout of a value-major table [R][G]: row stride 32 * seg floats, seg = groups per lane (multiple of 4);
// logical group g = L * seg + 4 k + j  lives at  128 k + 4 L + j ; pads hold -inf (they vanish from max / exp)
__host__ __device__ __forceinline__ int hot_seg(int G) { return ((G + 31) / 32 + 3) / 4 * 4; }
__host__ __device__ __forceinline__ int hot_pos(int g, int seg) {
    const int L = g / seg, w = g - L * seg;
    return 128 * (w >> 2) + 4 * L + (w & 3);
}

// one warp per table row: row maximum of prior + score, then the scaled, max-relative hot row (pads -inf)
__global__ void __launch_bounds__(256) table_hot_fold_kernel(int R, int G, int seg, const float *__restrict__ table,
                                                             const float *__restrict__ prior, float *__restrict__ hot) {
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= R) return;
    const float *src = table + static_cast<size_t>(r) * G;
    float m = -INFINITY;
    for (int g = lane; g < G; g += 32) m = fmaxf(m, (prior ? prior[g] : 0.f) + src[g]);
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    const int stride = 32 * seg;
    float *dst = hot + static_cast<size_t>(r) * stride;
    for (int p = lane; p < stride; p += 32) {
        // inverse of hot_pos: p = 128 k + 4 L + j
        const int k = p >> 7, L = (p >> 2) & 31, j = p & 3;
        const int g = L * seg + 4 * k + j;
        dst[p] = (4 * k + j < seg && g < G) ? ((prior ? prior[g] : 0.f) + src[g] - m) * kLog2e : -INFINITY;
    }
}

size_t table_hot_floats(int R, int G) { return static_cast<size_t>(R) * 32 * hot_seg(G); }

struct TableRowsArgs {
    int G;
    KeyMap km;
    size_t N;
    const float *hot;        // [(V+1)][32 * seg]: (prior + score - row max) * log2 e
    const uint32_t *values;
    const float *u;
    int32_t *assign;
};

constexpr int kTableWarps = 8;

// kStage: only the OWNING lane's segment matters for the walk, yet with the walk inside the row loop all 32 lanes
// execute it (2 instructions per cell).  Staged form: the owner parks its 4 K4 likelihoods and the draw left for them in
// a per-warp shared-memory slot of the row (predicated stores, one lane active), and after the 32 rows of the iteration
// lane i walks row i's slot -- 32 walks in one pass of 4 K4 steps instead of 32 passes (c4: 1.719 -> 1.664 ms, same draws).
// kPoly: of a lane's K4 quads, the first kPoly are exponentiated on the FMA pipe (poly_ex2_pair, numerics.cuh).
template <int K4, bool kStage = true, int kPoly = 0>
__global__ void __launch_bounds__(kTableWarps * 32) table_rows_kernel(const TableRowsArgs a) {
    constexpr int SEG = 4 * K4;
    constexpr int SLOT = SEG + 4;  // floats per staged row: SEG likelihoods + the draw (16-byte aligned, bank-skewed)
    __shared__ __align__(16) float stage_s[kStage ? kTableWarps * 32 * SLOT : 4];
    float *stage = stage_s + (threadIdx.x >> 5) * 32 * SLOT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int G = a.G;
    const unsigned full = 0xffffffffu;
    const size_t stride4 = 32 * K4;  // float4 per table row
    const float4 *hot4 = reinterpret_cast<const float4 *>(a.hot) + lane;
    const size_t step = static_cast<size_t>(gridDim.x) * kTableWarps * 32;
    for (size_t n0 = (static_cast<size_t>(blockIdx.x) * kTableWarps + warp) * 32; n0 < a.N; n0 += step) {
        const size_t n = n0 + lane < a.N ? n0 + lane : a.N - 1;
        const int my_row = key_row(a.km, a.values[n]);
        const float my_u = a.u[n];
        int my_res = 0;
        // always 32 iterations (rows past the end are clamped copies): a compile-time trip count keeps the warp
        // provably converged, so the shuffles / vote / CREDUX need no WARPSYNC guards
#pragma unroll 2
        for (int i = 0; i < 32; ++i) {
            const int r = __shfl_sync(full, my_row, i);
            const float uu = __shfl_sync(full, my_u, i);
            const float4 *src = hot4 + static_cast<size_t>(r) * stride4;
            float s[SEG];
#pragma unroll
            for (int k = 0; k < K4; ++k) {
                const float4 q = __ldg(src + 32 * k);
                if (k < kPoly) {
                    f2_unpack(poly_ex2_pair(f2_pack(q.x, q.y)), s[4 * k + 0], s[4 * k + 1]);
                    f2_unpack(poly_ex2_pair(f2_pack(q.z, q.w)), s[4 * k + 2], s[4 * k + 3]);
                    continue;
                }
                s[4 * k + 0] = mufu_ex2(q.x);  // exp(prior + scores_[v][g] - shift[g] - max)
                s[4 * k + 1] = mufu_ex2(q.y);
                s[4 * k + 2] = mufu_ex2(q.z);
                s[4 * k + 3] = mufu_ex2(q.w);
            }
            float part = 0.f;
#pragma unroll
            for (int j = 0; j < SEG; ++j) part += s[j];
            float incl = part;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const float v = __shfl_up_sync(full, incl, o);
                if (lane >= o) incl += v;
            }
            const float total = __shfl_sync(full, incl, 31);
            const float t0 = total * uu;
            const unsigned hit = __ballot_sync(full, incl >= t0);
            const int owner = hit ? __ffs(hit) - 1 : 31;
            if (kStage) {
                if (lane == owner) {
                    float4 *dst = reinterpret_cast<float4 *>(stage + i * SLOT);
#pragma unroll
                    for (int k = 0; k < K4; ++k) dst[k] = make_float4(s[4 * k], s[4 * k + 1], s[4 * k + 2], s[4 * k + 3]);
                    stage[i * SLOT + SEG] = t0 - (incl - part);
                }
                if (lane == i) my_res = hit ? owner : -1;  // resolved after the loop
                continue;
            }
            // every lane walks its own segment (only the owner's count is used): t -= l[j]; stop at t <= 0
            float t = t0 - (incl - part);
            unsigned neg = 0;
#pragma unroll
            for (int j = 0; j < SEG; ++j) {
                t -= s[j];
                neg += __float_as_uint(t) >> 31;  // LEA.HI: counts t < 0 (an exact +0 continues: a near-tie)
            }
            const int idx = lane * SEG + min(SEG - static_cast<int>(neg), SEG - 1);
            int res = __shfl_sync(full, idx, owner);
            res = hit ? min(res, G - 1) : G - 1;
            if (lane == i) my_res = res;
        }
        if (kStage) {
            __syncwarp();
            const float4 *src = reinterpret_cast<const float4 *>(stage + lane * SLOT);
            float t = stage[lane * SLOT + SEG];
            unsigned neg = 0;
#pragma unroll
            for (int k = 0; k < K4; ++k) {
                const float4 q = src[k];
                t -= q.x;
                neg += __float_as_uint(t) >> 31;
                t -= q.y;
                neg += __float_as_uint(t) >> 31;
                t -= q.z;
                neg += __float_as_uint(t) >> 31;
                t -= q.w;
                neg += __float_as_uint(t) >> 31;
            }
            const int owner = my_res;
            my_res = owner < 0 ? G - 1 : min(owner * SEG + min(SEG - static_cast<int>(neg), SEG - 1), G - 1);
            __syncwarp();  // the slots are rewritten by the next 32 rows
        }
        if (n0 + lane < a.N) a.assign[n0 + lane] = my_res;
    }
}

template <int K4, bool kStage = true, int kPoly = 0>
static int launch_table_rows_k(dist_b200_ctx *ctx, const TableRowsArgs &a, cudaStream_t s) {
    auto kern = table_rows_kernel<K4, kStage, kPoly>;
    int per_sm = 0;
    DISTB200_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kTableWarps * 32, 0));
    if (per_sm < 1) per_sm = 1;
    const size_t want = (a.N + kTableWarps * 32 - 1) / (kTableWarps * 32);
    const size_t cap = static_cast<size_t>(ctx->sm_count) * per_sm;
    kern<<<static_cast<unsigned>(want < cap ? want : cap), kTableWarps * 32, 0, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("table_rows launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

// dpd, sampling only, G <= 1024; DIST_B200_ERR_UNSUPPORTED -> the caller takes the generic gather kernel
int launch_table_rows(dist_b200_ctx *ctx, const dist_b200_feature *f, const void *column, size_t N, const float *prior,
                      const float *u, int32_t *assign, cudaStream_t s) {
    if (N == 0 || f->G == 0) return DIST_B200_OK;
    // the per-call re-layout costs O(V G): only worth it for batches well beyond the table itself
    if (!f->dpd_hot || f->G > 1024 || N < 4 * static_cast<size_t>(f->dim + 1)) return DIST_B200_ERR_UNSUPPORTED;
    {
        const int R = f->dim + 1;
        table_hot_fold_kernel<<<(R + 7) / 8, 256, 0, s>>>(R, f->G, hot_seg(f->G), static_cast<const float *>(f->params), prior, f->dpd_hot);
    }
    TableRowsArgs a{};
    a.G = f->G;
    a.km = KeyMap{f->dim, f->keys_dense ? 1 : 0, f->keys_dev, f->key_rows_dev};
    a.N = N;
    a.hot = f->dpd_hot;
    a.values = static_cast<const uint32_t *>(column);
    a.u = u;
    a.assign = assign;
    // a quarter of a lane's cells (one of its four quads at c4) are exponentiated on the FMA pipe (poly_ex2_pair): with the walk
    // staged the kernel has the issue slots for it -- same-box A/B at c4: 0 / 1 / 2 of 4 quads 1.664 / 1.553 / 1.715 ms.
    // DIST_B200_OPT_TABLE_KERNEL = 2 (A/B runs): walk inside the row loop, every exp2 on the MUFU pipe (G in (384, 512])
    switch (hot_seg(f->G) / 4) {
        case 1: return launch_table_rows_k<1>(ctx, a, s);
        case 2: return launch_table_rows_k<2>(ctx, a, s);
        case 3: return launch_table_rows_k<3>(ctx, a, s);
        case 4:
            if (ctx->opt[DIST_B200_OPT_TABLE_KERNEL] == 2) return launch_table_rows_k<4, false>(ctx, a, s);
            if (ctx->opt[DIST_B200_OPT_EXP_OFFLOAD] == 1) return launch_table_rows_k<4, true, 0>(ctx, a, s);
            return launch_table_rows_k<4, true, 1>(ctx, a, s);
        case 5: return launch_table_rows_k<5, true, 1>(ctx, a, s);
        case 6: return launch_table_rows_k<6, true, 1>(ctx, a, s);
        case 7: return launch_table_rows_k<7, true, 2>(ctx, a, s);
        default: return launch_table_rows_k<8, true, 2>(ctx, a, s);
    }
}

// ------------------------------------------------------------------------------------------------
// (2) per-value CDF trees.
// Tree of one table row: L levels of fan-out 8 over Gp = 8^L >= G leaves.  Level l (1-based) holds 8^l floats:
// entry i = inclusive prefix sum of the likelihoods up to the END of its block of 8^(L-l) groups; pads +inf.
// Levels are stored back to back: offset(l) = 8 + 64 + ... + 8^(l-1) = (8^l - 8) / 7.  total[r] = sum of the row.
struct CdfArgs {
    int model, G, R, L, vdim;
    size_t tree_floats;      // floats per row
    const void *params;      // dpd: table [R][G]; dd: table [g][vdim]; bb: float4 {heads, tails} per group
    const float *prior;
    float *tree;             // [R][tree_floats]
    float *total;            // [R]
};

__device__ __forceinline__ float table_score(const CdfArgs &a, int r, int g) {
    switch (a.model) {
        case DIST_B200_DPD: return static_cast<const float *>(a.params)[static_cast<size_t>(r) * a.G + g];
        case DIST_B200_DD: return static_cast<const float *>(a.params)[static_cast<size_t>(g) * a.vdim + r];
        default: {  // bb: row 1 = heads (value != 0), row 0 = tails
            const float4 q = static_cast<const float4 *>(a.params)[g];
            return r ? q.x : q.y;
        }
    }
}

// one warp per table row: max, likelihoods, inclusive prefix sums (chunks of 32 groups carried left to right),
// then the upper tree levels are strided views of the leaf prefix
__global__ void __launch_bounds__(256) value_cdf_build_kernel(const CdfArgs a) {
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= a.R) return;
    const unsigned full = 0xffffffffu;
    const int G = a.G;
    int Gp = 1;
    for (int l = 0; l < a.L; ++l) Gp *= 8;
    float m = -INFINITY;
    for (int g = lane; g < G; g += 32) m = fmaxf(m, (a.prior ? a.prior[g] : 0.f) + table_score(a, r, g));
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(full, m, o));
    const float nm = -m * kLog2e;
    float *row = a.tree + static_cast<size_t>(r) * a.tree_floats;
    float *leaf = row + (Gp - 8) / 7;  // offset of level L
    float carry = 0.f;
    for (int g0 = 0; g0 < Gp; g0 += 32) {
        const int g = g0 + lane;
        float l = 0.f;
        if (g < G) l = mufu_ex2(fmaf((a.prior ? a.prior[g] : 0.f) + table_score(a, r, g), kLog2e, nm));
        float incl = l;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float v = __shfl_up_sync(full, incl, o);
            if (lane >= o) incl += v;
        }
        incl += carry;
        carry = __shfl_sync(full, incl, 31);
        if (g < Gp) {
            const float p = g < G ? incl : INFINITY;
            leaf[g] = p;
            // upper levels: this leaf closes a block of 8^(L-l) groups when (g + 1) is a multiple of it
            int blk = 8, off = (Gp / 8 - 8) / 7;  // level L-1
            for (int l2 = a.L - 1; l2 >= 1; --l2) {
                if (((g + 1) & (blk - 1)) == 0) row[off + (g + 1) / blk - 1] = p;
                blk *= 8;
                off = (Gp / blk - 8) / 7;
            }
        }
    }
    if (lane == 0) a.total[r] = carry;  // sum over the G real groups (pads contributed 0)
}

struct CdfSampleArgs {
    int G, L;
    KeyMap km;
    size_t N, tree_floats;
    const float *tree, *total;
    const uint32_t *values;  // dpd uint32 / dd int32; bb: bytes (value_bytes = 1)
    int value_bytes;
    const float *u;
    int32_t *assign;
};

// 8 lanes per data row (one 32-byte sector per tree node), 4 rows per warp step, 32 rows per warp iteration
template <int L>
__global__ void __launch_bounds__(256) value_cdf_sample_kernel(const CdfSampleArgs a) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, sub = lane >> 3, l8 = lane & 7;
    const unsigned full = 0xffffffffu;
    const size_t step = static_cast<size_t>(gridDim.x) * (blockDim.x >> 5) * 32;
    for (size_t n0 = (static_cast<size_t>(blockIdx.x) * (blockDim.x >> 5) + warp) * 32; n0 < a.N; n0 += step) {
        const size_t n = n0 + lane < a.N ? n0 + lane : a.N - 1;
        const uint32_t v = a.value_bytes == 1 ? (reinterpret_cast<const uint8_t *>(a.values)[n] ? 1u : 0u) : a.values[n];
        const int my_row = key_row(a.km, v);
        const float my_t = a.u[n] * __ldg(a.total + my_row);
        int my_res = 0;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            const int j = 4 * it + sub;  // the data row (within the 32) this 8-lane group resolves
            const int r = __shfl_sync(full, my_row, j);
            const float t = __shfl_sync(full, my_t, j);
            const float *row = a.tree + static_cast<size_t>(r) * a.tree_floats;
            int idx = 0, off = 0, width = 8;
#pragma unroll
            for (int l = 0; l < L; ++l) {
                const float p = __ldg(row + off + 8 * idx + l8);
                const unsigned lt = (__ballot_sync(full, p < t) >> (8 * sub)) & 0xffu;
                idx = 8 * idx + min(__popc(lt), 7);  // first node whose prefix reaches t (block ends hold the parent's prefix)
                off += width;
                width *= 8;
            }
            const int got = __shfl_sync(full, idx, 8 * (lane & 3));  // lane j <- group j & 3 of iteration j >> 2
            if ((lane >> 2) == it) my_res = got;
        }
        if (n0 + lane < a.N) a.assign[n0 + lane] = min(my_res, a.G - 1);
    }
}

// ------------------------------------------------------------------------------------------------
// (2b) per-value CDF + guide table (the default of the shortcut for G <= 1024): same likelihoods and inclusive prefix
// sums as the trees, stored as a plain row cdf[r][Gs], plus guide[r][k] = first group whose prefix reaches
// (k / K) * total, K a power of two >= 2 G.  A data row is ONE THREAD: k = floor(u K) (exact: K is a power of two),
// start at guide[r][k] and step forward while cdf < t -- on average G / K + 1 < 2 probes, no warp-wide votes, 32
// independent rows per warp in flight where the tree search had 4.  Exactness of the start: u >= k / K, products by
// `total` round monotonically, so t = fl(u total) >= fl((k / K) total) = the threshold the guide entry was built for,
// and the first prefix >= t cannot lie before it.  Same result as the tree search (first g with cdf[g] >= t, clamped
// to G - 1) wherever the prefix sums are monotone, i.e. up to near-ties.
struct GuideArgs {
    int model, G, R, Gs, K, vdim;
    const void *params;
    const float *prior;
    float *cdf;        // [R][Gs]
    float *total;      // [R]
    uint16_t *guide;   // [R][K]
};
__device__ __forceinline__ float guide_table_score(const GuideArgs &a, int r, int g) {
    CdfArgs c{};
    c.model = a.model;
    c.G = a.G;
    c.vdim = a.vdim;
    c.params = a.params;
    return table_score(c, r, g);
}

constexpr int kGuideWarps = 8;

// one warp per table row; the row's prefix sums stay in shared memory for the K binary searches of the guide
__global__ void __launch_bounds__(kGuideWarps * 32) value_guide_build_kernel(const GuideArgs a) {
    extern __shared__ float guide_smem[];  // [kGuideWarps][Gs]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int r = blockIdx.x * kGuideWarps + warp;
    if (r >= a.R) return;
    const unsigned full = 0xffffffffu;
    const int G = a.G;
    float *mine = guide_smem + warp * a.Gs;
    float m = -INFINITY;
    for (int g = lane; g < G; g += 32) m = fmaxf(m, (a.prior ? a.prior[g] : 0.f) + guide_table_score(a, r, g));
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(full, m, o));
    const float nm = -m * kLog2e;
    float *row = a.cdf + static_cast<size_t>(r) * a.Gs;
    float carry = 0.f;
    for (int g0 = 0; g0 < a.Gs; g0 += 32) {  // identical arithmetic to value_cdf_build_kernel: same prefix sums
        const int g = g0 + lane;
        float l = 0.f;
        if (g < G) l = mufu_ex2(fmaf((a.prior ? a.prior[g] : 0.f) + guide_table_score(a, r, g), kLog2e, nm));
        float incl = l;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float v = __shfl_up_sync(full, incl, o);
            if (lane >= o) incl += v;
        }
        incl += carry;
        carry = __shfl_sync(full, incl, 31);
        const float p = g < G ? incl : INFINITY;
        row[g] = p;
        mine[g] = p;
    }
    if (lane == 0) a.total[r] = carry;
    __syncwarp();
    uint16_t *gd = a.guide + static_cast<size_t>(r) * a.K;
    const float inv_k = 1.f / static_cast<float>(a.K);
    for (int k = lane; k < a.K; k += 32) {
        const float thr = (static_cast<float>(k) * inv_k) * carry;  // = fl(u total) at u = k / K
        int lo = 0, hi = G - 1;  // first g in [0, G - 1] with cdf[g] >= thr, G - 1 when none
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (mine[mid] < thr) lo = mid + 1;
            else hi = mid;
        }
        gd[k] = static_cast<uint16_t>(lo);
    }
}

struct GuideSampleArgs {
    int G, Gs, K;
    KeyMap km;
    size_t N;
    const float *cdf, *total;
    const uint16_t *guide;
    const uint32_t *values;
    int value_bytes;
    const float *u;
    int32_t *assign;
};

__device__ __forceinline__ int guide_draw(const GuideSampleArgs &a, uint32_t v, float uu, float kf) {
    const int r = key_row(a.km, v);
    const float t = uu * __ldg(a.total + r);
    const int k = max(0, min(static_cast<int>(uu * kf), a.K - 1));
    int g = __ldg(a.guide + static_cast<size_t>(r) * a.K + k);
    const float *c = a.cdf + static_cast<size_t>(r) * a.Gs;
    while (g < a.G - 1 && __ldg(c + g) < t) ++g;
    return g;
}

// kVec = 4: four consecutive rows per thread (16-byte loads of the values / uniforms, one 16-byte store of the indices;
// four independent gather chains in flight per thread); the last N % 4 rows and unaligned buffers take the scalar form
template <int kVec>
__global__ void __launch_bounds__(256) value_guide_sample_kernel(const GuideSampleArgs a) {
    const size_t step = static_cast<size_t>(gridDim.x) * blockDim.x;
    const float kf = static_cast<float>(a.K);
    const size_t first = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (kVec == 4) {
        const size_t nq = a.N / 4;
        for (size_t q = first; q < nq; q += step) {
            uint32_t v[4];
            if (a.value_bytes == 1) {
                const uchar4 b = reinterpret_cast<const uchar4 *>(a.values)[q];
                v[0] = b.x ? 1u : 0u, v[1] = b.y ? 1u : 0u, v[2] = b.z ? 1u : 0u, v[3] = b.w ? 1u : 0u;
            } else {
                const uint4 w = reinterpret_cast<const uint4 *>(a.values)[q];
                v[0] = w.x, v[1] = w.y, v[2] = w.z, v[3] = w.w;
            }
            const float4 u4 = reinterpret_cast<const float4 *>(a.u)[q];
            const float uu[4] = {u4.x, u4.y, u4.z, u4.w};
            int g[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) g[i] = guide_draw(a, v[i], uu[i], kf);
            reinterpret_cast<int4 *>(a.assign)[q] = make_int4(g[0], g[1], g[2], g[3]);
        }
        const size_t n = nq * 4 + first;  // the ragged tail
        if (n < a.N) {
            const uint32_t v = a.value_bytes == 1 ? (reinterpret_cast<const uint8_t *>(a.values)[n] ? 1u : 0u) : a.values[n];
            a.assign[n] = guide_draw(a, v, a.u[n], kf);
        }
    } else {
        for (size_t n = first; n < a.N; n += step) {
            const uint32_t v = a.value_bytes == 1 ? (reinterpret_cast<const uint8_t *>(a.values)[n] ? 1u : 0u) : a.values[n];
            a.assign[n] = guide_draw(a, v, a.u[n], kf);
        }
    }
}

static int guide_k(int G) {
    int K = 64;
    while (K < 2 * G) K *= 2;
    return K;
}
static int guide_gs(int G) { return (G + 31) / 32 * 32; }
static size_t guide_floats(int R, int G) {
    return static_cast<size_t>(R) * guide_gs(G) + static_cast<size_t>(R) + (static_cast<size_t>(R) * guide_k(G) + 1) / 2;
}

static int cdf_levels(int G) {
    int L = 1, cap = 8;
    while (cap < G) {
        cap *= 8;
        ++L;
    }
    return L;
}
size_t value_cdf_floats(int R, int G) {
    const int L = cdf_levels(G);
    size_t per = 0, w = 8;
    for (int l = 0; l < L; ++l) {
        per += w;
        w *= 8;
    }
    const size_t trees = static_cast<size_t>(R) * per + static_cast<size_t>(R);  // trees + totals
    const size_t guided = G <= 1024 ? guide_floats(R, G) : 0;                     // cdf rows + totals + guide tables
    return trees > guided ? trees : guided;
}
static size_t value_cdf_tree_floats(int R, int G) {
    const int L = cdf_levels(G);
    size_t per = 0, w = 8;
    for (int l = 0; l < L; ++l) {
        per += w;
        w *= 8;
    }
    return per;
}

// ------------------------------------------------------------------------------------------------
// (3) the logp form of (2): per table row r, lse[r] = log sum_g exp(prior_g + T[r][g]) (one warp per row: the reduction
// of value_guide_build_kernel without the prefix sums and guide), then logp[n] = lse[key_row(value n)].
__global__ void __launch_bounds__(kGuideWarps * 32) value_logp_build_kernel(const GuideArgs a) {
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * kGuideWarps + (threadIdx.x >> 5);
    if (r >= a.R) return;
    const unsigned full = 0xffffffffu;
    float m = -INFINITY;
    for (int g = lane; g < a.G; g += 32) m = fmaxf(m, (a.prior ? a.prior[g] : 0.f) + guide_table_score(a, r, g));
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(full, m, o));
    const float nm = fminf(-m * kLog2e, 3.0e38f);  // finite when the whole row is -inf: the sum is then 0
    float sum = 0.f;
    for (int g = lane; g < a.G; g += 32) sum += mufu_ex2(fmaf((a.prior ? a.prior[g] : 0.f) + guide_table_score(a, r, g), kLog2e, nm));
#pragma unroll
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(full, sum, o);
    if (lane == 0) a.total[r] = logp_finish(nm, sum);
}

struct ValueLogpArgs {
    KeyMap km;
    size_t N;
    const float *lse;
    const uint32_t *values;
    int value_bytes;
    float *logp;
};

__device__ __forceinline__ uint32_t table_value(const ValueLogpArgs &a, size_t n) {
    return a.value_bytes == 1 ? (reinterpret_cast<const uint8_t *>(a.values)[n] ? 1u : 0u) : a.values[n];
}

// kVec = 4: four consecutive rows per thread with 16-byte loads and stores, as value_guide_sample_kernel
template <int kVec>
__global__ void __launch_bounds__(256) value_logp_gather_kernel(const ValueLogpArgs a) {
    const size_t step = static_cast<size_t>(gridDim.x) * blockDim.x;
    const size_t first = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (kVec == 4) {
        const size_t nq = a.N / 4;
        for (size_t q = first; q < nq; q += step) {
            uint32_t v[4];
            if (a.value_bytes == 1) {
                const uchar4 b = reinterpret_cast<const uchar4 *>(a.values)[q];
                v[0] = b.x ? 1u : 0u, v[1] = b.y ? 1u : 0u, v[2] = b.z ? 1u : 0u, v[3] = b.w ? 1u : 0u;
            } else {
                const uint4 w = reinterpret_cast<const uint4 *>(a.values)[q];
                v[0] = w.x, v[1] = w.y, v[2] = w.z, v[3] = w.w;
            }
            float lp[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) lp[i] = __ldg(a.lse + key_row(a.km, v[i]));
            reinterpret_cast<float4 *>(a.logp)[q] = make_float4(lp[0], lp[1], lp[2], lp[3]);
        }
        const size_t n = nq * 4 + first;  // the ragged tail
        if (n < a.N) a.logp[n] = __ldg(a.lse + key_row(a.km, table_value(a, n)));
    } else {
        for (size_t n = first; n < a.N; n += step) a.logp[n] = __ldg(a.lse + key_row(a.km, table_value(a, n)));
    }
}

// value -> table row of a single table feature (dd values are clamped to dim - 1 like the row-mapped kernel does)
static int table_key_map(const dist_b200_feature *f, int &R, KeyMap &km) {
    switch (f->model) {
        case DIST_B200_DPD:
            R = f->dim + 1;
            km = KeyMap{f->dim, f->keys_dense ? 1 : 0, f->keys_dev, f->key_rows_dev};
            return DIST_B200_OK;
        case DIST_B200_DD:
            R = f->dim;
            km = KeyMap{f->dim - 1, 1, nullptr, nullptr};
            return DIST_B200_OK;
        case DIST_B200_BB:
            R = 2;
            km = KeyMap{1, 1, nullptr, nullptr};
            return DIST_B200_OK;
        default: return DIST_B200_ERR_UNSUPPORTED;
    }
}

// single table feature, logp only.  `buf` holds R floats (feature-owned scratch).  DIST_B200_ERR_UNSUPPORTED below 4 R rows
// (the same threshold as the sampler): the caller takes the per-cell kernels
int launch_value_logp(dist_b200_ctx *ctx, const dist_b200_feature *f, float *buf, const void *column, size_t N,
                      const float *prior, float *logp, cudaStream_t s) {
    if (N == 0 || f->G == 0) return DIST_B200_OK;
    int R;
    KeyMap km{};
    if (table_key_map(f, R, km)) return DIST_B200_ERR_UNSUPPORTED;
    if (N < 4 * static_cast<size_t>(R)) return DIST_B200_ERR_UNSUPPORTED;
    GuideArgs b{};
    b.model = f->model;
    b.G = f->G;
    b.R = R;
    b.vdim = f->dim;
    b.params = f->params;
    b.prior = prior;
    b.total = buf;
    value_logp_build_kernel<<<(R + kGuideWarps - 1) / kGuideWarps, kGuideWarps * 32, 0, s>>>(b);
    ValueLogpArgs a{};
    a.km = km;
    a.N = N;
    a.lse = buf;
    a.values = static_cast<const uint32_t *>(column);
    a.value_bytes = f->model == DIST_B200_BB ? 1 : 4;
    a.logp = logp;
    const bool vec = N >= 1024 && ((reinterpret_cast<uintptr_t>(column) | reinterpret_cast<uintptr_t>(logp)) & 15) == 0;
    const size_t want = ((vec ? N / 4 : N) + 255) / 256;
    const size_t cap = static_cast<size_t>(ctx->sm_count) * 8;
    const unsigned grid = static_cast<unsigned>(want < cap ? want : cap);
    if (vec) value_logp_gather_kernel<4><<<grid, 256, 0, s>>>(a);
    else value_logp_gather_kernel<1><<<grid, 256, 0, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("value_logp launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

// single table feature, sampling only.  `buf` holds value_cdf_floats(R, G) floats (feature-owned scratch).
int launch_value_cdf(dist_b200_ctx *ctx, const dist_b200_feature *f, float *buf, const void *column, size_t N,
                     const float *prior, const float *u, int32_t *assign, cudaStream_t s) {
    if (N == 0 || f->G == 0) return DIST_B200_OK;
    const int G = f->G;
    const int L = cdf_levels(G);
    if (L > 4) return DIST_B200_ERR_UNSUPPORTED;
    int R;
    // the trees cost O(R G) per call: only worth it for batches well beyond the number of distinct values
    if (N < 4 * static_cast<size_t>(f->model == DIST_B200_DPD ? f->dim + 1 : (f->model == DIST_B200_DD ? f->dim : 2)))
        return DIST_B200_ERR_UNSUPPORTED;
    KeyMap km{};
    switch (f->model) {
        case DIST_B200_DPD:
            R = f->dim + 1;
            km = KeyMap{f->dim, f->keys_dense ? 1 : 0, f->keys_dev, f->key_rows_dev};
            break;
        case DIST_B200_DD:  // values are clamped to dim - 1 like the row-mapped kernel does
            R = f->dim;
            km = KeyMap{f->dim - 1, 1, nullptr, nullptr};
            break;
        case DIST_B200_BB:
            R = 2;
            km = KeyMap{1, 1, nullptr, nullptr};
            break;
        default: return DIST_B200_ERR_UNSUPPORTED;
    }
    // DIST_B200_OPT_VALUE_CDF = 2 (A/B runs): the tree search also where the guide-table kernels apply
    if (G <= 1024 && ctx->opt[DIST_B200_OPT_VALUE_CDF] != 2) {
        GuideArgs b{};
        b.model = f->model;
        b.G = G;
        b.R = R;
        b.Gs = guide_gs(G);
        b.K = guide_k(G);
        b.vdim = f->dim;
        b.params = f->params;
        b.prior = prior;
        b.cdf = buf;
        b.total = buf + static_cast<size_t>(R) * b.Gs;
        b.guide = reinterpret_cast<uint16_t *>(b.total + R);
        value_guide_build_kernel<<<(R + kGuideWarps - 1) / kGuideWarps, kGuideWarps * 32, kGuideWarps * b.Gs * sizeof(float), s>>>(b);
        GuideSampleArgs a{};
        a.G = G;
        a.Gs = b.Gs;
        a.K = b.K;
        a.km = km;
        a.N = N;
        a.cdf = b.cdf;
        a.total = b.total;
        a.guide = b.guide;
        a.values = static_cast<const uint32_t *>(column);
        a.value_bytes = f->model == DIST_B200_BB ? 1 : 4;
        a.u = u;
        a.assign = assign;
        const bool vec = N >= 1024 && ((reinterpret_cast<uintptr_t>(column) | reinterpret_cast<uintptr_t>(u) | reinterpret_cast<uintptr_t>(assign)) & 15) == 0;
        const size_t want = ((vec ? N / 4 : N) + 255) / 256;
        const size_t cap = static_cast<size_t>(ctx->sm_count) * 8;
        const unsigned grid = static_cast<unsigned>(want < cap ? want : cap);
        if (vec) value_guide_sample_kernel<4><<<grid, 256, 0, s>>>(a);
        else value_guide_sample_kernel<1><<<grid, 256, 0, s>>>(a);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("value_guide launch: ") + cudaGetErrorString(e));
        return DIST_B200_OK;
    }
    CdfArgs b{};
    b.model = f->model;
    b.G = G;
    b.R = R;
    b.L = L;
    b.vdim = f->dim;
    b.tree_floats = value_cdf_tree_floats(R, G);
    b.params = f->params;
    b.prior = prior;
    b.tree = buf;
    b.total = buf + static_cast<size_t>(R) * b.tree_floats;
    value_cdf_build_kernel<<<(R + 7) / 8, 256, 0, s>>>(b);
    CdfSampleArgs a{};
    a.G = G;
    a.L = L;
    a.km = km;
    a.N = N;
    a.tree_floats = b.tree_floats;
    a.tree = b.tree;
    a.total = b.total;
    a.values = static_cast<const uint32_t *>(column);
    a.value_bytes = f->model == DIST_B200_BB ? 1 : 4;
    a.u = u;
    a.assign = assign;
    const size_t want = (N + 255) / 256;
    const size_t cap = static_cast<size_t>(ctx->sm_count) * 8;
    const unsigned grid = static_cast<unsigned>(want < cap ? want : cap);
    switch (L) {
        case 1: value_cdf_sample_kernel<1><<<grid, 256, 0, s>>>(a); break;
        case 2: value_cdf_sample_kernel<2><<<grid, 256, 0, s>>>(a); break;
        case 3: value_cdf_sample_kernel<3><<<grid, 256, 0, s>>>(a); break;
        default: value_cdf_sample_kernel<4><<<grid, 256, 0, s>>>(a); break;
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("value_cdf launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

}  // namespace distb200
