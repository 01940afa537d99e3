// score_rows.cuh -- the row-mapped fused score(+prior)(+sample) kernel (instantiated per model in score_rows_*.cu).
//
// Replaces, for N rows at once, the per-value stack of SURVEY.md §3.2:
//   PitmanYor::Mixture::score_value (clustering.hpp:195-208, overwrite with the prior vector)
//   -> Model::Mixture::score_value for every feature (accumulate; src/models/nich.cc:33-66,
//      src/models/gp.cc:32-67, bb.hpp:303-313, dd.hpp:433-445)
//   -> sample_from_scores_overwrite (random.hpp:360-366 = random.cc:94-106 + random.hpp:315-333).
//
// Mapping (B200): one ROW per lane, groups walked in register tiles of CHUNK.  The per-group caches
// sit in shared memory and every lane of a warp reads the same group at the same time, so a cache
// entry is one conflict-free broadcast LDS.128 shared by 32 rows; row values are read with coalesced
// loads from feature-major columns.  Everything the reference does in three passes over a G-float
// buffer (score, max/exp/sum, scan) happens in registers, in the reference's own left-to-right
// order within a tile: no warp shuffles, and no [N][G] round trip through HBM unless the caller
// asks for the scores.
//
//   G <= CHUNK  : the whole score row lives in registers; max, exp, running total and the
//                 `t -= l[i]; t <= 0` walk are the reference's loops verbatim.
//   logp mode   : neither sample nor scores: per row an online (negated scaled max, sum of exp) pair is merged across
//                 the tiles (no slots, no walk) and log sum_g exp(score) is written.
//   G  > CHUNK  : per tile (negated scaled max, sum of exp) pairs are merged into at most kSlots
//                 slots kept in shared memory; a walk over the slots finds the one holding
//                 u * total, then each thread re-scores just that slot's tiles for its own row
//                 (same code path as the main pass, with a per-lane group offset) and finishes with
//                 the reference's walk.
//
// Group caches are staged with cp.async: resident for the whole kernel when all features fit in
// shared memory, otherwise double-buffered per (feature, tile) behind the math of the previous
// feature.  KIND >= 0 instantiates the single-feature kernels (model known at compile time, prior
// folded into the resident caches); KIND = -1 is the cross-cat kernel (any feature list).
#pragma once
#include "common.cuh"

namespace distb200 {

// internal single-feature kind: NormalInverseChiSq with the block's cache copy re-laid out in PAIRS of groups,
// {-mean_a, -mean_b, prec_a, prec_b | coef_a, coef_b, score_a, score_b}, so that the hot loop runs on packed
// fp32x2 instructions (two cells per FADD2 / FMUL2 / FFMA2: 8 issue slots per cell instead of 11.5)
constexpr int kKindNichPacked = 17;
// internal single-feature kind: DirichletDiscrete, G <= 128, sampling only.  The block's cache copy holds, per
// (group, value), (prior[g] + scores_[v][g] - shift[g] - m_v) * log2(e) with m_v the maximum over groups for that
// value -- what scores_to_likelihoods would subtract for any row carrying v (random.cc:94-106) -- so a cell is one
// shared-memory gather + MUFU.EX2, and the walk runs over pair sums (half the registers: five blocks per SM).
constexpr int kKindDdScaled = 18;
// the same with dim = 16 known at compile time (DirichletDiscrete<16>, the c1 shape): the per-cell gather address
// becomes base + immediate, which takes an IMAD and a LEA out of a 7.6-instruction cell (profiles/r02_c1_dd_steady.txt)
constexpr int kKindDdScaled16 = 19;
__host__ __device__ constexpr bool is_dd_scaled(int kind) { return kind == kKindDdScaled || kind == kKindDdScaled16; }

constexpr int kSlots = 16;
constexpr int kStages = 3;  // cp.async ring depth of the streaming mode
constexpr size_t kResidentBudget = 96 * 1024;  // bytes of group caches kept resident in smem

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gmem_src) {
    const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

__host__ __device__ __forceinline__ int kind_stride(int kind, int vdim) {  // floats of cache per group
    return (kind == DIST_B200_DD || kind == kKindGpTable || is_dd_scaled(kind)) ? vdim : 4;
}

// GammaPoisson term of one (value, group) cell -- the single definition shared by the direct path, the
// table builder and the out-of-table fallback, so all three produce the same bits  (gp.cc:56-66)
__device__ __forceinline__ float gp_term(const float4 q, uint32_t xb, const float *__restrict__ coeff,
                                         const float *__restrict__ logfact) {
    const float xf = static_cast<float>(xb);
    const float lf = xb < 64 ? logfact[xb] : fast_lgamma_cell(static_cast<float>(xb + 1u), coeff);
    const float lg = fast_lgamma_cell(q.x + xf, coeff);
    return fmaf(q.y, xf, (q.z + lg) - lf);
}

// BetaNegativeBinomial term (bnb.hpp:308-319): q = {post_beta, alpha, score, -}
__device__ __forceinline__ float bnb_term(const float4 q, uint32_t xb, const float *__restrict__ coeff) {
    const float beta = q.x + static_cast<float>(xb);
    return (q.z + fast_lgamma_cell(beta, coeff)) - fast_lgamma_cell(beta + q.y, coeff);
}

// raw 32-bit value of row `row` of a feature column
__device__ __forceinline__ uint32_t load_value(int kind, const void *column, size_t row) {
    if (kind == DIST_B200_BB) return static_cast<const uint8_t *>(column)[row];
    return static_cast<const uint32_t *>(column)[row];
}

// one cell with caches behind a generic pointer: identical arithmetic to the tiled loop below
__device__ __forceinline__ float cell_score(int kind, uint32_t xb, const float *__restrict__ p, int vdim,
                                            const float *__restrict__ coeff, const float *__restrict__ logfact) {
    switch (kind) {
        case DIST_B200_NICH: {
            const float4 q = *reinterpret_cast<const float4 *>(p);
            const float d = __uint_as_float(xb) - q.x;
            const float z = __fadd_rn(1.f, __fmul_rn(q.y, __fmul_rn(d, d)));
            return fmaf(q.z, fast_log2_cell(z), q.w);  // q.z = log_coeff * ln 2
        }
        case DIST_B200_GP:
            return gp_term(*reinterpret_cast<const float4 *>(p), xb, coeff, logfact);
        case DIST_B200_BNB:
            return bnb_term(*reinterpret_cast<const float4 *>(p), xb, coeff);
        case DIST_B200_BB: {
            const float2 q = *reinterpret_cast<const float2 *>(p);
            return xb ? q.x : q.y;
        }
        case kKindGpTable:  // p points at this group's table row; out-of-table values handled by the caller
            return p[min(xb, static_cast<uint32_t>(kGpTableX - 1))];
        default: {  // DD
            const int v = min(static_cast<int>(xb), vdim - 1);
            return p[v];
        }
    }
}

// acc[j] (+)= model term of groups pb[0..CHUNK) for one row value.  kAssign: first feature of a
// single-feature kernel, whose caches already carry the prior.
template <int CHUNK, bool kAssign>
__device__ __forceinline__ void accumulate_feature(int kind, uint32_t xb, const float *__restrict__ pb, int vdim,
                                                   float (&acc)[CHUNK], const float *__restrict__ coeff,
                                                   const float *__restrict__ logfact,
                                                   const float4 *__restrict__ aux = nullptr) {
    switch (kind) {
        case kKindGpTable: {
            // tabulated GammaPoisson: one conflict-free gather per cell (lanes differ only in the value
            // column of a 32-wide row).  Counts beyond the table take the direct formula from `aux`.
            if (xb < static_cast<uint32_t>(kGpTableX)) {
#pragma unroll
                for (int j = 0; j < CHUNK; ++j) {
                    const float v = pb[j * kGpTableX + xb];
                    acc[j] = kAssign ? v : acc[j] + v;
                }
            } else {
#pragma unroll 1
                for (int j = 0; j < CHUNK; ++j) {
                    const float v = gp_term(aux[j], xb, coeff, logfact);
#pragma unroll
                    for (int jj = 0; jj < CHUNK; ++jj)
                        if (jj == j) acc[jj] = kAssign ? v : acc[jj] + v;
                }
            }
        } break;
        case kKindNichPacked: {
            // the same cell, two groups per instruction: d = x + (-mean); z = 1 + prec * (d * d) with every product
            // and sum rounded separately (the reference's unfused order, so the fast_log table step is the oracle's)
            const float4 *p4 = reinterpret_cast<const float4 *>(pb);
            const uint64_t x2 = f2_pack(__uint_as_float(xb), __uint_as_float(xb)), one2 = f2_pack(1.f, 1.f);
#pragma unroll
            for (int j = 0; j < CHUNK; j += 2) {
                const float4 qa = p4[j], qb = p4[j + 1];
                const uint64_t d2 = f2_add(x2, f2_pack(qa.x, qa.y));
                // (ptxas 12.9 contracts mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 despite the explicit rounding
                // modifiers; w * 1 + 1 as an explicit fma is the unfused sum and still a single FFMA2)
                const uint64_t z2 = f2_fma(f2_mul(f2_pack(qa.z, qa.w), f2_mul(d2, d2)), one2, one2);
                float za, zb;
                f2_unpack(z2, za, zb);
                const uint64_t v2 = f2_fma(f2_pack(qb.x, qb.y), f2_pack(fast_log2_cell(za), fast_log2_cell(zb)), f2_pack(qb.z, qb.w));
                float va, vb;
                f2_unpack(v2, va, vb);
                acc[j] = kAssign ? va : acc[j] + va;
                acc[j + 1] = kAssign ? vb : acc[j + 1] + vb;
            }
        } break;
        case DIST_B200_NICH: {
            // score + log_coeff * fast_log(1 + precision * (v - mean)^2)   (nich.cc:59-65)
            const float4 *p4 = reinterpret_cast<const float4 *>(pb);
            const float x = __uint_as_float(xb);
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) {
                const float4 q = p4[j];
                const float d = x - q.x;
                const float z = __fadd_rn(1.f, __fmul_rn(q.y, __fmul_rn(d, d)));
                const float v = fmaf(q.z, fast_log2_cell(z), q.w);  // q.z = log_coeff * ln 2
                acc[j] = kAssign ? v : acc[j] + v;
            }
        } break;
        case DIST_B200_GP: {
            // score + fast_lgamma(post_alpha + v) - fast_log_factorial(v) + score_coeff * v  (gp.cc:56-66)
            const float4 *p4 = reinterpret_cast<const float4 *>(pb);
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) {
                const float v = gp_term(p4[j], xb, coeff, logfact);
                acc[j] = kAssign ? v : acc[j] + v;
            }
        } break;
        case DIST_B200_BNB: {
            // score + fast_lgamma(post_beta + v) - fast_lgamma(post_beta + v + alpha)   (bnb.hpp:308-319)
            const float4 *p4 = reinterpret_cast<const float4 *>(pb);
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) {
                const float v = bnb_term(p4[j], xb, coeff);
                acc[j] = kAssign ? v : acc[j] + v;
            }
        } break;
        case DIST_B200_BB: {
            // value ? heads[g] : tails[g]   (bb.hpp:303-313)
            const float4 *p4 = reinterpret_cast<const float4 *>(pb);
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) {
                const float2 q = *reinterpret_cast<const float2 *>(p4 + j);
                const float v = xb ? q.x : q.y;
                acc[j] = kAssign ? v : acc[j] + v;
            }
        } break;
        default: {  // DD: scores_[value][g] - scores_shift_[g], pre-subtracted table (dd.hpp:433-445)
            const int vi = min(static_cast<int>(xb), vdim - 1);
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) {
                const float v = pb[j * vdim + vi];
                acc[j] = kAssign ? v : acc[j] + v;
            }
        } break;
    }
}

struct RowsArgs {
    int G;
    int resident;        // all caches resident in smem
    int stage_floats;    // floats per staging buffer (streaming mode)
    int accumulate;
    size_t N;
    const float *prior;
    const float *u;
    int32_t *assign;
    float *scores;
    NumericTables t;
    // peer push (feature shards): row r of this launch is global row row0 + r; it belongs to owner
    // (row0 + r) / block_rows and is stored into that owner's slot for this rank, push[owner] (a peer
    // device pointer mapped over NVLink), at local row (row0 + r) % block_rows
    int n_push;
    size_t row0, block_rows;
    float *push[kMaxPushOwners];
    float *logp;  // logp mode (kSample = kScores = false): logp[n] = log sum_g exp(score of row n, group g)
};

// kSub (feature lists whose caches stream, more groups than one register tile, sampling only): per tile the row keeps
// the tile's maximum and the sums of exp over SUB-SLOTS of 16 groups, so that the draw is located down to 16 groups
// from the main pass and only those are re-scored (from global memory, through the transposed GammaPoisson tables).
constexpr int kSubGroups = 16;
// Missing cells (feature lists only, MaskList in common.cuh).  A warp's 32 rows share one mask word: row tiles are
// multiples of 32 rows.
__device__ __forceinline__ bool cell_observed(const uint32_t *m, size_t row) {
    return !m || ((__ldg(m + (row >> 5)) >> (row & 31)) & 1u);
}
// mask of feature f: none without masks (the unmasked kernel), else read from the kernel's MaskList parameter
__device__ __forceinline__ const uint32_t *mask_of(int) { return nullptr; }
__device__ __forceinline__ const uint32_t *mask_of(int f, const MaskList &ml) { return ml.m[f]; }

// (logp mode: no minimum of resident blocks -- the register cap the others take would make its online pair spill)
// Masks: empty, or one MaskList (score_rows_masked*.cu, feature lists with missing cells: a lane whose cell is missing
// sits that feature out).  Without masks the kernel is the unmasked one instruction for instruction.
template <int CHUNK, int KIND, bool kSample, bool kScores, int THREADS, bool kSub = false, typename... Masks>
__global__ void __launch_bounds__(THREADS, (!kSample && !kScores) ? 1 : THREADS == 128 ? (is_dd_scaled(KIND) ? 5 : 3) : (CHUNK <= 32 ? (KIND >= 0 ? 4 : 3) : (CHUNK <= 64 ? 2 : 1)))
score_rows_kernel(const __grid_constant__ FeatList feats, const RowsArgs a, Masks... masks) {
    constexpr bool kMask = sizeof...(Masks) > 0;
    constexpr int kThreads = THREADS;  // block size of this instantiation
    static_assert(!kSub || (KIND < 0 && kSample && !kScores && CHUNK % kSubGroups == 0), "kSub: streaming feature lists, sampling only");
    static_assert(!kMask || KIND < 0, "masks: feature-list kernels only");
    constexpr int kSubPer = CHUNK / kSubGroups;  // sub-slots per tile
    extern __shared__ __align__(16) float smem[];
    // layout: coeff[33*8] | logfact[64] | prior[Gpad] | tile[8 warps][32][33] (kScores) |
    //         slots[kSlots][kThreads] float2 (kSample, multi-tile) | caches
    constexpr bool kSingle = KIND >= 0;  // one feature of a known model; caches resident
    // prior folded into the resident caches (first feature ASSIGNS): not for gp, whose score[g] cancels
    // against lgamma(post_alpha + v) -- adding the prior before that cancellation would cost ~1e-5
    constexpr bool kFold = kSingle && KIND != DIST_B200_GP && KIND != DIST_B200_BNB;
    constexpr bool kNich = KIND == DIST_B200_NICH || KIND == kKindNichPacked;
    constexpr bool kLogp = !kSample && !kScores;
    const int G = a.G;
    const int nchunks = (G + CHUNK - 1) / CHUNK;
    const int Gpad = nchunks * CHUNK;
    const bool multi = nchunks > 1;
    float *coeff = smem;
    float *logfact = coeff + 33 * kLgammaRowStride;
    float *prior_s = logfact + 64;
    float *cursor = prior_s + Gpad;
    float *tile = cursor;
    if (kScores) cursor += (kThreads / 32) * 32 * 33;
    float2 *slots = reinterpret_cast<float2 *>(cursor);
    float *subs = cursor;  // kSub: [nchunks][kSubPer + 1][kThreads] -- sub-slot sums, then the tile's negated scaled max
    if (kSub) cursor += nchunks * (kSubPer + 1) * kThreads;
    else if (kSample && multi) cursor += 2 * kSlots * kThreads;
    float *caches = cursor;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int F = kSingle ? 1 : feats.n;
    const bool resident = kSingle ? true : (a.resident != 0);

    if (!is_dd_scaled(KIND)) {  // (table lookups need neither; the dd kernel reuses the area as scratch)
        for (int i = tid; i < 33 * kLgammaRowStride; i += kThreads) coeff[i] = a.t.lgamma5[i];
        if (tid < 64) logfact[tid] = a.t.log_factorial[tid];
    }
    // the prior vector (clustering's overwrite) seeds every accumulator; padded groups get -inf
    for (int g = tid; g < Gpad; g += kThreads)
        prior_s[g] = g < G ? ((a.prior && !a.accumulate) ? a.prior[g] : 0.f) : -INFINITY;
    if (resident) {
        size_t off = 0;
        for (int f = 0; f < F; ++f) {
            const int n = Gpad * kind_stride(kSingle ? KIND : feats.f[f].kind, feats.f[f].vdim);
            const float *src = static_cast<const float *>(feats.f[f].params);
            for (int i = tid * 4; i < n; i += kThreads * 4) cp_async16(caches + off + i, src + i);
            off += n;
        }
        cp_async_commit();
        cp_async_wait<0>();
    }
    __syncthreads();
    if (kFold) {
        // fold the prior into this block's private copy of the caches: the first (only) feature then
        // ASSIGNS prior + term in one FFMA instead of seeding accumulators and adding
        const int vdim = feats.f[0].vdim;
        // Padded groups (g >= G) become -inf for every row here, so the hot loop needs no per-cell mask:
        // their prior is -inf, and nich borrows group 0's (mean, precision, coeff) so that the term is finite
        // or -inf exactly when a real group's is (zeroed parameters would give 0 * inf = NaN for |x| > 1e19).
        for (int g = tid; g < Gpad; g += kThreads) {
            const float p = prior_s[g];
            if (kNich) {
                if (g >= G) {
                    caches[g * 4 + 0] = caches[0];
                    caches[g * 4 + 1] = caches[1];
                    caches[g * 4 + 2] = caches[2];
                }
                caches[g * 4 + 3] += p;
            } else if (KIND == DIST_B200_GP) caches[g * 4 + 2] += p;
            else if (KIND == DIST_B200_BB) {
                caches[g * 4 + 0] += p;
                caches[g * 4 + 1] += p;
            } else {
                for (int v = 0; v < vdim; ++v) caches[g * vdim + v] += p;
            }
        }
        __syncthreads();
        if (is_dd_scaled(KIND)) {
            // per value: the maximum over groups, then (score - max) * log2e in place (a thread owns its value's column;
            // padded groups stay -inf)
            const int vdim = feats.f[0].vdim;
            // threads cover (value, slice of the groups): with one thread per value the 2 x Gpad dependent shared-memory
            // accesses of 16 threads were most of a small launch's time (c1 at 1e5 rows: ~9 us of prologue in a 17 us kernel).
            // Partial maxima go through the lgamma coefficient area, which a dd kernel never reads.
            const int nsl = vdim <= kThreads ? min(kThreads / vdim, (33 * kLgammaRowStride) / vdim) : 1;
            if (nsl > 1) {
                float *part = coeff;
                const int v = tid % vdim, sl = tid / vdim;
                const int per = (Gpad + nsl - 1) / nsl, ga = sl * per, gb = min(Gpad, ga + per);
                if (sl < nsl) {
                    float m = -INFINITY;
                    for (int g = ga; g < gb; ++g) m = fmaxf(m, caches[g * vdim + v]);
                    part[sl * vdim + v] = m;
                }
                __syncthreads();
                if (sl < nsl) {
                    float m = part[v];
                    for (int k = 1; k < nsl; ++k) m = fmaxf(m, part[k * vdim + v]);
                    for (int g = ga; g < gb; ++g) caches[g * vdim + v] = (caches[g * vdim + v] - m) * kLog2e;
                }
            } else {
                for (int v = tid; v < vdim; v += kThreads) {
                    float m = -INFINITY;
                    for (int g = 0; g < Gpad; ++g) m = fmaxf(m, caches[g * vdim + v]);
                    for (int g = 0; g < Gpad; ++g) caches[g * vdim + v] = (caches[g * vdim + v] - m) * kLog2e;
                }
            }
            __syncthreads();
        }
        if (KIND == kKindNichPacked) {
            // re-lay the private copy out in pairs of groups (in place: a thread owns its pair's eight floats)
            for (int p = tid; p < Gpad / 2; p += kThreads) {
                float4 *c4 = reinterpret_cast<float4 *>(caches) + 2 * p;
                const float4 a4 = c4[0], b4 = c4[1];
                c4[0] = make_float4(-a4.x, -b4.x, a4.y, b4.y);
                c4[1] = make_float4(a4.z, b4.z, a4.w, b4.w);
            }
            __syncthreads();
        }
    }

    const int chunks_per_slot = (nchunks + kSlots - 1) / kSlots;
    const int nslots = (nchunks + chunks_per_slot - 1) / chunks_per_slot;
    // the selected slot is re-scored in-thread through the main loop body when caches are resident
    const int extra = (kSample && multi && resident) ? chunks_per_slot : 0;
    // Row tiles are strided over the blocks: neighbouring blocks stream neighbouring rows (DRAM / TLB
    // locality for the many column streams of a cross-cat kind).  Splitting the last, partial round at
    // warp granularity was measured and dropped: same-box A/B at c2 0.7315 ms plain vs 0.7380 ms balanced
    // (blocks that finish early free MUFU issue slots for their neighbours on the SM), and the extra loop
    // state cost the register-capped cross-cat kernel 8%.
    const size_t ntiles = (a.N + kThreads - 1) / kThreads;
    // dd scaled-table kind (a tile of rows is ~3 us of work): the next tile's value and uniform are requested while the
    // current tile is evaluated, so the load latency is not left to the other resident blocks
    constexpr bool kPrefetch = kSample && is_dd_scaled(KIND);
    uint32_t pre_v = 0;
    float pre_u = 0.f;
    if (kPrefetch && blockIdx.x < ntiles) {
        const size_t r0 = min(static_cast<size_t>(blockIdx.x) * kThreads + tid, a.N - 1);
        pre_v = load_value(DIST_B200_DD, feats.f[0].column, r0);
        pre_u = a.u[r0];
    }
    for (size_t tile_id = blockIdx.x; tile_id < ntiles; tile_id += gridDim.x) {
        const size_t tile_base = tile_id * kThreads;
        const size_t row_end = a.N;
        size_t row = tile_base + tid;
        const bool valid = row < row_end;
        if (!valid) row = row_end - 1;  // clamp: compute on a real row, discard the result
        float slot_m = INFINITY, slot_s = 0.f;  // slot being merged: negated scaled max, sum of exp
        float nmax = 0.f, tres = 0.f;           // finalisation state: row's negated scaled max, remaining draw
        float lp_m = INFINITY, lp_s = 0.f;      // logp mode: the row's negated scaled max and sum of exp so far
        int sel = 0, count = 0, result = 0;
        const float urow = kPrefetch ? pre_u : (kSample ? a.u[row] : 0.f);
        const uint32_t vrow = pre_v;
        if (kPrefetch && tile_id + gridDim.x < ntiles) {
            const size_t rn = min((tile_id + gridDim.x) * kThreads + tid, a.N - 1);
            pre_v = load_value(DIST_B200_DD, feats.f[0].column, rn);
            pre_u = a.u[rn];
        }

        for (int it = 0; it < nchunks + extra; ++it) {
            const bool fin = it >= nchunks;  // block-uniform: re-scoring the selected slot
            // group offset of this thread's tile: uniform in the main pass, per lane when finalising
            int g0 = it * CHUNK;
            if (fin) g0 = min((sel * chunks_per_slot + (it - nchunks)) * CHUNK, Gpad - CHUNK);
            // streaming mode: a kStages-deep cp.async ring; stage (f % kStages) holds feature f's caches for
            // this tile of groups followed by this block's row values of feature f (one word per thread),
            // so both arrive kStages-1 features ahead of their use
            const int ring_floats = a.stage_floats + kThreads;
            auto issue = [&](int f) {
                const FeatDesc &fd = feats.f[f];
                const int st = kind_stride(fd.kind, fd.vdim);
                const float *src = static_cast<const float *>(fd.params) + static_cast<size_t>(g0) * st;
                float *dst = caches + (f % kStages) * ring_floats;
                for (int i = tid * 4; i < CHUNK * st; i += kThreads * 4) cp_async16(dst + i, src + i);
                const char *xp = static_cast<const char *>(fd.column) + (fd.kind == DIST_B200_BB ? row : 4 * row);
                cp_async4(dst + a.stage_floats + tid, reinterpret_cast<const void *>(reinterpret_cast<uintptr_t>(xp) & ~uintptr_t(3)));
            };
            if (!resident) {
#pragma unroll
                for (int f = 0; f < kStages - 1; ++f) {
                    if (f < F) issue(f);
                    cp_async_commit();
                }
            }

            float acc[CHUNK];
            if (!kFold) {
#pragma unroll
                for (int j = 0; j < CHUNK; j += 4) {
                    const float4 p = *reinterpret_cast<const float4 *>(prior_s + g0 + j);
                    acc[j] = p.x;
                    acc[j + 1] = p.y;
                    acc[j + 2] = p.z;
                    acc[j + 3] = p.w;
                }
            }

            if (is_dd_scaled(KIND)) {
                // gather + exp + pair sums fused below (the sampler of this kind reads the block's table itself)
            } else if (kSingle) {
                const uint32_t xb = load_value(KIND == kKindNichPacked ? DIST_B200_NICH : KIND, feats.f[0].column, row);
                const int vdim = feats.f[0].vdim;
                accumulate_feature<CHUNK, kFold>(KIND, xb, caches + static_cast<size_t>(g0) * kind_stride(KIND, vdim), vdim,
                                                 acc, coeff, logfact);
            } else {
                uint32_t xb = resident ? load_value(feats.f[0].kind, feats.f[0].column, row) : 0u;
                size_t res_off = 0;
                for (int f = 0; f < F; ++f) {
                    const FeatDesc &fd = feats.f[f];
                    const int st = kind_stride(fd.kind, fd.vdim);
                    uint32_t xn = 0;
                    const float *pb;
                    const bool obs = kMask ? cell_observed(mask_of(f, masks...), row) : true;
                    if (resident) {
                        if (f + 1 < F) xn = load_value(feats.f[f + 1].kind, feats.f[f + 1].column, row);
                        pb = caches + res_off + static_cast<size_t>(g0) * st;
                        res_off += static_cast<size_t>(Gpad) * st;
                    } else {
                        cp_async_wait<kStages - 2>();  // this thread's copies of feature f have landed
                        __syncthreads();               // ... everyone's have, and stage (f-1) % kStages is free
                        if (f + kStages - 1 < F) issue(f + kStages - 1);
                        cp_async_commit();
                        pb = caches + (f % kStages) * ring_floats;
                        const uint32_t word = reinterpret_cast<const uint32_t *>(pb + a.stage_floats)[tid];
                        if (fd.kind == DIST_B200_BB) {
                            const uintptr_t addr = reinterpret_cast<uintptr_t>(fd.column) + row;
                            xb = (word >> (8 * (addr & 3))) & 0xffu;
                        } else {
                            xb = word;
                        }
                    }
                    // a missing cell adds nothing: its lane sits out this feature (no arithmetic on the value it holds, so
                    // an inf / NaN term of that value cannot reach the sum)
                    if (!kMask || obs)
                        accumulate_feature<CHUNK, false>(fd.kind, xb, pb, fd.vdim, acc, coeff, logfact,
                                                         static_cast<const float4 *>(fd.aux) + g0);
                    if (resident) xb = xn;
                }
                if (!resident) __syncthreads();  // the ring is refilled by the next tile's prologue
            }

            if (!kFold && g0 + CHUNK > G) {
                // ragged last tile: padded groups carry zeroed caches, whose model terms may be inf/NaN
                // (lgamma(0)); pin them to -inf so they vanish from max / exp / the walk.  With the prior
                // folded into the caches (kFold) the padded entries are -inf by construction.
#pragma unroll
                for (int j = 0; j < CHUNK; ++j)
                    if (g0 + j >= G) acc[j] = -INFINITY;
            }

            if (kScores && !fin) {
                // [32 rows][32 groups] transposes through a padded per-warp tile -> every store instruction
                // writes one full 128-byte line of a row.  Everything row-invariant is hoisted: the loop body
                // is one LDS, one STG and a pointer step.
                float *tw = tile + warp * 32 * 33;
                const size_t wrow0 = tile_base + warp * 32;
                const int nrows = wrow0 < row_end ? static_cast<int>(row_end - wrow0 < 32 ? row_end - wrow0 : 32) : 0;
#pragma unroll
                for (int sb = 0; sb < CHUNK / 32; ++sb) {
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 32; ++j) tw[lane * 33 + j] = acc[sb * 32 + j];
                    __syncwarp();
                    if (((G & 3) == 0) && g0 + sb * 32 + 32 <= G && !a.accumulate && (!a.n_push || a.block_rows >= 32)) {
                        // 16-byte stores: lane (r, c) = (lane / 8, lane % 8) writes groups [4c, 4c + 4) of rows r, r + 4, ...
                        // -- four conflict-free scalar LDS, one ST.128; a store instruction covers four 128-byte row
                        // segments (a quarter of the store instructions, 16 B per lane on the NVLink path).  A push
                        // takes them only with blocks of >= 32 rows, where the warp's 32 rows span at most two owners;
                        // smaller blocks take the scalar path below, which walks any number of owners.
                        const int r = lane >> 3, c = lane & 7;
                        const int gq = g0 + sb * 32 + 4 * c;
                        const size_t grow0 = a.row0 + wrow0;
                        const int owner0 = a.n_push ? static_cast<int>(grow0 / a.block_rows) : 0;
                        const size_t off0 = a.n_push ? grow0 - static_cast<size_t>(owner0) * a.block_rows : 0;
                        const int first = a.n_push ? static_cast<int>(a.block_rows - off0 < 32 ? a.block_rows - off0 : 32) : 32;
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int row = 4 * i + r;
                            if (row >= nrows) continue;
                            const float *sp = tw + row * 33 + 4 * c;
                            const float4 v = make_float4(sp[0], sp[1], sp[2], sp[3]);
                            float *base;
                            if (a.n_push)
                                base = row < first ? a.push[owner0] + (off0 + row) * G : a.push[owner0 + 1] + static_cast<size_t>(row - first) * G;
                            else
                                base = a.scores + (wrow0 + row) * G;
                            *reinterpret_cast<float4 *>(base + gq) = v;
                        }
                        continue;
                    }
                    const int g = g0 + sb * 32 + lane;
                    if (g >= G) continue;
                    const float *src = tw + lane;
                    if (a.n_push) {
                        // rows of this warp tile land in as many owners' slots as its 32 rows span
                        const size_t grow0 = a.row0 + wrow0;
                        int owner = static_cast<int>(grow0 / a.block_rows);
                        size_t off = grow0 - static_cast<size_t>(owner) * a.block_rows;
                        float *dst = a.push[owner] + off * G + g;
                        for (int i = 0; i < nrows; ++i) {
                            if (off == a.block_rows) {
                                ++owner;
                                off = 0;
                                dst = a.push[owner] + g;
                            }
                            *dst = src[i * 33];
                            dst += G;
                            ++off;
                        }
                    } else {
                        float *dst = a.scores + wrow0 * G + g;
                        if (a.accumulate) {
                            for (int i = 0; i < nrows; ++i, dst += G) *dst += src[i * 33];
                        } else if (nrows == 32) {
#pragma unroll
                            for (int i = 0; i < 32; ++i, dst += G) *dst = src[i * 33];
                        } else {
                            for (int i = 0; i < nrows; ++i, dst += G) *dst = src[i * 33];
                        }
                    }
                }
            }

            if (kLogp) {
                // the tile's (negated scaled max, sum of exp) pair merged into the row's, as the multi-tile sampler merges
                // a slot; nm is finite also when every group of the tile sits at -inf (its sum is then 0, not NaN)
                float m = acc[0];
#pragma unroll
                for (int j = 1; j < CHUNK; ++j) m = fmaxf(m, acc[j]);
                const float nm = fminf(-m * kLog2e, 3.0e38f);
                const uint64_t l2e2 = f2_pack(kLog2e, kLog2e), nm2 = f2_pack(nm, nm);
                uint64_t s2 = f2_pack(0.f, 0.f);
#pragma unroll
                for (int j = 0; j < CHUNK; j += 2) {
                    float ea, eb;
                    f2_unpack(f2_fma(f2_pack(acc[j], acc[j + 1]), l2e2, nm2), ea, eb);
                    s2 = f2_add(s2, f2_pack(mufu_ex2(ea), mufu_ex2(eb)));
                }
                float se, so;
                f2_unpack(s2, se, so);
                const float s = se + so;
                const float dlt = lp_m - nm;
                const float e = mufu_ex2(-fabsf(dlt));
                lp_s = dlt > 0.f ? fmaf(lp_s, e, s) : fmaf(s, e, lp_s);
                lp_m = fminf(lp_m, nm);
            }

            if (kSample && is_dd_scaled(KIND)) {
                // One gather + MUFU.EX2 per cell; likelihoods are kept as PAIR sums, in four contiguous segments
                // (four independent chains for the total and for the walk `t -= l; stop at t <= 0`, random.hpp:315-333).
                // The walk stops on a pair; the pair's first likelihood is then recomputed (one more gather) to place the
                // stop inside it.  Sign-bit counting as everywhere: an exact +0 continues (a near-tie).
                const int vdim = KIND == kKindDdScaled16 ? 16 : feats.f[0].vdim;
                const int vi = min(static_cast<int>(vrow), vdim - 1);
                const float *pb = caches + vi;
                constexpr int PAIRS = CHUNK / 2, SEGP = PAIRS / 4;
                static_assert(CHUNK % 8 == 0, "register tile: four segments of whole pairs");
                float p[PAIRS];
                float seg[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int k = 0; k < SEGP; ++k) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int j = 2 * (q * SEGP + k);
                        p[q * SEGP + k] = mufu_ex2(pb[j * vdim]) + mufu_ex2(pb[(j + 1) * vdim]);
                        seg[q] += p[q * SEGP + k];
                    }
                }
                const float p1 = seg[0], p2 = p1 + seg[1], p3 = p2 + seg[2];
                const float t0 = (p3 + seg[3]) * urow;
                float t[4] = {t0, t0 - p1, t0 - p2, t0 - p3};
                // the draw left in front of the first pair that is not passed = the smallest t >= +0 seen so far.  As unsigned
                // integers the non-negative floats keep their order and every negative one is larger than all of them: one
                // unsigned min per pair (a segment that starts at t < 0 is never the stopping one, its value is unused)
                unsigned last[4] = {__float_as_uint(t[0]), __float_as_uint(t[1]), __float_as_uint(t[2]), __float_as_uint(t[3])};
                unsigned neg[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                for (int k = 0; k < SEGP; ++k) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        t[q] -= p[q * SEGP + k];
                        neg[q] += __float_as_uint(t[q]) >> 31;
                        last[q] = min(last[q], __float_as_uint(t[q]));
                    }
                }
                // pairs passed in front of the stop; a segment after the stopping one starts at t <= 0 and passes none
                int passed = 0, qs = 3;
                bool open = true;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int c = SEGP - static_cast<int>(neg[q]);
                    if (open) {
                        passed += c;
                        if (c < SEGP) {
                            qs = q;
                            open = false;
                        }
                    }
                }
                const float before = __uint_as_float(qs == 0 ? last[0] : (qs == 1 ? last[1] : (qs == 2 ? last[2] : last[3])));
                const int kp = min(passed, PAIRS - 1);
                const float first = mufu_ex2(pb[(2 * kp) * vdim]);
                const int idx = 2 * kp + ((before - first > 0.f) ? 1 : 0);
                result = min(open ? CHUNK - 1 : idx, G - 1);
            } else if (kSample) {
                if (!multi) {
                    // scores_to_likelihoods + sample_from_likelihoods (random.cc:94-106, random.hpp:315-333) on the
                    // register row.  exp(s - m) = 2^(s log2e - m log2e): one packed FFMA2 per two cells + MUFU.EX2.
                    // The row is cut into four contiguous segments: four independent partial sums, then four
                    // independent walks `t -= l[i]` that start from the draw minus the mass of the segments before
                    // (a thread's only parallelism is ILP here: one 128-deep dependent chain per phase would leave the
                    // few resident warps waiting on FADD latency).  The stop `t <= 0` is counted from t's sign bit
                    // (one LEA.HI per cell; an exact +0 continues: a near-tie); segments after the stop count 0.
                    float m = acc[0];
#pragma unroll
                    for (int j = 1; j < CHUNK; ++j) m = fmaxf(m, acc[j]);
                    const float nm = -m * kLog2e;
                    const uint64_t l2e2 = f2_pack(kLog2e, kLog2e), nm2 = f2_pack(nm, nm);
                    constexpr int SEGLEN = CHUNK / 4;
                    static_assert(CHUNK % 8 == 0, "register tile: four segments of an even number of groups");
                    float seg[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                    for (int j = 0; j < SEGLEN; j += 2) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            float ea, eb;
                            f2_unpack(f2_fma(f2_pack(acc[q * SEGLEN + j], acc[q * SEGLEN + j + 1]), l2e2, nm2), ea, eb);
                            acc[q * SEGLEN + j] = mufu_ex2(ea);
                            acc[q * SEGLEN + j + 1] = mufu_ex2(eb);
                            seg[q] = (seg[q] + acc[q * SEGLEN + j]) + acc[q * SEGLEN + j + 1];
                        }
                    }
                    const float p1 = seg[0], p2 = p1 + seg[1], p3 = p2 + seg[2];
                    const float t0 = (p3 + seg[3]) * urow;
                    float t[4] = {t0, t0 - p1, t0 - p2, t0 - p3};
                    unsigned neg[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                    for (int j = 0; j < SEGLEN; ++j) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            t[q] -= acc[q * SEGLEN + j];
                            neg[q] += __float_as_uint(t[q]) >> 31;
                        }
                    }
                    result = min(CHUNK - static_cast<int>((neg[0] + neg[1]) + (neg[2] + neg[3])), G - 1);
                } else if (kSub) {
                    float m = acc[0];
#pragma unroll
                    for (int j = 1; j < CHUNK; ++j) m = fmaxf(m, acc[j]);
                    const float nm = fminf(-m * kLog2e, 3.0e38f);  // finite also when every group of the tile sits at -inf (a masked-out prior): its weights are then 0, not NaN
                    const uint64_t l2e2 = f2_pack(kLog2e, kLog2e), nm2 = f2_pack(nm, nm);
#pragma unroll
                    for (int k = 0; k < kSubPer; ++k) {
                        float sk = 0.f;  // summed left to right, as the re-score walk subtracts
#pragma unroll
                        for (int j = 0; j < kSubGroups; j += 2) {
                            float ea, eb;
                            f2_unpack(f2_fma(f2_pack(acc[k * kSubGroups + j], acc[k * kSubGroups + j + 1]), l2e2, nm2), ea, eb);
                            sk += mufu_ex2(ea);
                            sk += mufu_ex2(eb);
                        }
                        subs[(it * (kSubPer + 1) + k) * kThreads + tid] = sk;
                    }
                    subs[(it * (kSubPer + 1) + kSubPer) * kThreads + tid] = nm;
                } else if (!fin) {
                    float m = acc[0];
#pragma unroll
                    for (int j = 1; j < CHUNK; ++j) m = fmaxf(m, acc[j]);
                    // slots carry nm = -(max * log2 e), rounded ONCE: every later rescale is a
                    // difference of these rounded values, so tile sums stay mutually consistent
                    const float nm = -m * kLog2e;
                    const uint64_t l2e2 = f2_pack(kLog2e, kLog2e), nm2 = f2_pack(nm, nm);
                    uint64_t s2 = f2_pack(0.f, 0.f);
#pragma unroll
                    for (int j = 0; j < CHUNK; j += 2) {  // one FFMA2 + one FADD2 per two cells
                        float ea, eb;
                        f2_unpack(f2_fma(f2_pack(acc[j], acc[j + 1]), l2e2, nm2), ea, eb);
                        s2 = f2_add(s2, f2_pack(mufu_ex2(ea), mufu_ex2(eb)));
                    }
                    float se, so;
                    f2_unpack(s2, se, so);
                    const float s = se + so;
                    // rescale to the smaller nm (the larger maximum): one of the two factors is 2^0 = 1, so a
                    // single EX2 of -|difference| serves (slot_m = +inf on a fresh slot gives e = 0, slot_s = 0)
                    const float dlt = slot_m - nm;
                    const float e = mufu_ex2(-fabsf(dlt));
                    slot_s = dlt > 0.f ? fmaf(slot_s, e, s) : fmaf(s, e, slot_s);
                    slot_m = fminf(slot_m, nm);
                    if ((it + 1) % chunks_per_slot == 0 || it + 1 == nchunks) {
                        slots[(it / chunks_per_slot) * kThreads + tid] = make_float2(slot_m, slot_s);
                        slot_m = INFINITY;
                        slot_s = 0.f;
                    }
                    if (it + 1 == nchunks) {
                        // total over slots, then the walk over slots to the one holding u * total
                        float mm = INFINITY;
                        for (int k = 0; k < nslots; ++k) mm = fminf(mm, slots[k * kThreads + tid].x);
                        float total = 0.f;
                        for (int k = 0; k < nslots; ++k) {
                            const float2 ms = slots[k * kThreads + tid];
                            const float w = ms.y * mufu_ex2(mm - ms.x);
                            slots[k * kThreads + tid].y = w;  // the walk below reads the rescaled mass back: no second EX2
                            total += w;
                        }
                        float t = total * urow;
                        sel = nslots - 1;
                        for (int k = 0; k < nslots; ++k) {
                            const float w = slots[k * kThreads + tid].y;
                            if (t <= w) {
                                sel = k;
                                break;
                            }
                            if (k + 1 < nslots) t -= w;
                        }
                        nmax = mm;
                        tres = t;
                        count = 0;
                    }
                } else {
                    // finalisation: this tile belongs to the selected slot of this thread's row
                    const bool live = (sel * chunks_per_slot + (it - nchunks)) * CHUNK < Gpad;
                    if (live) {
#pragma unroll
                        for (int j = 0; j < CHUNK; ++j) {
                            tres -= mufu_ex2(fmaf(acc[j], kLog2e, nmax));
                            count += 1 - static_cast<int>(__float_as_uint(tres) >> 31);  // tres >= +0 continues
                        }
                    }
                }
            }
        }  // tiles of groups

        if (kSub) {
            // tiles -> the tile holding u * total -> its sub-slot -> re-score that sub-slot's 16 groups
            float mm = INFINITY;
            for (int c = 0; c < nchunks; ++c) mm = fminf(mm, subs[(c * (kSubPer + 1) + kSubPer) * kThreads + tid]);
            float total = 0.f;
            for (int c = 0; c < nchunks; ++c) {
                float sc = 0.f;
                for (int k = 0; k < kSubPer; ++k) sc += subs[(c * (kSubPer + 1) + k) * kThreads + tid];
                total += sc * mufu_ex2(mm - subs[(c * (kSubPer + 1) + kSubPer) * kThreads + tid]);
            }
            float t = total * urow;
            int csel = nchunks - 1;
            float fsel = 1.f;
            for (int c = 0; c < nchunks; ++c) {
                float sc = 0.f;
                for (int k = 0; k < kSubPer; ++k) sc += subs[(c * (kSubPer + 1) + k) * kThreads + tid];
                const float fc = mufu_ex2(mm - subs[(c * (kSubPer + 1) + kSubPer) * kThreads + tid]);
                const float w = sc * fc;
                fsel = fc;
                if (t <= w) {
                    csel = c;
                    break;
                }
                if (c + 1 < nchunks) t -= w;
            }
            t = fsel > 0.f ? t / fsel : 0.f;  // the remaining draw on the selected tile's own scale
            int ksel = kSubPer - 1;
            for (int k = 0; k < kSubPer; ++k) {
                const float w = subs[(csel * (kSubPer + 1) + k) * kThreads + tid];
                if (t <= w) {
                    ksel = k;
                    break;
                }
                if (k + 1 < kSubPer) t -= w;
            }
            const float nm = subs[(csel * (kSubPer + 1) + kSubPer) * kThreads + tid];
            const int gb = csel * CHUNK + ksel * kSubGroups;
            // the same sums in the same order as the main pass: prior, then the features left to right
            float sc16[kSubGroups];
#pragma unroll
            for (int j = 0; j < kSubGroups; ++j) sc16[j] = prior_s[gb + j];
            for (int f = 0; f < F; ++f) {
                const FeatDesc &fd = feats.f[f];
                if (kMask && !cell_observed(mask_of(f, masks...), row)) continue;  // the main pass added 0 for this cell
                const uint32_t xv = load_value(fd.kind, fd.column, row);
                if (fd.kind == kKindGpTable && xv < static_cast<uint32_t>(kGpTableX)) {
                    // transposed table [value][capacity] behind the [capacity][value] one: 64 contiguous bytes
                    const float4 *tp = reinterpret_cast<const float4 *>(static_cast<const float *>(fd.params) +
                                                                        static_cast<size_t>(kGpTableX + xv) * fd.cap + gb);
#pragma unroll
                    for (int q = 0; q < kSubGroups / 4; ++q) {
                        const float4 v = __ldg(tp + q);
                        sc16[4 * q] += v.x;
                        sc16[4 * q + 1] += v.y;
                        sc16[4 * q + 2] += v.z;
                        sc16[4 * q + 3] += v.w;
                    }
                } else if (fd.kind == kKindGpTable) {
#pragma unroll 1
                    for (int j = 0; j < kSubGroups; ++j) {
                        const float v = gp_term(static_cast<const float4 *>(fd.aux)[gb + j], xv, coeff, logfact);
#pragma unroll
                        for (int jj = 0; jj < kSubGroups; ++jj)
                            if (jj == j) sc16[jj] += v;
                    }
                } else if (fd.kind == DIST_B200_BB) {
                    // compact copy [heads[Gpad] | tails[Gpad]] made for this launch (bb_compact_kernel): 64 contiguous bytes
                    const float4 *bp = reinterpret_cast<const float4 *>(static_cast<const float *>(fd.aux) + (xv ? 0 : fd.cap) + gb);
#pragma unroll
                    for (int q = 0; q < kSubGroups / 4; ++q) {
                        const float4 v = __ldg(bp + q);
                        sc16[4 * q] += v.x;
                        sc16[4 * q + 1] += v.y;
                        sc16[4 * q + 2] += v.z;
                        sc16[4 * q + 3] += v.w;
                    }
                } else {
                    const int st = kind_stride(fd.kind, fd.vdim);
#pragma unroll
                    for (int j = 0; j < kSubGroups; ++j)
                        sc16[j] += cell_score(fd.kind, xv, static_cast<const float *>(fd.params) + static_cast<size_t>(gb + j) * st, fd.vdim, coeff, logfact);
                }
            }
            int cnt = 0;
#pragma unroll
            for (int j = 0; j < kSubGroups; ++j) {
                const float sj = gb + j < G ? sc16[j] : -INFINITY;  // padded groups: as in the main pass
                t -= mufu_ex2(fmaf(sj, kLog2e, nm));
                cnt += 1 - static_cast<int>(__float_as_uint(t) >> 31);  // t >= +0 continues (an exact 0: a near-tie)
            }
            result = min(gb + cnt, G - 1);
        } else if (kSample && multi) {
            if (resident) {
                result = min(sel * chunks_per_slot * CHUNK + count, G - 1);
            } else {
                // streaming caches: re-score the selected slot cell by cell from global memory -- or read the scores back
                // where this launch has just written them (the row's scores were stored by lanes of this warp)
                int idx = G - 1;
                const int gb = sel * chunks_per_slot * CHUNK, ge = min(G, gb + chunks_per_slot * CHUNK);
                float t = tres;
                const bool readback = kScores && !a.accumulate && !a.n_push;
                if (readback) __syncwarp();
                for (int g = gb; g < ge; ++g) {
                    float s = prior_s[g];
                    if (readback) {
                        s = a.scores[row * static_cast<size_t>(G) + g];
                    } else
                    for (int f = 0; f < F; ++f) {
                        const FeatDesc &fd = feats.f[f];
                        if (kMask && !cell_observed(mask_of(f, masks...), row)) continue;
                        const uint32_t xv = load_value(fd.kind, fd.column, row);
                        if (fd.kind == kKindGpTable && xv >= static_cast<uint32_t>(kGpTableX))
                            s += gp_term(static_cast<const float4 *>(fd.aux)[g], xv, coeff, logfact);
                        else
                            s += cell_score(fd.kind, xv,
                                            static_cast<const float *>(fd.params) +
                                                static_cast<size_t>(g) * kind_stride(fd.kind, fd.vdim),
                                            fd.vdim, coeff, logfact);
                    }
                    t -= mufu_ex2(fmaf(s, kLog2e, nmax));
                    if (t <= 0.f) {
                        idx = g;
                        break;
                    }
                }
                result = idx;
            }
        }
        if (kSample && valid) a.assign[row] = result;
        if (kLogp && valid) a.logp[row] = logp_finish(lp_m, lp_s);
    }  // row tiles
}


// ---------------------------------------------------------------------------------------------
// launchers (header templates: every score_rows_*.cu instantiates the variants of its own model)
template <int CHUNK, int KIND, bool kSample, bool kScores, int THREADS, bool kSub = false, bool kMask = false>
static int launch_variant(dist_b200_ctx *ctx, const FeatList &feats, RowsArgs a, cudaStream_t s, const MaskList *masks = nullptr) {
    constexpr int kThreads = THREADS;
    const int G = a.G;
    const int nchunks = (G + CHUNK - 1) / CHUNK;
    const int Gpad = nchunks * CHUNK;
    size_t cache_floats = 0;
    int max_stride = 4;
    for (int f = 0; f < feats.n; ++f) {
        const int st = kind_stride(feats.f[f].kind, feats.f[f].vdim);
        cache_floats += static_cast<size_t>(Gpad) * st;
        if (st > max_stride) max_stride = st;
    }
    size_t fixed = (33 * kLgammaRowStride + 64 + Gpad) * sizeof(float);
    if (kScores) fixed += (kThreads / 32) * 32 * 33 * sizeof(float);
    if (kSub) fixed += sizeof(float) * nchunks * (CHUNK / kSubGroups + 1) * kThreads;
    else if (kSample && nchunks > 1) fixed += sizeof(float2) * kSlots * kThreads;
    a.resident = (!kSub && cache_floats * sizeof(float) <= kResidentBudget) ? 1 : 0;
    if (KIND >= 0 && !a.resident) return DIST_B200_ERR_UNSUPPORTED;  // caller falls back to the generic kernel
    a.stage_floats = CHUNK * max_stride;
    const size_t smem = fixed + (a.resident ? cache_floats : kStages * (static_cast<size_t>(a.stage_floats) + kThreads)) * sizeof(float);
    if (smem > 227 * 1024) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "score_rows: group caches exceed shared memory");
    auto run = [&](auto kern, auto... extra) -> int {
        DISTB200_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        int per_sm = 0;
        DISTB200_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, smem));
        if (per_sm < 1) per_sm = 1;
        const size_t ntiles = (a.N + kThreads - 1) / kThreads;
        const size_t max_blocks = static_cast<size_t>(ctx->sm_count) * per_sm;
        const unsigned grid = static_cast<unsigned>(ntiles < max_blocks ? ntiles : max_blocks);
        kern<<<grid, kThreads, smem, s>>>(feats, a, extra...);
        return DIST_B200_OK;
    };
    int rc;
    if constexpr (kMask) {
        void (*kern)(FeatList, RowsArgs, MaskList) = score_rows_kernel<CHUNK, KIND, kSample, kScores, kThreads, kSub, MaskList>;
        rc = run(kern, *masks);
    } else {
        void (*kern)(FeatList, RowsArgs) = score_rows_kernel<CHUNK, KIND, kSample, kScores, kThreads, kSub>;
        rc = run(kern);
    }
    if (rc) return rc;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("score_rows launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

int launch_crosscat_tile32(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s);
int launch_crosscat_tile64(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s);
int launch_crosscat_ksub(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s);

template <int CHUNK, int KIND, int THREADS>
static int launch_modes(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s) {
    const bool sample = a.assign != nullptr, scores = a.scores != nullptr;
    if (a.logp) {
        // a feature list does not fit a 128-group logp tile in registers: two 64-group tiles instead
        if constexpr (KIND < 0 && CHUNK == 128) return launch_crosscat_tile64(ctx, feats, a, s);
        else return launch_variant<CHUNK, KIND, false, false, THREADS>(ctx, feats, a, s);
    }
    if (sample && scores) return launch_variant<CHUNK, KIND, true, true, THREADS>(ctx, feats, a, s);
    if (sample) return launch_variant<CHUNK, KIND, true, false, THREADS>(ctx, feats, a, s);
    return launch_variant<CHUNK, KIND, false, true, THREADS>(ctx, feats, a, s);
}

// kSub launches: heads / tails of every BetaBernoulli feature of the list as two contiguous rows (the float4 caches hold
// them 16 bytes apart: the 16-group re-score would touch eight sectors per feature instead of two)
static __global__ void __launch_bounds__(256) bb_compact_kernel(const __grid_constant__ FeatList feats, int Gpad) {
    const FeatDesc &fd = feats.f[blockIdx.y];
    if (fd.kind != DIST_B200_BB) return;
    float *out = const_cast<float *>(static_cast<const float *>(fd.aux));
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < Gpad; g += gridDim.x * blockDim.x) {
        const float4 q = static_cast<const float4 *>(fd.params)[g];
        out[g] = q.x;
        out[Gpad + g] = q.y;
    }
}

// the kSub kernel serves feature lists whose 32-group-tile caches do not fit the resident budget
static bool ksub_wanted(const FeatList &feats, int G) {
    size_t cache_bytes = 0;
    for (int f = 0; f < feats.n; ++f)
        cache_bytes += sizeof(float) * static_cast<size_t>((G + 31) / 32 * 32) * kind_stride(feats.f[f].kind, feats.f[f].vdim);
    return cache_bytes > kResidentBudget;
}

// `local` = `feats` with every BetaBernoulli feature pointed at a compact copy of its caches for the kSub re-score
static int ksub_list(dist_b200_ctx *ctx, const FeatList &feats, int G, FeatList &local, cudaStream_t s) {
    const int Gpad = (G + 127) / 128 * 128;  // <= every feature's capacity (ensure_params pads to 128 groups)
    int n_bb = 0;
    for (int f = 0; f < feats.n; ++f) n_bb += feats.f[f].kind == DIST_B200_BB ? 1 : 0;
    if (int rc = grow(ctx, ctx->bbt, ctx->bbt_bytes, sizeof(float) * n_bb * 2 * Gpad)) return rc;
    local = feats;
    for (int f = 0, k = 0; f < local.n; ++f)
        if (local.f[f].kind == DIST_B200_BB) {
            local.f[f].aux = ctx->bbt + static_cast<size_t>(k++) * 2 * Gpad;
            local.f[f].cap = Gpad;
        }
    if (n_bb) {
        bb_compact_kernel<<<dim3((Gpad + 255) / 256, local.n), 256, 0, s>>>(local, Gpad);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("bb_compact launch: ") + cudaGetErrorString(e));
    }
    return DIST_B200_OK;
}

// Register tile.  G <= 128: the whole row in one tile (the sampler is then the reference's loops on registers);
// 64 < G <= 128 of a single feature runs 128-thread blocks, three per SM (12 warps instead of the 8 of one
// 256-thread block: the row-wide dependent chains of max / total / walk need the extra warps to hide their
// latency) -- DIST_B200_OPT_SMALL_TILE selects the alternatives for A/B runs.  G > 128: 32-group tiles.
// the feature-list (KIND = -1) instantiations are the heaviest to compile: they live in three translation units
// (score_rows.cu: 128-group tiles; score_rows_cc32.cu: 32-group tiles + kSub; score_rows_cc64.cu: 64-group tiles)
template <int KIND>
static int launch_tile32(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s) {
    if constexpr (KIND < 0) return launch_crosscat_tile32(ctx, feats, a, s);
    else return launch_modes<32, KIND, 256>(ctx, feats, a, s);
}
template <int KIND>
static int launch_tile64(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s) {
    if constexpr (KIND < 0) return launch_crosscat_tile64(ctx, feats, a, s);
    else return launch_modes<64, KIND, 256>(ctx, feats, a, s);
}

template <int KIND>
static int launch_tiers(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s) {
    if (a.G <= 32) return launch_tile32<KIND>(ctx, feats, a, s);
    if (a.G <= 64) return launch_tile64<KIND>(ctx, feats, a, s);
    if (a.G <= 128) {
        if (KIND < 0) return launch_modes<128, KIND, 128>(ctx, feats, a, s);
        const int v = ctx->opt[DIST_B200_OPT_SMALL_TILE];
        if (v == 1) return launch_modes<128, KIND, 256>(ctx, feats, a, s);
        if (v == 3) return launch_tile32<KIND>(ctx, feats, a, s);
        if (v != 2 && a.assign && !a.scores) {
            // sampling only: the register tile is G rounded up to 16 groups (G = 100 pads to 112 instead of 128:
            // every padded group is a wasted MUFU.EX2)
            if (a.G <= 80) return launch_variant<80, KIND, true, false, 128>(ctx, feats, a, s);
            if (a.G <= 96) return launch_variant<96, KIND, true, false, 128>(ctx, feats, a, s);
            if (a.G <= 112) return launch_variant<112, KIND, true, false, 128>(ctx, feats, a, s);
        }
        return launch_modes<128, KIND, 128>(ctx, feats, a, s);
    }
    // measured at c2, sampling only: 32-group tiles 0.748 ms, 64-group tiles 0.774 ms; with the [N][G] scores also written
    // (HBM-store bound): 32-group tiles 1.215 ms, 64-group tiles 1.098 ms -- a store instruction then covers 256-byte runs of
    // a row instead of 128-byte ones (DIST_B200_OPT_ROW_TILE = 32 / 64 forces either for A/B runs)
    if constexpr (KIND < 0) if (a.assign && !a.scores && !a.n_push && ctx->opt[DIST_B200_OPT_ROW_TILE] == 0) {
        // feature lists too large to keep resident (a cross-cat kind): the 128-group streaming tiles of the G <= 128 case
        // with sub-slot bookkeeping (kSub); measured at 256 features against the 32-group tiles + per-cell re-score of a whole
        // slot from global memory: G = 256, 1M rows 53.4 -> 14.9 ms; G = 1024, 100k rows 15.3 -> 7.19 ms
        if (ksub_wanted(feats, a.G)) {
            FeatList local;
            if (int rc = ksub_list(ctx, feats, a.G, local, s)) return rc;
            const int rc = launch_crosscat_ksub(ctx, local, a, s);
            if (rc != DIST_B200_ERR_UNSUPPORTED) return rc;  // (too many groups for the sub-slot sums in shared memory)
        }
    }
    const int tile = ctx->opt[DIST_B200_OPT_ROW_TILE] ? ctx->opt[DIST_B200_OPT_ROW_TILE] : (a.scores ? 64 : 32);
    if (tile == 64) return launch_tile64<KIND>(ctx, feats, a, s);
    return launch_tile32<KIND>(ctx, feats, a, s);
}

// one per model, each in its own translation unit (parallel compilation)
int launch_single_nich(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s);
int launch_single_gp(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s);
int launch_single_bnb(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s);
int launch_single_bb(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s);
int launch_single_dd(dist_b200_ctx *ctx, const FeatList &feats, const RowsArgs &a, cudaStream_t s);

}  // namespace distb200
