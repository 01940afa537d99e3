// nich_rows.cu -- NormalInverseChiSq, one feature, G > 128, sampling only: the c2 shape (1M rows x 1024 groups).
//
// Same algorithm as score_rows_kernel<32, nich packed> (score_rows.cuh: rows on lanes, 32-group register tiles,
// per-tile (max, sum exp) pairs merged into 16 slots, walk over the slots, re-score of the selected slot), rebuilt
// around what its ncu capture showed (profiles/r02_c2_nich_packed.txt): the MUFU pipe it is bound by was 77 % busy
// while the stall reasons were MIO throttle + short scoreboard, because the shared-memory pipe was almost as loaded
// as the MUFU pipe -- a warp-wide LDS.128 occupies it for four wavefronts even when all lanes read the same address,
// i.e. 4 cycles per (warp, cell) against MUFU's 16 cycles per (warp, cell) / 4 sub-partitions, and the re-score pass
// read with up to 32-way bank conflicts (every lane its own slot, all slots at the same bank offset).  Here
//   * every thread carries TWO rows, so a group's parameters are loaded once per two cells (half the wavefronts);
//   * the block's parameter copy is skewed by 16 bytes per slot, so the lanes of the re-score pass, which sit in
//     different slots, mostly hit different banks;
//   * 6 of every 16 pairs of softmax exponentials are evaluated on the FMA pipe (poly_ex2_pair, numerics.cuh): with two
//     MUFU per cell (LG2 + EX2) the kernel sat at 89 % XU-pipe activity while the FMA pipe idled at 20 %
//     (profiles/r02_c2_nich_rows.txt); same-box A/B 0.571 -> 0.521 ms;
//   * rows are dealt to the blocks in half-tiles, so the per-SM loads differ by half a tile (see the kernel).
// The default is now nich_rows2_kernel below (static softmax reference, four rows per thread: 0.522 -> 0.482 ms);
// nich_rows_kernel stays selectable (DIST_B200_OPT_NICH_PACKED = 3) and is what the paragraphs above describe.
// Cell arithmetic is the packed fp32x2 form of nich.cc:59-65 (see accumulate_feature, kKindNichPacked): two groups per
// FADD2 / FMUL2 / FFMA2, every product and sum rounded as the reference's unfused expression.
#include "score_rows.cuh"

namespace distb200 {

constexpr int kNrThreads = 256;
constexpr int kNrChunk = 32;
constexpr int kNrRows = 2;  // rows per thread
constexpr int kNrPolyDefault = 6;  // pairs of every 16 whose exp2 runs on the FMA pipe (poly_ex2_pair)

struct NichRowsArgs {
    int G;
    size_t N;
    const float4 *params;  // {mean, precision, log_coeff * ln 2, score} per group (capacity padded to 128 groups)
    const float *prior;    // [G] or nullptr
    const float *values;
    const float *u;
    int32_t *assign;
    float *logp;           // nich_logp_kernel: log sum_g exp(prior + score) per row
};

// geometry of the block-private parameter copy and the per-row slot pairs
struct NichGeom {
    int G, nchunks, cps, nslots, slot_groups;
    const float4 *caches;  // pair p of groups at float4 index 2 p + (2 p) / slot_groups (one float4 of skew per slot)
    float2 *slots;         // [R][kSlots][kNrThreads] {negated scaled max, sum}
};

// R rows per thread (row r of the thread = half-tile r of the tile: 256 consecutive rows) against all groups, then the
// draw.  R = 2 is the steady state; R = 1 evaluates a block's odd last half-tile at half the cost (see the kernel).
template <int kPoly, int R>
__device__ __forceinline__ void nich_tile(const NichGeom &g, const float (&xrow)[R], const float (&urow)[R], const size_t (&row)[R],
                                          size_t N, int32_t *__restrict__ assign) {
    const int tid = threadIdx.x;
    const uint64_t one2 = f2_pack(1.f, 1.f), l2e2 = f2_pack(kLog2e, kLog2e);
    uint64_t x2[R];
    float slot_m[R], slot_s[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        x2[r] = f2_pack(xrow[r], xrow[r]);
        slot_m[r] = INFINITY;  // negated scaled max of the slot being merged
        slot_s[r] = 0.f;
    }
    // one 32-group tile of one row: acc[j] = prior + score + log_coeff * fast_log(1 + precision * (x - mean)^2)
    auto score_tile = [&](const float4 *p4, int r, float (&acc)[kNrChunk]) {
#pragma unroll
        for (int j = 0; j < kNrChunk; j += 2) {
            const float4 qa = p4[j], qb = p4[j + 1];
            const uint64_t d2 = f2_add(x2[r], f2_pack(qa.x, qa.y));
            const uint64_t z2 = f2_fma(f2_mul(f2_pack(qa.z, qa.w), f2_mul(d2, d2)), one2, one2);  // unfused 1 + w (see score_rows.cuh)
            float za, zb;
            f2_unpack(z2, za, zb);
            f2_unpack(f2_fma(f2_pack(qb.x, qb.y), f2_pack(fast_log2_cell(za), fast_log2_cell(zb)), f2_pack(qb.z, qb.w)), acc[j], acc[j + 1]);
        }
    };
    for (int c = 0; c < g.nchunks; ++c) {
        const float4 *p4 = g.caches + c * kNrChunk + c / g.cps;
        float acc[R][kNrChunk];
#pragma unroll
        for (int j = 0; j < kNrChunk; j += 2) {  // parameters once, all rows
            const float4 qa = p4[j], qb = p4[j + 1];
            const uint64_t nm2 = f2_pack(qa.x, qa.y), pr2 = f2_pack(qa.z, qa.w), co2 = f2_pack(qb.x, qb.y), sc2 = f2_pack(qb.z, qb.w);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const uint64_t d2 = f2_add(x2[r], nm2);
                const uint64_t z2 = f2_fma(f2_mul(pr2, f2_mul(d2, d2)), one2, one2);
                float za, zb;
                f2_unpack(z2, za, zb);
                f2_unpack(f2_fma(co2, f2_pack(fast_log2_cell(za), fast_log2_cell(zb)), sc2), acc[r][j], acc[r][j + 1]);
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float m = acc[r][0];
#pragma unroll
            for (int j = 1; j < kNrChunk; ++j) m = fmaxf(m, acc[r][j]);
            const float nm = -m * kLog2e;  // rounded once: every later rescale is a difference of these values
            const uint64_t nm2 = f2_pack(nm, nm);
            uint64_t s2 = f2_pack(0.f, 0.f);
#pragma unroll
            for (int j = 0; j < kNrChunk; j += 2) {
                const uint64_t e2 = f2_fma(f2_pack(acc[r][j], acc[r][j + 1]), l2e2, nm2);
                if (((j / 2) * kPoly) % 16 < kPoly) {  // kPoly of 16 pairs, evenly spread between the MUFU pairs
                    s2 = f2_add(s2, poly_ex2_pair(e2));
                } else {
                    float ea, eb;
                    f2_unpack(e2, ea, eb);
                    s2 = f2_add(s2, f2_pack(mufu_ex2(ea), mufu_ex2(eb)));
                }
            }
            float se, so;
            f2_unpack(s2, se, so);
            const float s = se + so;
            const float dlt = slot_m[r] - nm;
            const float e = mufu_ex2(-fabsf(dlt));
            slot_s[r] = dlt > 0.f ? fmaf(slot_s[r], e, s) : fmaf(s, e, slot_s[r]);
            slot_m[r] = fminf(slot_m[r], nm);
            if ((c + 1) % g.cps == 0 || c + 1 == g.nchunks) {
                g.slots[(r * kSlots + c / g.cps) * kNrThreads + tid] = make_float2(slot_m[r], slot_s[r]);
                slot_m[r] = INFINITY;
                slot_s[r] = 0.f;
            }
        }
    }
    // per row: total over the slots, walk to the slot holding u * total, re-score that slot, walk its cells
#pragma unroll
    for (int r = 0; r < R; ++r) {
        float2 *sl = g.slots + (r * kSlots) * kNrThreads + tid;
        float mm = INFINITY;
        for (int k = 0; k < g.nslots; ++k) mm = fminf(mm, sl[k * kNrThreads].x);
        float total = 0.f;
        for (int k = 0; k < g.nslots; ++k) {
            const float2 ms = sl[k * kNrThreads];
            const float w = ms.y * mufu_ex2(mm - ms.x);
            sl[k * kNrThreads].y = w;
            total += w;
        }
        float t = total * urow[r];
        int sel = g.nslots - 1;
        for (int k = 0; k < g.nslots; ++k) {
            const float w = sl[k * kNrThreads].y;
            if (t <= w) {
                sel = k;
                break;
            }
            if (k + 1 < g.nslots) t -= w;
        }
        int count = 0;
        for (int cc = 0; cc < g.cps; ++cc) {
            const int c = sel * g.cps + cc;
            if (c >= g.nchunks) break;
            float acc[kNrChunk];
            score_tile(g.caches + c * kNrChunk + sel, r, acc);
#pragma unroll
            for (int j = 0; j < kNrChunk; ++j) {
                t -= mufu_ex2(fmaf(acc[j], kLog2e, mm));
                count += 1 - static_cast<int>(__float_as_uint(t) >> 31);  // t >= +0 continues (an exact 0: a near-tie)
            }
        }
        if (row[r] < N) assign[row[r]] = min(sel * g.slot_groups + count, g.G - 1);
    }
}

// Work split: the rows are cut into HALF-TILES of 256 (one row per thread) and every block takes a contiguous run of
// them, as even as the count allows (the runs differ by at most one half-tile).  A block evaluates its run two
// half-tiles at a time (two rows per thread) and an odd last one alone at half the cost, so the blocks' loads differ by
// half a tile at most instead of a whole one: at c2 (1M rows, 296 blocks: 13.2 half-tiles per block) the slowest SM
// runs 13.5 tile-halves instead of 14.
template <int kPoly>
__global__ void __launch_bounds__(kNrThreads, 2) nich_rows_kernel(const NichRowsArgs a) {
    extern __shared__ __align__(16) float smem[];
    NichGeom g;
    g.G = a.G;
    g.nchunks = (a.G + kNrChunk - 1) / kNrChunk;
    const int Gpad = g.nchunks * kNrChunk;
    g.cps = (g.nchunks + kSlots - 1) / kSlots;  // chunks per slot
    g.nslots = (g.nchunks + g.cps - 1) / g.cps;
    g.slot_groups = g.cps * kNrChunk;
    float4 *caches = reinterpret_cast<float4 *>(smem);
    g.caches = caches;
    g.slots = reinterpret_cast<float2 *>(caches + Gpad + g.nslots);
    const int tid = threadIdx.x;

    // block-private parameter copy: prior folded into the score, padded groups -inf (they borrow group 0's mean /
    // precision / coefficient so the term stays finite-or-(-inf) exactly as for a real group), pairs interleaved
    for (int p = tid; p < Gpad / 2; p += kNrThreads) {
        float4 q[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int gi = 2 * p + k;
            q[k] = a.params[gi < a.G ? gi : 0];
            q[k].w = gi < a.G ? q[k].w + (a.prior ? a.prior[gi] : 0.f) : -INFINITY;
        }
        const int at = 2 * p + (2 * p) / g.slot_groups;
        caches[at] = make_float4(-q[0].x, -q[1].x, q[0].y, q[1].y);
        caches[at + 1] = make_float4(q[0].z, q[1].z, q[0].w, q[1].w);
    }
    __syncthreads();

    const size_t nhalf = (a.N + kNrThreads - 1) / kNrThreads;
    const size_t base = nhalf / gridDim.x, rem = nhalf % gridDim.x;
    const size_t h0 = blockIdx.x * base + (blockIdx.x < rem ? blockIdx.x : rem);
    const size_t h1 = h0 + base + (blockIdx.x < rem ? 1 : 0);
    // the next tile's rows are requested while the current tile is evaluated (2 048 cells per row: the load latency --
    // HBM, or PCIe when the host entry hands the kernel page-locked host buffers -- disappears behind them)
    float xnext[kNrRows], unext[kNrRows];
    auto fetch = [&](size_t h) {
#pragma unroll
        for (int r = 0; r < kNrRows; ++r) {
            const size_t rw = (h + r) * kNrThreads + tid;
            const size_t rr = rw < a.N ? rw : a.N - 1;  // clamp: compute on a real row, discard the result
            xnext[r] = __ldg(a.values + rr);
            unext[r] = __ldg(a.u + rr);
        }
    };
    if (h0 < h1) fetch(h0);
    size_t h = h0;
    for (; h + kNrRows <= h1; h += kNrRows) {
        size_t row[kNrRows];
        float xrow[kNrRows], urow[kNrRows];
#pragma unroll
        for (int r = 0; r < kNrRows; ++r) {
            row[r] = (h + r) * kNrThreads + tid;
            xrow[r] = xnext[r];
            urow[r] = unext[r];
        }
        if (h + kNrRows < h1) fetch(h + kNrRows);
        nich_tile<kPoly, kNrRows>(g, xrow, urow, row, a.N, a.assign);
    }
    if (h < h1) {  // odd half-tile left: one row per thread
        const size_t row[1] = {h * kNrThreads + tid};
        const float xrow[1] = {xnext[0]}, urow[1] = {unext[0]};
        nich_tile<kPoly, 1>(g, xrow, urow, row, a.N, a.assign);
    }
}

// ------------------------------------------------------------------------------------------------
// nich_rows2_kernel: the same cells against a STATIC reference instead of the row's running maximum.
//   score_g(x) = sc_g + co_g ln z <= sc_g   (co_g < 0, z >= 1),   sc_g = prior_g + score_g of the group,
// so M* = max_g sc_g bounds every score of every row, and the softmax weights can be formed directly as
//   e_g = 2^(co_g lg2 z + (sc_g - M*) log2 e)  in (0, 1]
// in the FFMA2 that used to produce the score: no per-tile maximum (FMNMX3), no second FFMA2 for the exponent, no
// (max, sum) merges, no 64 live score registers -- a thread carries FOUR rows (a group's parameters are loaded once
// per four cells) and a slot is a plain sum.  Ratios of weights do not depend on the reference, and for every term that
// matters (exponent near 0) both summands of the FFMA2 are small, so it is rounded finer than a score near -50 was.
// What a static reference cannot promise is range: a row whose best score lies far below M* (an outlier to every group)
// would lose its small terms to underflow.  Rows whose total comes out below 2^-40 (flushed terms are then < 2^-86 of
// the total) are therefore re-evaluated by nich2_row_exact with their own maximum; with the empty group a Pitman-Yor
// mixture always carries (broad prior predictive), such rows do not occur in practice.
constexpr int kN2Rows = 4;
constexpr int kN2PolyDefault = 5;  // same-box sweep at c2: 0 / 3 / 4 / 5 / 6 / 8 / 10 / 12 of 16 -> 0.534 / 0.502 / 0.494 / 0.482 / 0.507 / 0.502 / 0.504 / 0.537 ms
constexpr float kN2Redo = 9.094947e-13f;  // 2^-40

struct Nich2Geom {
    int G, nchunks, cps, nslots, slot_groups;
    const float4 *caches;  // pair p at float4 index 2 p + (2 p) / slot_groups: {-mean a, -mean b, prec a, prec b}, {co a, co b, sc' a, sc' b}
    float *slots;          // [R][kSlots][kNrThreads] sums of weights
};

// exponent of one cell: co lg2(fast_log argument) + sc'  (the unfused 1 + prec d^2 of nich.cc:59-65, table-step mantissa)
__device__ __forceinline__ float nich2_arg(const Nich2Geom &g, int gi, float x) {
    const int p = gi >> 1, at = 2 * p + (2 * p) / g.slot_groups;
    const float4 qa = g.caches[at], qb = g.caches[at + 1];
    const bool hi = gi & 1;
    const float d = x + (hi ? qa.y : qa.x);
    const float z = __fadd_rn(1.f, __fmul_rn(hi ? qa.w : qa.z, __fmul_rn(d, d)));
    return fmaf(hi ? qb.y : qb.x, fast_log2_cell(z), hi ? qb.w : qb.z);
}

// scores_to_likelihoods + sample_from_likelihoods with the row's own maximum (random.cc:94-106, random.hpp:315-333)
__device__ __noinline__ int nich2_row_exact(const Nich2Geom &g, float x, float u) {
    float m = -INFINITY;
    for (int gi = 0; gi < g.G; ++gi) m = fmaxf(m, nich2_arg(g, gi, x));
    float total = 0.f;
    for (int gi = 0; gi < g.G; ++gi) total += mufu_ex2(nich2_arg(g, gi, x) - m);
    float t = total * u;
    int count = 0;
    for (int gi = 0; gi < g.G; ++gi) {
        t -= mufu_ex2(nich2_arg(g, gi, x) - m);
        count += 1 - static_cast<int>(__float_as_uint(t) >> 31);
    }
    return min(count, g.G - 1);
}

template <int kPoly, int R>
__device__ __forceinline__ void nich2_tile(const Nich2Geom &g, const float (&xrow)[R], const float (&urow)[R], const size_t (&row)[R],
                                           size_t N, int32_t *__restrict__ assign) {
    const int tid = threadIdx.x;
    const uint64_t one2 = f2_pack(1.f, 1.f);
    uint64_t x2[R], sa[R], sb[R];  // two partial sums per row: even / odd pairs
#pragma unroll
    for (int r = 0; r < R; ++r) {
        x2[r] = f2_pack(xrow[r], xrow[r]);
        sa[r] = sb[r] = f2_pack(0.f, 0.f);
    }
    // weights of one pair of groups for row r; kPoly of every 16 pairs on the FMA pipe (same choice in both passes)
    auto pair_weights = [&](const float4 &qa, const float4 &qb, int r, int j) {
        const uint64_t d2 = f2_add(x2[r], f2_pack(qa.x, qa.y));
        const uint64_t z2 = f2_fma(f2_mul(f2_pack(qa.z, qa.w), f2_mul(d2, d2)), one2, one2);  // unfused 1 + w (see score_rows.cuh)
        float za, zb;
        f2_unpack(z2, za, zb);
        const uint64_t a2 = f2_fma(f2_pack(qb.x, qb.y), f2_pack(fast_log2_cell(za), fast_log2_cell(zb)), f2_pack(qb.z, qb.w));
        if (((j / 2) * kPoly) % 16 < kPoly) return poly_ex2_pair(a2);
        float ea, eb;
        f2_unpack(a2, ea, eb);
        return f2_pack(mufu_ex2(ea), mufu_ex2(eb));
    };
    for (int c = 0; c < g.nchunks; ++c) {
        const float4 *p4 = g.caches + c * kNrChunk + c / g.cps;
#pragma unroll
        for (int j = 0; j < kNrChunk; j += 2) {  // parameters once, all rows
            const float4 qa = p4[j], qb = p4[j + 1];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const uint64_t e2 = pair_weights(qa, qb, r, j);
                if (j & 2) sb[r] = f2_add(sb[r], e2);
                else sa[r] = f2_add(sa[r], e2);
            }
        }
        if ((c + 1) % g.cps == 0 || c + 1 == g.nchunks) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                float a0, a1;
                f2_unpack(f2_add(sa[r], sb[r]), a0, a1);
                g.slots[(r * kSlots + c / g.cps) * kNrThreads + tid] = a0 + a1;
                sa[r] = sb[r] = f2_pack(0.f, 0.f);
            }
        }
    }
    // per row: total over the slots, walk to the slot holding u * total, re-form that slot's weights, walk its cells
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const float *sl = g.slots + (r * kSlots) * kNrThreads + tid;
        float total = 0.f;
        for (int k = 0; k < g.nslots; ++k) total += sl[k * kNrThreads];
        int result;
        if (!(total >= kN2Redo)) {
            result = nich2_row_exact(g, xrow[r], urow[r]);  // an outlier to every group: its own maximum
        } else {
            float t = total * urow[r];
            int sel = g.nslots - 1;
            for (int k = 0; k < g.nslots; ++k) {
                const float w = sl[k * kNrThreads];
                if (t <= w) {
                    sel = k;
                    break;
                }
                if (k + 1 < g.nslots) t -= w;
            }
            int count = 0;
            for (int cc = 0; cc < g.cps; ++cc) {
                const int c = sel * g.cps + cc;
                if (c >= g.nchunks) break;
                const float4 *p4 = g.caches + c * kNrChunk + sel;
#pragma unroll
                for (int j = 0; j < kNrChunk; j += 2) {
                    float ea, eb;
                    f2_unpack(pair_weights(p4[j], p4[j + 1], r, j), ea, eb);
                    t -= ea;
                    count += 1 - static_cast<int>(__float_as_uint(t) >> 31);  // t >= +0 continues (an exact 0: a near-tie)
                    t -= eb;
                    count += 1 - static_cast<int>(__float_as_uint(t) >> 31);
                }
            }
            result = min(sel * g.slot_groups + count, g.G - 1);
        }
        if (row[r] < N) assign[row[r]] = result;
    }
}

// rows are dealt in units of 256 (one row per thread) as in nich_rows_kernel; a block evaluates its run four units at a
// time and the remainder with the two- and one-row forms
template <int kPoly, int RT, int kBlocks>
__global__ void __launch_bounds__(kNrThreads, kBlocks) nich_rows2_kernel(const NichRowsArgs a) {
    extern __shared__ __align__(16) float smem[];
    __shared__ float red[kNrThreads / 32];
    Nich2Geom g;
    g.G = a.G;
    g.nchunks = (a.G + kNrChunk - 1) / kNrChunk;
    const int Gpad = g.nchunks * kNrChunk;
    g.cps = (g.nchunks + kSlots - 1) / kSlots;
    g.nslots = (g.nchunks + g.cps - 1) / g.cps;
    g.slot_groups = g.cps * kNrChunk;
    float4 *caches = reinterpret_cast<float4 *>(smem);
    g.caches = caches;
    g.slots = reinterpret_cast<float *>(caches + Gpad + g.nslots);
    const int tid = threadIdx.x;

    // this block's run of 256-row units, and the request for its first piece before anything else
    const size_t nunits = (a.N + kNrThreads - 1) / kNrThreads;
    const size_t base = nunits / gridDim.x, rem = nunits % gridDim.x;
    const size_t h0 = blockIdx.x * base + (blockIdx.x < rem ? blockIdx.x : rem);
    const size_t h1 = h0 + base + (blockIdx.x < rem ? 1 : 0);
    float xnext[RT], unext[RT];
    auto fetch = [&](size_t hh, int cnt) {
#pragma unroll
        for (int r = 0; r < RT; ++r) {
            if (r < cnt) {
                const size_t rw = (hh + r) * kNrThreads + tid;
                const size_t rr = rw < a.N ? rw : a.N - 1;  // clamp: compute on a real row, discard the result
                xnext[r] = __ldg(a.values + rr);
                unext[r] = __ldg(a.u + rr);
            }
        }
    };
    auto piece = [&](size_t hh, int lead_left) -> int {  // units of the next piece: 2 / 1 while leading units remain, then RT
        if (hh >= h1) return 0;
        if (RT >= 4 && lead_left >= 2) return 2;
        if (lead_left >= 1) return 1;
        return RT;
    };
    size_t h = h0;
    int lead = static_cast<int>((h1 - h0) % RT);
    int n = piece(h, lead);
#pragma unroll
    for (int r = 0; r < RT; ++r) xnext[r] = unext[r] = 0.f;
    if (n) fetch(h, n);

    // M* = max over the real groups of prior + score (the same value in every block)
    float m = -INFINITY;
    for (int gi = tid; gi < a.G; gi += kNrThreads) m = fmaxf(m, a.params[gi].w + (a.prior ? a.prior[gi] : 0.f));
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((tid & 31) == 0) red[tid >> 5] = m;
    __syncthreads();
    m = red[0];
#pragma unroll
    for (int w = 1; w < kNrThreads / 32; ++w) m = fmaxf(m, red[w]);
    // block-private parameter copy: padded groups get sc' = -inf and borrow group 0's mean / precision / coefficient
    for (int p = tid; p < Gpad / 2; p += kNrThreads) {
        float4 q[2];
        float sc[2], co[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int gi = 2 * p + k;
            q[k] = a.params[gi < a.G ? gi : 0];
            const float s = q[k].w + (a.prior ? a.prior[gi < a.G ? gi : 0] : 0.f);
            sc[k] = gi < a.G ? (s - m) * kLog2e : -INFINITY;
            co[k] = static_cast<float>(static_cast<double>(q[k].z) * 1.4426950408889634);  // log_coeff ln 2 -> log_coeff (lg2 scale)
        }
        const int at = 2 * p + (2 * p) / g.slot_groups;
        caches[at] = make_float4(-q[0].x, -q[1].x, q[0].y, q[1].y);
        caches[at + 1] = make_float4(co[0], co[1], sc[0], sc[1]);
    }
    __syncthreads();

    // the short leading pieces (run length mod RT: two units, then one) come FIRST: the block's first request for rows is
    // small -- when the rows live in page-locked host memory every block's first fetch crosses PCIe with nothing to hide
    // behind -- and the first full tile's rows arrive while the leading piece is evaluated
    while (n) {
        size_t row[RT];
        float xrow[RT], urow[RT];
#pragma unroll
        for (int r = 0; r < RT; ++r) {
            row[r] = (h + r) * kNrThreads + tid;
            xrow[r] = xnext[r];
            urow[r] = unext[r];
        }
        const int nc = n;
        h += nc;
        if (nc < RT) lead -= nc;
        n = piece(h, lead);
        if (n) fetch(h, n);
        if (nc == RT) {
            nich2_tile<kPoly, RT>(g, xrow, urow, row, a.N, a.assign);
        } else if (nc == 2) {
            const size_t row2[2] = {row[0], row[1]};
            const float x2[2] = {xrow[0], xrow[1]}, u2[2] = {urow[0], urow[1]};
            nich2_tile<kPoly, 2>(g, x2, u2, row2, a.N, a.assign);
        } else {
            const size_t row1[1] = {row[0]};
            const float x1[1] = {xrow[0]}, u1[1] = {urow[0]};
            nich2_tile<kPoly, 1>(g, x1, u1, row1, a.N, a.assign);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// nich_logp_kernel: the row log-normaliser with nich_rows2_kernel's static reference.  The weights it sums are
// e_g = 2^((s_g - M*) log2 e), so logp = M* + ln(sum_g e_g) needs no slots and no walk, and a thread carries its four rows
// across all the tiles.  Rows whose sum falls below 2^-40 are re-evaluated with their own maximum (nich2_row_logp).
__device__ __noinline__ float nich2_row_logp(const Nich2Geom &g, float x) {  // ln sum_g 2^(arg_g), arg on the lg2 scale
    float m = -INFINITY;
    for (int gi = 0; gi < g.G; ++gi) m = fmaxf(m, nich2_arg(g, gi, x));
    if (m == -INFINITY) return -INFINITY;
    float total = 0.f;
    for (int gi = 0; gi < g.G; ++gi) total += mufu_ex2(nich2_arg(g, gi, x) - m);
    return (m + log2f(total)) * kLn2;
}

template <int kPoly>
__global__ void __launch_bounds__(kNrThreads, 2) nich_logp_kernel(const NichRowsArgs a) {
    extern __shared__ __align__(16) float smem[];
    __shared__ float red[kNrThreads / 32];
    constexpr int R = kN2Rows;
    Nich2Geom g;
    g.G = a.G;
    g.nchunks = (a.G + kNrChunk - 1) / kNrChunk;
    const int Gpad = g.nchunks * kNrChunk;
    g.cps = (g.nchunks + kSlots - 1) / kSlots;
    g.nslots = (g.nchunks + g.cps - 1) / g.cps;
    g.slot_groups = g.cps * kNrChunk;
    float4 *caches = reinterpret_cast<float4 *>(smem);
    g.caches = caches;
    g.slots = nullptr;
    const int tid = threadIdx.x;
    // M* as in nich_rows2_kernel; 0 when every group sits at -inf, so that the weights are 0 and not NaN
    float m = -INFINITY;
    for (int gi = tid; gi < a.G; gi += kNrThreads) m = fmaxf(m, a.params[gi].w + (a.prior ? a.prior[gi] : 0.f));
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((tid & 31) == 0) red[tid >> 5] = m;
    __syncthreads();
    m = red[0];
#pragma unroll
    for (int w = 1; w < kNrThreads / 32; ++w) m = fmaxf(m, red[w]);
    if (m == -INFINITY) m = 0.f;
    for (int p = tid; p < Gpad / 2; p += kNrThreads) {  // the block-private copy of nich_rows2_kernel
        float4 q[2];
        float sc[2], co[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int gi = 2 * p + k;
            q[k] = a.params[gi < a.G ? gi : 0];
            const float s = q[k].w + (a.prior ? a.prior[gi < a.G ? gi : 0] : 0.f);
            sc[k] = gi < a.G ? (s - m) * kLog2e : -INFINITY;
            co[k] = static_cast<float>(static_cast<double>(q[k].z) * 1.4426950408889634);
        }
        const int at = 2 * p + (2 * p) / g.slot_groups;
        caches[at] = make_float4(-q[0].x, -q[1].x, q[0].y, q[1].y);
        caches[at + 1] = make_float4(co[0], co[1], sc[0], sc[1]);
    }
    __syncthreads();

    const uint64_t one2 = f2_pack(1.f, 1.f);
    const size_t tile_rows = static_cast<size_t>(kNrThreads) * R;
    const size_t ntiles = (a.N + tile_rows - 1) / tile_rows;
    for (size_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        size_t row[R];
        float x[R];
        uint64_t x2[R], sa[R], sb[R];  // two partial sums per row: even / odd pairs
#pragma unroll
        for (int r = 0; r < R; ++r) {
            row[r] = t * tile_rows + static_cast<size_t>(r) * kNrThreads + tid;
            x[r] = __ldg(a.values + (row[r] < a.N ? row[r] : a.N - 1));  // clamp: compute on a real row, discard the result
            x2[r] = f2_pack(x[r], x[r]);
            sa[r] = sb[r] = f2_pack(0.f, 0.f);
        }
        for (int c = 0; c < g.nchunks; ++c) {
            const float4 *p4 = g.caches + c * kNrChunk + c / g.cps;
#pragma unroll
            for (int j = 0; j < kNrChunk; j += 2) {  // parameters once, all rows; the weights of nich2_tile
                const float4 qa = p4[j], qb = p4[j + 1];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const uint64_t d2 = f2_add(x2[r], f2_pack(qa.x, qa.y));
                    const uint64_t z2 = f2_fma(f2_mul(f2_pack(qa.z, qa.w), f2_mul(d2, d2)), one2, one2);
                    float za, zb;
                    f2_unpack(z2, za, zb);
                    const uint64_t a2 = f2_fma(f2_pack(qb.x, qb.y), f2_pack(fast_log2_cell(za), fast_log2_cell(zb)), f2_pack(qb.z, qb.w));
                    uint64_t e2;
                    if (((j / 2) * kPoly) % 16 < kPoly) {
                        e2 = poly_ex2_pair(a2);
                    } else {
                        float ea, eb;
                        f2_unpack(a2, ea, eb);
                        e2 = f2_pack(mufu_ex2(ea), mufu_ex2(eb));
                    }
                    if (j & 2) sb[r] = f2_add(sb[r], e2);
                    else sa[r] = f2_add(sa[r], e2);
                }
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float a0, a1;
            f2_unpack(f2_add(sa[r], sb[r]), a0, a1);
            const float total = a0 + a1;
            const float lp = total >= kN2Redo ? m + logf(total) : m + nich2_row_logp(g, x[r]);  // an outlier to every group
            if (row[r] < a.N) a.logp[row[r]] = lp;
        }
    }
}

int launch_nich_logp(dist_b200_ctx *ctx, const float4 *params, const void *column, int G, size_t N, const float *prior,
                     float *logp, cudaStream_t s) {
    if (G <= 128 || !logp) return DIST_B200_ERR_UNSUPPORTED;
    const int nchunks = (G + kNrChunk - 1) / kNrChunk;
    const int cps = (nchunks + kSlots - 1) / kSlots;
    const int nslots = (nchunks + cps - 1) / cps;
    const size_t smem = sizeof(float4) * (nchunks * kNrChunk + nslots);
    if (smem > 220 * 1024) return DIST_B200_ERR_UNSUPPORTED;
    NichRowsArgs a{};
    a.G = G;
    a.N = N;
    a.params = params;
    a.prior = prior;
    a.values = static_cast<const float *>(column);
    a.logp = logp;
    auto kern = nich_logp_kernel<kN2PolyDefault>;
    DISTB200_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    int per_sm = 0;
    DISTB200_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kNrThreads, smem));
    if (per_sm < 1) per_sm = 1;
    const size_t tile_rows = static_cast<size_t>(kNrThreads) * kN2Rows;
    const size_t ntiles = (N + tile_rows - 1) / tile_rows;
    const size_t cap = static_cast<size_t>(ctx->sm_count) * per_sm;
    kern<<<static_cast<unsigned>(ntiles < cap ? ntiles : cap), kNrThreads, smem, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("nich_logp launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

template <int kPoly, int RT = kN2Rows, int kBlocks = 2>
static int launch_nich_rows2_t(dist_b200_ctx *ctx, const NichRowsArgs &a, size_t smem, cudaStream_t s) {
    smem -= sizeof(float) * (kN2Rows - RT) * kSlots * kNrThreads;
    DISTB200_CUDA(ctx, cudaFuncSetAttribute(nich_rows2_kernel<kPoly, RT, kBlocks>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    int per_sm = 0;
    DISTB200_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nich_rows2_kernel<kPoly, RT, kBlocks>, kNrThreads, smem));
    if (per_sm < 1) per_sm = 1;
    const size_t tile_rows = static_cast<size_t>(kNrThreads) * RT;
    const size_t ntiles = (a.N + tile_rows - 1) / tile_rows;
    const size_t cap = static_cast<size_t>(ctx->sm_count) * per_sm;
    nich_rows2_kernel<kPoly, RT, kBlocks><<<static_cast<unsigned>(ntiles < cap ? ntiles : cap), kNrThreads, smem, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("nich_rows2 launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

template <int kPoly>
static int launch_nich_rows_t(dist_b200_ctx *ctx, const NichRowsArgs &a, size_t smem, cudaStream_t s) {
    DISTB200_CUDA(ctx, cudaFuncSetAttribute(nich_rows_kernel<kPoly>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    int per_sm = 0;
    DISTB200_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nich_rows_kernel<kPoly>, kNrThreads, smem));
    if (per_sm < 1) per_sm = 1;
    const size_t tile_rows = static_cast<size_t>(kNrThreads) * kNrRows;
    const size_t ntiles = (a.N + tile_rows - 1) / tile_rows;
    const size_t cap = static_cast<size_t>(ctx->sm_count) * per_sm;
    nich_rows_kernel<kPoly><<<static_cast<unsigned>(ntiles < cap ? ntiles : cap), kNrThreads, smem, s>>>(a);  // N > 0: the callers return early on an empty batch
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("nich_rows launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

// DIST_B200_ERR_UNSUPPORTED: the caller takes the generic kernel
int launch_nich_rows(dist_b200_ctx *ctx, const float4 *params, const void *column, int G, size_t N, const float *prior,
                     const float *u, int32_t *assign, cudaStream_t s) {
    if (G <= 128 || !assign) return DIST_B200_ERR_UNSUPPORTED;
    const int nchunks = (G + kNrChunk - 1) / kNrChunk;
    const int Gpad = nchunks * kNrChunk;
    const int cps = (nchunks + kSlots - 1) / kSlots;
    const int nslots = (nchunks + cps - 1) / cps;
    const size_t smem = sizeof(float4) * (Gpad + nslots) + sizeof(float2) * kNrRows * kSlots * kNrThreads;
    NichRowsArgs a{};
    a.G = G;
    a.N = N;
    a.params = params;
    a.prior = prior;
    a.values = static_cast<const float *>(column);
    a.u = u;
    a.assign = assign;
    // default: the static-reference kernel, four rows per thread (nich_rows2_kernel); DIST_B200_OPT_NICH_PACKED = 3 (A/B runs):
    // the two-row kernel with per-tile maxima it replaced.  DIST_B200_OPT_EXP_OFFLOAD: 0 = default, 1 = every exp2 on the
    // MUFU pipe, 1 + k = k of every 16 pairs on the FMA pipe
    if (ctx->opt[DIST_B200_OPT_NICH_PACKED] != 3) {
        const size_t smem2 = sizeof(float4) * (Gpad + nslots) + sizeof(float) * kN2Rows * kSlots * kNrThreads;
        if (smem2 > 220 * 1024) return DIST_B200_ERR_UNSUPPORTED;  // (one block per SM beyond ~2 800 groups)
        switch (ctx->opt[DIST_B200_OPT_EXP_OFFLOAD]) {
            case 1: return launch_nich_rows2_t<0>(ctx, a, smem2, s);
            case 5: return launch_nich_rows2_t<4>(ctx, a, smem2, s);
            case 7: return launch_nich_rows2_t<6>(ctx, a, smem2, s);
            case 9: return launch_nich_rows2_t<8>(ctx, a, smem2, s);
            default: return launch_nich_rows2_t<kN2PolyDefault>(ctx, a, smem2, s);
        }
    }
    if (smem > 110 * 1024) return DIST_B200_ERR_UNSUPPORTED;  // two blocks per SM
    // DIST_B200_OPT_EXP_OFFLOAD (A/B runs): 0 = default, 1 = every exp2 on the MUFU pipe, 1 + k = k of 16 pairs on the FMA pipe
    switch (ctx->opt[DIST_B200_OPT_EXP_OFFLOAD]) {
        case 1: return launch_nich_rows_t<0>(ctx, a, smem, s);
        case 5: return launch_nich_rows_t<4>(ctx, a, smem, s);
        case 9: return launch_nich_rows_t<8>(ctx, a, smem, s);
        default: return launch_nich_rows_t<kNrPolyDefault>(ctx, a, smem, s);
    }
}

}  // namespace distb200
