// niw_tc_wide.cu -- NormalInverseWishart<d>, 32 < d <= 128, on the 5th-generation tensor cores: [N][G] scores.
//
// The contraction of niw_tc.cu at a padded dimension DP in {64, 128}: for every (row n, group g)
//   y = W_g (x_n - mu0) - b_g,   b_g = W_g (mu'_g - mu0),   q = |y|^2,
//   score = C_g - 0.5 (dof_g + d) fast_log(1 + q / dof_g)
// where mu0 = Shared.mu centres the rows (the pack kernel subtracts it before splitting) and b_g is formed in double by
// niw_prep_wide_kernel.  Centring makes the split error follow |W (x - mu0)| + |W (mu' - mu0)|, i.e. the spread of the data
// around the prior mean, instead of |W x| + |W mu'|, which grows with the data's offset (DESIGN.md section 6, "d > 32").
//
// One MMA stage is 128 B rows = 128 / DP groups (2 at DP = 64, 1 at DP = 128), so every tcgen05.mma is M = 128, N = 128,
// K = 16:  D[128 rows][128] = X[128][K] * Wstage[128][K]^T,  K = DP + 16.
// Precision as niw_tc.cu: x 2^ex = x_hi + x_lo per 128-row tile, W 2^ew = W_hi + W_lo per group, the tile accumulates
// hi hi + lo hi + hi lo in fp32; -b rides in column DP of the hi images (its high term against one copy of the scaled
// constant 1 in A, its low term in column DP + 1 against a second copy), so the accumulator holds (y - b) 2^(ex + ew).
// MMAs per (row tile, stage): 3 DP / 16 + 1.
//
// Nothing is fused: the scores go to [N][G] (prior or accumulate as launch_niw_scores takes them) and the sampler,
// score_logp_batch and mixed lists run over them.  At DP = 128 the contraction is ~16x the d = 32 work per cell while
// writing and re-reading [N][G] costs the same, so a fused walk would buy little here.
//
// Shared memory (DP = 128): one resident 128-row A tile (hi | lo, 68 KB) + a 2-stage ring of stage records (68 KB each)
// = 204 KB; DP = 64: three resident tiles (108 KB) + two 36 KB stages.  TMEM: two 128-column fp32 accumulators.
// Warps: 0 loader (cp.async.bulk), 1 MMA issuer, 2..5 epilogue (one per TMEM lane quarter: tcgen05.ld 32 columns at a
// time, sums of squares, MUFU.LG2, the score).
#include <cuda_fp16.h>

#include "common.cuh"

namespace distb200 {

namespace {

constexpr int kWRows = 128;  // rows per tile (M) and B rows per stage (N)
constexpr int kWEpiWarps = 4;
constexpr int kWThreads = 64 + 32 * kWEpiWarps;
constexpr int kWBStages = 2;

template <int DP>
struct Wide {
    static constexpr int K = DP + 16;                    // d + the b columns, padded to the k-step of 16
    static constexpr int GPS = kWRows / DP;              // groups per stage
    static constexpr int AHi = kWRows * K * 2;           // hi image of a row tile
    static constexpr int ALo = kWRows * DP * 2;          // its lo image (the augmented columns have no low part)
    static constexpr int ATile = AHi + ALo;
    static constexpr int BHi = kWRows * K * 2;
    static constexpr int BLo = kWRows * DP * 2;
    static constexpr int BImages = BHi + BLo;
    static constexpr int BRec = BImages + GPS * 16;      // W_hi | W_lo | consts[GPS][4]
    static constexpr int CT = DP == 64 ? 3 : 1;          // resident row tiles per chunk
    static constexpr size_t Smem = static_cast<size_t>(CT) * ATile + static_cast<size_t>(kWBStages) * BRec + 32 * 8 + 1024;
};

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// no-swizzle K-major canonical layout (as niw_tc.cu): core matrix = 8 rows x 8 halves, core (row group j, k core c) at
// half offset (c * 16 + j) * 64 for 128-row operands
__host__ __device__ __forceinline__ int core_off(int row, int k) { return ((k >> 3) * (kWRows / 8) + (row >> 3)) * 64 + (row & 7) * 8 + (k & 7); }

__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>(((kWRows / 8) * 128 >> 4) & 0x3FFFu) << 16;  // K-adjacent cores: 16 row groups apart
    d |= static_cast<uint64_t>((128 >> 4) & 0x3FFFu) << 32;                 // M/N-adjacent cores: 128 bytes apart
    d |= static_cast<uint64_t>(1) << 46;
    return d;
}

__device__ __forceinline__ void w_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void w_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void w_mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void w_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0, spins = 0;
    while (!done) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(done)
                     : "r"(bar), "r"(parity)
                     : "memory");
        if (!done && ++spins > (1u << 26)) __trap();  // never hang the device on a protocol error
    }
}
__device__ __forceinline__ void w_bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint32_t bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;\n" ::"r"(
                     smem_addr(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(bar), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ uint64_t w_policy(bool keep) {
    uint64_t p;
    if (keep) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(p));
    else asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}
__device__ __forceinline__ void w_umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d),
                 "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
                 : "memory");
}
__device__ __forceinline__ void w_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void w_tmem_ld32(uint32_t taddr, uint32_t *r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ uint64_t w_pack2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ uint64_t w_fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ float w_sum2(uint64_t a) {
    float lo, hi;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a));
    return lo + hi;
}

// 2^(13 - e) for maxabs = m 2^e, m in [0.5, 1): the scaled operand's largest magnitude lands in [2^12, 2^13) (niw_tc.cu)
__device__ __forceinline__ float w_split_scale(float maxabs) {
    if (!(maxabs > 0.f) || !isfinite(maxabs)) return 1.f;
    int e;
    frexpf(maxabs, &e);
    return ldexpf(1.f, 13 - e);
}

// ---------------------------------------------------------------------------------------------
// Stage records from the group records of niw_prep_wide_kernel (b[DP] | W[DP][DP] | consts[4]): one block per stage of GPS
// groups; B row (j DP + i) = [W_g[i][:] | -b_g[i] hi | -b_g[i] lo | 0] 2^ew_g split in two fp16 images (the lo image stops at
// K = DP), consts {C_g, -0.5 (dof + d) ln 2, 1 / dof, 2^-ew_g}.  Groups past G: zero images, C = -inf.
template <int DP>
__global__ void __launch_bounds__(256) niw_tc_wide_prep_kernel(int G, const float *__restrict__ recs, unsigned char *__restrict__ out) {
    using C = Wide<DP>;
    constexpr int REC = DP + DP * DP + 4;
    __shared__ float scale[C::GPS];
    __shared__ float red[8];
    const int st = blockIdx.x, tid = threadIdx.x;
    for (int j = 0; j < C::GPS; ++j) {  // the group's largest magnitude among W and b: they share its scale
        const int g = st * C::GPS + j;
        float m = 0.f;
        if (g < G)
            for (int e = tid; e < DP + DP * DP; e += blockDim.x) m = fmaxf(m, fabsf(recs[static_cast<size_t>(g) * REC + e]));
#pragma unroll
        for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((tid & 31) == 0) red[tid >> 5] = m;
        __syncthreads();
        if (tid == 0) {
            float mm = red[0];
            for (int w = 1; w < 8; ++w) mm = fmaxf(mm, red[w]);
            scale[j] = w_split_scale(mm);
        }
        __syncthreads();
    }
    unsigned char *rec_out = out + static_cast<size_t>(st) * C::BRec;
    __half *w_hi = reinterpret_cast<__half *>(rec_out), *w_lo = w_hi + kWRows * C::K;
    float *consts = reinterpret_cast<float *>(rec_out + C::BImages);
    for (int e = tid; e < kWRows * C::K; e += blockDim.x) {
        const int n = e / C::K, k = e - n * C::K;  // B row n = j DP + i, column k
        const int j = n / DP, i = n - j * DP, g = st * C::GPS + j;
        const float *rec = recs + static_cast<size_t>(g < G ? g : 0) * REC;
        const int off = core_off(n, k);
        if (k < DP) {
            const float w = g < G ? rec[DP + i * DP + k] * scale[j] : 0.f;
            const __half hi = __float2half_rn(w);
            w_hi[off] = hi;
            w_lo[off] = __float2half_rn(w - __half2float(hi));
        } else {
            const float w = g < G ? -rec[i] * scale[j] : 0.f;
            const __half hi = __float2half_rn(w);
            w_hi[off] = k == DP ? hi : k == DP + 1 ? __float2half_rn(w - __half2float(hi)) : __float2half_rn(0.f);
        }
    }
    if (tid < C::GPS) {
        const int g = st * C::GPS + tid;
        const float *k4 = recs + static_cast<size_t>(g < G ? g : 0) * REC + DP + DP * DP;
        consts[tid * 4 + 0] = g < G ? k4[0] : -INFINITY;
        consts[tid * 4 + 1] = g < G ? k4[1] : 0.f;
        consts[tid * 4 + 2] = g < G ? k4[2] : 0.f;
        consts[tid * 4 + 3] = 1.f / scale[tid];
    }
}

// ---------------------------------------------------------------------------------------------
// Row tiles -> A images: one block per 128-row tile; [x - mu0 | 1 | 1 | 0] 2^ex = hi + lo in fp16 (core-matrix order, K = DP + 16
// for hi, DP for lo), zero rows past N; ex from the tile's largest |x - mu0| (and 1: the constant columns); sx[tile] = 2^-ex.
template <int DP>
__global__ void __launch_bounds__(256) niw_tc_wide_pack_kernel(size_t N, int d, const float *__restrict__ values, const float *__restrict__ mu0,
                                                               __half *__restrict__ xpack, float *__restrict__ sx) {
    using C = Wide<DP>;
    __shared__ float red[8];
    __shared__ float s_scale;
    const size_t tile = blockIdx.x;
    const int tid = threadIdx.x;
    const size_t row0 = tile * kWRows;
    const int nr = static_cast<int>(N - row0 < static_cast<size_t>(kWRows) ? N - row0 : kWRows);
    float m = 0.f;
    for (int e = tid; e < nr * d; e += blockDim.x) m = fmaxf(m, fabsf(__ldg(values + row0 * d + e) - __ldg(mu0 + e % d)));
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((tid & 31) == 0) red[tid >> 5] = m;
    __syncthreads();
    if (tid == 0) {
        float mm = red[0];
        for (int w = 1; w < 8; ++w) mm = fmaxf(mm, red[w]);
        const float sc = w_split_scale(fmaxf(mm, 1.f));
        s_scale = sc;
        sx[tile] = 1.f / sc;
    }
    __syncthreads();
    const float sc = s_scale;
    __half *hi_img = xpack + tile * (C::ATile / 2), *lo_img = hi_img + kWRows * C::K;
    constexpr int kCores = C::K / 8;  // 16-byte core rows per row
    for (int it = tid; it < kWRows * kCores; it += blockDim.x) {
        const int r = it / kCores, c = it - r * kCores, k0 = 8 * c;
        const bool live = r < nr;
        __align__(16) __half hi[8], lo[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int k = k0 + i;
            float v = 0.f;
            if (k < DP) {
                if (live && k < d) v = (__ldg(values + (row0 + r) * d + k) - __ldg(mu0 + k)) * sc;
            } else if (live && (k == DP || k == DP + 1)) {
                v = sc;  // the scaled constant 1 (a power of two: exact), once for -b's high term, once for its low term
            }
            hi[i] = __float2half_rn(v);
            lo[i] = __float2half_rn(v - __half2float(hi[i]));
        }
        const int off = core_off(r, k0);
        *reinterpret_cast<uint4 *>(hi_img + off) = *reinterpret_cast<const uint4 *>(hi);
        if (k0 < DP) *reinterpret_cast<uint4 *>(lo_img + off) = *reinterpret_cast<const uint4 *>(lo);
    }
}

struct WideArgs {
    int G, n_stages, accumulate;
    size_t N, ntiles;
    const unsigned char *stagerecs;  // [n_stages][BRec]
    const __half *xpack;             // [ntiles][ATile / 2]
    const float *sx;                 // [ntiles]
    const float *prior;              // [G] or nullptr
    float *scores;                   // [N][G]
};

template <int DP>
__global__ void __launch_bounds__(kWThreads, 1) niw_tc_wide_kernel(const WideArgs a) {
    using C = Wide<DP>;
    constexpr int CT = C::CT;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *As = smem_raw;                          // [CT][hi | lo]
    unsigned char *Bs = As + CT * C::ATile;                // [kWBStages][stage record]
    uint64_t *bars = reinterpret_cast<uint64_t *>(Bs + kWBStages * C::BRec);
    const uint32_t bars_s = smem_addr(bars);
    auto a_full = [&](int i) { return bars_s + 8u * i; };
    auto a_empty = [&](int i) { return bars_s + 8u * (CT + i); };
    auto b_full = [&](int i) { return bars_s + 8u * (2 * CT + i); };
    auto b_empty = [&](int i) { return bars_s + 8u * (2 * CT + kWBStages + i); };
    auto t_full = [&](int i) { return bars_s + 8u * (2 * CT + 2 * kWBStages + i); };
    auto t_empty = [&](int i) { return bars_s + 8u * (2 * CT + 2 * kWBStages + 2 + i); };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * CT + 2 * kWBStages + 4);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ns = a.n_stages;
    if (tid == 0) {
        for (int i = 0; i < CT; ++i) {
            w_mbar_init(a_full(i), 1);
            w_mbar_init(a_empty(i), 1);
        }
        for (int i = 0; i < kWBStages; ++i) {
            w_mbar_init(b_full(i), 1);
            w_mbar_init(b_empty(i), kWEpiWarps);  // the record also carries the epilogue's constants
        }
        for (int i = 0; i < 2; ++i) {
            w_mbar_init(t_full(i), 1);
            w_mbar_init(t_empty(i), kWEpiWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;\n" ::"r"(smem_addr(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    // D = F32, A = B = F16, both K-major, M = 128, N = 128
    const uint32_t idesc = (1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
    const size_t nchunks = (a.ntiles + CT - 1) / CT;

    if (warp == 0) {
        // ===================== loader =====================
        if (lane == 0) {
            uint32_t bstage = 0, bphase = 0, aphase = 0;
            const uint64_t pol_stream = w_policy(false), pol_keep = w_policy(true);
            for (size_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
                const size_t t0 = chunk * CT;
                const int nt = static_cast<int>(a.ntiles - t0 < static_cast<size_t>(CT) ? a.ntiles - t0 : CT);
                auto load_a = [&](int t) {
                    w_mbar_wait(a_empty(t), aphase ^ 1);  // the previous chunk's MMAs on this tile have retired
                    w_mbar_expect_tx(a_full(t), C::ATile);
                    w_bulk_g2s(As + t * C::ATile, a.xpack + (t0 + t) * (C::ATile / 2), C::ATile, a_full(t), pol_stream);
                };
                load_a(0);
                for (int st = 0; st < ns; ++st) {
                    w_mbar_wait(b_empty(bstage), bphase ^ 1);
                    w_mbar_expect_tx(b_full(bstage), C::BRec);
                    w_bulk_g2s(Bs + bstage * C::BRec, a.stagerecs + static_cast<size_t>(st) * C::BRec, C::BRec, b_full(bstage), pol_keep);
                    if (++bstage == kWBStages) {
                        bstage = 0;
                        bphase ^= 1;
                    }
                    if (st == 0)
                        for (int t = 1; t < nt; ++t) load_a(t);
                }
                aphase ^= 1;
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            uint32_t bstage = 0, bphase = 0, aphase = 0, tphase = 0;
            int tb = 0;
            for (size_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
                const size_t t0 = chunk * CT;
                const int nt = static_cast<int>(a.ntiles - t0 < static_cast<size_t>(CT) ? a.ntiles - t0 : CT);
                for (int st = 0; st < ns; ++st) {
                    w_mbar_wait(b_full(bstage), bphase);
                    const uint32_t b_hi = smem_addr(Bs + bstage * C::BRec), b_lo = b_hi + C::BHi;
                    for (int t = 0; t < nt; ++t) {
                        if (st == 0) w_mbar_wait(a_full(t), aphase);
                        w_mbar_wait(t_empty(tb), ((tphase >> tb) & 1u) ^ 1u);
                        tphase ^= 1u << tb;
                        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                        const uint32_t d_addr = tmem_base + tb * kWRows;
                        const uint32_t a_hi = smem_addr(As + t * C::ATile), a_lo = a_hi + C::AHi;
                        uint32_t acc = 0;
#pragma unroll
                        for (int ks = 0; ks < C::K / 16; ++ks) {  // K = 16 per instruction = two 8-half cores
                            const uint32_t o = ks * 2 * (kWRows / 8) * 128;
                            w_umma(d_addr, smem_desc(a_hi + o), smem_desc(b_hi + o), idesc, acc);
                            acc = 1;
                            if (ks == DP / 16) continue;  // the augmented k-step: both terms of -b are in the hi images
                            w_umma(d_addr, smem_desc(a_lo + o), smem_desc(b_hi + o), idesc, 1);
                            w_umma(d_addr, smem_desc(a_hi + o), smem_desc(b_lo + o), idesc, 1);
                        }
                        if (st == ns - 1) w_commit(a_empty(t));
                        w_commit(t_full(tb));
                        tb ^= 1;
                    }
                    if (++bstage == kWBStages) {
                        bstage = 0;
                        bphase ^= 1;
                    }
                }
                aphase ^= 1;
            }
        }
    } else {
        // ===================== epilogue =====================
        const int q = warp & 3;  // TMEM lane quarter this warp may access
        const int r_in_tile = q * 32 + lane;
        uint32_t bstage = 0, bphase = 0, fphase = 0;
        int tb = 0;
        for (size_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
            const size_t t0 = chunk * CT;
            const int nt = static_cast<int>(a.ntiles - t0 < static_cast<size_t>(CT) ? a.ntiles - t0 : CT);
            float sxt[CT];
#pragma unroll
            for (int t = 0; t < CT; ++t) sxt[t] = t < nt ? __ldg(a.sx + t0 + t) : 1.f;
            for (int st = 0; st < ns; ++st) {
                w_mbar_wait(b_full(bstage), bphase);
                const float *cs = reinterpret_cast<const float *>(Bs + bstage * C::BRec + C::BImages);
                float pr[C::GPS];
#pragma unroll
                for (int j = 0; j < C::GPS; ++j) {
                    const int g = st * C::GPS + j;
                    pr[j] = (g < a.G && a.prior && !a.accumulate) ? __ldg(a.prior + g) : 0.f;
                }
#pragma unroll
                for (int t = 0; t < CT; ++t) {
                    if (t >= nt) break;
                    w_mbar_wait(t_full(tb), (fphase >> tb) & 1u);
                    fphase ^= 1u << tb;
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + tb * kWRows;
                    float qs[C::GPS];
#pragma unroll
                    for (int j = 0; j < C::GPS; ++j) {
                        uint64_t qa = 0ull, qb = 0ull;
#pragma unroll
                        for (int c = 0; c < DP / 32; ++c) {
                            uint32_t yr[32];
                            w_tmem_ld32(t_row + j * DP + 32 * c, yr);
                            asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
                            for (int i = 0; i < 32; i += 4) {
                                const uint64_t d0 = w_pack2(__uint_as_float(yr[i]), __uint_as_float(yr[i + 1]));
                                const uint64_t d1 = w_pack2(__uint_as_float(yr[i + 2]), __uint_as_float(yr[i + 3]));
                                qa = w_fma2(d0, d0, qa);
                                qb = w_fma2(d1, d1, qb);
                            }
                        }
                        qs[j] = w_sum2(qa) + w_sum2(qb);
                    }
                    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
                    if (lane == 0) w_mbar_arrive(t_empty(tb));
                    tb ^= 1;
                    const size_t row = (t0 + t) * kWRows + r_in_tile;
                    if (row < a.N) {
#pragma unroll
                        for (int j = 0; j < C::GPS; ++j) {
                            const int g = st * C::GPS + j;
                            if (g >= a.G) continue;
                            const float4 c = *reinterpret_cast<const float4 *>(cs + j * 4);
                            const float unscale = sxt[t] * c.w;  // 2^-(ex + ew): exact
                            const float qq = qs[j] * (unscale * unscale);
                            const float arg = __fadd_rn(1.f, __fmul_rn(c.z, qq));
                            const float v = fmaf(c.y, fast_log2_cell(arg), c.x) + pr[j];
                            float *dst = a.scores + row * a.G + g;
                            *dst = a.accumulate ? *dst + v : v;
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) w_mbar_arrive(b_empty(bstage));
                if (++bstage == kWBStages) {
                    bstage = 0;
                    bphase ^= 1;
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;\n" ::"r"(tmem_base) : "memory");
}

template <int DP>
int stages_of(int G) { return (G + Wide<DP>::GPS - 1) / Wide<DP>::GPS; }

template <int DP>
int launch_wide_prep_t(dist_b200_ctx *ctx, int G, const float *recs, float *tc_buf, cudaStream_t s) {
    const int ns = stages_of<DP>(G);
    if (ns == 0) return DIST_B200_OK;
    niw_tc_wide_prep_kernel<DP><<<ns, 256, 0, s>>>(G, recs, reinterpret_cast<unsigned char *>(tc_buf));
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("niw_tc_wide_prep launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

template <int DP>
int launch_wide_t(dist_b200_ctx *ctx, int G, int d, const float *tc_buf, const float *mu0, const void *values, size_t N,
                  const float *prior, float *scores, int accumulate, cudaStream_t s) {
    using C = Wide<DP>;
    const size_t ntiles = (N + kWRows - 1) / kWRows;
    const size_t nchunks = (ntiles + C::CT - 1) / C::CT;
    const unsigned grid = static_cast<unsigned>(nchunks < static_cast<size_t>(ctx->sm_count) ? nchunks : ctx->sm_count);
    const size_t xbytes = ntiles * C::ATile;
    const size_t sxbytes = (ntiles * sizeof(float) + 255) / 256 * 256;
    if (int rc = grow(ctx, ctx->xpack, ctx->xpack_bytes, xbytes + sxbytes)) return rc;
    unsigned char *base = static_cast<unsigned char *>(ctx->xpack);
    WideArgs a{};
    a.G = G;
    a.n_stages = stages_of<DP>(G);
    a.accumulate = accumulate;
    a.N = N;
    a.ntiles = ntiles;
    a.stagerecs = reinterpret_cast<const unsigned char *>(tc_buf);
    a.xpack = reinterpret_cast<const __half *>(base);
    a.sx = reinterpret_cast<const float *>(base + xbytes);
    a.prior = prior;
    a.scores = scores;
    niw_tc_wide_pack_kernel<DP><<<static_cast<unsigned>(ntiles), 256, 0, s>>>(N, d, static_cast<const float *>(values), mu0,
                                                                            reinterpret_cast<__half *>(base), reinterpret_cast<float *>(base + xbytes));
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaFuncSetAttribute(niw_tc_wide_kernel<DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(C::Smem));
    if (e == cudaSuccess) {
        niw_tc_wide_kernel<DP><<<grid, kWThreads, C::Smem, s>>>(a);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("niw_tc_wide launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

}  // namespace

size_t niw_tc_wide_floats(int G, int d) {
    const size_t bytes = niw_padded_dim(d) == 64 ? static_cast<size_t>(stages_of<64>(G)) * Wide<64>::BRec
                                                 : static_cast<size_t>(stages_of<128>(G)) * Wide<128>::BRec;
    return (bytes + 3) / 4;
}

int launch_niw_tc_wide_prep(dist_b200_ctx *ctx, int G, int d, const float *recs, float *tc_buf, cudaStream_t s) {
    if (niw_padded_dim(d) == 64) return launch_wide_prep_t<64>(ctx, G, recs, tc_buf, s);
    return launch_wide_prep_t<128>(ctx, G, recs, tc_buf, s);
}

int launch_niw_tc_wide(dist_b200_ctx *ctx, int G, int d, const float *tc_buf, const float *mu0, const void *values, size_t N,
                       const float *prior, float *scores, int accumulate, cudaStream_t s) {
    if (N == 0 || G == 0) return DIST_B200_OK;
    if (!tc_buf || !scores) return fail(ctx, DIST_B200_ERR_STATE, "niw_tc_wide: no operand images or no score buffer");
    if (niw_padded_dim(d) == 64) return launch_wide_t<64>(ctx, G, d, tc_buf, mu0, values, N, prior, scores, accumulate, s);
    return launch_wide_t<128>(ctx, G, d, tc_buf, mu0, values, N, prior, scores, accumulate, s);
}

}  // namespace distb200
