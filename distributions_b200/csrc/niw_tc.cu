// niw_tc.cu -- NormalInverseWishart<32> on the 5th-generation tensor cores: quadratic forms, Student-t scores and
// (fused) sample_from_scores in ONE persistent kernel.
//
// The only dense contraction on the hot path (SURVEY.md 8 a11): for every (row n, group g)
//   y = W_g x_n   (W_g = L_g^-1, d x d),    q = |y - W_g mu'_g|^2,
//   score = C_g - 0.5 (dof_g + d) fast_log(1 + q / dof_g)          (niw.hpp:353-360, random.hpp:160-185)
// Stacking the W_g of 8 groups gives a B operand of 256 rows, so one tcgen05.mma tile is
//   D[128 rows][256 = 8 groups x 32 dims] = X[128][32] * Wstack[256][32]^T
// with the fp32 accumulator in TMEM (2 x 256 columns, double buffered).  A TMEM lane is a data row and a
// 32-column slice is exactly one cell's y vector.
//
// Precision.  One low-precision pass is not enough: y - b cancels |W mu'| ~ 17 down to |y - b| ~ 1, so 10-bit
// operands cost ~0.04 absolute on a score.  Both operands are therefore split in two fp16 terms
//   x 2^ex = x_hi + x_lo,   W 2^ew = W_hi + W_lo        (11 + 11 significant bits, fp16 x fp16 products are exact in fp32)
// and the tile accumulates x_hi W_hi + x_lo W_hi + x_hi W_lo (the dropped x_lo W_lo is ~2^-22 relative).  The power-of-two
// scales keep fp16 in range whatever the data: ex per 128-row tile (chosen by the pack kernel from the tile's largest
// |x|), ew per group (from its largest |W|); the epilogue undoes them inside the FFMA2 that subtracts b, so they cost
// nothing.  kind::f16 issues K = 16 per instruction.
//
// The subtraction of b rides in the GEMM: the operands carry a 33rd column, x_aug = 2^ex (i.e. the scaled constant 1)
// and W_aug = -b 2^ew (split like W; ew covers max(|W|, |b|)), padded to K = 48, so the accumulator already holds
// (y - b) 2^(ex + ew) and the epilogue is a plain sum of squares.  Measured why: with b read from shared memory the
// epilogue issued 32 broadcast LDS.128 per thread per tile, and a warp-wide LDS.128 occupies the shared-memory pipe for
// four wavefronts even when every lane reads the same address -- 1 000 of the pipe's cycles per (tile, block), on top
// of the 600 the tensor core needs for its own operand reads: the kernel sat at 35 % tensor-pipe activity
// (profiles/r02_c5_niw_v1_lds_bound.txt).  -b is split like W, and both of its terms sit in the hi image (columns 32 and
// 33, against two copies of the constant in A), so the augmented k-step is ONE MMA: 7 MMAs per (tile, block) = two k-steps x
// {hi hi, lo hi, hi lo} + the augmented hi hi; the lo images stop at K = 32.  3xTF32 (round 1) needed 12 at twice the bytes.
// W = L^-1 is LOWER TRIANGULAR: the k-step over x[16..32) only feeds the upper 16 dims of every group.  The B rows
// (= accumulator columns) are ordered (low dims of the 8 groups | high dims of the 8 groups), and that k-step's three
// MMAs run with N = 128 on columns [128, 256): 5.5 MMA-equivalents per (tile, block).
//
// Schedule (per CTA, one per SM, persistent over chunks of kChunkTiles row tiles; 18 warps):
//   warp 0 (one lane)  loader   -- cp.async.bulk of the chunk's A images (resident for the whole chunk) and of the
//                                  32 block records {W_hi, W_lo, constants} through a 2-stage ring
//   warp 1 (one lane)  issuer   -- for every block, for every resident tile: 7 x tcgen05.mma (three of them N = 128), tcgen05.commit
//   warps 2..17        epilogue -- four warps per TMEM lane quarter, each owns two groups (2 x 32 accumulator columns):
//                                  tcgen05.ld, sums of squares on packed fp32x2, MUFU.LG2, the score; per row an ONLINE
//                                  (max, sum of exp) pair; the chunk's scores go to a per-CTA scratch block
//                                  (512 KB, reused every chunk: it lives in L2; pair-major, so a warp stores and later
//                                  walks whole lines), and after the last block the same warps walk one row each:
//                                  t = u * total, first group with t - sum exp <= 0 (random.hpp:315-333).
// L2 -> SM traffic: the A images once (160 MB) + 1.3 MB of block records per chunk (2.5 GB at c5) -- round 1 re-streamed
// the rows for every block (8 GB) and round-tripped 2 GB of scores through HBM for a separate sampler.
// Without a sampler request (score_batch, accumulate, mixed feature lists) the same kernel writes [N][G] scores.
//
// What bounds it (profiles/r02_c5_power.txt): launched back to back, the board's 1 000 W power cap -- nvidia-smi shows
// sw_power_cap active and the SM clock at 1.65 - 1.8 GHz instead of 1.965; with the MMAs alone (debug 4) the kernel runs at
// the tensor pipe's rate.  Every removed MMA, shared-memory operand read, L2 round trip or instruction is therefore time:
// 8 -> 7 -> 5.5 MMAs, K = 32 lo images, whole-line scratch accesses, and an epilogue without per-tile overhead (the profiling
// modes are template instantiations: as runtime branches they cost 27 % of all executed instructions) took the kernel from
// 1.97 to 1.22 ms (profiles/r02_c5_niw_fused.txt).
#include <cuda_fp16.h>

#include "common.cuh"

namespace distb200 {

constexpr int kTcDim = 32;                 // d
constexpr int kTcK = 48;                   // K of the GEMM: d + the b column, padded to the k-step of 16
constexpr int kTcGroupsPerBlock = 8;       // groups per B tile (N = 256)
constexpr int kTcRows = 128;               // rows per tile (M)
constexpr int kAImageBytes = kTcRows * kTcK * 2;            // the hi image of a row tile (K = 48): 12 KB
constexpr int kALoBytes = kTcRows * kTcDim * 2;             // its lo image (K = 32: the augmented columns have no low part): 8 KB
constexpr int kATileBytes = kAImageBytes + kALoBytes;       // hi | lo
constexpr int kBImageBytes = 256 * kTcK * 2;                // the hi image of a block (K = 48): 24 KB
constexpr int kBLoBytes = 256 * kTcDim * 2;                 // its lo image (K = 32): 16 KB
constexpr int kBImagesBytes = kBImageBytes + kBLoBytes;
constexpr int kBlockRecBytes = kBImagesBytes + kTcGroupsPerBlock * 4 * 4;  // W_hi | W_lo | consts[8][4]
constexpr int kChunkTiles = 4;             // resident row tiles per chunk (512 rows)
constexpr int kBStages = 2;
constexpr int kEpiWarps = 16;            // epilogue warps: four per TMEM lane quarter, each owns a quarter of the columns
constexpr int kFusedThreads = 64 + 32 * kEpiWarps;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// no-swizzle K-major canonical layout of an fp16 operand: core matrix = 8 rows x 16 bytes (8 halves along K), rows
// 16 B apart; core (row group j, k core c) at byte offset (c * n_row_groups + j) * 128.  Offset in HALVES:
__host__ __device__ __forceinline__ int core_offset_halves(int row, int k, int n_row_groups) {
    return ((k >> 3) * n_row_groups + (row >> 3)) * 64 + (row & 7) * 8 + (k & 7);
}

__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);           // start address, bits [0,14)
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;  // leading (K) byte offset, bits [16,30)
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;  // stride (M/N) byte offset, bits [32,46)
    d |= static_cast<uint64_t>(1) << 46;                           // descriptor version (Blackwell)
    return d;                                                      // layout type 0 = no swizzle
}

// mbarriers are addressed by their shared-space address, computed once per kernel (a generic -> shared conversion per
// call shows up in an epilogue that hands over a TMEM buffer every few hundred cycles)
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    uint32_t spins = 0;
    while (!done) {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (!done && ++spins > (1u << 26)) __trap();  // never hang the device on a protocol error
    }
}
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(bar)
                 : "memory");
}
// L2 eviction policies: the per-CTA score scratch and the block records are re-used (evict last), the row images stream
// through once (evict first) -- without them the streaming rows push dirty scratch lines out to HBM
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_g2s_hint(void *smem_dst, const void *gmem_src, uint32_t bytes, uint32_t bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;\n" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(bar), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ void st_f2_hint(float2 *p, float2 v, uint64_t policy) {
    asm volatile("st.global.L2::cache_hint.v2.f32 [%0], {%1, %2}, %3;\n" ::"l"(p), "f"(v.x), "f"(v.y), "l"(policy) : "memory");
}
__device__ __forceinline__ float2 ld_f2_hint(const float2 *p, uint64_t policy) {
    float2 v;
    asm volatile("ld.global.L2::cache_hint.v2.f32 {%0, %1}, [%2], %3;\n" : "=f"(v.x), "=f"(v.y) : "l"(p), "l"(policy) : "memory");
    return v;
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar) : "memory");
}
// 32 columns: one half (16 dims) of two cells
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t *r) {
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

// Blackwell packed fp32 pairs: one instruction, two lanes of the FMA pipe (halves the epilogue's issue count)
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ float sum2(uint64_t a) {
    float lo, hi;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a));
    return lo + hi;
}

// 2^e with e = 12 - floor(log2(maxabs)): the scaled operand's largest magnitude lands in [2^12, 2^13) -- far from
// fp16's 65504, and its low-order term (2^-11 of that) still has all of its bits above fp16's subnormal quantum
__device__ __forceinline__ float split_scale(float maxabs) {
    if (!(maxabs > 0.f) || !isfinite(maxabs)) return 1.f;
    int e;
    frexpf(maxabs, &e);          // maxabs = m 2^e, m in [0.5, 1)  ->  floor(log2) = e - 1
    return ldexpf(1.f, 13 - e);
}

// ---------------------------------------------------------------------------------------------
// Block records.  From the group records of niw_prep_kernel (mu'[32] | W[32][32] | consts[4]) build, per block of
// 8 groups: [W | -b | 0] 2^ew split in two fp16 images (core-matrix order, K = 48) and {C_g, -0.5 (dof + d) ln 2, 1 / dof,
// 2^-ew_g}.  Groups past G are padding: zero W, C = -inf (they vanish from max / exp).
__global__ void __launch_bounds__(256) niw_tc_prep_kernel(int G, const float *__restrict__ recs, unsigned char *__restrict__ blockrecs) {
    constexpr int REC = kTcDim + kTcDim * kTcDim + 4;
    __shared__ float scale[kTcGroupsPerBlock];
    __shared__ float nb[256];  // -b = -(W mu'), unscaled
    const int blk = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    {
        const int g = blk * kTcGroupsPerBlock + (tid >> 5), i = tid & 31;
        double b = 0.0;
        if (g < G) {
            const float *rec = recs + static_cast<size_t>(g) * REC;
            for (int k = 0; k <= i; ++k) b += static_cast<double>(rec[kTcDim + i * kTcDim + k]) * static_cast<double>(rec[k]);
        }
        nb[tid] = static_cast<float>(-b);
    }
    __syncthreads();
    {   // one warp per group: largest magnitude among W and b (they share the group's scale)
        const int g = blk * kTcGroupsPerBlock + warp;
        float m = g < G ? fabsf(nb[warp * 32 + lane]) : 0.f;
        if (g < G)
            for (int e = lane; e < kTcDim * kTcDim; e += 32) m = fmaxf(m, fabsf(recs[static_cast<size_t>(g) * REC + kTcDim + e]));
#pragma unroll
        for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) scale[warp] = split_scale(m);
    }
    __syncthreads();
    unsigned char *rec_out = blockrecs + static_cast<size_t>(blk) * kBlockRecBytes;
    __half *w_hi = reinterpret_cast<__half *>(rec_out), *w_lo = w_hi + 256 * kTcK;
    float *consts = reinterpret_cast<float *>(rec_out + kBImagesBytes);
    for (int e = tid; e < 256 * kTcK; e += blockDim.x) {
        const int n = e / kTcK, k = e - n * kTcK;  // B row n = (group in block) * 32 + i, column k
        const int g = blk * kTcGroupsPerBlock + (n >> 5), i = n & 31;
        // B row (= accumulator column) of (group, dim i): the low 16 dims of the 8 groups, then the high 16 dims -- W is lower
        // triangular, so the k-step over x[16..32) only feeds the high half and its MMAs run with N = 128
        const int brow = (i >> 4) * 128 + (n >> 5) * 16 + (i & 15);
        const int off = core_offset_halves(brow, k, 32);
        if (k < kTcDim) {
            const float w = g < G ? recs[static_cast<size_t>(g) * REC + kTcDim + i * kTcDim + k] * scale[n >> 5] : 0.f;
            const __half hi = __float2half_rn(w);
            w_hi[off] = hi;
            w_lo[off] = __float2half_rn(w - __half2float(hi));
        } else {  // augmented columns of the hi image: -b's high term in column 32, its low term in column 33, zeros after
            const float w = g < G ? nb[n] * scale[n >> 5] : 0.f;
            const __half hi = __float2half_rn(w);
            w_hi[off] = k == kTcDim ? hi : k == kTcDim + 1 ? __float2half_rn(w - __half2float(hi)) : __float2half_rn(0.f);
        }
    }
    if (tid < kTcGroupsPerBlock) {
        const int g = blk * kTcGroupsPerBlock + tid;
        const float *k4 = recs + static_cast<size_t>(g < G ? g : 0) * REC + kTcDim + kTcDim * kTcDim;
        consts[tid * 4 + 0] = g < G ? k4[0] : -INFINITY;
        consts[tid * 4 + 1] = g < G ? k4[1] : 0.f;
        consts[tid * 4 + 2] = g < G ? k4[2] : 0.f;
        consts[tid * 4 + 3] = 1.f / scale[tid];
    }
}

// ---------------------------------------------------------------------------------------------
// Row tiles -> A-operand images: one block per 128-row tile; tile-wide power-of-two scale, [x | 1 | 0] 2^ex = hi + lo in
// fp16, core-matrix order (K = 48), zero rows past N; sx[tile] = 2^-ex.
__global__ void __launch_bounds__(256) niw_tc_pack_x_kernel(size_t N, const float *__restrict__ values, __half *__restrict__ xpack,
                                                            float *__restrict__ sx) {
    __shared__ float wmax[8];
    __shared__ float s_scale;
    const size_t tile = blockIdx.x;
    const int tid = threadIdx.x, r = tid >> 1, k0 = (tid & 1) * 16;  // thread: 16 consecutive dims of one row
    const size_t row = tile * kTcRows + r;
    float4 x[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) x[c] = row < N ? __ldg(reinterpret_cast<const float4 *>(values + row * kTcDim + k0) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    float m = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) m = fmaxf(fmaxf(m, fmaxf(fabsf(x[c].x), fabsf(x[c].y))), fmaxf(fabsf(x[c].z), fabsf(x[c].w)));
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((tid & 31) == 0) wmax[tid >> 5] = m;
    __syncthreads();
    if (tid == 0) {
        float mm = wmax[0];
        for (int w = 1; w < 8; ++w) mm = fmaxf(mm, wmax[w]);
        const float sc = split_scale(fmaxf(mm, 1.f));  // the constant column (1) takes part in the tile's range
        s_scale = sc;
        sx[tile] = 1.f / sc;
    }
    __syncthreads();
    const float sc = s_scale;
    __half *hi_img = xpack + tile * (kATileBytes / 2), *lo_img = hi_img + kTcRows * kTcK;
    const float *xf = reinterpret_cast<const float *>(x);
#pragma unroll
    for (int kc = 0; kc < 2; ++kc) {  // one 16-byte core row (8 halves) per store
        __align__(16) __half hi[8], lo[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float v = xf[kc * 8 + i] * sc;
            hi[i] = __float2half_rn(v);
            lo[i] = __float2half_rn(v - __half2float(hi[i]));
        }
        const int off = core_offset_halves(r, k0 + 8 * kc, kTcRows / 8);
        *reinterpret_cast<uint4 *>(hi_img + off) = *reinterpret_cast<const uint4 *>(hi);
        *reinterpret_cast<uint4 *>(lo_img + off) = *reinterpret_cast<const uint4 *>(lo);
    }
    {   // columns 32..47 of the hi image: the scaled constant 1 (exact in fp16: a power of two) twice, then zeros
        __align__(16) __half aug[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) aug[i] = __float2half_rn(0.f);
        if ((tid & 1) == 0) aug[0] = aug[1] = __float2half_rn(row < N ? sc : 0.f);  // one for -b's high term, one for its low term
        const int off = core_offset_halves(r, kTcDim + 8 * (tid & 1), kTcRows / 8);
        *reinterpret_cast<uint4 *>(hi_img + off) = *reinterpret_cast<const uint4 *>(aug);
    }
}

struct NiwTcArgs {
    int G, n_blocks, accumulate, Gpad;
    size_t N, ntiles;
    const unsigned char *blockrecs;  // [n_blocks][kBlockRecBytes]
    const __half *xpack;             // [ntiles][2][128 * 48]
    const float *sx;                 // [ntiles]
    const float *prior;              // [G] or nullptr
    float *scores;                   // materialising mode: [N][G]
    float *scratch;                  // fused mode: [grid][Gpad / 4][kChunkTiles * 128] float4 (four groups of one row)
    const float *u;                  // fused mode
    int32_t *assign;                 // fused mode
};

// kDebug (DIST_B200_OPT_NIW_DEBUG, profiling builds of the same kernel whose results are WRONG by construction): 1 = no
// sampling walk, 2 = also no epilogue math, 4 = barrier hand-offs only (loader + MMA stream alone), 5 = and 3 of the 7 MMAs.
// A template parameter, not a runtime flag: as a runtime branch the debug paths cost the production kernel 64 register
// initialisations per thread per tile (28 % of its instructions, profiles/r02_c5_niw_fused.txt)
template <bool kFused, int kDebug>
__global__ void __launch_bounds__(kFusedThreads, 1) niw_tc_fused_kernel(const NiwTcArgs a) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *As = smem_raw;                                        // [kChunkTiles][hi | lo]  64 KB
    unsigned char *Bs = As + kChunkTiles * kATileBytes;                  // [kBStages][block record]
    constexpr int kParts = kEpiWarps / 4;                                        // column parts of a block (one per epilogue warp of a lane quarter)
    float *half_m = reinterpret_cast<float *>(Bs + kBStages * kBlockRecBytes);   // [kParts][kChunkTiles * 128] online max per column part
    float *half_s = half_m + kParts * kChunkTiles * kTcRows;                     // [kParts][kChunkTiles * 128] online sum
    uint64_t *bars = reinterpret_cast<uint64_t *>(half_s + kParts * kChunkTiles * kTcRows);
    // shared-space addresses of the mbarriers: X(i) = the i-th barrier of ring X
    const uint32_t bars_s = smem_u32(bars);
    auto a_full = [&](int i) { return bars_s + 8u * i; };
    auto a_empty = [&](int i) { return bars_s + 8u * (kChunkTiles + i); };
    auto b_full = [&](int i) { return bars_s + 8u * (2 * kChunkTiles + i); };
    auto b_empty = [&](int i) { return bars_s + 8u * (2 * kChunkTiles + kBStages + i); };
    auto t_full = [&](int i) { return bars_s + 8u * (2 * kChunkTiles + 2 * kBStages + i); };
    auto t_empty = [&](int i) { return bars_s + 8u * (2 * kChunkTiles + 2 * kBStages + 2 + i); };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * kChunkTiles + 2 * kBStages + 4);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nb = a.n_blocks;
    if (tid == 0) {
        for (int i = 0; i < kChunkTiles; ++i) {
            mbar_init(a_full(i), 1);
            mbar_init(a_empty(i), 1);
        }
        for (int i = 0; i < kBStages; ++i) {
            mbar_init(b_full(i), 1);
            mbar_init(b_empty(i), kEpiWarps);  // one arrival per epilogue warp: the record also carries their constants
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(t_full(i), 1);
            mbar_init(t_empty(i), kEpiWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    // instruction descriptors: D = F32, A = B = F16, both K-major, M = 128, N = 256 / 128 (the high-dims half alone)
    const uint32_t idesc = (1u << 4) | (0u << 7) | (0u << 10) | ((256u >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t idesc_half = (1u << 4) | (0u << 7) | (0u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

    const size_t nchunks = (a.ntiles + kChunkTiles - 1) / kChunkTiles;

    if (warp == 0) {
        // ===================== loader =====================
        if (lane == 0) {
            uint32_t bstage = 0, bphase = 0, aphase = 0;
            const uint64_t pol_stream = l2_policy_evict_first(), pol_keep = l2_policy_evict_last();
            for (size_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
                const size_t t0 = chunk * kChunkTiles;
                const int nt = static_cast<int>(a.ntiles - t0 < kChunkTiles ? a.ntiles - t0 : kChunkTiles);
                auto load_a = [&](int t) {
                    mbar_wait(a_empty(t), aphase ^ 1);  // the previous chunk's MMAs on this tile have retired
                    mbar_expect_tx(a_full(t), kATileBytes);
                    bulk_g2s_hint(As + t * kATileBytes, a.xpack + (t0 + t) * (kATileBytes / 2), kATileBytes, a_full(t), pol_stream);
                };
                // in consumption order: tile 0, block 0, the remaining tiles, the remaining blocks
                load_a(0);
                for (int blk = 0; blk < nb; ++blk) {
                    mbar_wait(b_empty(bstage), bphase ^ 1);
                    mbar_expect_tx(b_full(bstage), kBlockRecBytes);
                    bulk_g2s_hint(Bs + bstage * kBlockRecBytes, a.blockrecs + static_cast<size_t>(blk) * kBlockRecBytes, kBlockRecBytes, b_full(bstage), pol_keep);
                    if (++bstage == kBStages) {
                        bstage = 0;
                        bphase ^= 1;
                    }
                    if (blk == 0)
                        for (int t = 1; t < nt; ++t) load_a(t);
                }
                aphase ^= 1;
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            uint32_t bstage = 0, bphase = 0, aphase = 0, tphase = 0;  // tphase / fphase: bit tb = phase of accumulator tb
            int tb = 0;
            for (size_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
                const size_t t0 = chunk * kChunkTiles;
                const int nt = static_cast<int>(a.ntiles - t0 < kChunkTiles ? a.ntiles - t0 : kChunkTiles);
                for (int blk = 0; blk < nb; ++blk) {
                    mbar_wait(b_full(bstage), bphase);
                    const uint32_t b_hi = smem_u32(Bs + bstage * kBlockRecBytes), b_lo = b_hi + kBImageBytes;
                    for (int t = 0; t < nt; ++t) {
                        if (blk == 0) mbar_wait(a_full(t), aphase);
                        mbar_wait(t_empty(tb), ((tphase >> tb) & 1u) ^ 1u);  // epilogue has drained this accumulator
                        tphase ^= 1u << tb;
                        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                        const uint32_t d_addr = tmem_base + tb * 256;
                        const uint32_t a_hi = smem_u32(As + t * kATileBytes), a_lo = a_hi + kAImageBytes;
                        uint32_t acc = 0;
#pragma unroll
                        for (int ks = 0; ks < kTcK / 16; ++ks) {  // K = 16 per instruction = two 8-half cores
                            const uint32_t ao = ks * 2 * (kTcRows / 8) * 128;
                            // k-step 1 (x[16..32)) meets zeros in the low-dims half of the lower-triangular W: N = 128, B rows and
                            // accumulator columns [128, 256) only
                            const bool half = ks == 1;
                            const uint32_t bo = ks * 2 * 32 * 128 + (half ? 16 * 128 : 0), dd = d_addr + (half ? 128 : 0);
                            const uint32_t id = half ? idesc_half : idesc;
                            umma_f16(dd, make_smem_desc(a_hi + ao, (kTcRows / 8) * 128, 128), make_smem_desc(b_hi + bo, 32 * 128, 128), id, acc);
                            acc = 1;
                            // the augmented k-step carries both terms of -b in the hi images: one MMA
                            if (kDebug >= 5 || ks == kTcDim / 16) continue;  // (debug 5: hi x hi only)
                            umma_f16(dd, make_smem_desc(a_lo + ao, (kTcRows / 8) * 128, 128), make_smem_desc(b_hi + bo, 32 * 128, 128), id, 1);
                            umma_f16(dd, make_smem_desc(a_hi + ao, (kTcRows / 8) * 128, 128), make_smem_desc(b_lo + bo, 32 * 128, 128), id, 1);
                        }
                        if (blk == nb - 1) umma_commit(a_empty(t));  // tile reusable by the next chunk once these retire
                        umma_commit(t_full(tb));                     // accumulator ready for the epilogue
                        tb ^= 1;
                    }
                    if (++bstage == kBStages) {
                        bstage = 0;
                        bphase ^= 1;
                    }
                }
                aphase ^= 1;
            }
        }
    } else {
        // ===================== epilogue + sampler (kEpiWarps warps) =====================
        const int e = warp - 2;
        const int q = warp & 3;        // TMEM lane quarter this warp may access
        const int h = e >> 2;          // column part: groups [kPer h, kPer h + kPer) of the block
        const int r_in_tile = q * 32 + lane;
        constexpr int kPer = kTcGroupsPerBlock / kParts;
        static_assert(kPer == 2, "the epilogue below loads 64 columns (two cells) per thread");
        uint32_t bstage = 0, bphase = 0, fphase = 0;
        int tb = 0;
        float *scratch = kFused ? a.scratch + static_cast<size_t>(blockIdx.x) * kChunkTiles * kTcRows * a.Gpad : nullptr;
        const uint64_t pol_keep = l2_policy_evict_last();
        for (size_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
            const size_t t0 = chunk * kChunkTiles;
            const int nt = static_cast<int>(a.ntiles - t0 < kChunkTiles ? a.ntiles - t0 : kChunkTiles);
            float sxt[kChunkTiles], om[kChunkTiles], os[kChunkTiles];  // tile scales; online (max * log2e, sum) of this row x half
#pragma unroll
            for (int t = 0; t < kChunkTiles; ++t) {
                sxt[t] = t < nt ? __ldg(a.sx + t0 + t) : 1.f;
                om[t] = -INFINITY;
                os[t] = 0.f;
            }
            for (int blk = 0; blk < nb; ++blk) {
                mbar_wait(b_full(bstage), bphase);
                const float *cs = reinterpret_cast<const float *>(Bs + bstage * kBlockRecBytes + kBImagesBytes);
                float pr[kPer];
#pragma unroll
                for (int jj = 0; jj < kPer; ++jj) {
                    const int g = blk * kTcGroupsPerBlock + h * kPer + jj;
                    pr[jj] = (g < a.G && a.prior && !a.accumulate) ? __ldg(a.prior + g) : 0.f;
                }
#pragma unroll
                for (int t = 0; t < kChunkTiles; ++t) {
                    if (t >= nt) break;
                    mbar_wait(t_full(tb), (fphase >> tb) & 1u);
                    fphase ^= 1u << tb;
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    if (kDebug >= 4) {  // barrier hand-offs only: the rate of the loader + MMA stream alone
                        asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
                        if (lane == 0) mbar_arrive(t_empty(tb));
                        tb ^= 1;
                        continue;
                    }
                    uint32_t yr[64];
                    // this thread's two groups: their low 16 dims at columns [32 h, 32 h + 32), their high 16 dims 128 further
                    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + tb * 256 + h * kPer * 16;
                    tmem_ld32_nowait(t_row, yr);
                    tmem_ld32_nowait(t_row + 128, yr + 32);
                    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
                    if (lane == 0) mbar_arrive(t_empty(tb));  // accumulator drained by this warp: one of the 8 arrivals
                    tb ^= 1;
                    float out[kPer];
                    if (kDebug >= 2) {
#pragma unroll
                        for (int jj = 0; jj < kPer; ++jj) out[jj] = __uint_as_float(yr[jj * 16]);
                    } else
#pragma unroll
                    for (int jj = 0; jj < kPer; ++jj) {
                        const int j = h * kPer + jj;
                        const uint32_t *ylo = &yr[jj * 16], *yhi = &yr[32 + jj * 16];  // (y - b) 2^(ex + ew): dims [0, 16) and [16, 32)
                        const float4 c = *reinterpret_cast<const float4 *>(cs + j * 4);
                        const float unscale = sxt[t] * c.w;  // 2^-(ex + ew): exact
                        uint64_t qa = 0ull, qb = 0ull;
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const uint32_t *y = i < 4 ? ylo + 4 * i : yhi + 4 * (i - 4);
                            const uint64_t d0 = pack2(__uint_as_float(y[0]), __uint_as_float(y[1]));
                            const uint64_t d1 = pack2(__uint_as_float(y[2]), __uint_as_float(y[3]));
                            qa = fma2(d0, d0, qa);
                            qb = fma2(d1, d1, qb);
                        }
                        const float qq = (sum2(qa) + sum2(qb)) * (unscale * unscale);  // power-of-two factor: exact
                        const float arg = __fadd_rn(1.f, __fmul_rn(c.z, qq));
                        out[jj] = fmaf(c.y, fast_log2_cell(arg), c.x) + pr[jj];
                    }
                    const size_t row = (t0 + t) * kTcRows + r_in_tile;
                    if (kFused) {
                        // the chunk's scores stay on chip (L2), quad-major so that a warp stores / walks whole lines; online (max, sum exp) of this row x half
                        st_f2_hint(reinterpret_cast<float2 *>(scratch) + static_cast<size_t>(blk * kParts + h) * (kChunkTiles * kTcRows) + t * kTcRows + r_in_tile,
                                   make_float2(out[0], out[1]), pol_keep);
                        const float m4 = fmaxf(out[0], out[1]) * kLog2e;
                        const float mn = fmaxf(fmaxf(om[t], m4), -3.0e38f);  // finite even when both groups are padding
                        float s4 = 0.f;
#pragma unroll
                        for (int jj = 0; jj < kPer; ++jj) s4 += mufu_ex2(fmaf(out[jj], kLog2e, -mn));
                        os[t] = fmaf(os[t], mufu_ex2(om[t] - mn), s4);  // om = -inf on the first block: factor 0
                        om[t] = mn;
                    } else if (row < a.N) {
                        const int gbase = blk * kTcGroupsPerBlock + h * kPer;
                        float *dst = a.scores + row * a.G + gbase;
                        if (gbase + kPer <= a.G && (a.G & 1) == 0) {
                            float2 o0 = make_float2(out[0], out[1]);
                            if (a.accumulate) {
                                const float2 p0 = *reinterpret_cast<float2 *>(dst);
                                o0 = make_float2(o0.x + p0.x, o0.y + p0.y);
                            }
                            *reinterpret_cast<float2 *>(dst) = o0;
                        } else {
#pragma unroll
                            for (int jj = 0; jj < kPer; ++jj)
                                if (gbase + jj < a.G) dst[jj] = a.accumulate ? dst[jj] + out[jj] : out[jj];
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(b_empty(bstage));  // this warp is done with the record's -b / constants
                if (++bstage == kBStages) {
                    bstage = 0;
                    bphase ^= 1;
                }
            }
            if (kFused) {
                // ---- sample_from_scores for the chunk's rows: combine the column parts, then every thread walks one row
#pragma unroll
                for (int t = 0; t < kChunkTiles; ++t) {
                    half_m[h * kChunkTiles * kTcRows + t * kTcRows + r_in_tile] = om[t];
                    half_s[h * kChunkTiles * kTcRows + t * kTcRows + r_in_tile] = os[t];
                }
                asm volatile("bar.sync 1, %0;\n" ::"n"(32 * kEpiWarps) : "memory");  // scratch and the part pairs are complete (CTA-scope visibility)
                const int et = tid - 64;
                for (int rc = et; rc < nt * kTcRows; rc += 32 * kEpiWarps) {
                    const size_t row = t0 * kTcRows + rc;
                    if (row >= a.N || kDebug >= 1) continue;
                    float mm = half_m[rc];  // max score * log2e
#pragma unroll
                    for (int p = 1; p < kParts; ++p) mm = fmaxf(mm, half_m[p * kChunkTiles * kTcRows + rc]);
                    float total = 0.f;
#pragma unroll
                    for (int p = 0; p < kParts; ++p)
                        total = fmaf(half_s[p * kChunkTiles * kTcRows + rc], mufu_ex2(half_m[p * kChunkTiles * kTcRows + rc] - mm), total);
                    float tt = total * __ldg(a.u + row);
                    const float2 *src = reinterpret_cast<const float2 *>(scratch) + rc;  // pair j of this row: src[j * rows per chunk]
                    const float2 ninf = make_float2(-INFINITY, -INFINITY);
                    const int npairs = a.Gpad / 2;
                    unsigned neg = 0;
                    for (int j2 = 0; j2 < npairs; j2 += 16) {  // 32 cells per step, sixteen loads in flight
                        float2 v[16];
#pragma unroll
                        for (int k = 0; k < 16; ++k) v[k] = j2 + k < npairs ? ld_f2_hint(src + static_cast<size_t>(j2 + k) * (kChunkTiles * kTcRows), pol_keep) : ninf;
#pragma unroll
                        for (int k = 0; k < 16; ++k) {
                            tt -= mufu_ex2(fmaf(v[k].x, kLog2e, -mm));
                            neg += __float_as_uint(tt) >> 31;
                            tt -= mufu_ex2(fmaf(v[k].y, kLog2e, -mm));
                            neg += __float_as_uint(tt) >> 31;
                        }
                    }
                    const int walked = (npairs + 15) / 16 * 32;  // cells walked, incl. the -inf fill of a ragged last step
                    a.assign[row] = min(walked - static_cast<int>(neg), a.G - 1);
                }
                asm volatile("bar.sync 1, %0;\n" ::"n"(32 * kEpiWarps) : "memory");  // nobody overwrites the scratch while a row is still being walked
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" ::"r"(tmem_base) : "memory");
}

// ---------------------------------------------------------------------------------------------
size_t niw_tc_floats(int G) {
    const size_t nb = (G + kTcGroupsPerBlock - 1) / kTcGroupsPerBlock;
    return (nb * kBlockRecBytes + 3) / 4;
}

int launch_niw_tc_prep(dist_b200_ctx *ctx, int G, const float *recs, float *tc_buf, cudaStream_t s) {
    const int nb = (G + kTcGroupsPerBlock - 1) / kTcGroupsPerBlock;
    if (nb == 0) return DIST_B200_OK;
    niw_tc_prep_kernel<<<nb, 256, 0, s>>>(G, recs, reinterpret_cast<unsigned char *>(tc_buf));
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("niw_tc_prep launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

// scores != nullptr: [N][G] scores (optionally accumulated); else the fused sampler writes assign[N]
int launch_niw_tc(dist_b200_ctx *ctx, int G, const float *tc_buf, const void *values, size_t N, const float *prior,
                  float *scores, int accumulate, const float *u, int32_t *assign, cudaStream_t s) {
    if (N == 0 || G == 0) return DIST_B200_OK;
    const int nb = (G + kTcGroupsPerBlock - 1) / kTcGroupsPerBlock;
    const bool fused = scores == nullptr;
    if (fused && (!u || !assign)) return fail(ctx, DIST_B200_ERR_INVALID, "niw_tc: nothing to produce");
    const size_t ntiles = (N + kTcRows - 1) / kTcRows;
    const size_t nchunks = (ntiles + kChunkTiles - 1) / kChunkTiles;
    const unsigned grid = static_cast<unsigned>(nchunks < static_cast<size_t>(ctx->sm_count) ? nchunks : ctx->sm_count);
    // per-call buffers: packed rows | tile scales | (fused) per-CTA score scratch
    const size_t xbytes = ntiles * kATileBytes;
    const size_t sxbytes = (ntiles * sizeof(float) + 255) / 256 * 256;
    const size_t Gpad = static_cast<size_t>(nb) * kTcGroupsPerBlock;
    const size_t scratch_bytes = fused ? static_cast<size_t>(grid) * kChunkTiles * kTcRows * Gpad * sizeof(float) : 0;
    if (int rc = grow(ctx, ctx->xpack, ctx->xpack_bytes, xbytes + sxbytes + scratch_bytes)) return rc;
    unsigned char *base = static_cast<unsigned char *>(ctx->xpack);
    NiwTcArgs a{};
    a.G = G;
    a.n_blocks = nb;
    a.accumulate = accumulate;
    a.Gpad = static_cast<int>(Gpad);
    a.N = N;
    a.ntiles = ntiles;
    a.blockrecs = reinterpret_cast<const unsigned char *>(tc_buf);
    a.xpack = reinterpret_cast<const __half *>(base);
    a.sx = reinterpret_cast<const float *>(base + xbytes);
    a.prior = prior;
    a.scores = scores;
    a.scratch = reinterpret_cast<float *>(base + xbytes + sxbytes);
    a.u = u;
    a.assign = assign;
    niw_tc_pack_x_kernel<<<static_cast<unsigned>(ntiles), 256, 0, s>>>(N, static_cast<const float *>(values), reinterpret_cast<__half *>(base),
                                                                   reinterpret_cast<float *>(base + xbytes));
    const size_t smem = static_cast<size_t>(kChunkTiles) * kATileBytes + static_cast<size_t>(kBStages) * kBlockRecBytes +
                        2 * (kEpiWarps / 4) * kChunkTiles * kTcRows * sizeof(float) + 32 * sizeof(uint64_t) + 1024;
    cudaError_t e;
    auto launch = [&](auto kern) {
        cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (err == cudaSuccess) kern<<<grid, kFusedThreads, smem, s>>>(a);
        return err;
    };
    if (fused) {
        switch (ctx->opt[DIST_B200_OPT_NIW_DEBUG]) {  // profiling variants, see the kernel's comment
            case 0: e = launch(niw_tc_fused_kernel<true, 0>); break;
            case 1: e = launch(niw_tc_fused_kernel<true, 1>); break;
            case 2: case 3: e = launch(niw_tc_fused_kernel<true, 2>); break;
            case 4: e = launch(niw_tc_fused_kernel<true, 4>); break;
            default: e = launch(niw_tc_fused_kernel<true, 5>); break;
        }
    } else {
        e = launch(niw_tc_fused_kernel<false, 0>);
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("niw_tc launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

}  // namespace distb200
