// numerics.cuh -- device restatements of the reference's fast math (special.hpp, vendor/fmath.hpp),
// fused into the score kernels instead of living behind vector_math.cc loops.
//
// Two forms of fast_log exist on purpose:
//   fast_log_table : the literal 2^14-entry table (special.hpp:57-67).  Used by the cache-rebuild
//                    kernels, which are O(G*dim) and off the hot path, so dd/dpd/bb caches and every
//                    fast_log inside a Scorer::init are bit-identical to the restated algorithm.
//   fast_log_cell  : the per-cell form for arguments that are positive, finite and normal (nich/niw:
//                    1 + precision*d^2 >= 1).  The reference's table is indexed by the top 14 mantissa
//                    bits, i.e. it evaluates log2 of the argument with its low 9 mantissa bits cleared.
//                    Clearing those bits and issuing one MUFU.LG2 reproduces that step function --
//                    including its truncation bias -- to within the MUFU error (<= 2^-22 absolute in
//                    log2 for arguments in [1,2), 2^-22 relative elsewhere) without a 64 KB gather.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace distb200 {

constexpr float kLn2 = 0.69314718055994529f;   // special.hpp:66
constexpr float kLog2e = 1.4426950408889634f;
constexpr int kLgammaRowStride = 8;            // lgamma_approx_coeff5 rows padded 6 -> 8 floats

// device-resident tables owned by the context
struct NumericTables {
    const float *log2_table;   // [1 << 14]  special.cc:35-44
    const float *lgamma5;      // [33][8]    special.cc:144-211 (a5..a0, 2 pad)
    const float *lgamma_nu3;   // [18][4]    special.cc:232-269 (a3..a0)
    const float *log_factorial;  // [64]     special.cc:213-230
};

__device__ __forceinline__ float mufu_lg2(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));  // ftz: no denormal fix-up code around the MUFU
    return y;
}
__device__ __forceinline__ float mufu_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// special.hpp:57-67, any input (sign ignored, 0 -> -127 ln 2, inf -> 128 ln 2)
__device__ __forceinline__ float fast_log_table(float x, const float *__restrict__ log2_table) {
    const int intx = __float_as_int(x);
    const int e = ((intx >> 23) & 255) - 127;
    const int man = (intx & 0x7FFFFF) >> 9;
    return __fmul_rn(__fadd_rn(static_cast<float>(e), __ldg(log2_table + man)), kLn2);
}

// per-cell form; x must be positive, finite, normal.  fast_log2_cell is the table's log2 part; the
// hot loops fold the trailing `* ln 2` into the per-group coefficient (one FMUL less per cell).
__device__ __forceinline__ float fast_log2_cell(float x) {
    return mufu_lg2(__uint_as_float(__float_as_uint(x) & 0xFFFFFE00u));
}
__device__ __forceinline__ float fast_log_cell(float x) { return fast_log2_cell(x) * kLn2; }

// The log-determinant of an NIW scale matrix (score_mv_student_t's constant, Group::score_data): fast_log(det) as the
// reference writes it while det is a normal float; beyond that (the reference's float determinant() has overflowed to
// inf or flushed to 0, and its result is meaningless) the log of the determinant itself, logdet = sum_i 2 ln L_ii, as the
// reference's exact-math Python flavour computes it (dbg/models/niw.py:213,216).  At d = 32 the window is a geometric-mean
// per-dimension variance in about [0.065, 16].
__device__ __forceinline__ float niw_log_det(double det, double logdet, const float *__restrict__ log2_table) {
    const float f = static_cast<float>(det);
    if (isfinite(f) && f >= 1.17549435e-38f) return fast_log_table(f, log2_table);
    return static_cast<float>(logdet);
}

// fast_exp as used by scores_to_likelihoods (random.cc:94-106): argument = score - max <= 0.
// fmath::exp is exp() to 4e-7 (source) / 5e-6 (the -ffast-math build); MUFU.EX2 of x*log2(e) is
// within 2^-22 + the rounding of the product.  Results below 2^-126 flush to 0 (the reference
// returns garbage denormals there, fmath.hpp:455-458; both are < 1.2e-38 of the row maximum).
__device__ __forceinline__ float fast_exp_neg(float x) { return mufu_ex2(x * kLog2e); }

// log sum_g exp(s_g) from a reference nm = -(m log2 e) and sum = sum_g 2^(s_g log2 e + nm): ln(sum) - nm ln 2.  A row
// whose every term is -inf has sum = 0 (nm finite: the callers clamp it) and gets -inf, never NaN.
__device__ __forceinline__ float logp_finish(float nm, float sum) { return fmaf(-nm, kLn2, logf(sum)); }

// floor(log2 y) for positive y from the exponent field (special.hpp:127-146; subnormals via clz)
__device__ __forceinline__ int float_exponent(float y) {
    const int x = __float_as_int(y);
    const int c = x >> 23;
    return c ? c - 127 : (31 - __clz(x)) - 149;
}

// special.hpp:114-171.  Hot form: fp32 Horner (the reference accumulates explicit powers in double;
// measured difference <= 4.1e-7 relative).  y < 2.5 or >= 2^32 defers to lgammaf like the reference.
static __device__ __noinline__ float lgammaf_slow(float y) { return lgammaf(y); }

__device__ __forceinline__ float fast_lgamma_cell(float y, const float *__restrict__ coeff /* [33][8] */) {
    if (y < 2.5f || 4294967295.0f <= y) return lgammaf_slow(y);
    const int c = (__float_as_int(y) >> 23) - 127;
    const float4 hi = *reinterpret_cast<const float4 *>(coeff + c * kLgammaRowStride);      // a5 a4 a3 a2
    const float2 lo = *reinterpret_cast<const float2 *>(coeff + c * kLgammaRowStride + 4);  // a1 a0
    float s = fmaf(hi.x, y, hi.y);
    s = fmaf(s, y, hi.z);
    s = fmaf(s, y, hi.w);
    s = fmaf(s, y, lo.x);
    return fmaf(s, y, lo.y);
}

// exact restatement for the cache rebuilds: double power sums as written (special.hpp:154-170)
__device__ inline float fast_lgamma_exact(float y, const float *__restrict__ coeff) {
    if (y < 2.5f || 4294967295.0f <= y) return lgammaf(y);
    const float *a = coeff + float_exponent(y) * kLgammaRowStride;
    double yprod = y;
    double sum = a[5];
    sum += a[4] * yprod;
    yprod *= y;
    sum += a[3] * yprod;
    yprod *= y;
    sum += a[2] * yprod;
    yprod *= y;
    sum += a[1] * yprod;
    yprod *= y;
    sum += a[0] * yprod;
    return static_cast<float>(sum);
}

// special.hpp:208-214
__device__ __forceinline__ float fast_log_factorial(uint32_t n, const float *__restrict__ table64,
                                                    const float *__restrict__ coeff) {
    if (n < 64) return table64[n];
    return fast_lgamma_exact(static_cast<float>(n + 1u), coeff);
}

// special.hpp:224-235,239-273 (cache rebuild only: nich Scorer::init)
__device__ inline float fast_lgamma_nu(float nu, const float *__restrict__ coeff3 /* [18][4] */) {
    if (nu < 0.0625f || 4294967295.0f <= nu) {
        return __fsub_rn(lgammaf(__fadd_rn(__fmul_rn(nu, 0.5f), 0.5f)), lgammaf(__fmul_rn(nu, 0.5f)));
    }
    const int c = float_exponent(nu);
    const float *a = coeff3 + ((c + 4) / 2) * 4;
    // a0 + x*a1 + x*x*a2 + x*x*x*a3, left to right, no contraction
    float r = __fadd_rn(a[3], __fmul_rn(nu, a[2]));
    r = __fadd_rn(r, __fmul_rn(__fmul_rn(nu, nu), a[1]));
    r = __fadd_rn(r, __fmul_rn(__fmul_rn(__fmul_rn(nu, nu), nu), a[0]));
    return r;
}

// Blackwell packed fp32 pairs (one issue slot, two lanes of the FMA pipe); every element is IEEE-rounded like
// the scalar __fadd_rn / __fmul_rn / fmaf it replaces
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

// exp2 of a pair on the FMA pipe (Cody-Waite split + degree-5 polynomial, <= 2.21e-7 relative over every fp32
// argument in [-1, 0], hence over every reachable fractional part: the accuracy class of MUFU.EX2's 2^-22; the constant
// term is exactly 1, so integer arguments give exact powers of two), for arguments <= ~0.  The sampling kernels are bound by the MUFU pipe (16 lanes / clock / SM) while the
// FMA pipe idles: a share of their exp2 takes this route instead of MUFU.EX2 (the softmax trick of recent attention
// kernels; nich_rows.cu: kPoly of every 16 pairs).  x + 1.5 * 2^23 rounds x to the nearest integer n in the low mantissa bits, f = x - n lies
// in [-0.5, 0.5], and 2^n is applied by adding n to the exponent field; below -125 the argument is clamped (2^-125 of
// the row maximum: the MUFU route flushes those cells to 0, both are < 3e-38 of the total).
__device__ __forceinline__ uint64_t poly_ex2_pair(uint64_t x2) {
    float xa, xb;
    f2_unpack(x2, xa, xb);
    x2 = f2_pack(fmaxf(xa, -125.f), fmaxf(xb, -125.f));
    const float magic = 12582912.f;
    const uint64_t r2 = f2_add(x2, f2_pack(magic, magic));
    const uint64_t f2 = f2_add(x2, f2_fma(r2, f2_pack(-1.f, -1.f), f2_pack(magic, magic)));  // x - n, exact
    uint64_t p2 = f2_fma(f2_pack(0.0013276472454890609f, 0.0013276472454890609f), f2, f2_pack(0.009675540961325169f, 0.009675540961325169f));
    p2 = f2_fma(p2, f2, f2_pack(0.05550713092088699f, 0.05550713092088699f));
    p2 = f2_fma(p2, f2, f2_pack(0.24022120237350464f, 0.24022120237350464f));
    p2 = f2_fma(p2, f2, f2_pack(0.6931469440460205f, 0.6931469440460205f));
    p2 = f2_fma(p2, f2, f2_pack(1.f, 1.f));
    float pa, pb, ra, rb;
    f2_unpack(p2, pa, pb);
    f2_unpack(r2, ra, rb);
    return f2_pack(__uint_as_float(__float_as_uint(pa) + (__float_as_uint(ra) << 23)),
                   __uint_as_float(__float_as_uint(pb) + (__float_as_uint(rb) << 23)));
}

}  // namespace distb200
