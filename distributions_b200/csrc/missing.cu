// missing.cu -- the two small kernels behind the masked entries that reuse unmasked kernels (api.cu):
//   mask_assign: an assignment vector with -1 wherever a feature's cell is (not) observed, so that add / remove rows and
//                sample_values skip exactly those rows of that feature through their existing kernels;
//   masked_accumulate: one dpd / niw feature's [N][G] scores added into the list's scores where the cell is observed.
#include <algorithm>

#include "common.cuh"

namespace distb200 {

__global__ void __launch_bounds__(256) mask_assign_kernel(const int32_t *__restrict__ assign, const uint32_t *__restrict__ observed,
                                                          size_t N, uint32_t keep, int32_t *__restrict__ out) {
    const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
    for (size_t n = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; n < N; n += stride) {
        const uint32_t bit = (__ldg(observed + (n >> 5)) >> (n & 31)) & 1u;
        out[n] = bit == keep ? assign[n] : -1;
    }
}

int launch_mask_assign(dist_b200_ctx *ctx, const int32_t *assign, const uint32_t *observed, size_t N, int keep, int32_t *out,
                       cudaStream_t s) {
    if (N == 0) return DIST_B200_OK;
    const size_t blocks = std::min<size_t>((N + 255) / 256, static_cast<size_t>(ctx->sm_count) * 8);
    mask_assign_kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(assign, observed, N, keep ? 1u : 0u, out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("mask_assign launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

// one thread per 4 groups of a row (16-byte accesses when G % 4 == 0, scalar otherwise).  A missing cell selects 0,
// never 0 * tmp: the missing row's tmp may be inf or NaN (its value was scored like any other)
template <bool kVec>
__global__ void __launch_bounds__(256) masked_accumulate_kernel(float *__restrict__ scores, const float *__restrict__ tmp,
                                                                const uint32_t *__restrict__ observed, size_t N, int G,
                                                                const float *__restrict__ prior, int accumulate) {
    const int q = (G + 3) / 4;
    const size_t total = N * static_cast<size_t>(q);
    const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride) {
        const size_t n = i / q;
        const int g0 = static_cast<int>(i - n * q) * 4;
        const bool obs = (__ldg(observed + (n >> 5)) >> (n & 31)) & 1u;
        float *dst = scores + n * G + g0;
        const float *src = tmp + n * G + g0;
        if (kVec) {
            float4 b = accumulate ? *reinterpret_cast<const float4 *>(dst)
                                  : (prior ? *reinterpret_cast<const float4 *>(prior + g0) : make_float4(0.f, 0.f, 0.f, 0.f));
            if (obs) {
                const float4 t = *reinterpret_cast<const float4 *>(src);
                b.x += t.x;
                b.y += t.y;
                b.z += t.z;
                b.w += t.w;
            }
            *reinterpret_cast<float4 *>(dst) = b;
        } else {
            for (int k = 0; k < 4 && g0 + k < G; ++k) {
                float b = accumulate ? dst[k] : (prior ? prior[g0 + k] : 0.f);
                if (obs) b += src[k];
                dst[k] = b;
            }
        }
    }
}

int launch_masked_accumulate(dist_b200_ctx *ctx, float *scores, const float *tmp, const uint32_t *observed, size_t N, int G,
                             const float *prior, int accumulate, cudaStream_t s) {
    if (N == 0) return DIST_B200_OK;
    const size_t total = N * static_cast<size_t>((G + 3) / 4);
    const unsigned blocks = static_cast<unsigned>(std::min<size_t>((total + 255) / 256, static_cast<size_t>(ctx->sm_count) * 16));
    const bool vec = G % 4 == 0 && reinterpret_cast<uintptr_t>(scores) % 16 == 0 && reinterpret_cast<uintptr_t>(tmp) % 16 == 0 &&
                     (!prior || reinterpret_cast<uintptr_t>(prior) % 16 == 0);
    if (vec) masked_accumulate_kernel<true><<<blocks, 256, 0, s>>>(scores, tmp, observed, N, G, prior, accumulate);
    else masked_accumulate_kernel<false><<<blocks, 256, 0, s>>>(scores, tmp, observed, N, G, prior, accumulate);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("masked_accumulate launch: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

}  // namespace distb200
