// gbxq_generic.cu -- shape-agnostic quantized matmul (any M,N; K % 32 == 0; bf16/f16/f32).
//
// Serves every argument combination the fast kernels decline (f16/f32 activations, rows whose
// byte length is not 16-byte aligned, tiny K) with the same numerical contract as the fast paths:
// fp32 accumulate of x*q per group, y += scale*sum(x q) + bias*sum(x), one final rounding to T,
// optional bias as a second rounded add (quantized_linear_gba.py:195-205).
// One warp per output row, lanes stride over 8-code octets, up to 4 rows of x per pass.
#include "gbxq_common.cuh"

namespace gbxq {

template <int BITS, typename T, int MT>
__global__ void __launch_bounds__(256) generic_kernel(const T* __restrict__ x, const uint32_t* __restrict__ w,
                                                      const T* __restrict__ scales, const T* __restrict__ biases,
                                                      const T* __restrict__ bias, T* __restrict__ y, int64_t M,
                                                      int64_t N, int64_t K, int gs) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t wpr = K * BITS / 32;
    const int64_t G = K / gs;
    const int64_t octets = K >> 3;
    const int64_t m0 = (int64_t)blockIdx.y * MT;

    for (int64_t n = warp; n < N; n += nwarps) {
        const uint32_t* row = w + n * wpr;
        float acc[MT];
#pragma unroll
        for (int m = 0; m < MT; m++) acc[m] = 0.f;
        for (int64_t k8 = lane; k8 < octets; k8 += 32) {
            uint32_t q[8];
            extract_octet<BITS>(row, k8, wpr, q);
            const int64_t g = (k8 << 3) / gs;
            const float s = to_f32(scales[n * G + g]);
            const float b = to_f32(biases[n * G + g]);
#pragma unroll
            for (int m = 0; m < MT; m++) {
                if (m0 + m < M) {
                    const T* xr = x + (m0 + m) * K + (k8 << 3);
                    float qs = 0.f, xs = 0.f;
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const float xv = to_f32(xr[i]);
                        qs = fmaf(xv, (float)q[i], qs);
                        xs += xv;
                    }
                    acc[m] = fmaf(s, qs, acc[m]);
                    acc[m] = fmaf(b, xs, acc[m]);
                }
            }
        }
#pragma unroll
        for (int m = 0; m < MT; m++) {
            const float v = warp_sum(acc[m]);
            if (lane == 0 && m0 + m < M) {
                float r = round_to<T>(v);
                if (bias != nullptr) r = __fadd_rn(r, to_f32(bias[n]));
                y[(m0 + m) * N + n] = from_f32<T>(r);
            }
        }
    }
}

template <int BITS, typename T>
static int launch_t(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y,
                    int64_t M, int64_t N, int64_t K, int gs, cudaStream_t st) {
    if (M == 0 || N == 0) return GBXQ_OK;
    constexpr int MT = 4;
    const int threads = 256;
    int64_t blocks = (N + 7) / 8;
    const int64_t cap = (int64_t)device_sm_count() * 8;
    if (blocks > cap) blocks = cap;
    const int64_t mtiles = (M + MT - 1) / MT;
    if (mtiles > 65535) return GBXQ_EUNSUPPORTED;
    dim3 grid((unsigned)blocks, (unsigned)mtiles);
    return launch(generic_kernel<BITS, T, MT>, grid, dim3(threads), 0, st, false, (const T*)x, w, (const T*)s, (const T*)b,
                  (const T*)bias, (T*)y, M, N, K, gs);
}

template <int BITS>
static int launch_b(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y,
                    int64_t M, int64_t N, int64_t K, int gs, int dtype, cudaStream_t st) {
    switch (dtype) {
        case GBXQ_BF16: return launch_t<BITS, __nv_bfloat16>(x, w, s, b, bias, y, M, N, K, gs, st);
        case GBXQ_F16: return launch_t<BITS, __half>(x, w, s, b, bias, y, M, N, K, gs, st);
        default: return launch_t<BITS, float>(x, w, s, b, bias, y, M, N, K, gs, st);
    }
}

int launch_generic(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y,
                   int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, cudaStream_t st) {
    switch (bits) {
        case 2: return launch_b<2>(x, w, s, b, bias, y, M, N, K, gs, dtype, st);
        case 3: return launch_b<3>(x, w, s, b, bias, y, M, N, K, gs, dtype, st);
        case 4: return launch_b<4>(x, w, s, b, bias, y, M, N, K, gs, dtype, st);
        case 6: return launch_b<6>(x, w, s, b, bias, y, M, N, K, gs, dtype, st);
        case 8: return launch_b<8>(x, w, s, b, bias, y, M, N, K, gs, dtype, st);
    }
    return GBXQ_EINVAL_BITS;
}

}  // namespace gbxq
