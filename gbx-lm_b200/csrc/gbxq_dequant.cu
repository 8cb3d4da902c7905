// gbxq_dequant.cu -- bit-exact mx.dequantize replacement (reference callers: gbx_lm/tuner/lora.py:62-68,
// gbx_lm/tuner/utils.py:214-220, gbx_lm/tuner/dora.py:101).
//
//   W[n,k] = T( T(scale * T(q)) + bias )   -- two roundings, the multiply and the add are separate
//   T-typed operations in MLX's op graph (no FMA); q <= 255 is exact in bf16/f16/f32.
//
// HBM-bound: reads bits/8 B and writes sizeof(T) B per weight.  One thread converts one octet
// (8 codes -> 16 B of bf16/f16 or 32 B of f32) so that a warp writes 512 contiguous bytes.
#include "gbxq_common.cuh"

namespace gbxq {

template <int BITS, typename T>
__global__ void __launch_bounds__(256) dequant_kernel(const uint32_t* __restrict__ w, const T* __restrict__ scales,
                                                      const T* __restrict__ biases, T* __restrict__ out, int64_t N,
                                                      int64_t K, int gs) {
    const int64_t octets_per_row = K >> 3;
    const int64_t total = N * octets_per_row;
    const int64_t wpr = K * BITS / 32;
    const int64_t G = K / gs;
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += (int64_t)gridDim.x * blockDim.x) {
        const int64_t n = o / octets_per_row;
        const int64_t k8 = o - n * octets_per_row;
        uint32_t q[8];
        extract_octet<BITS>(w + n * wpr, k8, wpr, q);
        const int64_t g = (k8 << 3) / gs;  // gs % 8 == 0: an octet never crosses a group
        const float s = to_f32(scales[n * G + g]);
        const float b = to_f32(biases[n * G + g]);
        T vals[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const float prod = round_to<T>(__fmul_rn(s, (float)q[i]));  // T(scale * q)
            vals[i] = from_f32<T>(__fadd_rn(prod, b));                  // T(prod + bias)
        }
        T* dst = out + n * K + (k8 << 3);
        if constexpr (sizeof(T) == 2) {
            *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(vals);
        } else {
            reinterpret_cast<uint4*>(dst)[0] = reinterpret_cast<const uint4*>(vals)[0];
            reinterpret_cast<uint4*>(dst)[1] = reinterpret_cast<const uint4*>(vals)[1];
        }
    }
}

template <int BITS, typename T>
static int launch_t(const uint32_t* w, const void* s, const void* b, void* out, int64_t N, int64_t K, int gs,
                    cudaStream_t st) {
    const int64_t total = N * (K >> 3);
    if (total == 0) return GBXQ_OK;
    const int threads = 256;
    int64_t blocks = (total + threads - 1) / threads;
    const int64_t cap = (int64_t)device_sm_count() * 16;
    if (blocks > cap) blocks = cap;
    return launch(dequant_kernel<BITS, T>, dim3((unsigned)blocks), dim3(threads), 0, st, false, w, (const T*)s, (const T*)b,
                  (T*)out, N, K, gs);
}

template <int BITS>
static int launch_b(const uint32_t* w, const void* s, const void* b, void* out, int64_t N, int64_t K, int gs,
                    int dtype, cudaStream_t st) {
    switch (dtype) {
        case GBXQ_BF16: return launch_t<BITS, __nv_bfloat16>(w, s, b, out, N, K, gs, st);
        case GBXQ_F16: return launch_t<BITS, __half>(w, s, b, out, N, K, gs, st);
        default: return launch_t<BITS, float>(w, s, b, out, N, K, gs, st);
    }
}

int launch_dequantize(const uint32_t* w, const void* s, const void* b, void* out, int64_t N, int64_t K, int bits,
                      int gs, int dtype, cudaStream_t st) {
    switch (bits) {
        case 2: return launch_b<2>(w, s, b, out, N, K, gs, dtype, st);
        case 3: return launch_b<3>(w, s, b, out, N, K, gs, dtype, st);
        case 4: return launch_b<4>(w, s, b, out, N, K, gs, dtype, st);
        case 6: return launch_b<6>(w, s, b, out, N, K, gs, dtype, st);
        case 8: return launch_b<8>(w, s, b, out, N, K, gs, dtype, st);
    }
    return GBXQ_EINVAL_BITS;
}

}  // namespace gbxq
