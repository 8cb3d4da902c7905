// gbxq_gather.cu -- the two quantized matmul forms either side of the QuantizedLinear path (SURVEY.md 8f-3 / 8f-4):
//
//   * mx.gather_qmm(x, w, scales, biases, rhs_indices=idx, transpose=True): the expert-indexed quantized matmul of
//     QuantizedSwitchLinear.__call__ (gbx_lm/models/switch_layers.py:78-92): batch item r multiplies the [M, K] matrix
//     x[lhs[r]] with expert rhs[r] of the stacked [E, N, K*bits/32] weights.
//   * mx.quantized_matmul(x, w, scales, biases, transpose=False): x[.., M, K] @ dequant(w)[K, N] with w quantized along
//     its last axis N -- `scores @ V` on the quantized KV cache (gbx_lm/models/base.py:90-92); batched through the same
//     index arrays (a GQA broadcast of V over the repeated query heads is rhs[r] = r / n_repeats).
//
// Both are batched by (lhs, rhs) index arrays that live on the DEVICE (router output / arange): no host round trip.
// Numerical contract as the other kernels: fp32 accumulation, one rounding to T, optional bias as a second rounded add.
// These are correct, coalesced CUDA kernels for decode-sized work (a few rows per batch item); they are not tuned
// against the roofline like the QuantizedLinear kernels.
#include "gbxq_common.cuh"

namespace gbxq {

namespace {

__device__ __forceinline__ int64_t clamp_index(const int32_t* idx, int64_t r, int64_t limit) {
    int64_t v = idx != nullptr ? (int64_t)idx[r] : r;
    if (v < 0) v = 0;
    if (v >= limit) v = limit - 1;
    return v;
}

// transpose = True: one warp per output feature n, lanes stride over 8-code octets of the expert's row n.
template <int BITS, typename T, int MT>
__global__ void __launch_bounds__(256) gather_t_kernel(const T* __restrict__ x, const uint32_t* __restrict__ w,
                                                       const T* __restrict__ scales, const T* __restrict__ biases,
                                                       const T* __restrict__ bias, const int32_t* __restrict__ lhs,
                                                       const int32_t* __restrict__ rhs, T* __restrict__ y, int64_t XB,
                                                       int64_t E, int64_t M, int64_t N, int64_t K, int gs) {
    const int lane = threadIdx.x & 31;
    const int64_t r = blockIdx.z;
    const int64_t xi = clamp_index(lhs, r, XB), e = clamp_index(rhs, r, E);
    const int64_t wpr = K * BITS / 32, G = K / gs, octets = K >> 3;
    const int64_t m0 = (int64_t)blockIdx.y * MT;
    const T* xb = x + xi * M * K;
    const uint32_t* wb = w + e * N * wpr;
    const T* sb = scales + e * N * G;
    const T* bb = biases + e * N * G;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t n = warp; n < N; n += nwarps) {
        const uint32_t* row = wb + n * wpr;
        float acc[MT];
#pragma unroll
        for (int m = 0; m < MT; m++) acc[m] = 0.f;
        for (int64_t k8 = lane; k8 < octets; k8 += 32) {
            uint32_t q[8];
            extract_octet<BITS>(row, k8, wpr, q);
            const int64_t g = (k8 << 3) / gs;
            const float s = to_f32(sb[n * G + g]), b = to_f32(bb[n * G + g]);
#pragma unroll
            for (int m = 0; m < MT; m++) {
                if (m0 + m < M) {
                    const T* xr = xb + (m0 + m) * K + (k8 << 3);
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
                float o = round_to<T>(v);
                if (bias != nullptr) o = __fadd_rn(o, to_f32(bias[e * N + n]));
                y[(r * M + m0 + m) * N + n] = from_f32<T>(o);
            }
        }
    }
}

// transpose = False: w[e] is [K, N*bits/32], quantized along N.  A thread owns one octet of 8 output columns and a
// slice of k; a block = OCT octets x (256 / OCT) k slices, partial sums meet in shared memory.  Loads of one k row are
// coalesced across the octets; x[m, k] is a broadcast.
template <int BITS, typename T, int MT>
__global__ void __launch_bounds__(256) gather_n_kernel(const T* __restrict__ x, const uint32_t* __restrict__ w,
                                                       const T* __restrict__ scales, const T* __restrict__ biases,
                                                       const int32_t* __restrict__ lhs, const int32_t* __restrict__ rhs,
                                                       T* __restrict__ y, int64_t XB, int64_t E, int64_t M, int64_t N,
                                                       int64_t K, int gs, int oct) {
    __shared__ float red[256 * 8];
    const int64_t r = blockIdx.z;
    const int64_t xi = clamp_index(lhs, r, XB), e = clamp_index(rhs, r, E);
    const int64_t wpr = N * BITS / 32, G = N / gs;
    const int64_t m0 = (int64_t)blockIdx.y * MT;
    const int o_in = threadIdx.x % oct, ks = threadIdx.x / oct, nks = 256 / oct;
    const int64_t o = (int64_t)blockIdx.x * oct + o_in;  // octet of output columns 8o .. 8o+7
    const bool live = (o << 3) < N;
    const T* xb = x + xi * M * K;
    const uint32_t* wb = w + e * K * wpr;
    const T* sb = scales + e * K * G;
    const T* bb = biases + e * K * G;
    float acc[MT][8];
#pragma unroll
    for (int m = 0; m < MT; m++)
#pragma unroll
        for (int i = 0; i < 8; i++) acc[m][i] = 0.f;
    if (live) {
        const int64_t g = (o << 3) / gs;
        for (int64_t k = ks; k < K; k += nks) {
            uint32_t q[8];
            extract_octet<BITS>(wb + k * wpr, o, wpr, q);
            const float s = to_f32(sb[k * G + g]), b = to_f32(bb[k * G + g]);
            float wv[8];
#pragma unroll
            for (int i = 0; i < 8; i++) wv[i] = fmaf(s, (float)q[i], b);
#pragma unroll
            for (int m = 0; m < MT; m++) {
                if (m0 + m < M) {
                    const float xv = to_f32(xb[(m0 + m) * K + k]);
#pragma unroll
                    for (int i = 0; i < 8; i++) acc[m][i] = fmaf(xv, wv[i], acc[m][i]);
                }
            }
        }
    }
    // reduce the k slices (fixed order: deterministic), slice 0 writes
#pragma unroll 1
    for (int m = 0; m < MT; m++) {
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 8; i++) red[threadIdx.x * 8 + i] = acc[m][i];
        __syncthreads();
        if (ks == 0 && live && m0 + m < M) {
#pragma unroll
            for (int i = 0; i < 8; i++) {
                float t = 0.f;
                for (int j = 0; j < nks; j++) t += red[(j * oct + o_in) * 8 + i];
                const int64_t n = (o << 3) + i;
                if (n < N) y[(r * M + m0 + m) * N + n] = from_f32<T>(t);
            }
        }
    }
}

template <int BITS, typename T>
int launch_t(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, const int32_t* lhs,
             const int32_t* rhs, void* y, int64_t R, int64_t XB, int64_t E, int64_t M, int64_t N, int64_t K, int transpose,
             int gs, cudaStream_t st) {
    constexpr int MT = 4;
    const int64_t mtiles = (M + MT - 1) / MT;
    if (mtiles > 65535 || R > 65535) return GBXQ_EUNSUPPORTED;
    if (transpose) {
        int64_t blocks = (N + 7) / 8;
        const int64_t cap = (int64_t)device_sm_count() * 8;
        if (blocks > cap) blocks = cap;
        dim3 grid((unsigned)blocks, (unsigned)mtiles, (unsigned)R);
        return launch(gather_t_kernel<BITS, T, MT>, grid, dim3(256), 0, st, false, (const T*)x, w, (const T*)s, (const T*)b,
                      (const T*)bias, lhs, rhs, (T*)y, XB, E, M, N, K, gs);
    } else {
        const int64_t octs = (N + 7) / 8;
        int oct = 32;
        while (oct > 1 && oct / 2 >= octs) oct /= 2;  // narrow N (head_dim 64 / 128): more k slices per block
        dim3 grid((unsigned)((octs + oct - 1) / oct), (unsigned)mtiles, (unsigned)R);
        return launch(gather_n_kernel<BITS, T, MT>, grid, dim3(256), 0, st, false, (const T*)x, w, (const T*)s, (const T*)b, lhs,
                      rhs, (T*)y, XB, E, M, N, K, gs, oct);
    }
}

template <int BITS>
int launch_b(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, const int32_t* lhs,
             const int32_t* rhs, void* y, int64_t R, int64_t XB, int64_t E, int64_t M, int64_t N, int64_t K, int transpose,
             int gs, int dtype, cudaStream_t st) {
    switch (dtype) {
        case GBXQ_BF16: return launch_t<BITS, __nv_bfloat16>(x, w, s, b, bias, lhs, rhs, y, R, XB, E, M, N, K, transpose, gs, st);
        case GBXQ_F16: return launch_t<BITS, __half>(x, w, s, b, bias, lhs, rhs, y, R, XB, E, M, N, K, transpose, gs, st);
        default: return launch_t<BITS, float>(x, w, s, b, bias, lhs, rhs, y, R, XB, E, M, N, K, transpose, gs, st);
    }
}

}  // namespace

int launch_gather_qmm(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, const int32_t* lhs,
                      const int32_t* rhs, void* y, int64_t R, int64_t XB, int64_t E, int64_t M, int64_t N, int64_t K,
                      int transpose, int bits, int gs, int dtype, cudaStream_t st) {
    // grid.z carries the batch: split long batches
    for (int64_t r0 = 0; r0 < R; r0 += 32768) {
        const int64_t rn = R - r0 < 32768 ? R - r0 : 32768;
        const size_t esz = dtype == GBXQ_F32 ? 4 : 2;
        void* yo = reinterpret_cast<uint8_t*>(y) + (size_t)r0 * M * N * esz;
        const int32_t* l = lhs ? lhs + r0 : nullptr;
        const int32_t* rr = rhs ? rhs + r0 : nullptr;
        // without index arrays item r reads x[r] / w[r]: shift the bases instead
        const void* xo = lhs ? x : reinterpret_cast<const uint8_t*>(x) + (size_t)r0 * M * K * esz;
        const int64_t xb = lhs ? XB : XB - r0;
        int rc;
        if (rhs == nullptr && r0 > 0) return GBXQ_EUNSUPPORTED;  // > 32768 experts addressed by position: not a real case
        switch (bits) {
            case 2: rc = launch_b<2>(xo, w, s, b, bias, l, rr, yo, rn, xb, E, M, N, K, transpose, gs, dtype, st); break;
            case 3: rc = launch_b<3>(xo, w, s, b, bias, l, rr, yo, rn, xb, E, M, N, K, transpose, gs, dtype, st); break;
            case 4: rc = launch_b<4>(xo, w, s, b, bias, l, rr, yo, rn, xb, E, M, N, K, transpose, gs, dtype, st); break;
            case 6: rc = launch_b<6>(xo, w, s, b, bias, l, rr, yo, rn, xb, E, M, N, K, transpose, gs, dtype, st); break;
            case 8: rc = launch_b<8>(xo, w, s, b, bias, l, rr, yo, rn, xb, E, M, N, K, transpose, gs, dtype, st); break;
            default: return GBXQ_EINVAL_BITS;
        }
        if (rc != GBXQ_OK) return rc;
    }
    return GBXQ_OK;
}

}  // namespace gbxq
