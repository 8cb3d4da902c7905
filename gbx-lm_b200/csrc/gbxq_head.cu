// gbxq_head.cu -- the UNQUANTIZED vocabulary projection of the decode step (SURVEY.md 8f rank 1):
//     logits[M, V] = x[M, K] . W[V, K]^T        W = lm_head.weight, or embed_tokens.weight when tied
// (reference: `out = self.lm_head(out)` / `self.model.embed_tokens.as_linear(out)`, gbx_lm/models/qllama.py:183-184,
// 194-198).  bf16 [V, K] is 21 % (8B) to 49 % (1B) of the bytes of a decode step, so once the quantized projections are
// fast this GEMV bounds tokens/s.  Pure HBM streaming: a warp owns whole rows of W, its lanes read the row as 16-byte
// vectors (8 bf16, coalesced 512 bytes per warp instruction, 8 vectors in flight per lane), multiply against the
// activations held in shared memory, accumulate in fp32 and reduce with warp shuffles; one rounding to bf16.
// Programmatic dependent launch as in the quantized decode kernels: the first weight vectors of a warp are requested
// BEFORE griddepcontrol.wait (the head's weights are frozen), x is read after it.
#include "gbxq_common.cuh"

namespace gbxq {

namespace {

constexpr int kHeadWarps = 16;
constexpr int kHeadThreads = kHeadWarps * 32;
constexpr int kInFlight = 8;  // 16-byte vectors a lane keeps in flight

__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

// MT tokens (1, 2, 4, 8).  x lives in shared memory as bf16 [MT][K]; nvec = K / 8 vectors per row, a multiple of 32.
template <int MT>
__global__ void __launch_bounds__(kHeadThreads, 2)
head_gemv_kernel(const __nv_bfloat16* __restrict__ x, const uint4* __restrict__ w, __nv_bfloat16* __restrict__ y, int M,
                 int64_t V, int K) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    uint4* xs = reinterpret_cast<uint4*>(smem_raw);  // [MT][K/8]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nvec = K >> 3;
    const int per_lane = nvec >> 5;  // vectors of a row per lane
    const int64_t nwarps = (int64_t)gridDim.x * kHeadWarps;
    const int64_t gw = (int64_t)blockIdx.x * kHeadWarps + warp;
    // contiguous row ranges per warp (a warp streams one long contiguous piece of W)
    const int64_t r0 = gw * V / nwarps, r1 = (gw + 1) * V / nwarps;

    if (threadIdx.x == 0) griddep_launch_dependents();
    // first vectors of the first row: requested before the dependency wait (frozen parameters)
    uint4 wv[kInFlight];
    const uint4* row = w + (size_t)r0 * nvec;
    if (r0 < r1) {
#pragma unroll
        for (int u = 0; u < kInFlight; u++)
            if (u < per_lane) wv[u] = ldg_stream(row + lane + 32 * u);
    }
    griddep_wait();
    for (int i = threadIdx.x; i < MT * nvec; i += kHeadThreads) {
        const int m = i / nvec;
        xs[i] = m < M ? reinterpret_cast<const uint4*>(x)[i] : make_uint4(0u, 0u, 0u, 0u);
    }
    __syncthreads();

    for (int64_t r = r0; r < r1; r++) {
        float acc[MT];
#pragma unroll
        for (int m = 0; m < MT; m++) acc[m] = 0.f;
        row = w + (size_t)r * nvec;
        for (int c0 = 0; c0 < per_lane; c0 += kInFlight) {
            if (c0 > 0 || r > r0) {
#pragma unroll
                for (int u = 0; u < kInFlight; u++)
                    if (c0 + u < per_lane) wv[u] = ldg_stream(row + lane + 32 * (c0 + u));
            }
#pragma unroll
            for (int u = 0; u < kInFlight; u++) {
                if (c0 + u < per_lane) {
                    const uint32_t ww[4] = {wv[u].x, wv[u].y, wv[u].z, wv[u].w};
                    float wf[8];
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        wf[2 * i] = __uint_as_float(ww[i] << 16);
                        wf[2 * i + 1] = __uint_as_float(ww[i] & 0xffff0000u);
                    }
#pragma unroll
                    for (int m = 0; m < MT; m++) {
                        const uint4 xv = xs[m * nvec + lane + 32 * (c0 + u)];
                        const uint32_t xw[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            acc[m] = fmaf(wf[2 * i], __uint_as_float(xw[i] << 16), acc[m]);
                            acc[m] = fmaf(wf[2 * i + 1], __uint_as_float(xw[i] & 0xffff0000u), acc[m]);
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int m = 0; m < MT; m++) acc[m] = warp_sum(acc[m]);
        if (lane == 0) {
#pragma unroll
            for (int m = 0; m < MT; m++)
                if (m < M) y[(size_t)m * V + r] = __float2bfloat16_rn(acc[m]);
        }
    }
}

template <int MT> int launch_mt(const void* x, const void* w, void* y, int M, int64_t V, int K, cudaStream_t st) {
    constexpr auto kern = head_gemv_kernel<MT>;
    const size_t smem = (size_t)MT * K * 2;
    const int rc = allow_dynamic_smem<kern>(100 * 1024);
    if (rc != GBXQ_OK) return rc;
    if (smem > 100 * 1024) return GBXQ_EUNSUPPORTED;
    return launch(kern, dim3((unsigned)(2 * device_sm_count())), dim3(kHeadThreads), smem, st, true,
                  reinterpret_cast<const __nv_bfloat16*>(x), reinterpret_cast<const uint4*>(w),
                  reinterpret_cast<__nv_bfloat16*>(y), M, V, K);
}

}  // namespace

int launch_head_gemv(const void* x, const void* w, void* y, int64_t M, int64_t V, int64_t K, cudaStream_t st) {
    if (M < 1 || M > 8 || V < 1 || K < 256 || (K % 256) || K > (1 << 20)) return GBXQ_EUNSUPPORTED;
    if (((uintptr_t)x | (uintptr_t)w) & 15) return GBXQ_EALIGN;
    if ((uintptr_t)y & 1) return GBXQ_EALIGN;
    if (M == 1) return launch_mt<1>(x, w, y, (int)M, V, (int)K, st);
    if (M == 2) return launch_mt<2>(x, w, y, (int)M, V, (int)K, st);
    if (M <= 4) return launch_mt<4>(x, w, y, (int)M, V, (int)K, st);
    return launch_mt<8>(x, w, y, (int)M, V, (int)K, st);
}

}  // namespace gbxq
