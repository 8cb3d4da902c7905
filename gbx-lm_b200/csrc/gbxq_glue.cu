// gbxq_glue.cu -- the step-either-side fusions of a batch-1..4 DECODE step (SURVEY.md 8f rank 2): what sits between the
// QuantizedLinear forwards of a block in the reference's callers (gbx_lm/models/qllama.py:76-141) as four small kernels
// instead of ~45 framework launches per block:
//   rope_cache        q, k <- RoPE(q, k) (mx.fast.rope, traditional=False; qllama.py:83-88), k / v written into the static
//                     KV cache at the step's position (cache.update_and_fetch, qllama.py:85), or, on a rotating cache, at
//                     the ring slot of that position (RotatingKVCache, gbx_lm/models/cache.py:280-420; kv_cache_row)
//   decode_attention  one query row per head against the cache, causal over absolute positions, GQA
//                     (scaled_dot_product_attention, qllama.py:90-93)
//   add_rmsnorm       h = x + r (residual, qllama.py:137-141) and y = RMSNorm(h) * w (nn.RMSNorm) in one pass
//   silu_mul          silu(gate) * up (qllama.py:115)
// All bf16 in / out, fp32 inside, position read from DEVICE memory (CUDA-graph replayable).  They are launch-latency
// bound (a few KB each); the point is the launch count of the decode step, not bandwidth.
#include <math.h>

#include "gbxq_common.cuh"

namespace gbxq {

namespace {

__device__ __forceinline__ float bf(const __nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ __nv_bfloat16 tobf(float v) { return __float2bfloat16_rn(v); }

// grid (Hq + 2 Hkv, B * T), block D/2 threads.  Row r = b * T + t of q / k / v is token t of batch row b, at position
// p_b + t (T > 1: a verify block of consecutive tokens; cache row b receives all of them).  Head h < Hq: rotate q in
// place; Hq <= h < Hq+Hkv: rotate k into the cache; else copy v into the cache.
__global__ void rope_cache_kernel(__nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                                  const __nv_bfloat16* __restrict__ v, const int64_t* __restrict__ pos_p,
                                  const float* __restrict__ inv_freq, __nv_bfloat16* __restrict__ kc,
                                  __nv_bfloat16* __restrict__ vc, int Hq, int Hkv, int D, int64_t max_len, int64_t keep,
                                  int pos_stride, int T) {
    const int h = blockIdx.x, r = blockIdx.y, b = r / T, i = threadIdx.x, half = D / 2;
    pdl_wait_then_trigger();
    // the RoPE angle is the absolute position's; k / v go to its cache row.  pos_stride 0: one position for every row
    const int64_t pos = pos_p[(size_t)b * pos_stride] + r % T;
    const int64_t row = kv_cache_row(pos, max_len, keep);
    if (row < 0) return;  // never write outside the cache
    if (h < Hq + Hkv) {
        const bool isq = h < Hq;
        const __nv_bfloat16* src = isq ? q + ((size_t)r * Hq + h) * D : k + ((size_t)r * Hkv + (h - Hq)) * D;
        __nv_bfloat16* dst = isq ? q + ((size_t)r * Hq + h) * D : kc + (((size_t)b * Hkv + (h - Hq)) * max_len + row) * D;
        const float ang = __fmul_rn((float)pos, inv_freq[i]);
        const float c = cosf(ang), s = sinf(ang);
        const float x1 = bf(src[i]), x2 = bf(src[i + half]);
        // separate roundings of the four products, as the unfused elementwise graph computes them
        const float o1 = __fsub_rn(__fmul_rn(x1, c), __fmul_rn(x2, s));
        const float o2 = __fadd_rn(__fmul_rn(x1, s), __fmul_rn(x2, c));
        dst[i] = tobf(o1);
        dst[i + half] = tobf(o2);
    } else {
        const int hv = h - Hq - Hkv;
        const __nv_bfloat16* src = v + ((size_t)r * Hkv + hv) * D;
        __nv_bfloat16* dst = vc + (((size_t)b * Hkv + hv) * max_len + row) * D;
        dst[i] = src[i];
        dst[i + half] = src[i + half];
    }
}

// grid (Hq, B * T), block 256 threads, dynamic shared memory = one float per visible key.  Query row r = b * T + t reads
// cache row b with keys 0 .. p_b + t visible: a verify block's t-th query is exactly a single query at p_b + t.
// Phase 1: one THREAD per key (keys tid, tid + 256, ...): the 16-byte loads of a key row are independent, so a block
// has thousands of bytes in flight instead of one dependent load per warp and key (the first version of this kernel
// walked the keys with an online softmax per warp and was latency-bound: +0.5 ms per 8B token at 100 keys).  Block max /
// sum, probabilities back to shared memory.  Phase 2: thread = (key split, head-dim element), coalesced V rows.
template <int D>
__global__ void __launch_bounds__(256) decode_attention_kernel(const __nv_bfloat16* __restrict__ q,
                                                               const __nv_bfloat16* __restrict__ kc,
                                                               const __nv_bfloat16* __restrict__ vc,
                                                               const int64_t* __restrict__ pos_p,
                                                               __nv_bfloat16* __restrict__ out, int Hq, int Hkv,
                                                               int64_t max_len, int64_t attend_len, float scale,
                                                               int pos_stride, int T) {
    constexpr int SPLITS = 256 / D;
    extern __shared__ float sc[];
    __shared__ float qs[D], red[8], part[SPLITS][D];
    const int h = blockIdx.x, r = blockIdx.y, b = r / T, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int hk = h / (Hq / Hkv);
    pdl_wait_then_trigger();
    int64_t last = pos_p[(size_t)b * pos_stride] + r % T;  // keys 0 .. pos of this query are visible
    if (last >= attend_len) last = attend_len - 1;
    const int n = (int)(last + 1);
    const __nv_bfloat16* kp = kc + ((size_t)b * Hkv + hk) * max_len * D;
    const __nv_bfloat16* vp = vc + ((size_t)b * Hkv + hk) * max_len * D;
    if (tid < D) qs[tid] = bf(q[((size_t)r * Hq + h) * D + tid]) * scale;
    __syncthreads();
    float lmax = -INFINITY;
    for (int j = tid; j < n; j += 256) {
        const uint4* kr = reinterpret_cast<const uint4*>(kp + (size_t)j * D);
        float s = 0.f;
#pragma unroll
        for (int v = 0; v < D / 8; v++) {
            const uint4 u = kr[v];
            const __nv_bfloat16* uv = reinterpret_cast<const __nv_bfloat16*>(&u);
#pragma unroll
            for (int e = 0; e < 8; e++) s = fmaf(qs[8 * v + e], bf(uv[e]), s);
        }
        sc[j] = s;
        lmax = fmaxf(lmax, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    if (lane == 0) red[warp] = lmax;
    __syncthreads();
    float m = red[0];
#pragma unroll
    for (int w = 1; w < 8; w++) m = fmaxf(m, red[w]);
    __syncthreads();
    float lsum = 0.f;
    for (int j = tid; j < n; j += 256) {
        const float p = __expf(sc[j] - m);
        sc[j] = p;
        lsum += p;
    }
    lsum = warp_sum(lsum);
    if (lane == 0) red[warp] = lsum;
    __syncthreads();
    float l = 0.f;
#pragma unroll
    for (int w = 0; w < 8; w++) l += red[w];
    const int split = tid / D, d = tid % D;
    float acc = 0.f;
#pragma unroll 4
    for (int j = split; j < n; j += SPLITS) acc = fmaf(sc[j], bf(vp[(size_t)j * D + d]), acc);
    part[split][d] = acc;
    __syncthreads();
    if (tid < D) {
        float o = 0.f;
#pragma unroll
        for (int sp = 0; sp < SPLITS; sp++) o += part[sp][tid];
        out[((size_t)r * Hq + h) * D + tid] = tobf(n > 0 && l > 0.f ? o / l : 0.f);
    }
}

// one block (256 threads) per row of H elements (H % 8 == 0): h = bf16(x + r) (r may be null: h = x), y = bf16(h * rstd * w)
__global__ void __launch_bounds__(256) add_rmsnorm_kernel(const __nv_bfloat16* __restrict__ x,
                                                          const __nv_bfloat16* __restrict__ r,
                                                          const __nv_bfloat16* __restrict__ w, float eps,
                                                          __nv_bfloat16* __restrict__ h_out,
                                                          __nv_bfloat16* __restrict__ y_out, int H) {
    const size_t row = blockIdx.x;
    const int nv = H / 8;
    pdl_wait_then_trigger();
    const uint4* xv = reinterpret_cast<const uint4*>(x + row * H);
    const uint4* rv = r ? reinterpret_cast<const uint4*>(r + row * H) : nullptr;
    float ss = 0.f;
    // pass 1: residual sum (kept in h_out) and sum of squares
    for (int i = threadIdx.x; i < nv; i += 256) {
        uint4 a = xv[i];
        __nv_bfloat16* av = reinterpret_cast<__nv_bfloat16*>(&a);
        if (rv) {
            uint4 c = rv[i];
            const __nv_bfloat16* cv = reinterpret_cast<const __nv_bfloat16*>(&c);
#pragma unroll
            for (int e = 0; e < 8; e++) av[e] = tobf(__fadd_rn(bf(av[e]), bf(cv[e])));
        }
#pragma unroll
        for (int e = 0; e < 8; e++) ss = fmaf(bf(av[e]), bf(av[e]), ss);
        if (h_out) reinterpret_cast<uint4*>(h_out + row * H)[i] = a;
        else if (rv) reinterpret_cast<uint4*>(y_out + row * H)[i] = a;  // no h wanted: park it in y for pass 2
    }
    __shared__ float red[8];
    ss = warp_sum(ss);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) tot += red[i];
    const float rstd = rsqrtf(tot / (float)H + eps);
    const uint4* hv = h_out ? reinterpret_cast<const uint4*>(h_out + row * H)
                            : (rv ? reinterpret_cast<const uint4*>(y_out + row * H) : xv);
    const uint4* wv = reinterpret_cast<const uint4*>(w);
    for (int i = threadIdx.x; i < nv; i += 256) {  // the same thread re-reads what it wrote in pass 1
        uint4 a = hv[i], g = wv[i];
        __nv_bfloat16* av = reinterpret_cast<__nv_bfloat16*>(&a);
        const __nv_bfloat16* gv = reinterpret_cast<const __nv_bfloat16*>(&g);
#pragma unroll
        for (int e = 0; e < 8; e++) av[e] = tobf(bf(av[e]) * rstd * bf(gv[e]));
        reinterpret_cast<uint4*>(y_out + row * H)[i] = a;
    }
}

// out = bf16(bf16(silu(g)) * u): the two roundings of the unfused F.silu(gate) * up
__global__ void __launch_bounds__(256) silu_mul_kernel(const __nv_bfloat16* __restrict__ g, const __nv_bfloat16* __restrict__ u,
                                                       __nv_bfloat16* __restrict__ out, int64_t nvec) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    pdl_wait_then_trigger();
    if (i >= nvec) return;
    uint4 a = reinterpret_cast<const uint4*>(g)[i], b = reinterpret_cast<const uint4*>(u)[i];
    __nv_bfloat16* av = reinterpret_cast<__nv_bfloat16*>(&a);
    const __nv_bfloat16* bv = reinterpret_cast<const __nv_bfloat16*>(&b);
#pragma unroll
    for (int e = 0; e < 8; e++) {
        const float x = bf(av[e]);
        const float s = bf(tobf(x / (1.f + expf(-x))));
        av[e] = tobf(s * bf(bv[e]));
    }
    reinterpret_cast<uint4*>(out)[i] = a;
}

}  // namespace

int launch_rope_cache(void* q, const void* k, const void* v, const int64_t* pos, int pos_stride, const float* inv_freq,
                      void* kc, void* vc, int B, int T, int Hq, int Hkv, int D, int64_t max_len, int64_t keep, cudaStream_t st) {
    if (!q || !k || !v || !pos || !inv_freq || !kc || !vc) return GBXQ_ENULL;
    if (B < 1 || Hq < 1 || Hkv < 1 || D < 2 || (D & 1) || D / 2 > 1024 || max_len < 1 || keep >= max_len) return GBXQ_ESHAPE;
    if (pos_stride != 0 && pos_stride != 1) return GBXQ_ESHAPE;
    if (T < 1 || T > kMaxBlockTokens || (int64_t)B * T > 65535) return GBXQ_ESHAPE;  // B * T: grid.y
    return launch(rope_cache_kernel, dim3(Hq + 2 * Hkv, B * T), dim3(D / 2), 0, st, true,
        reinterpret_cast<__nv_bfloat16*>(q), reinterpret_cast<const __nv_bfloat16*>(k), reinterpret_cast<const __nv_bfloat16*>(v),
        pos, inv_freq, reinterpret_cast<__nv_bfloat16*>(kc), reinterpret_cast<__nv_bfloat16*>(vc), Hq, Hkv, D, max_len, keep, pos_stride, T);
}

int launch_decode_attention(const void* q, const void* kc, const void* vc, const int64_t* pos, int pos_stride, void* out,
                            int B, int T, int Hq, int Hkv, int D, int64_t max_len, int64_t attend_len, float scale,
                            cudaStream_t st) {
    if (!q || !kc || !vc || !pos || !out) return GBXQ_ENULL;
    if (B < 1 || Hq < 1 || Hkv < 1 || Hq % Hkv || max_len < 1 || attend_len < 1 || attend_len > max_len) return GBXQ_ESHAPE;
    if (pos_stride != 0 && pos_stride != 1) return GBXQ_ESHAPE;
    if (T < 1 || T > kMaxBlockTokens || (int64_t)B * T > 65535) return GBXQ_ESHAPE;  // B * T: grid.y
    const dim3 grid(Hq, B * T);
    auto Q = reinterpret_cast<const __nv_bfloat16*>(q);
    auto K = reinterpret_cast<const __nv_bfloat16*>(kc);
    auto V = reinterpret_cast<const __nv_bfloat16*>(vc);
    auto O = reinterpret_cast<__nv_bfloat16*>(out);
    if (attend_len > 49152) return GBXQ_EUNSUPPORTED;  // one float of shared memory per visible key
    const size_t smem = (size_t)attend_len * sizeof(float);
    int rc = allow_dynamic_smem<decode_attention_kernel<64>>(49152 * 4);
    if (rc == GBXQ_OK) rc = allow_dynamic_smem<decode_attention_kernel<128>>(49152 * 4);
    if (rc != GBXQ_OK) return rc;
    switch (D) {
        case 64: return launch(decode_attention_kernel<64>, grid, dim3(256), smem, st, true, Q, K, V, pos, O, Hq, Hkv, max_len, attend_len, scale, pos_stride, T);
        case 128: return launch(decode_attention_kernel<128>, grid, dim3(256), smem, st, true, Q, K, V, pos, O, Hq, Hkv, max_len, attend_len, scale, pos_stride, T);
    }
    return GBXQ_EUNSUPPORTED;
}

int launch_add_rmsnorm(const void* x, const void* r, const void* w, float eps, void* h_out, void* y_out, int64_t rows, int H,
                       cudaStream_t st) {
    if (rows < 1 || H < 8 || H % 8) return GBXQ_ESHAPE;
    return launch(add_rmsnorm_kernel, dim3((unsigned)rows), dim3(256), 0, st, true,
        reinterpret_cast<const __nv_bfloat16*>(x), reinterpret_cast<const __nv_bfloat16*>(r),
        reinterpret_cast<const __nv_bfloat16*>(w), eps, reinterpret_cast<__nv_bfloat16*>(h_out),
        reinterpret_cast<__nv_bfloat16*>(y_out), H);
}

int launch_silu_mul(const void* g, const void* u, void* out, int64_t n, cudaStream_t st) {
    if (n < 8 || n % 8) return GBXQ_ESHAPE;
    const int64_t nvec = n / 8;
    return launch(silu_mul_kernel, dim3((unsigned)((nvec + 255) / 256)), dim3(256), 0, st, true,
                  reinterpret_cast<const __nv_bfloat16*>(g), reinterpret_cast<const __nv_bfloat16*>(u),
                  reinterpret_cast<__nv_bfloat16*>(out), nvec);
}

}  // namespace gbxq
