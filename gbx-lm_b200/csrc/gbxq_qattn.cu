// gbxq_qattn.cu -- the decode step of a group-quantized KV cache (the reference's kv_bits path: generate_step ->
// maybe_quantize_kv_cache, gbx_lm/utils.py:204-214, QuantizedKVCache.update_and_fetch, gbx_lm/models/cache.py:172-185,
// quantized_scaled_dot_product_attention, gbx_lm/models/base.py:65-98) as three launches per layer:
//
//   rope_cache_quantized   q rotated in place; k rotated and v copied, each quantized into its (codes, scales, biases)
//                          triple at row *pos -- the quantized counterpart of gbxq_rope_cache.  The rotated k is rounded
//                          to bf16 first and the groups go through the recipe of gbxq_quantize (gbxq_affine.cuh), so the
//                          triples are bit-identical to gbxq_rope_cache into a bf16 row followed by gbxq_quantize_rows.
//                          On a rotating cache the row is the ring slot of the position (kv_cache_row).
//   qattn_partial          flash-decoding over the codes: one CTA per (key chunk of 256, kv head, batch) serves all
//                          Hq/Hkv query heads of the group, so K and V are read from HBM once.  The chunk's K and V codes
//                          (contiguous: the cache is position-major) are brought in with cp.async; scores use the
//                          algebra of the matmul kernels, score = scale_g * sum(q * code) + bias_g * sum(q) per group,
//                          and P.V folds the V scale into the probability, out = sum(p * s * code) + sum(p * b).
//                          Each CTA leaves (max, sum, o) of its chunk per query head in the caller's workspace.
//   qattn_combine          per (query head, batch): the partials of the chunks that hold visible keys, combined in chunk
//                          order.
//
// Chunk borders are multiples of 256 keys whatever attend_len / max_len / the position, and the combine reads only the
// chunks below the position, so the result is bitwise the same for an eager call (attend_len = pos + 1) and a graph
// replay (attend_len = max_len).  No shared memory grows with the context: there is no context cap.
//
// A verify block (T > 1 consecutive tokens per batch row, at p_b .. p_b + T - 1; the `_multi` entry points): the write
// covers the B * T tokens, and one qattn_partial CTA serves the G * T query rows of its kv head, one token after the
// other over the chunk it has brought into shared memory once -- so the codes are read from HBM once per verify step,
// not T times.  Each query runs the single-query code on its own visible keys, so it is bitwise the single query.
// bf16 in and out, fp32 inside; every width (2/3/4/6/8), group sizes 32/64/128 <= D, D in {64, 128}, Hq/Hkv <= 8.
#include <math.h>

#include "gbxq_affine.cuh"
#include "gbxq_common.cuh"

namespace gbxq {

namespace {

constexpr int kChunk = 256;    // keys per CTA of qattn_partial (fixed: the combine order must not depend on attend_len)
constexpr int kThreads = 256;
constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ float bf(const __nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ __nv_bfloat16 tobf(float v) { return __float2bfloat16_rn(v); }

// exact float of a code (< 2^23) without the conversion pipe: 2^23 + c, minus 2^23
__device__ __forceinline__ float code_f(uint32_t c) { return __uint_as_float(0x4B000000u | c) - 8388608.f; }

__device__ __forceinline__ void cp_async16(void* s, const void* g) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(s)), "l"(__cvta_generic_to_global(g)) : "memory");
}
__device__ __forceinline__ void cp_async4(void* s, const void* g) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(s)), "l"(__cvta_generic_to_global(g)) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// `bytes` (a multiple of 4) from global to shared memory by the whole block, 16 bytes a copy where alignment allows
__device__ __forceinline__ void copy_async(void* dst, const void* src, uint32_t bytes) {
    if ((((uintptr_t)src) & 15) == 0 && (bytes & 15) == 0) {
        for (uint32_t i = threadIdx.x; i < bytes / 16; i += kThreads)
            cp_async16((char*)dst + 16 * i, (const char*)src + 16 * i);
    } else {
        for (uint32_t i = threadIdx.x; i < bytes / 4; i += kThreads) cp_async4((char*)dst + 4 * i, (const char*)src + 4 * i);
    }
}

// ------------------------------------------------------------------------------------------ RoPE + quantized cache write
// grid (Hq + 2 Hkv, B * T), one warp per row of D; lane owns the D/32 consecutive elements lane*EPL ...  Row r = b * T + t
// of q / k / v is token t of batch row b, at position p_b + t.  Head h < Hq: q rotated in place; Hq <= h < Hq+Hkv: k
// rotated, rounded to bf16 and quantized into row kv_cache_row(p_b + t) of cache row b; else v quantized.
template <int D, int BITS>
__global__ void __launch_bounds__(32) rope_cache_q_kernel(__nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                                                          const __nv_bfloat16* __restrict__ v, const int64_t* __restrict__ pos_p,
                                                          const float* __restrict__ inv_freq, uint32_t* __restrict__ kq,
                                                          __nv_bfloat16* __restrict__ ks, __nv_bfloat16* __restrict__ kb,
                                                          uint32_t* __restrict__ vq, __nv_bfloat16* __restrict__ vs,
                                                          __nv_bfloat16* __restrict__ vb, int Hq, int Hkv, int64_t max_len,
                                                          int64_t keep, int gs, int pos_stride, int T) {
    constexpr int EPL = D / 32, HALF = D / 2, W = D * BITS / 32;
    __shared__ uint32_t codes_s[D];
    __shared__ __align__(8) uint8_t bytes_s[D * BITS / 8 + 8];
    const int h = blockIdx.x, r = blockIdx.y, b = r / T, lane = threadIdx.x;
    pdl_wait_then_trigger();
    // the RoPE angle is the absolute position's; k / v go to its cache row.  pos_stride 0: one position for every row
    const int64_t pos = pos_p[(size_t)b * pos_stride] + r % T;
    const int64_t slot = kv_cache_row(pos, max_len, keep);
    if (slot < 0) return;  // never write outside the cache
    float val[EPL];
    int hh;  // kv head of a k / v row
    if (h < Hq + Hkv) {
        const bool isq = h < Hq;
        hh = h - Hq;
        __nv_bfloat16* src = isq ? q + ((size_t)r * Hq + h) * D : const_cast<__nv_bfloat16*>(k) + ((size_t)r * Hkv + hh) * D;
#pragma unroll
        for (int e = 0; e < EPL; e++) {
            // the expressions of gbxq_rope_cache, element by element
            const int d = lane * EPL + e, i = d < HALF ? d : d - HALF;
            const float ang = __fmul_rn((float)pos, inv_freq[i]);
            const float c = cosf(ang), s = sinf(ang);
            const float x1 = bf(src[i]), x2 = bf(src[i + HALF]);
            const float o = d < HALF ? __fsub_rn(__fmul_rn(x1, c), __fmul_rn(x2, s)) : __fadd_rn(__fmul_rn(x1, s), __fmul_rn(x2, c));
            val[e] = bf(tobf(o));
        }
        if (isq) {
            __syncwarp();  // every lane has read its partners' inputs before q is overwritten
#pragma unroll
            for (int e = 0; e < EPL; e++) src[lane * EPL + e] = tobf(val[e]);
            return;
        }
    } else {
        hh = h - Hq - Hkv;
#pragma unroll
        for (int e = 0; e < EPL; e++) val[e] = bf(v[((size_t)r * Hkv + hh) * D + lane * EPL + e]);
    }
    const bool isk = h < Hq + Hkv;
    uint32_t* cq = isk ? kq : vq;
    __nv_bfloat16* cs = isk ? ks : vs;
    __nv_bfloat16* cb = isk ? kb : vb;
    // groups are aligned runs of seg lanes
    const int seg = gs / EPL;
    float mx = val[0], mn = val[0];
#pragma unroll
    for (int e = 1; e < EPL; e++) {
        mx = fmaxf(mx, val[e]);
        mn = fminf(mn, val[e]);
    }
    for (int o = 1; o < seg; o <<= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    }
    const AffineGroup grp = affine_group<BITS>(mx, mn);
#pragma unroll
    for (int e = 0; e < EPL; e++) codes_s[lane * EPL + e] = affine_code<BITS>(val[e], grp);
    const size_t row = ((size_t)b * Hkv + hh) * (size_t)max_len + (size_t)slot;
    const int ng = D / gs;
    if (lane % seg == 0) {
        cs[row * ng + lane / seg] = tobf(grp.scale);
        cb[row * ng + lane / seg] = tobf(grp.bias);
    }
    __syncwarp();
    if (lane < D / 8) {  // octet `lane` of the row: BITS bytes of the LSB-first stream
        uint32_t c8[8];
#pragma unroll
        for (int i = 0; i < 8; i++) c8[i] = codes_s[lane * 8 + i];
        const uint64_t pack = pack_octet<BITS>(c8);
#pragma unroll
        for (int i = 0; i < BITS; i++) bytes_s[lane * BITS + i] = (uint8_t)(pack >> (8 * i));
    }
    __syncwarp();
    if (lane < W) cq[row * W + lane] = reinterpret_cast<const uint32_t*>(bytes_s)[lane];
}

// ------------------------------------------------------------------------------------------ split-K decode attention
// the BITS words of one 32-code run (always whole words: 32 * BITS bits)
template <int BITS>
__device__ __forceinline__ void load_run(const uint32_t* p, uint32_t (&w)[BITS]) {
    if constexpr (BITS % 4 == 0) {
#pragma unroll
        for (int i = 0; i < BITS / 4; i++) {
            const uint4 u = reinterpret_cast<const uint4*>(p)[i];
            w[4 * i] = u.x; w[4 * i + 1] = u.y; w[4 * i + 2] = u.z; w[4 * i + 3] = u.w;
        }
    } else if constexpr (BITS == 2 || BITS == 6) {
#pragma unroll
        for (int i = 0; i < BITS / 2; i++) {
            const uint2 u = reinterpret_cast<const uint2*>(p)[i];
            w[2 * i] = u.x; w[2 * i + 1] = u.y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < BITS; i++) w[i] = p[i];
    }
}

// code i (0..31) of a run
template <int BITS>
__device__ __forceinline__ uint32_t run_code(const uint32_t (&w)[BITS], int i) {
    const int bit = i * BITS, wi = bit >> 5, off = bit & 31;
    uint32_t c = w[wi] >> off;
    if (off + BITS > 32) c |= w[wi + 1] << (32 - off);
    return c & ((1u << BITS) - 1u);
}

// shared-memory plan of qattn_partial (bytes; every offset a multiple of 16).  MULTI: the cross-warp reduction gets its
// own space, because the codes stay in use for the block's next query.
template <int D, int BITS, int GMAX, bool MULTI>
struct QAttnPlan {
    static constexpr int W = D * BITS / 32;   // words per cache row
    static constexpr int RUNS = D / 32;        // 32-code runs per row
    static constexpr int NGMAX = D / 32;       // groups per row at most (gs >= 32)
    static constexpr int CODES = kChunk * W * 4;
    static constexpr int RED = 8 * GMAX * D * 4;  // per-warp partial outputs, after the codes are consumed
    static constexpr int UNION = MULTI || 2 * CODES > RED ? 2 * CODES : RED;
    static constexpr int KS = UNION, KB = KS + kChunk * NGMAX * 4, VS = KB + kChunk * NGMAX * 4, VB = VS + kChunk * NGMAX * 4;
    static constexpr int QF = VB + kChunk * NGMAX * 4;   // q * scale * log2(e), [d % 32][d / 32][head]
    static constexpr int QRS = QF + D * GMAX * 4;        // per (run, head) sums of QF
    static constexpr int SC = QRS + RUNS * GMAX * 4;     // scores, then probabilities, [key][head]
    static constexpr int ML = SC + kChunk * GMAX * 4;    // (max, sum) per head
    static constexpr int RD = MULTI ? ML + GMAX * 2 * 4 : 0;  // the reduction: after ML, or over the consumed codes
    static constexpr int BYTES = MULTI ? RD + RED : ML + GMAX * 2 * 4;
};

// grid (nch, Hkv, B), kThreads threads.  Writes ws[((r * Hq + hq) * nch + chunk) * (D + 2) + {0: max (log2 domain),
// 1: sum, 2..: o[D]}] for the G = Hq / Hkv query heads of kv head blockIdx.y and the query rows r = b * T + t of batch
// row b (T = 1 unless MULTI).
template <int D, int BITS, int GMAX, bool MULTI>
__global__ void __launch_bounds__(kThreads, 2) qattn_partial_kernel(
    const __nv_bfloat16* __restrict__ q, const uint32_t* __restrict__ kq, const __nv_bfloat16* __restrict__ ks,
    const __nv_bfloat16* __restrict__ kb, const uint32_t* __restrict__ vq, const __nv_bfloat16* __restrict__ vs,
    const __nv_bfloat16* __restrict__ vb, const int64_t* __restrict__ pos_p, float* __restrict__ ws, int Hq, int Hkv,
    int64_t max_len, int64_t attend_len, int nch, int gs, float qscale, int pos_stride, int T) {
    using P = QAttnPlan<D, BITS, GMAX, MULTI>;
    constexpr int W = P::W, RUNS = P::RUNS;
    extern __shared__ __align__(16) uint8_t smem[];
    uint32_t* kc = reinterpret_cast<uint32_t*>(smem);
    uint32_t* vc = reinterpret_cast<uint32_t*>(smem + P::CODES);
    float* red = reinterpret_cast<float*>(smem + P::RD);
    float* ksf = reinterpret_cast<float*>(smem + P::KS);
    float* kbf = reinterpret_cast<float*>(smem + P::KB);
    float* vsf = reinterpret_cast<float*>(smem + P::VS);
    float* vbf = reinterpret_cast<float*>(smem + P::VB);
    float* qf = reinterpret_cast<float*>(smem + P::QF);
    float* qrs = reinterpret_cast<float*>(smem + P::QRS);
    float* sc = reinterpret_cast<float*>(smem + P::SC);
    float* ml = reinterpret_cast<float*>(smem + P::ML);

    const int chunk = blockIdx.x, hk = blockIdx.y, b = blockIdx.z;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int G = Hq / Hkv, ng = D / gs, nt = MULTI ? T : 1;
    pdl_wait_then_trigger();
    const int64_t p0 = pos_p[(size_t)b * pos_stride];  // query tq of this row sees keys 0 .. p0 + tq
    const int64_t j0 = (int64_t)chunk * kChunk;
    const size_t head_stride = (size_t)nch * (D + 2);
    int64_t last_all = p0 + nt - 1;  // the block's last query sees the most keys
    if (last_all >= attend_len) last_all = attend_len - 1;
    const int64_t n_all = last_all + 1;
    if (j0 >= n_all) {  // no visible key in this chunk: empty partials (the combine does not read them)
        for (int i = t; i < nt * G; i += kThreads) {
            float* w = ws + ((((size_t)b * nt + i / G) * Hq + (size_t)hk * G + i % G) * nch + chunk) * (D + 2);
            w[0] = -INFINITY;
            w[1] = 0.f;
        }
        return;
    }
    const int nload = (int)min((int64_t)kChunk, n_all - j0);
    const size_t plane = ((size_t)b * Hkv + hk) * (size_t)max_len + (size_t)j0;  // first row of the chunk
    copy_async(kc, kq + plane * W, (uint32_t)nload * W * 4);
    cp_async_commit();
    copy_async(vc, vq + plane * W, (uint32_t)nload * W * 4);
    cp_async_commit();
    for (int i = t; i < nload * ng; i += kThreads) {
        ksf[i] = bf(ks[plane * ng + i]);
        kbf[i] = bf(kb[plane * ng + i]);
        vsf[i] = bf(vs[plane * ng + i]);
        vbf[i] = bf(vb[plane * ng + i]);
    }
#pragma unroll 1
    for (int tq = 0; tq < nt; tq++) {  // the block's queries over the chunk in shared memory (one pass unless MULTI)
        const size_t row = (size_t)b * nt + tq;
        int64_t last = p0 + tq;  // keys 0 .. pos of this query are visible
        if (last >= attend_len) last = attend_len - 1;
        const int64_t n = last + 1;
        float* wsb = ws + ((row * Hq + (size_t)hk * G) * nch + chunk) * (D + 2);
        if (j0 >= n) {  // an empty partial for this query (uniform over the block)
            if (t < G) {
                wsb[t * head_stride] = -INFINITY;
                wsb[t * head_stride + 1] = 0.f;
            }
            continue;
        }
        const int nvalid = (int)min((int64_t)kChunk, n - j0);
        for (int i = t; i < D * GMAX; i += kThreads) {  // i = (d % 32, d / 32, head)
            const int h = i % GMAX, r = (i / GMAX) % RUNS, d = (i / GMAX / RUNS) + 32 * r;
            qf[i] = h < G ? bf(q[(row * Hq + (size_t)hk * G + h) * D + d]) * qscale : 0.f;
        }
        __syncthreads();
        if (t < RUNS * GMAX) {
            const int r = t / GMAX, h = t % GMAX;
            float s = 0.f;
            for (int i = 0; i < 32; i++) s += qf[(i * RUNS + r) * GMAX + h];
            qrs[t] = s;
        }
        cp_async_wait<1>();  // K codes of this thread landed
        __syncthreads();

        // ---- scores: thread = (key, 32-code run); the runs of a key are adjacent lanes
        {
            constexpr int KPP = kThreads / RUNS;
            const int run = t % RUNS, g_run = run * 32 / gs;
#pragma unroll 1
            for (int p = 0; p < kChunk / KPP; p++) {
                const int j = p * KPP + t / RUNS;
                const bool live = j < nvalid;
                float acc[GMAX];
#pragma unroll
                for (int h = 0; h < GMAX; h++) acc[h] = 0.f;
                if (live) {
                    uint32_t w[BITS];
                    load_run<BITS>(kc + j * W + run * BITS, w);
#pragma unroll
                    for (int i = 0; i < 32; i++) {
                        const float cf = code_f(run_code<BITS>(w, i));
                        const float4* qq = reinterpret_cast<const float4*>(qf + (i * RUNS + run) * GMAX);
#pragma unroll
                        for (int h4 = 0; h4 < GMAX / 4; h4++) {
                            const float4 x = qq[h4];
                            acc[4 * h4] = fmaf(x.x, cf, acc[4 * h4]);
                            acc[4 * h4 + 1] = fmaf(x.y, cf, acc[4 * h4 + 1]);
                            acc[4 * h4 + 2] = fmaf(x.z, cf, acc[4 * h4 + 2]);
                            acc[4 * h4 + 3] = fmaf(x.w, cf, acc[4 * h4 + 3]);
                        }
                    }
                    const float s = ksf[j * ng + g_run], bb = kbf[j * ng + g_run];
#pragma unroll
                    for (int h = 0; h < GMAX; h++) acc[h] = fmaf(s, acc[h], bb * qrs[run * GMAX + h]);
                }
#pragma unroll
                for (int o = 1; o < RUNS; o <<= 1)
#pragma unroll
                    for (int h = 0; h < GMAX; h++) acc[h] += __shfl_xor_sync(0xffffffffu, acc[h], o);
                if (run == 0) {
#pragma unroll
                    for (int h = 0; h < GMAX; h++) sc[j * GMAX + h] = live ? acc[h] : -INFINITY;
                }
            }
        }
        __syncthreads();
        // ---- chunk softmax: warp h owns query head h
        if (warp < G) {
            const int h = warp;
            float m = -INFINITY;
            for (int j = lane; j < kChunk; j += 32) m = fmaxf(m, sc[j * GMAX + h]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            float l = 0.f;
            for (int j = lane; j < kChunk; j += 32) {
                const float p = exp2f(sc[j * GMAX + h] - m);
                sc[j * GMAX + h] = p;
                l += p;
            }
            l = warp_sum(l);
            if (lane == 0) {
                ml[2 * h] = m;
                ml[2 * h + 1] = l;
            }
        }
        cp_async_wait<0>();
        __syncthreads();

        // ---- P.V: thread = (8-code octet of the row, key split); lanes of one key are adjacent
        constexpr int OCT = D / 8, SPL = kThreads / OCT;
        const int oct = t % OCT, split = t / OCT, g_oct = oct * 8 / gs;
        float acc[GMAX][8], pb[GMAX];
#pragma unroll
        for (int h = 0; h < GMAX; h++) {
            pb[h] = 0.f;
#pragma unroll
            for (int i = 0; i < 8; i++) acc[h][i] = 0.f;
        }
#pragma unroll 1
        for (int j = split; j < nvalid; j += SPL) {
            uint32_t c[8];
            extract_octet<BITS>(vc + j * W, oct, W, c);
            float cf[8];
#pragma unroll
            for (int i = 0; i < 8; i++) cf[i] = code_f(c[i]);
            const float sv = vsf[j * ng + g_oct], bv = vbf[j * ng + g_oct];
            const float4* pp = reinterpret_cast<const float4*>(sc + j * GMAX);
#pragma unroll
            for (int h4 = 0; h4 < GMAX / 4; h4++) {
                const float4 p4 = pp[h4];
                const float pr[4] = {p4.x, p4.y, p4.z, p4.w};
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const int h = 4 * h4 + e;
                    const float ps = pr[e] * sv;
                    pb[h] = fmaf(pr[e], bv, pb[h]);
#pragma unroll
                    for (int i = 0; i < 8; i++) acc[h][i] = fmaf(ps, cf[i], acc[h][i]);
                }
            }
        }
#pragma unroll
        for (int h = 0; h < GMAX; h++)
#pragma unroll
            for (int i = 0; i < 8; i++) {
                float a = acc[h][i] + pb[h];
#pragma unroll
                for (int o = OCT; o < 32; o <<= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
                acc[h][i] = a;
            }
        __syncthreads();  // the P.V reads are done (and unless MULTI the codes are consumed: `red` reuses their space)
        if (lane < OCT) {
#pragma unroll
            for (int h = 0; h < GMAX; h++) {
                float4* dst = reinterpret_cast<float4*>(red + (warp * GMAX + h) * D + oct * 8);
                dst[0] = make_float4(acc[h][0], acc[h][1], acc[h][2], acc[h][3]);
                dst[1] = make_float4(acc[h][4], acc[h][5], acc[h][6], acc[h][7]);
            }
        }
        __syncthreads();
        for (int i = t; i < G * D; i += kThreads) {
            const int h = i / D, d = i % D;
            float o = 0.f;
#pragma unroll
            for (int w = 0; w < 8; w++) o += red[(w * GMAX + h) * D + d];
            wsb[h * head_stride + 2 + d] = o;
        }
        if (t < G) {
            wsb[t * head_stride] = ml[2 * t];
            wsb[t * head_stride + 1] = ml[2 * t + 1];
        }
    }  // tq: the next query rewrites qf / qrs / sc / ml / red only after the barriers that follow their last reads
}

// grid (Hq, B * T), D threads: the chunks with visible keys of query row r = b * T + t, in chunk order
template <int D>
__global__ void __launch_bounds__(D) qattn_combine_kernel(const float* __restrict__ ws, const int64_t* __restrict__ pos_p,
                                                          __nv_bfloat16* __restrict__ out, int Hq, int64_t attend_len, int nch,
                                                          int pos_stride, int T) {
    const int h = blockIdx.x, r = blockIdx.y, b = r / T, d = threadIdx.x;
    pdl_wait_then_trigger();
    int64_t last = pos_p[(size_t)b * pos_stride] + r % T;
    if (last >= attend_len) last = attend_len - 1;
    const int nv = last < 0 ? 0 : (int)((last + kChunk) / kChunk);
    const float* base = ws + ((size_t)r * Hq + h) * (size_t)nch * (D + 2);
    float m = -INFINITY;
    for (int c = 0; c < nv; c++) m = fmaxf(m, base[(size_t)c * (D + 2)]);
    float o = 0.f, l = 0.f;
    for (int c = 0; c < nv; c++) {
        const float* pc = base + (size_t)c * (D + 2);
        const float e = exp2f(pc[0] - m);
        l = fmaf(e, pc[1], l);
        o = fmaf(e, pc[2 + d], o);
    }
    out[((size_t)r * Hq + h) * D + d] = tobf(nv > 0 && l > 0.f ? o / l : 0.f);
}

int check_common(int B, int T, int Hq, int Hkv, int D, int64_t max_len, int bits, int gs) {
    if (bits != 2 && bits != 3 && bits != 4 && bits != 6 && bits != 8) return GBXQ_EINVAL_BITS;
    if (gs != 32 && gs != 64 && gs != 128) return GBXQ_EINVAL_GROUP;
    if (B < 1 || Hq < 1 || Hkv < 1 || Hq % Hkv || max_len < 1 || B > 65535 || Hkv > 65535) return GBXQ_ESHAPE;
    if (T < 1 || T > kMaxBlockTokens || B * T > 65535) return GBXQ_ESHAPE;
    if ((D != 64 && D != 128) || gs > D || Hq / Hkv > 8) return GBXQ_EUNSUPPORTED;
    return GBXQ_OK;
}

int64_t chunks_of(int64_t attend_len) { return (attend_len + kChunk - 1) / kChunk; }

template <int D, int BITS>
int launch_rope_q(const QCacheWrite& a, cudaStream_t st) {
    return launch(rope_cache_q_kernel<D, BITS>, dim3(a.Hq + 2 * a.Hkv, a.B * a.T), dim3(32), 0, st, true,
        reinterpret_cast<__nv_bfloat16*>(a.q), reinterpret_cast<const __nv_bfloat16*>(a.k),
        reinterpret_cast<const __nv_bfloat16*>(a.v), a.pos, a.inv_freq, a.kq, reinterpret_cast<__nv_bfloat16*>(a.ks),
        reinterpret_cast<__nv_bfloat16*>(a.kb), a.vq, reinterpret_cast<__nv_bfloat16*>(a.vs),
        reinterpret_cast<__nv_bfloat16*>(a.vb), a.Hq, a.Hkv, a.max_len, a.keep, a.gs, a.pos_stride, a.T);
}

template <int D>
int rope_q_bits(const QCacheWrite& a, cudaStream_t st) {
    switch (a.bits) {
        case 2: return launch_rope_q<D, 2>(a, st);
        case 3: return launch_rope_q<D, 3>(a, st);
        case 4: return launch_rope_q<D, 4>(a, st);
        case 6: return launch_rope_q<D, 6>(a, st);
        default: return launch_rope_q<D, 8>(a, st);
    }
}

template <int D, int BITS, int GMAX, bool MULTI>
int launch_qattn_t(const QAttn& a, cudaStream_t st) {
    using P = QAttnPlan<D, BITS, GMAX, MULTI>;
    constexpr auto kern = qattn_partial_kernel<D, BITS, GMAX, MULTI>;
    int rc = allow_dynamic_smem<kern>(P::BYTES);
    if (rc != GBXQ_OK) return rc;
    const int nch = (int)chunks_of(a.attend_len);
    float* ws = reinterpret_cast<float*>(a.ws);
    const float qscale = a.scale * kLog2e;
    rc = launch(kern, dim3(nch, a.Hkv, a.B), dim3(kThreads), (size_t)P::BYTES, st, true,
        reinterpret_cast<const __nv_bfloat16*>(a.q), a.kq, reinterpret_cast<const __nv_bfloat16*>(a.ks),
        reinterpret_cast<const __nv_bfloat16*>(a.kb), a.vq, reinterpret_cast<const __nv_bfloat16*>(a.vs),
        reinterpret_cast<const __nv_bfloat16*>(a.vb), a.pos, ws, a.Hq, a.Hkv, a.max_len, a.attend_len, nch, a.gs, qscale, a.pos_stride,
        a.T);
    if (rc != GBXQ_OK) return rc;
    return launch(qattn_combine_kernel<D>, dim3(a.Hq, a.B * a.T), dim3(D), 0, st, true, (const float*)ws, a.pos,
                  reinterpret_cast<__nv_bfloat16*>(a.out), a.Hq, a.attend_len, nch, a.pos_stride, a.T);
}

template <int D, int BITS, bool MULTI>
int qattn_gm(const QAttn& a, cudaStream_t st) {
    return a.Hq / a.Hkv <= 4 ? launch_qattn_t<D, BITS, 4, MULTI>(a, st) : launch_qattn_t<D, BITS, 8, MULTI>(a, st);
}

template <int D, int BITS>
int qattn_g(const QAttn& a, cudaStream_t st) {
    return a.T > 1 ? qattn_gm<D, BITS, true>(a, st) : qattn_gm<D, BITS, false>(a, st);
}

template <int D>
int qattn_bits(const QAttn& a, cudaStream_t st) {
    switch (a.bits) {
        case 2: return qattn_g<D, 2>(a, st);
        case 3: return qattn_g<D, 3>(a, st);
        case 4: return qattn_g<D, 4>(a, st);
        case 6: return qattn_g<D, 6>(a, st);
        default: return qattn_g<D, 8>(a, st);
    }
}

}  // namespace

int launch_rope_cache_quantized(const QCacheWrite& a, cudaStream_t st) {
    const int rc = check_common(a.B, a.T, a.Hq, a.Hkv, a.D, a.max_len, a.bits, a.gs);
    if (rc != GBXQ_OK) return rc;
    if (a.keep >= a.max_len) return GBXQ_ESHAPE;
    if (a.pos_stride != 0 && a.pos_stride != 1) return GBXQ_ESHAPE;
    if (!a.q || !a.k || !a.v || !a.pos || !a.inv_freq || !a.kq || !a.ks || !a.kb || !a.vq || !a.vs || !a.vb) return GBXQ_ENULL;
    if (((uintptr_t)a.kq | (uintptr_t)a.vq) & 3) return GBXQ_EALIGN;
    return a.D == 64 ? rope_q_bits<64>(a, st) : rope_q_bits<128>(a, st);
}

size_t qattn_workspace_bytes(int B, int Hq, int Hkv, int D, int64_t attend_len) {
    if (B < 1 || Hq < 1 || Hkv < 1 || Hq % Hkv || (D != 64 && D != 128) || attend_len < 1) return 0;
    return (size_t)B * Hq * (size_t)chunks_of(attend_len) * (D + 2) * sizeof(float);
}

int launch_decode_attention_quantized(const QAttn& a, cudaStream_t st) {
    const int rc = check_common(a.B, a.T, a.Hq, a.Hkv, a.D, a.max_len, a.bits, a.gs);
    if (rc != GBXQ_OK) return rc;
    if (a.attend_len < 1 || a.attend_len > a.max_len || chunks_of(a.attend_len) > 65535 * 64) return GBXQ_ESHAPE;
    if (a.pos_stride != 0 && a.pos_stride != 1) return GBXQ_ESHAPE;
    if (!a.q || !a.kq || !a.ks || !a.kb || !a.vq || !a.vs || !a.vb || !a.pos || !a.out || !a.ws) return GBXQ_ENULL;
    if (a.ws_bytes < qattn_workspace_bytes(a.B * a.T, a.Hq, a.Hkv, a.D, a.attend_len)) return GBXQ_EWORKSPACE;
    if (((uintptr_t)a.kq | (uintptr_t)a.vq) & 3 || ((uintptr_t)a.ws & 15)) return GBXQ_EALIGN;
    return a.D == 64 ? qattn_bits<64>(a, st) : qattn_bits<128>(a, st);
}

}  // namespace gbxq
