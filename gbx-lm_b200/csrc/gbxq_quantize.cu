// gbxq_quantize.cu -- mx.quantize on the device: group-affine quantisation of fresh activations into the packed layout
// the matmul kernels read.  Reference callers: the quantized KV cache quantises the new keys / values of every step
// (gbx_lm/models/cache.py:176-177, QuantizedKVCache.update_and_fetch) before
// quantized_scaled_dot_product_attention reads them (gbx_lm/models/base.py:65-98), and KVCache.to_quantized
// (cache.py:251-263) converts a whole dense cache at once.
//
// Arithmetic (oracle/MLX_SPEC.md R6, fp32 throughout, every operation separately rounded -- no FMA can form because
// no multiply feeds an add), in gbxq_affine.cuh so that the fused cache write of gbxq_qattn.cu computes the same bits:
//     w_max, w_min over the group;  mask = |w_min| > |w_max|
//     scale = max((w_max - w_min) / (2^bits - 1), 1e-7);  scale = mask ? scale : -scale;  edge = mask ? w_min : w_max
//     q0 = rint(edge / scale);  if (q0 != 0) { scale = edge / q0;  bias = edge; } else bias = 0
//     code = clamp(rint((w - bias) / scale), 0, 2^bits - 1)         <- from the UNROUNDED fp32 scale / bias
//     scales[g] = T(scale), biases[g] = T(bias)
// Codes, scales and biases are bit-exact against the restatement (tests/test_gpu_quantize.py).  The per-element
// quotient is the IEEE one computed from ONE reciprocal per lane (two FMAs of correction), rint + conversion are a
// magic-number add: the first version (a full division, FRND and F2I per element, no load ahead) ran at 0.19-0.22 of
// the HBM roofline on large inputs, bound by the quarter-rate pipe and by one load in flight per warp
// (profiles/r04a_quantbench.txt); with those two fixed 0.30-0.36, issue-bound on the per-lane work (min / max
// reduction, the three divisions of the statistics, index arithmetic: ~250 instructions per 8 elements,
// profiles/r04b_quantbench.txt), hence 16 elements per lane for the 16-bit types and the group size as a template
// parameter.
//
// HBM-bound byte work: reads sizeof(T) bytes and writes bits/8 bytes per element (+ 2 * sizeof(T) per group).  The
// problem is flat: groups never cross rows (K % group_size == 0) and rows of codes are whole words (K % 32 == 0), so
// a warp takes 512 consecutive elements of a 16-bit type (32 bytes = 16 elements per lane; 256 of fp32), reduces
// min / max inside the lanes of a group with xor shuffles, stages its codes in shared memory and writes them back as
// coalesced words.  Destination rows can be remapped (gbxq_quantize_rows): the cache update writes the rows
// of every (batch, head) at the current offset of a [.., capacity, ..] buffer without a second copy.
#include "gbxq_affine.cuh"
#include "gbxq_common.cuh"

namespace gbxq {
namespace {

// destination row of source row r: (r / inner) * outer_stride + offset + r % inner;  inner <= 0: identity
struct RowMap {
    int64_t inner, outer_stride, offset;
};

__device__ __forceinline__ int64_t map_row(const RowMap& m, int64_t r) {
    const int64_t o = r / m.inner;
    return o * m.outer_stride + m.offset + (r - o * m.inner);
}

// A lane owns 32 contiguous bytes of the input: 16 elements of a 2-byte type, 8 of fp32.  They are kept as raw
// registers and loaded one chunk AHEAD of their use (the conversion to fp32 happens at use, so that the in-order issue
// does not stall on the load it is meant to overlap).
template <typename T> struct Epl { static constexpr int v = 32 / (int)sizeof(T); };
struct Raw { uint4 a, b; };

__device__ __forceinline__ void load_raw(const void* p, Raw& r) {
    r.a = __ldg(reinterpret_cast<const uint4*>(p));
    r.b = __ldg(reinterpret_cast<const uint4*>(p) + 1);
}
__device__ __forceinline__ void zero_raw(Raw& r) {
    r.a = make_uint4(0, 0, 0, 0);
    r.b = make_uint4(0, 0, 0, 0);
}
__device__ __forceinline__ void to_f32(const Raw& r, float (&v)[16], const __nv_bfloat16*) {
    const uint32_t w[8] = {r.a.x, r.a.y, r.a.z, r.a.w, r.b.x, r.b.y, r.b.z, r.b.w};
#pragma unroll
    for (int i = 0; i < 8; i++) {
        v[2 * i] = __uint_as_float(w[i] << 16);
        v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}
__device__ __forceinline__ void to_f32(const Raw& r, float (&v)[16], const __half*) {
    const uint32_t w[8] = {r.a.x, r.a.y, r.a.z, r.a.w, r.b.x, r.b.y, r.b.z, r.b.w};
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
        v[2 * i] = __low2float(h);
        v[2 * i + 1] = __high2float(h);
    }
}
__device__ __forceinline__ void to_f32(const Raw& r, float (&v)[8], const float*) {
    v[0] = __uint_as_float(r.a.x); v[1] = __uint_as_float(r.a.y); v[2] = __uint_as_float(r.a.z); v[3] = __uint_as_float(r.a.w);
    v[4] = __uint_as_float(r.b.x); v[5] = __uint_as_float(r.b.y); v[6] = __uint_as_float(r.b.z); v[7] = __uint_as_float(r.b.w);
}

// destination index of flat index `i` (a word of codes or a group) whose rows hold `per_row` of them
__device__ __forceinline__ int64_t map_index(const RowMap& m, int64_t i, int64_t per_row, bool small) {
    if (small) {  // everything fits 32 bits: a 32-bit division is a fraction of the 64-bit one
        const uint32_t r = (uint32_t)i / (uint32_t)per_row;
        const uint32_t o = r / (uint32_t)m.inner;
        return ((int64_t)o * m.outer_stride + m.offset + (r - o * (uint32_t)m.inner)) * per_row +
               ((uint32_t)i - r * (uint32_t)per_row);
    }
    const int64_t r = i / per_row;
    return map_row(m, r) * per_row + (i - r * per_row);
}

constexpr int kWarps = 8;

template <int BITS, int GS, typename T>
__global__ void __launch_bounds__(kWarps * 32) quantize_kernel(const T* __restrict__ w, uint32_t* __restrict__ q,
                                                              T* __restrict__ scales, T* __restrict__ biases,
                                                              int64_t total, int64_t K, RowMap map) {
    constexpr int EPL = Epl<T>::v;        // elements per lane and chunk
    constexpr int CH = 32 * EPL;          // elements per warp and chunk: 512 / 256
    constexpr int SEG = GS / EPL;         // lanes per group: 2..8 / 4..16
    constexpr int BPL = EPL * BITS / 8;   // bytes of codes per lane
    constexpr int WPC = EPL * BITS;       // words of codes per chunk
    __shared__ __align__(16) uint8_t stage_all[kWarps][32 * BPL];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t* stage = stage_all[warp];
    const int64_t nchunks = (total + CH - 1) / CH;
    const int64_t wpr = K * BITS / 32;  // words per row of codes
    const int64_t gpr = K / GS;         // groups per row
    const int64_t total_words = total / 32 * BITS;
    const bool dense = map.inner <= 0;
    const bool small = total_words < (int64_t(1) << 31) && total < (int64_t(1) << 31);
    const int64_t stride = (int64_t)gridDim.x * kWarps;

    int64_t c = (int64_t)blockIdx.x * kWarps + warp;
    Raw cur, nxt;
    zero_raw(cur);
    if (c < nchunks && c * CH + lane * EPL < total) load_raw(w + c * CH + lane * EPL, cur);
    for (; c < nchunks; c += stride) {
        const int64_t e0 = c * CH + lane * EPL;
        const bool live = e0 < total;  // total % 32 == 0: a lane's elements are all inside or all outside
        {
            const int64_t en = e0 + stride * CH;  // the chunk of the next iteration, requested before this one is used
            zero_raw(nxt);
            if (en < total) load_raw(w + en, nxt);
        }
        float v[EPL];
        to_f32(cur, v, (const T*)nullptr);  // dead lanes hold zeros
        float mx = v[0], mn = v[0];
#pragma unroll
        for (int i = 1; i < EPL; i++) {
            mx = fmaxf(mx, v[i]);
            mn = fminf(mn, v[i]);
        }
        // groups are aligned runs of SEG lanes; dead lanes only ever share a group with dead lanes (total % GS == 0)
#pragma unroll
        for (int o = 1; o < SEG; o <<= 1) {
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        }
        // statistics and codes: the shared recipe (gbxq_affine.cuh)
        const AffineGroup grp = affine_group<BITS>(mx, mn);
        const float scale = grp.scale, bias = grp.bias;
#pragma unroll
        for (int h = 0; h < EPL / 8; h++) {
            uint32_t codes[8];
#pragma unroll
            for (int i = 0; i < 8; i++) codes[i] = affine_code<BITS>(v[h * 8 + i], grp);
            const uint64_t pack = pack_octet<BITS>(codes);
            // 8 codes are BITS bytes of the chunk's LSB-first stream; the lane's codes start at byte lane * BPL
            uint8_t* dst = stage + lane * BPL + h * BITS;
            if constexpr (BITS == 8) {
                *reinterpret_cast<uint64_t*>(dst) = pack;
            } else if constexpr (BITS == 4) {
                *reinterpret_cast<uint32_t*>(dst) = (uint32_t)pack;
            } else if constexpr (BITS == 2) {
                *reinterpret_cast<uint16_t*>(dst) = (uint16_t)pack;
            } else {
#pragma unroll
                for (int b = 0; b < BITS; b++) dst[b] = (uint8_t)(pack >> (8 * b));
            }
        }
        if (live && (lane & (SEG - 1)) == 0) {
            int64_t g = (int64_t)((uint64_t)e0 / GS);
            if (!dense) g = map_index(map, g, gpr, small);
            scales[g] = from_f32<T>(scale);
            biases[g] = from_f32<T>(bias);
        }
        __syncwarp();
        const int64_t w0 = c * WPC;
#pragma unroll
        for (int j0 = 0; j0 < WPC; j0 += 32) {
            const int j = j0 + lane;
            int64_t wi = w0 + j;
            if (j < WPC && wi < total_words) {
                const uint32_t word = reinterpret_cast<const uint32_t*>(stage)[j];
                if (!dense) wi = map_index(map, wi, wpr, small);
                q[wi] = word;
            }
        }
        __syncwarp();
        cur = nxt;
    }
}

// resident CTAs per SM of this instantiation (registers decide), asked once per process
template <int BITS, int GS, typename T> int ctas_per_sm() {
    static std::atomic<int> cached{0};
    int n = cached.load(std::memory_order_relaxed);
    if (n == 0) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, quantize_kernel<BITS, GS, T>, kWarps * 32, 0) != cudaSuccess || n < 1)
            n = 4;
        cached.store(n, std::memory_order_relaxed);
    }
    return n;
}

template <int BITS, int GS, typename T>
int launch_t(const void* w, uint32_t* q, void* s, void* b, int64_t total, int64_t K, const RowMap& map, cudaStream_t st) {
    constexpr int CH = 32 * Epl<T>::v;
    const int64_t nchunks = (total + CH - 1) / CH;
    int64_t blocks = (nchunks + kWarps - 1) / kWarps;
    const int64_t cap = (int64_t)device_sm_count() * ctas_per_sm<BITS, GS, T>();  // one resident wave, grid-stride beyond
    if (blocks > cap) blocks = cap;
    return launch(quantize_kernel<BITS, GS, T>, dim3((unsigned)blocks), dim3(kWarps * 32), 0, st, false, (const T*)w, q, (T*)s,
                  (T*)b, total, K, map);
}

template <int BITS, int GS>
int launch_g(const void* w, uint32_t* q, void* s, void* b, int64_t total, int64_t K, int dtype, const RowMap& map,
             cudaStream_t st) {
    switch (dtype) {
        case GBXQ_BF16: return launch_t<BITS, GS, __nv_bfloat16>(w, q, s, b, total, K, map, st);
        case GBXQ_F16: return launch_t<BITS, GS, __half>(w, q, s, b, total, K, map, st);
        default: return launch_t<BITS, GS, float>(w, q, s, b, total, K, map, st);
    }
}

template <int BITS>
int launch_b(const void* w, uint32_t* q, void* s, void* b, int64_t total, int64_t K, int gs, int dtype,
             const RowMap& map, cudaStream_t st) {
    switch (gs) {
        case 32: return launch_g<BITS, 32>(w, q, s, b, total, K, dtype, map, st);
        case 64: return launch_g<BITS, 64>(w, q, s, b, total, K, dtype, map, st);
        default: return launch_g<BITS, 128>(w, q, s, b, total, K, dtype, map, st);
    }
}

int quantize_checked(const void* w, uint32_t* q, void* s, void* b, int64_t rows, int64_t K, int bits, int gs,
                     int dtype, const RowMap& map, cudaStream_t st) {
    if (bits != 2 && bits != 3 && bits != 4 && bits != 6 && bits != 8) return GBXQ_EINVAL_BITS;
    if (gs != 32 && gs != 64 && gs != 128) return GBXQ_EINVAL_GROUP;
    if (dtype != GBXQ_BF16 && dtype != GBXQ_F16 && dtype != GBXQ_F32) return GBXQ_EDTYPE;
    if (rows < 0 || K <= 0 || K % gs != 0) return GBXQ_ESHAPE;
    if (map.inner > 0 && (rows % map.inner != 0 || map.offset < 0 || map.outer_stride < map.offset + map.inner))
        return GBXQ_ESHAPE;
    if (rows == 0) return GBXQ_OK;
    if (!w || !q || !s || !b) return GBXQ_ENULL;
    const uintptr_t elem = dtype == GBXQ_F32 ? 4 : 2;
    if (((uintptr_t)w & 15) || ((uintptr_t)q & 3) || ((uintptr_t)s & (elem - 1)) || ((uintptr_t)b & (elem - 1)))
        return GBXQ_EALIGN;
    const int64_t total = rows * K;
    switch (bits) {
        case 2: return launch_b<2>(w, q, s, b, total, K, gs, dtype, map, st);
        case 3: return launch_b<3>(w, q, s, b, total, K, gs, dtype, map, st);
        case 4: return launch_b<4>(w, q, s, b, total, K, gs, dtype, map, st);
        case 6: return launch_b<6>(w, q, s, b, total, K, gs, dtype, map, st);
        default: return launch_b<8>(w, q, s, b, total, K, gs, dtype, map, st);
    }
}

}  // namespace
}  // namespace gbxq

extern "C" {

int gbxq_quantize(const void* w, uint32_t* qweight, void* scales, void* biases, int64_t rows, int64_t K, int bits,
                  int group_size, int dtype, void* stream) {
    return gbxq::quantize_checked(w, qweight, scales, biases, rows, K, bits, group_size, dtype, gbxq::RowMap{0, 0, 0},
                                  (cudaStream_t)stream);
}

int gbxq_quantize_rows(const void* w, uint32_t* qweight, void* scales, void* biases, int64_t rows, int64_t K, int bits,
                       int group_size, int dtype, int64_t inner_rows, int64_t out_outer_stride_rows,
                       int64_t out_row_offset, void* stream) {
    if (inner_rows <= 0) return GBXQ_ESHAPE;
    return gbxq::quantize_checked(w, qweight, scales, biases, rows, K, bits, group_size, dtype,
                                  gbxq::RowMap{inner_rows, out_outer_stride_rows, out_row_offset}, (cudaStream_t)stream);
}

}  // extern "C"
