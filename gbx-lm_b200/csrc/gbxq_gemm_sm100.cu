// gbxq_gemm_sm100.cu -- prefill / large-batch quantized GEMM on the 5th-gen tensor cores
// (tcgen05.mma, accumulators in TMEM, activations by TMA) with in-kernel dequantisation.
//
// Reference call: QuantizedLinear.__call__ -> mx.quantized_matmul(transpose=True)
// (gbx_lm/models/quantized_linear_gba.py:195-203) with M = B*L rows of x; the reference prefills
// in chunks of up to 2048 tokens (gbx_lm/utils.py:226,312-319).  Above the ridge point
// (M ~ 40-140, SURVEY.md 8d) the path is a dense contraction bounded by the tensor pipe.
//
// Swap-AB formulation: the WEIGHT tile is the MMA "A" operand (M_mma = 128 output features fill the
// 128 TMEM lanes) and the TOKENS are the MMA N dimension (BN = 32..256 accumulator columns):
//     D[n, m] (TMEM, fp32) += A[n, k] (bf16 dequantised weights, smem) * B[k, m] (bf16 x, smem)
// so one dequantised 128 x 64 weight tile feeds up to 256 tokens, and skinny batches (M = 17..64)
// use the same kernel with a narrow N.
//
// Warp roles (576 threads, one CTA per SM, 3-4 stage ring, BLOCK_K = 64):
//   warp 0      TMA producer (cp.async.bulk.tensor.2d): the x tile [BN tokens x 64 k] (SWIZZLE_128B,
//               out-of-range tokens zero-filled), the PACKED weight tile [128 rows x 128 codes] for
//               two k-blocks at a time and the tile's scales / biases [128 rows x 8 groups], each on
//               its own mbarrier ring; also owns the TMEM allocation
//   warps 1-16  dequant producers: a thread owns a quarter of a weight row of the tile per k-block: reads its 16
//               packed codes and the group's scale/bias from the staging rings (no global loads, so the
//               proxy fence below never waits on HBM), unpacks with (w >> s) & mask | 0x4300 (two bf16
//               128+q per LOP3), applies scale*q+bias with one HFMA2.BF16 per pair (single rounding),
//               and stores the row into the canonical K-major 128B-swizzled layout the UMMA
//               descriptor expects (16-byte chunk c of row r at chunk position c ^ (r & 7));
//               fence.proxy.async, then arrive.  After the main loop the same warps are the epilogue:
//               tcgen05.ld 32x32b -> one rounding to bf16 (+ bias as a second rounded add) -> y
//   warp 17     MMA issuer: one thread issues 4 x tcgen05.mma (K = 16) per stage and commits the
//               stage's smem release and, at the end, the accumulator hand-off to the epilogue
#include <cuda.h>

#include <cstdlib>

#include "gbxq_common.cuh"

namespace gbxq {

namespace {

constexpr int kBlockK = 64;     // bf16 elements per k-block = one 128-byte swizzle atom
constexpr int kTileN = 128;     // output features per CTA (= UMMA M = TMEM lanes)
constexpr int kDequantWarps = 16;
constexpr int kThreads = (kDequantWarps + 2) * 32;
constexpr uint32_t kMagic = 0x43004300u;

// ------------------------------------------------------------------ tcgen05 / TMA PTX wrappers
__device__ __forceinline__ void tma_load_2d(void* dst, const void* tmap, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 format): rows of 128 bytes, 8-row
// core groups 1024 bytes apart (SBO), LBO unused for a swizzled K-major tile one atom wide.
__device__ __forceinline__ uint64_t make_sw128_kmajor_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);  // start address            bits [0,14)
    d |= (uint64_t)1 << 16;                        // leading byte offset (16 B; ignored) bits [16,30)
    d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset = 1024 B         bits [32,46)
    d |= (uint64_t)1 << 46;                        // descriptor version (sm_100)         bits [46,48)
    d |= (uint64_t)2 << 61;                        // layout type: SWIZZLE_128B           bits [61,64)
    return d;
}
// kind::f16 instruction descriptor: D = fp32, A = B = bf16, both K-major, M = 128, N = bn.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

struct GemmParams {
    const __nv_bfloat16* bias;
    __nv_bfloat16* y;
    int64_t M, N, K;
    int gs_shift;
    // split-K (skinny batches: 17..256 tokens leave only N/128 output tiles, a fraction of the 148 SMs): blockIdx.z
    // owns k-blocks [z*kb_per_split, ...), writes its fp32 partial tile to `ws` [splits][M][N]; the CTA that arrives
    // last at the tile's counter adds the partials in split order (deterministic) and rounds once to bf16.
    int splits, kb_per_split;  // kb_per_split is a multiple of 16 k-blocks (whole weight pairs and scale slots)
    float* ws;
    uint32_t* cnt;             // one counter per output tile, zero before and after the launch
};

// The 16 (3-bit: 32) consecutive codes of one row a dequant thread owns per k-block + the raw bf16
// scale / bias of their group.
template <int BITS> struct RowBlock {
    static constexpr int CODES = BITS == 3 ? 32 : 16;   // 3-bit quarters are not word aligned: use halves
    static constexpr int NW = CODES * BITS / 32;
    uint32_t w[NW];
    uint32_t s, b;
};

__device__ __forceinline__ uint32_t hsub2_bf16(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("sub.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ uint32_t hfma2_bf16(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("fma.rn.bf16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

// chunk c (codes 8c .. 8c+7 of the thread's block) as 4 packed bf16x2 registers in natural k order.
template <int BITS>
__device__ __forceinline__ uint4 dequant_chunk(const RowBlock<BITS>& rb, int c) {
    const uint32_t sraw = rb.s, braw = rb.b;
    uint4 out;
    if constexpr (BITS == 4 || BITS == 2) {
        const uint32_t s2 = sraw | (sraw << 16), b2 = braw | (braw << 16);
        uint32_t pr[4];  // pr[i] = (q_a, q_b) exact small integers in bf16
        if constexpr (BITS == 4) {
            const uint32_t word = rb.w[c];
#pragma unroll
            for (int i = 0; i < 4; i++)  // (nibble i, nibble i+4)
                pr[i] = hsub2_bf16(lop3_and_or(word >> (4 * i), 0x000f000fu, kMagic), kMagic);
        } else {
            // 2-bit: a word holds 16 codes; chunk c = fields 8*(c&1) .. +7 of word c>>1
            const uint32_t half = rb.w[c >> 1] >> (16 * (c & 1));  // the chunk's 8 fields now at bits 0..15
#pragma unroll
            for (int i = 0; i < 4; i++)  // (field i, field i+4): bits 2i and 2i+8 -> low bits of each half
                pr[i] = hsub2_bf16(lop3_and_or(__byte_perm(half >> (2 * i), 0u, 0x4140), 0x00030003u, kMagic), kMagic);
        }
        // re-pair (0,4),(1,5),(2,6),(3,7) -> (0,1),(2,3),(4,5),(6,7)
        const uint32_t q01 = __byte_perm(pr[0], pr[1], 0x5410), q45 = __byte_perm(pr[0], pr[1], 0x7632);
        const uint32_t q23 = __byte_perm(pr[2], pr[3], 0x5410), q67 = __byte_perm(pr[2], pr[3], 0x7632);
        out.x = hfma2_bf16(q01, s2, b2); out.y = hfma2_bf16(q23, s2, b2);
        out.z = hfma2_bf16(q45, s2, b2); out.w = hfma2_bf16(q67, s2, b2);
    } else {
        // generic widths (3, 6, 8): exact small integers via the fp32 magic number, fp32 FMA, one rounding
        const float s = __uint_as_float(sraw << 16), b = __uint_as_float(braw << 16);
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int bit = (8 * c + i) * BITS;
            const int wi = bit >> 5, off = bit & 31;
            uint32_t sh;
            if (off + BITS <= 32) sh = rb.w[wi] >> off;
            else sh = __funnelshift_r(rb.w[wi], rb.w[wi + 1], off);
            const float q = __uint_as_float(lop3_and_or(sh, (1u << BITS) - 1u, 0x4B000000u)) - 8388608.0f;
            v[i] = fmaf(s, q, b);
        }
        out.x = pack_bf16x2(v[0], v[1]); out.y = pack_bf16x2(v[2], v[3]);
        out.z = pack_bf16x2(v[4], v[5]); out.w = pack_bf16x2(v[6], v[7]);
    }
    return out;
}

template <int BITS, int BN> struct Cfg {
    // Two rings decoupled by depth: the x tiles (TMA, ~1 us latency) run 4-6 k-blocks ahead of the MMA,
    // the dequantised weight tiles (produced on-chip) only 3.
    static constexpr int XSTAGES = BN == 256 ? 4 : 6;
    static constexpr int ASTAGES = 3;
    static constexpr uint32_t A_BYTES = kTileN * kBlockK * 2;          // 16 KB
    static constexpr uint32_t B_BYTES = BN * kBlockK * 2;
    static constexpr uint32_t W_ROW_BYTES = 16 * BITS;                 // packed bytes of 128 codes (2 k-blocks)
    static constexpr uint32_t W_SLOT = kTileN * W_ROW_BYTES;           // 2*BITS KB
    static constexpr int W_SLOTS = (32 * 1024 / W_SLOT) >= 4 ? 4 : 2;  // packed-weight ring (pairs of k-blocks)
    static constexpr uint32_t S_SLOT = 2 * kTileN * 16;                // scales + biases, 8 groups per row
    static constexpr int S_SLOTS = 2;
    static constexpr uint32_t TMEM_COLS = BN < 32 ? 32 : BN;
    static constexpr size_t SMEM = (size_t)XSTAGES * B_BYTES + (size_t)ASTAGES * A_BYTES + (size_t)W_SLOTS * W_SLOT +
                                   (size_t)S_SLOTS * S_SLOT + (2 * XSTAGES + 2 * ASTAGES + 2 * W_SLOTS + 2 * S_SLOTS + 1) * 8 +
                                   16 + 1024;
};

template <int BITS, int BN>
__global__ void __launch_bounds__(kThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
            const __grid_constant__ CUtensorMap tmap_s, const __grid_constant__ CUtensorMap tmap_b, const GemmParams p) {
    using C = Cfg<BITS, BN>;
    constexpr int XS = C::XSTAGES, AS = C::ASTAGES, WS = C::W_SLOTS, SS = C::S_SLOTS;

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // 1024-byte alignment for the 128B-swizzled tiles
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* xring = smem;                                   // [XS][BN x 64] bf16, 128B-swizzled (TMA)
    uint8_t* aring = xring + (size_t)XS * C::B_BYTES;        // [AS][128 x 64] bf16, 128B-swizzled (dequant warps)
    uint8_t* wring = aring + (size_t)AS * C::A_BYTES;
    uint8_t* sring = wring + (size_t)WS * C::W_SLOT;
    uint64_t* full_a = reinterpret_cast<uint64_t*>(sring + (size_t)SS * C::S_SLOT);
    uint64_t* empty_a = full_a + AS;
    uint64_t* full_b = empty_a + AS;
    uint64_t* empty_b = full_b + XS;
    uint64_t* wfull = empty_b + XS;
    uint64_t* wempty = wfull + WS;
    uint64_t* sfull = wempty + WS;
    uint64_t* sempty = sfull + SS;
    uint64_t* tmem_full = sempty + SS;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * kTileN;
    const int m0 = blockIdx.y * BN;
    const int nkb_all = (int)(p.K / kBlockK);
    const int kb_lo = p.splits > 1 ? (int)blockIdx.z * p.kb_per_split : 0;   // first k-block of this split
    const int nkb = p.splits > 1 ? min(p.kb_per_split, nkb_all - kb_lo) : nkb_all;  // k-blocks of this CTA (loops are local)
    const int pr_lo = kb_lo >> 1;
    const int npair = (nkb + 1) >> 1;                     // packed-weight slots: 2 k-blocks each
    const int kb_per_s = p.gs_shift == 5 ? 4 : (p.gs_shift == 6 ? 8 : 16);  // k-blocks per scale slot (8 groups)
    const int nsl = (nkb + kb_per_s - 1) / kb_per_s;
    const int sl_lo = kb_lo / kb_per_s;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < AS; s++) {
            mbar_init(&full_a[s], kDequantWarps);  // one arrival per dequant warp
            mbar_init(&empty_a[s], 1);             // tcgen05.commit
        }
#pragma unroll
        for (int s = 0; s < XS; s++) {
            mbar_init(&full_b[s], 1);              // TMA producer (+ tx bytes)
            mbar_init(&empty_b[s], 1);             // tcgen05.commit
        }
#pragma unroll
        for (int s = 0; s < WS; s++) {
            mbar_init(&wfull[s], 1);
            mbar_init(&wempty[s], kDequantWarps);
        }
#pragma unroll
        for (int s = 0; s < SS; s++) {
            mbar_init(&sfull[s], 1);
            mbar_init(&sempty[s], kDequantWarps);
        }
        mbar_init(tmem_full, 1);
        fence_mbar_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, C::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            auto issue_w = [&](int pr) {  // packed weights of k-blocks 2pr, 2pr+1
                const int s = pr % WS;
                mbar_wait(&wempty[s], ((uint32_t)(pr / WS) & 1u) ^ 1u);
                mbar_arrive_expect_tx(&wfull[s], C::W_SLOT);
                tma_load_2d(wring + (size_t)s * C::W_SLOT, &tmap_w, (pr_lo + pr) * 4 * BITS, n0, &wfull[s]);
            };
            auto issue_s = [&](int sl) {  // scales + biases of groups 8sl .. 8sl+7
                const int s = sl % SS;
                mbar_wait(&sempty[s], ((uint32_t)(sl / SS) & 1u) ^ 1u);
                mbar_arrive_expect_tx(&sfull[s], C::S_SLOT);
                tma_load_2d(sring + (size_t)s * C::S_SLOT, &tmap_s, (sl_lo + sl) * 8, n0, &sfull[s]);
                tma_load_2d(sring + (size_t)s * C::S_SLOT + kTileN * 16, &tmap_b, (sl_lo + sl) * 8, n0, &sfull[s]);
            };
            // run the small streams ahead of the x stream: WS-1 weight slots and one scale slot in flight
            issue_s(0);
            for (int pr = 0; pr < WS - 1 && pr < npair; pr++) issue_w(pr);
            for (int kb = 0; kb < nkb; kb++) {
                if ((kb & 1) == 0 && (kb >> 1) + WS - 1 < npair) issue_w((kb >> 1) + WS - 1);
                if (kb % kb_per_s == 0 && kb / kb_per_s + 1 < nsl) issue_s(kb / kb_per_s + 1);
                const int s = kb % XS;
                mbar_wait(&empty_b[s], ((uint32_t)(kb / XS) & 1u) ^ 1u);
                mbar_arrive_expect_tx(&full_b[s], C::B_BYTES);
                tma_load_2d(xring + (size_t)s * C::B_BYTES, &tmap_x, (kb_lo + kb) * kBlockK, m0, &full_b[s]);
            }
        }
    } else if (warp == 1 + kDequantWarps) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc_bf16(kTileN, BN);
            for (int kb = 0; kb < nkb; kb++) {
                const int sa = kb % AS, sx = kb % XS;
                mbar_wait(&full_a[sa], (uint32_t)(kb / AS) & 1u);
                mbar_wait(&full_b[sx], (uint32_t)(kb / XS) & 1u);
                tc_fence_after();
                const uint32_t a_addr = smem_u32(aring + (size_t)sa * C::A_BYTES);
                const uint32_t b_addr = smem_u32(xring + (size_t)sx * C::B_BYTES);
#pragma unroll
                for (int k = 0; k < kBlockK / 16; k++) {
                    const uint64_t ad = make_sw128_kmajor_desc(a_addr + k * 32);
                    const uint64_t bd = make_sw128_kmajor_desc(b_addr + k * 32);
                    umma_f16(tmem_base, ad, bd, idesc, (kb | k) != 0 ? 1u : 0u);
                }
                umma_commit(&empty_a[sa]);  // both ring slots are free once these MMAs retire
                umma_commit(&empty_b[sx]);
            }
            umma_commit(tmem_full);      // accumulator complete -> epilogue
        }
    } else {
        // ===================== dequant producers (warps 1-16), then epilogue =====================
        const int dw = warp - 1;                 // 0..15
        const int r = dw * 8 + (lane >> 2);      // tile row this thread dequantises
        const int qk = lane & 3;                 // which 16-code quarter of the k-block
        using RB = RowBlock<BITS>;
        constexpr int CPT = RB::CODES / 8;       // 16-byte chunks this thread writes per k-block
        const bool lane_on = (BITS != 3) || ((qk & 1) == 0);
        const int c_base = (BITS == 3) ? (qk >> 1) * 4 : qk * 2;   // first chunk (of 8) this thread writes
        const uint32_t wring_u32 = smem_u32(wring), sring_u32 = smem_u32(sring);

        for (int kb = 0; kb < nkb; kb++) {
            const int pr = kb >> 1, ws = pr % WS;
            const int sl = kb / kb_per_s, ss = sl % SS;
            if ((kb & 1) == 0) mbar_wait(&wfull[ws], (uint32_t)(pr / WS) & 1u);
            if (kb % kb_per_s == 0) mbar_wait(&sfull[ss], (uint32_t)(sl / SS) & 1u);
            // ---- this thread's packed codes and their group's scale / bias, from the staging rings
            RB rb;
            if (lane_on) {
                const uint32_t wa = wring_u32 + (uint32_t)ws * C::W_SLOT + (uint32_t)r * C::W_ROW_BYTES +
                                    (uint32_t)((kb & 1) * 8 * BITS) + (uint32_t)(c_base * BITS);  // c_base*8 codes*BITS/8 bytes
                if constexpr (RB::NW == 4) {
                    const uint4 t = lds128(wa);
                    rb.w[0] = t.x; rb.w[1] = t.y; rb.w[2] = t.z; rb.w[3] = t.w;
                } else if constexpr (RB::NW == 2) {
                    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(rb.w[0]), "=r"(rb.w[1]) : "r"(wa));
                } else {
#pragma unroll
                    for (int i = 0; i < RB::NW; i++) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(rb.w[i]) : "r"(wa + 4 * i));
                }
                const int gl = ((kb * kBlockK + c_base * 8) >> p.gs_shift) & 7;  // group inside the 8-group slot
                const uint32_t sa = sring_u32 + (uint32_t)ss * C::S_SLOT + (uint32_t)r * 16 + (uint32_t)gl * 2;
                asm volatile("ld.shared.u16 %0, [%1];" : "=r"(rb.s) : "r"(sa));
                asm volatile("ld.shared.u16 %0, [%1];" : "=r"(rb.b) : "r"(sa + kTileN * 16));
            }
            const int s = kb % AS;
            mbar_wait(&empty_a[s], ((uint32_t)(kb / AS) & 1u) ^ 1u);
            if (lane_on) {
                uint8_t* a_row = aring + (size_t)s * C::A_BYTES + (size_t)r * 128;
#pragma unroll
                for (int c = 0; c < CPT; c++) {
                    const uint4 v = dequant_chunk<BITS>(rb, c);
                    *reinterpret_cast<uint4*>(a_row + (((c_base + c) ^ (r & 7)) << 4)) = v;
                }
            }
            fence_proxy_async();  // make the generic-proxy stores visible to the tensor core (async proxy)
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&full_a[s]);
                if ((kb & 1) == 1 || kb == nkb - 1) mbar_arrive(&wempty[ws]);
                if (kb % kb_per_s == kb_per_s - 1 || kb == nkb - 1) mbar_arrive(&sempty[ss]);
            }
        }

        // ---- epilogue: TMEM -> registers -> bf16 -> y[m, n]; warp drains TMEM lanes 32*(warp%4).. (its hardware
        //      quarter) and column quarter (dw >> 2) of the accumulator
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        const int q4 = warp & 3;
        const int er = q4 * 32 + lane;
        const int64_t n = (int64_t)n0 + er;
        const bool row_ok = n < p.N;
        const float bias_f = (p.bias != nullptr && row_ok) ? __bfloat162float(p.bias[n]) : 0.f;
        constexpr int QCOLS = BN / 4;
        constexpr int STEP = QCOLS >= 32 ? 32 : (QCOLS >= 16 ? 16 : 8);
        const int cq = dw >> 2;
#pragma unroll 1
        for (int c0 = cq * QCOLS; c0 < (cq + 1) * QCOLS; c0 += STEP) {
            uint32_t v[32];
            const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)c0;
            if constexpr (STEP == 32) tmem_ld32(taddr, v);
            else if constexpr (STEP == 16) tmem_ld16(taddr, v);
            else tmem_ld8(taddr, v);
            if (row_ok) {
#pragma unroll
                for (int j = 0; j < STEP; j++) {
                    const int64_t m = (int64_t)m0 + c0 + j;
                    if (m < p.M) {
                        if (p.splits > 1) {
                            p.ws[((size_t)blockIdx.z * p.M + m) * p.N + n] = __uint_as_float(v[j]);
                        } else {
                            float f = __bfloat162float(__float2bfloat16_rn(__uint_as_float(v[j])));
                            if (p.bias != nullptr) f = __fadd_rn(f, bias_f);
                            p.y[(size_t)m * p.N + n] = __float2bfloat16_rn(f);
                        }
                    }
                }
            }
        }
        tc_fence_before();
        if (p.splits > 1) {
            // the last split to arrive at this tile's counter adds the partial tiles in split order and writes y
            __threadfence();
            asm volatile("bar.sync 2, %0;" ::"n"(kDequantWarps * 32) : "memory");
            uint32_t* flag = tmem_slot + 1;  // shared scratch next to the TMEM address
            const uint32_t tile = blockIdx.y * gridDim.x + blockIdx.x;
            if (warp == 1 && lane == 0) *flag = atomicAdd(p.cnt + tile, 1u) == (uint32_t)p.splits - 1u ? 1u : 0u;
            asm volatile("bar.sync 2, %0;" ::"n"(kDequantWarps * 32) : "memory");
            if (*flag != 0u) {
                __threadfence();
                if (row_ok) {
                    for (int c = cq * QCOLS; c < (cq + 1) * QCOLS; c++) {
                        const int64_t m = (int64_t)m0 + c;
                        if (m < p.M) {
                            float acc = 0.f;
                            for (int z = 0; z < p.splits; z++) acc += __ldcg(p.ws + ((size_t)z * p.M + m) * p.N + n);
                            float f = __bfloat162float(__float2bfloat16_rn(acc));
                            if (p.bias != nullptr) f = __fadd_rn(f, bias_f);
                            p.y[(size_t)m * p.N + n] = __float2bfloat16_rn(f);
                        }
                    }
                }
                if (warp == 1 && lane == 0) p.cnt[tile] = 0u;  // left zero for the next launch
            }
        }
    }
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, C::TMEM_COLS);
    }
}

// ------------------------------------------------------------------ host side
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

bool encode_2d(CUtensorMap* tm, CUtensorMapDataType dt, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
               uint32_t box_inner, uint32_t box_outer, CUtensorMapSwizzle sw) {
    EncodeTiledFn enc = get_encode();
    if (enc == nullptr) return false;
    const cuuint64_t gdim[2] = {inner, outer};
    const cuuint64_t gstride[1] = {pitch_bytes};
    const cuuint32_t box[2] = {box_inner, box_outer};
    const cuuint32_t estr[2] = {1, 1};
    // GBXQ_TMA_L2PROMO = 0 / 64 / 128 / 256 (development switch; default 256 bytes)
    static const int promo = env_int("GBXQ_TMA_L2PROMO", 256);
    const CUtensorMapL2promotion pr = promo == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE
                                      : (promo == 64 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
                                                     : (promo == 128 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_256B));
    return enc(tm, dt, 2, const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, pr,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct Maps {
    CUtensorMap x, w, s, b;
};

template <int BITS, int BN>
int launch_inst(const Maps& mp, const GemmParams& p, cudaStream_t st) {
    constexpr size_t smem = Cfg<BITS, BN>::SMEM;
    static_assert(smem <= 227 * 1024, "shared memory budget");
    const int rc = allow_dynamic_smem<gemm_kernel<BITS, BN>>((int)smem);
    if (rc != GBXQ_OK) return rc;
    dim3 grid((unsigned)((p.N + kTileN - 1) / kTileN), (unsigned)((p.M + BN - 1) / BN), (unsigned)(p.splits > 1 ? p.splits : 1));
    return launch(gemm_kernel<BITS, BN>, grid, dim3(kThreads), smem, st, false, mp.x, mp.w, mp.s, mp.b, p);
}

template <int BITS>
int launch_bn(int bn, const Maps& mp, const GemmParams& p, cudaStream_t st) {
    switch (bn) {
        case 32: return launch_inst<BITS, 32>(mp, p, st);
        case 64: return launch_inst<BITS, 64>(mp, p, st);
        case 128: return launch_inst<BITS, 128>(mp, p, st);
        default: return launch_inst<BITS, 256>(mp, p, st);
    }
}

int pick_bn(int64_t M) { return M <= 32 ? 32 : (M <= 64 ? 64 : (M <= 128 ? 128 : 256)); }

}  // namespace

bool tma_encode_available() { return get_encode() != nullptr; }

bool encode_tensor_map_2d(void* tm, int dtype, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                          uint32_t box_inner, uint32_t box_outer, bool swizzle128) {
    return encode_2d(reinterpret_cast<CUtensorMap*>(tm), dtype == 0 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT32,
                     base, inner, outer, pitch_bytes, box_inner, box_outer,
                     swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE);
}

bool encode_tensor_map_2d_sw(void* tm, int dtype, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                             uint32_t box_inner, uint32_t box_outer, int swizzle_bytes) {
    const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                  : (swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                         : (swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE));
    return encode_2d(reinterpret_cast<CUtensorMap*>(tm), dtype == 0 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT32,
                     base, inner, outer, pitch_bytes, box_inner, box_outer, sw);
}

bool gemm_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                    const void* y) {
    if (dtype != GBXQ_BF16 || M < 1 || N < 1) return false;
    if (K % kBlockK) return false;
    if ((K * bits / 8) % 16) return false;      // TMA: packed row pitch must be a multiple of 16 bytes
    if (((K / gs) * 2) % 16) return false;      // TMA: scale row pitch must be a multiple of 16 bytes
    if (((uintptr_t)x | (uintptr_t)w) & 15) return false;
    if ((uintptr_t)y & 1) return false;
    if (M > (int64_t)1 << 24 || (N + kTileN - 1) / kTileN > 65535 * 32) return false;
    return get_encode() != nullptr;
}

// Split-K plan for a skinny batch: how many splits, k-blocks per split, workspace bytes (counter header + partials).
constexpr size_t kCntBytes = 16384;  // up to 4096 output tiles
void gemm_split_plan(int64_t M, int64_t N, int64_t K, int* splits, int* kb_per_split, size_t* ws_bytes) {
    *splits = 1;
    *kb_per_split = 0;
    *ws_bytes = 0;
    if (M > 256 || M < 1) return;
    const int bn = pick_bn(M);
    const int64_t tiles = ((N + kTileN - 1) / kTileN) * ((M + bn - 1) / bn);
    const int64_t nkb = K / kBlockK;
    const int sms = device_sm_count();
    if (tiles * 2 > sms || tiles > 4096) return;      // enough CTAs already
    int want = (int)(sms / tiles);
    if (want > 8) want = 8;
    const int chunks = (int)((nkb + 15) / 16);         // splits are whole 16-k-block chunks (weight pairs, scale slots)
    if (want > chunks) want = chunks;
    if (want < 2) return;
    const int per = (chunks + want - 1) / want * 16;
    const int s = (int)((nkb + per - 1) / per);
    if (s < 2) return;
    *splits = s;
    *kb_per_split = per;
    *ws_bytes = kCntBytes + (size_t)s * (size_t)M * (size_t)N * 4;
}

size_t gemm_workspace_bytes(int64_t M, int64_t N, int64_t K) {
    int s, per;
    size_t b;
    gemm_split_plan(M, N, K, &s, &per, &b);
    return b;
}

int launch_gemm(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                int64_t N, int64_t K, int bits, int gs, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    if (get_encode() == nullptr) return GBXQ_EUNSUPPORTED;
    if (((uintptr_t)s | (uintptr_t)b) & 15) return GBXQ_EUNSUPPORTED;
    const int bn = pick_bn(M);
    if ((M + bn - 1) / bn > 65535) return GBXQ_EUNSUPPORTED;
    Maps mp;
    const uint64_t words = (uint64_t)(K * bits / 32), G = (uint64_t)(K / gs);
    bool ok = encode_2d(&mp.x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, x, (uint64_t)K, (uint64_t)M, (uint64_t)K * 2, kBlockK, (uint32_t)bn,
                        CU_TENSOR_MAP_SWIZZLE_128B);
    ok = ok && encode_2d(&mp.w, CU_TENSOR_MAP_DATA_TYPE_UINT32, w, words, (uint64_t)N, words * 4, (uint32_t)(4 * bits), kTileN,
                         CU_TENSOR_MAP_SWIZZLE_NONE);
    ok = ok && encode_2d(&mp.s, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, s, G, (uint64_t)N, G * 2, 8, kTileN, CU_TENSOR_MAP_SWIZZLE_NONE);
    ok = ok && encode_2d(&mp.b, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, b, G, (uint64_t)N, G * 2, 8, kTileN, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (!ok) return GBXQ_EUNSUPPORTED;
    GemmParams p{};
    p.bias = reinterpret_cast<const __nv_bfloat16*>(bias);
    p.y = reinterpret_cast<__nv_bfloat16*>(y);
    p.M = M;
    p.N = N;
    p.K = K;
    p.gs_shift = gs == 32 ? 5 : (gs == 64 ? 6 : 7);
    p.splits = 1;
    {
        int sp, per;
        size_t need;
        gemm_split_plan(M, N, K, &sp, &per, &need);
        if (sp > 1 && workspace != nullptr && workspace_bytes >= need && !((uintptr_t)workspace & 15)) {
            p.splits = sp;
            p.kb_per_split = per;
            p.cnt = reinterpret_cast<uint32_t*>(workspace);
            p.ws = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + kCntBytes);
        }
    }
    switch (bits) {
        case 2: return launch_bn<2>(bn, mp, p, st);
        case 3: return launch_bn<3>(bn, mp, p, st);
        case 4: return launch_bn<4>(bn, mp, p, st);
        case 6: return launch_bn<6>(bn, mp, p, st);
        case 8: return launch_bn<8>(bn, mp, p, st);
    }
    return GBXQ_EINVAL_BITS;
}

}  // namespace gbxq
