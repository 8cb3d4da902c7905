// gbxq_gemm_ts_sm100.cu -- quantized GEMM with the dequantised weights fed to the tensor core FROM TENSOR MEMORY
// ("TS" form of tcgen05.mma: A in TMEM, B in shared memory).  Serves batches of 5..256 rows of x per tile (decode
// batches 8..64 of BASELINE configs 2-5 and prefill chunks, gbx_lm/utils.py:312-319) behind
// QuantizedLinear.__call__ -> mx.quantized_matmul(transpose=True) (gbx_lm/models/quantized_linear_gba.py:195-203).
//
// Why a second tensor-core kernel (gbxq_gemm_sm100.cu is the first): that kernel writes the dequantised bf16 tile to
// shared memory in the UMMA layout, k-block by k-block, with a proxy fence and a barrier round trip per 64 k: measured
// ~950 clocks per k-block (profiles/r01a_gemmbench.txt: 31-110 us per launch whatever the batch), 5x the HBM rate of
// 4-bit weights, and every dequantised byte crosses shared memory twice (STS + the tensor core's operand read).  Here
//   * a dequant thread owns ONE weight row (= one TMEM lane) and 32 consecutive k of a 128-k stage: one conflict-free
//     128-bit shared-memory load of packed codes (the packed tile is fetched by TMA with the swizzle that makes a
//     column of 16-byte pieces hit distinct banks), ~80 ALU instructions, ONE tcgen05.st of 16 columns -- no proxy
//     fence, no shared-memory store, half as many barrier round trips per k;
//   * swap-AB as before: weights are the MMA "A" operand (M = 128 output features = the 128 TMEM lanes, 8 columns per
//     K = 16 step), tokens are the MMA N dimension (BN = 16..256 accumulator columns), x tiles arrive by TMA in the
//     K-major 128B-swizzled layout;
//   * TMEM: accumulator at columns [0, BN), four A stages of 64 columns at [256, 512);
//   * x and packed weights have a producer warp each (x waits for the previous kernel of the stream -- programmatic
//     dependent launch --, weights and scales are immutable and stream ahead of it);
//   * split-K over blockIdx.z for skinny batches exactly as in gbxq_gemm_sm100.cu (deterministic reduction order).
#include <cstdlib>

//
// This file is compiled twice.  gbxq_gemm_ts_direct_sm100.cu includes it with GBXQ_TS_DIRECT defined: the variant for
// matrices whose row of scales is not a legal TMA row pitch (K / group_size not a multiple of 8: tensor-parallel K
// shards such as Qwen2.5-32B o_proj K/4 = 1280 = 10 groups of 128), where the dequant threads read their (row, group)
// scale and bias from global memory one stage ahead instead of from the TMA-fed scale ring.  Preprocessor blocks, not a
// template flag or a run-time branch: either of those changed the register allocation of the common kernel and cost
// prefill 3-5 % in same-box A/B runs (r03l-r03n).
#include "gbxq_umma.cuh"

namespace gbxq {

void gemm_split_plan(int64_t M, int64_t N, int64_t K, int* splits, int* kb_per_split, size_t* ws_bytes);
bool encode_tensor_map_2d_sw(void* tm, int dtype, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                             uint32_t box_inner, uint32_t box_outer, int swizzle_bytes);

#ifdef GBXQ_TS_DIRECT
#define TS_KERNEL gemm_ts_direct_kernel
#define TS_LAUNCH launch_gemm_ts_direct
#else
#define TS_KERNEL gemm_ts_kernel
#define TS_LAUNCH launch_gemm_ts
int launch_gemm_ts_direct(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                          int64_t N, int64_t K, int bits, int gs, void* workspace, size_t workspace_bytes, cudaStream_t st);
#endif

// A third compilation (gbxq_gemm_ts_grouped_sm100.cu, GBXQ_TS_GROUPED): up to three projections that read the same x
// (q|k|v, gate|up) and share bit width and group size as ONE launch -- the tiles of all segments in one grid, one
// tensor-map triple per segment.  The macros below keep the tokens of the plain compilation unchanged.
#ifdef GBXQ_TS_GROUPED
#undef TS_KERNEL
#define TS_KERNEL gemm_ts_grouped_kernel
#define TS_SIG const __grid_constant__ TsMaps maps, const TsParams p
#define TMAP_X &maps.x
#define TMAP_W &maps.w[seg]
#define TMAP_S &maps.s[seg]
#define TMAP_B &maps.b[seg]
#define P_N segN
#define P_BIAS seg_bias
#define P_Y seg_y
#define P_WS seg_ws
#define TILE_X ((int)blockIdx.x - tile_lo)
#else
#define TS_SIG                                                                                           \
    const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,              \
        const __grid_constant__ CUtensorMap tmap_s, const __grid_constant__ CUtensorMap tmap_b, const TsParams p
#define TMAP_X &tmap_x
#define TMAP_W &tmap_w
#define TMAP_S &tmap_s
#define TMAP_B &tmap_b
#define P_N p.N
#define P_BIAS p.bias
#define P_Y p.y
#define P_WS p.ws
#define TILE_X blockIdx.x
#endif

namespace {

using namespace umma;

constexpr int kHalfK = 128;    // one TMA box of packed codes: 128 rows x 128 codes
constexpr int kH = 2;          // boxes ("halves") per stage: the per-stage barrier traffic of the dequant warps (~120 of
                               // their ~195 instructions per 128 k, r02x SASS) is paid once per 256 k
constexpr int kStageK = kHalfK * kH;  // k per stage = 128 TMEM columns of A = 4 x tiles ("atoms") of 64 k
constexpr int kAtomK = 64;
constexpr int kTileN = 128;    // output features per CTA (= UMMA M = TMEM lanes)
constexpr int kDqWarps = 16;   // warps 1..16: (row quarter = warp % 4, k quarter = (warp - 1) / 4)
constexpr int kWarpMma = 17, kWarpW = 18;
constexpr int kThreads = 19 * 32;
constexpr int kAStages = 2;
constexpr int kAtomsPerStage = kStageK / 64;
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kTmemAOff = 256;
constexpr size_t kCntBytes = 16384;  // counter header of the split-K workspace (as gbxq_gemm_sm100.cu)

#ifdef GBXQ_TS_GROUPED
struct TsMaps {  // one x map, one (packed codes, scales, biases) triple per segment
    CUtensorMap x;
    CUtensorMap w[3], s[3], b[3];
};
#endif

struct TsParams {
    const __nv_bfloat16* bias;
    __nv_bfloat16* y;
    int64_t M, N, K;
    int gs_shift;
    int splits, kb_per_split;  // split-K: blockIdx.z owns k-blocks [z * kb_per_split, ...) (multiples of 16 k-blocks)
    float* ws;
    uint32_t* cnt;
    int early_w;               // 1: weights / scales are immutable while the call is in flight: fetch before griddepcontrol.wait
    const uint8_t* w_raw;      // packed weights (for the L2 prefetch of the CTA's rows)
    int64_t row_bytes;
    int rotate;                // 1: CTAs start their k loop at different stages (see stage_of)
#ifdef GBXQ_TS_GROUPED
    int nseg;                  // segments of the launch: segment i owns grid tiles [tile0[i], tile0[i + 1])
    int tile0[4];
    int64_t seg_n[3];
    const __nv_bfloat16* seg_bias[3];
    __nv_bfloat16* seg_y[3];
    int64_t seg_ws_off[3];     // floats: where the segment's split-K partials start in the workspace
#endif
#ifdef GBXQ_TS_DIRECT
    const uint16_t* s_raw;     // scales / biases [N, G] read directly by the dequant threads
    const uint16_t* b_raw;
    int64_t G;
#endif
    unsigned long long* dbg;   // development aid (gbxq_debug_ts_timeline): CTA 0 stamps %globaltimer, see tools/ts_timeline.py
};

template <int BITS, int BN> struct Cfg {
    static constexpr int XS = BN == 256 ? (BITS >= 8 ? 4 : 5) : 8;  // x atoms in flight (4 per stage)
    static constexpr uint32_t B_BYTES = BN * kAtomK * 2;
    static constexpr uint32_t W_ROW = 16 * BITS;                    // packed bytes of 128 codes
    static constexpr uint32_t W_HALF = kTileN * W_ROW;              // 2*BITS KB: one TMA box
    static constexpr uint32_t W_SLOT = kH * W_HALF;
    static constexpr int WS_RAW = (48 * 1024) / W_SLOT;
    static constexpr int WS = WS_RAW > 8 ? 8 : (WS_RAW < 2 ? 2 : WS_RAW);
    static constexpr uint32_t S_SLOT = 2 * kTileN * 16;             // scales + biases of 8 groups per row
    static constexpr int SS = 4;
    // Independent accumulators: the K = 16 steps of a tile go round-robin to NACC accumulators (TMEM columns j * BN) that
    // the epilogue adds in a fixed order.  A narrow MMA (N = 16: 8 clocks of tensor-pipe work) that accumulates into
    // the columns its predecessor has just written waits for that write-back: r02u/r02v timelines show ~100 ns per
    // dependent MMA, 0.8 us per 128-k stage whatever the width of the codes or the batch.
    static constexpr int NACC = BN <= 64 ? 4 : (BN == 128 ? 2 : 1);
    static constexpr int NBAR = 2 * XS + 2 * WS + 2 * SS + 2 * kAStages + 1;
    static constexpr size_t SMEM = (size_t)XS * B_BYTES + (size_t)WS * W_SLOT + (size_t)SS * S_SLOT + NBAR * 8 + 16 + 1024;
};

__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// timeline layout (CTA 0 only): [0] entry, [1] set-up done, [2] epilogue start, [3] exit, then per stage s (s < 64):
// [8 + 4s + 0] packed words landed (dequant warp 1), [.. + 1] A stage stored, [.. + 2] MMAs issued, [.. + 3] x tile landed
#define TS_STAMP(i)                                                                                        \
    do {                                                                                                   \
        if (p.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) p.dbg[(i)] = gtime(); \
    } while (0)

__device__ __forceinline__ uint32_t lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}

// The 32 codes (k quarter kq of the stage) of tile row r from a packed-weight slot.  The slot was written by TMA with
// Cfg::SWZ: 16-byte piece c of row r sits at piece c ^ f(r) so that the 8 lanes of an LDS wavefront (8 consecutive
// rows, same quarter) read distinct bank groups.
template <int BITS> __device__ __forceinline__ void load_codes(uint32_t slot, int r, int kq, uint32_t (&w)[BITS]) {
    if constexpr (BITS == 4) {
        const uint4 t = lds128(slot + (uint32_t)r * 64u + (uint32_t)((kq ^ ((r >> 1) & 3)) << 4));
        w[0] = t.x; w[1] = t.y; w[2] = t.z; w[3] = t.w;
    } else if constexpr (BITS == 2) {
        const uint2 t = lds64(slot + (uint32_t)r * 32u + (uint32_t)(((kq >> 1) ^ ((r >> 2) & 1)) << 4) + (uint32_t)(kq & 1) * 8u);
        w[0] = t.x; w[1] = t.y;
    } else if constexpr (BITS == 8) {
#pragma unroll
        for (int i = 0; i < 2; i++) {
            const uint4 t = lds128(slot + (uint32_t)r * 128u + (uint32_t)(((2 * kq + i) ^ (r & 7)) << 4));
            w[4 * i] = t.x; w[4 * i + 1] = t.y; w[4 * i + 2] = t.z; w[4 * i + 3] = t.w;
        }
    } else if constexpr (BITS == 3) {
#pragma unroll
        for (int i = 0; i < 3; i++) w[i] = lds32(slot + (uint32_t)r * 48u + (uint32_t)kq * 12u + 4u * i);
    } else {
#pragma unroll
        for (int i = 0; i < 3; i++) {
            const uint2 t = lds64(slot + (uint32_t)r * 96u + (uint32_t)kq * 24u + 8u * i);
            w[2 * i] = t.x; w[2 * i + 1] = t.y;
        }
    }
}

// 16-bit entry `g` (0..7) of a 16-byte row held in a uint4 (warp-uniform g)
__device__ __forceinline__ uint32_t pick16(const uint4& v, int g) {
    const int rs = g >> 1;
    const uint32_t wv = rs == 0 ? v.x : (rs == 1 ? v.y : (rs == 2 ? v.z : v.w));
    return (g & 1) ? (wv >> 16) : (wv & 0xffffu);
}

template <int BITS, int BN>
__global__ void __launch_bounds__(kThreads, 1)
TS_KERNEL(TS_SIG) {
    using C = Cfg<BITS, BN>;
    constexpr int XS = C::XS, WS = C::WS, SS = C::SS, AS = kAStages;

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* xring = smem;                                   // [XS][BN x 64] bf16, 128B-swizzled (TMA)
    uint8_t* wring = xring + (size_t)XS * C::B_BYTES;        // [WS][128 rows x 128 codes] packed (TMA, swizzled)
    uint8_t* sring = wring + (size_t)WS * C::W_SLOT;         // [SS][scales 128 x 8 | biases 128 x 8] bf16
    uint64_t* full_b = reinterpret_cast<uint64_t*>(sring + (size_t)SS * C::S_SLOT);
    uint64_t* empty_b = full_b + XS;
    uint64_t* wfull = empty_b + XS;
    uint64_t* wempty = wfull + WS;
    uint64_t* sfull = wempty + WS;
    uint64_t* sempty = sfull + SS;
    uint64_t* full_a = sempty + SS;
    uint64_t* empty_a = full_a + AS;
    uint64_t* tmem_full = empty_a + AS;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
#ifdef GBXQ_TS_GROUPED
    int seg = 0;
#pragma unroll
    for (int i = 1; i < 3; i++)
        if (i < p.nseg && (int)blockIdx.x >= p.tile0[i]) seg = i;
    const int tile_lo = p.tile0[seg];
    const int64_t segN = p.seg_n[seg];
    const __nv_bfloat16* seg_bias = p.seg_bias[seg];
    __nv_bfloat16* seg_y = p.seg_y[seg];
    float* seg_ws = p.ws + p.seg_ws_off[seg];
#endif
    const int n0 = TILE_X * kTileN;
    const int m0 = blockIdx.y * BN;
    const int st_all = (int)(p.K / kStageK);
    const int st_lo = p.splits > 1 ? (int)blockIdx.z * (p.kb_per_split >> 2) : 0;    // first stage of this split
    const int nst = p.splits > 1 ? min(p.kb_per_split >> 2, st_all - st_lo) : st_all;  // stages of this CTA
    const int sps_shift = p.gs_shift - 5;                                             // log2(stages per 8-group scale slot)
    const int st_per_s = 1 << sps_shift;                                              // 1, 2, 4 for group sizes 32, 64, 128
    const int sl_lo = st_lo >> sps_shift;
    (void)sl_lo;
    // Optional k rotation (GBXQ_TS_ROTATE=1): CTA b walks its stages starting at stage rot(b) and wraps around, so that
    // the CTAs of a grid do not all ask L2 for the same x tile at the same time.  Measured (r02v-r02y): no gain at small
    // batches (the loop is bound by the dequant warps' instruction issue, not by x) and -5 % on prefill tiles, where
    // lock-step CTAs share their x tiles in L2 -- off by default.  The order is fixed per CTA either way: deterministic.
    const int nrot = (p.rotate && nst % st_per_s == 0) ? nst / st_per_s : 1;
    const int rot = (int)(blockIdx.x % (unsigned)nrot) * st_per_s;
    auto stage_of = [&](int s) {  // loop index -> stage of this CTA's k range
        const int t = s + rot;
        return t >= nst ? t - nst : t;
    };

    if (threadIdx.x == 0) TS_STAMP(0);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < XS; s++) {
            mbar_init(&full_b[s], 1);    // x producer (+ tx bytes)
            mbar_init(&empty_b[s], 1);   // tcgen05.commit
        }
#pragma unroll
        for (int s = 0; s < WS; s++) {
            mbar_init(&wfull[s], 1);
            mbar_init(&wempty[s], kDqWarps);
        }
#pragma unroll
        for (int s = 0; s < SS; s++) {
            mbar_init(&sfull[s], 1);
            mbar_init(&sempty[s], kDqWarps);
        }
#pragma unroll
        for (int s = 0; s < AS; s++) {
            mbar_init(&full_a[s], kDqWarps);
            mbar_init(&empty_a[s], 1);   // tcgen05.commit
        }
        mbar_init(tmem_full, 1);
        fence_mbar_init();
    }
    if (warp == 0) {
        if (lane == 0) {
            tma_prefetch_desc(TMAP_X);
            tma_prefetch_desc(TMAP_W);
            tma_prefetch_desc(TMAP_S);
            tma_prefetch_desc(TMAP_B);
        }
        __syncwarp();
        tmem_alloc(tmem_slot, kTmemCols);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) griddep_launch_dependents();  // the next kernel of the stream may start its prologue when SMs free up
    if (threadIdx.x == 0) TS_STAMP(1);

    // The three single-issuer roles below run their loops with the WHOLE warp (uniform control flow, every lane polls
    // the barriers) and elect one lane per asynchronous instruction.  Written as `if (lane == 0) { loop }` each
    // tcgen05.mma cost ~16 SASS instructions (ELECT / R2UR.BROADCAST loops around every operand): ~150 clocks per MMA,
    // 0.77 us per 128-k stage -- the bound of r02r-r02w whatever the code width, the batch or the x / weight streams.
    if (warp == 0) {
        // ===================== x producer =====================
        griddep_wait();  // x belongs to the previous kernels of the stream
        const uint32_t xring_u32 = smem_u32(xring);
        for (int a = 0; a < kAtomsPerStage * nst; a++) {
            const int s = a % XS;
            mbar_wait(&empty_b[s], ((uint32_t)(a / XS) & 1u) ^ 1u);
            if (elect_one()) {
                mbar_arrive_expect_tx(&full_b[s], C::B_BYTES);
                tma_load_2d_u32(xring_u32 + (uint32_t)s * C::B_BYTES, TMAP_X, (kAtomsPerStage * (st_lo + stage_of(a / kAtomsPerStage)) + (a % kAtomsPerStage)) * kAtomK, m0,
                                smem_u32(&full_b[s]));
            }
            __syncwarp();
        }
    } else if (warp == kWarpW) {
        // ===================== packed-weight / scale producer =====================
        if (!p.early_w) griddep_wait();
        const uint32_t wring_b = smem_u32(wring), sring_b = smem_u32(sring);
        for (int s = 0; s < nst; s++) {
#ifndef GBXQ_TS_DIRECT
            if ((s & (st_per_s - 1)) == 0) {
                const int sl = s >> sps_shift, ss = sl % SS;
                mbar_wait(&sempty[ss], ((uint32_t)(sl / SS) & 1u) ^ 1u);
                if (elect_one()) {
                    const int gsl = sl_lo + (stage_of(s) >> sps_shift);  // the slot's place in the matrix
                    mbar_arrive_expect_tx(&sfull[ss], C::S_SLOT);
                    tma_load_2d_u32(sring_b + (uint32_t)ss * C::S_SLOT, TMAP_S, gsl * 8, n0, smem_u32(&sfull[ss]));
                    tma_load_2d_u32(sring_b + (uint32_t)ss * C::S_SLOT + kTileN * 16, TMAP_B, gsl * 8, n0, smem_u32(&sfull[ss]));
                }
                __syncwarp();
            }
#endif
            const int ws = s % WS;
            mbar_wait(&wempty[ws], ((uint32_t)(s / WS) & 1u) ^ 1u);
            if (elect_one()) {
                mbar_arrive_expect_tx(&wfull[ws], C::W_SLOT);
#pragma unroll
                for (int h = 0; h < kH; h++)
                    tma_load_2d_u32(wring_b + (uint32_t)ws * C::W_SLOT + (uint32_t)h * C::W_HALF, TMAP_W,
                                    ((st_lo + stage_of(s)) * kH + h) * 4 * BITS, n0, smem_u32(&wfull[ws]));
            }
            __syncwarp();
        }
    } else if (warp == kWarpMma) {
        // ===================== MMA issuer =====================
        constexpr uint32_t idesc = make_idesc_bf16(kTileN, BN);
        // K-major SWIZZLE_128B descriptor of an x tile: low word = address >> 4 | LBO(1) << 16, high word constant
        constexpr uint32_t kDescHi = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);
        const uint32_t xring_u32 = smem_u32(xring);
        for (int s = 0; s < nst; s++) {
            const int sa = s % AS;
            mbar_wait(&full_a[sa], (uint32_t)(s / AS) & 1u);
#pragma unroll
            for (int a = 0; a < kAtomsPerStage; a++) {
                const int ai = kAtomsPerStage * s + a, ax = ai % XS;
                mbar_wait(&full_b[ax], (uint32_t)(ai / XS) & 1u);
                tc_fence_after();
                const uint32_t b_lo = (((xring_u32 + (uint32_t)ax * C::B_BYTES) & 0x3FFFFu) >> 4) | (1u << 16);
                const uint32_t a_tmem = tmem_base + kTmemAOff + (uint32_t)(sa * (kStageK / 2) + a * 32);
                const uint32_t first = (s | a) != 0 ? 1u : 0u;
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < kAtomK / 16; k++)
                        mma_ts_f16_lohi(tmem_base + (uint32_t)((k % C::NACC) * BN), a_tmem + (uint32_t)(k * 8), b_lo + (uint32_t)(2 * k),
                                        kDescHi, idesc, k >= C::NACC ? 1u : first);
                    mma_commit(&empty_b[ax]);   // the x tile is free once these MMAs retire
                    if (a == kAtomsPerStage - 1) mma_commit(&empty_a[sa]);  // ... and so is the A stage
                }
                __syncwarp();
            }
        }
        if (elect_one()) mma_commit(tmem_full);  // accumulator complete -> epilogue
        __syncwarp();
    } else {
        // ===================== dequant warps (1..16), then epilogue =====================
        const int dw = warp - 1;
        const int rq = warp & 3;                 // TMEM lane quarter this warp may touch (hardware: warp id % 4)
        const int kq = dw >> 2;                  // k quarter of the stage
        const int r = rq * 32 + lane;            // tile row = TMEM lane
        const uint32_t wring_u32 = smem_u32(wring), sring_u32 = smem_u32(sring);
        const uint32_t a_lane = tmem_base + kTmemAOff + ((uint32_t)(rq * 32) << 16) + (uint32_t)(kq * 16);
        uint4 sreg = make_uint4(0u, 0u, 0u, 0u), breg = sreg;
        (void)sreg; (void)breg;
        // Software pipeline over the stages: the tcgen05.st of stage s is only waited for (and the stage handed to the
        // MMA warp) after the ALU work of stage s+1, and the packed words of stage s+1 are fetched from shared memory
        // while the store of stage s is in flight -- a warp's per-stage latency chain is its ~80 ALU instructions, not
        // load + ALU + store round trip (r02r: 0.8 us per stage with the serial chain).
        // Ring positions advance by increments (no divisions in the loop): fetch side (f*) runs one stage ahead of the
        // compute side (c*).  sin = stage inside its 8-group scale slot (the rotation keeps whole slots together).
        uint32_t w[kH][BITS];
        const int sps_mask = st_per_s - 1;
        const int gl_shift = 8 - p.gs_shift;                 // groups per stage = 1 << gl_shift
        int gl_base[kH];                                     // this thread's group inside the stage, per half
#pragma unroll
        for (int h = 0; h < kH; h++) gl_base[h] = (h * kHalfK + kq * 32) >> p.gs_shift;
        uint32_t f_w = wring_u32, f_s = sring_u32 + (uint32_t)r * 16u;
        uint32_t f_wbar = smem_u32(wfull), f_sbar = smem_u32(sfull);
        uint32_t f_wph = 0, f_sph = 0;
        int f_ws = 0, f_ss = 0, f_sin = 0;
        (void)f_s; (void)f_sbar; (void)f_sph; (void)f_ss;
#ifdef GBXQ_TS_DIRECT
        int f_idx = 0;
        uint32_t d_s[kH], d_b[kH];                           // the stage's raw scale / bias per half
        const bool d_row = (int64_t)n0 + r < P_N;
        const int64_t d_off = ((int64_t)n0 + r) * p.G;
#endif
        auto fetch = [&]() {
#ifdef GBXQ_TS_DIRECT
            {
                const int k0 = (st_lo + stage_of(f_idx)) * kStageK + kq * 32;
#pragma unroll
                for (int h = 0; h < kH; h++) {
                    const int64_t at = d_off + ((k0 + h * kHalfK) >> p.gs_shift);
                    d_s[h] = d_row ? (uint32_t)__ldg(p.s_raw + at) : 0u;
                    d_b[h] = d_row ? (uint32_t)__ldg(p.b_raw + at) : 0u;
                }
                f_idx++;
            }
#endif
            mbar_wait_u32(f_wbar + 8u * f_ws, f_wph);
#pragma unroll
            for (int h = 0; h < kH; h++) load_codes<BITS>(f_w + (uint32_t)f_ws * C::W_SLOT + (uint32_t)h * C::W_HALF, r, kq, w[h]);
#ifndef GBXQ_TS_DIRECT
            if (f_sin == 0) {
                mbar_wait_u32(f_sbar + 8u * f_ss, f_sph);
                sreg = lds128(f_s + (uint32_t)f_ss * C::S_SLOT);
                breg = lds128(f_s + (uint32_t)f_ss * C::S_SLOT + kTileN * 16u);
                if (++f_ss == SS) { f_ss = 0; f_sph ^= 1u; }
            }
#endif
            f_sin = (f_sin + 1) & sps_mask;
            if (++f_ws == WS) { f_ws = 0; f_wph ^= 1u; }
        };
        const uint32_t fa_bar = smem_u32(full_a), ea_bar = smem_u32(empty_a), we_bar = smem_u32(wempty), se_bar = smem_u32(sempty);
        int c_ws = 0, c_ss = 0, c_sin = 0, c_sa = 0;
        uint32_t c_aph = 1u;                                 // parity of "stage free" (fresh barriers pass a wait on 1)
        if (nst > 0) fetch();
        for (int s = 0; s < nst; s++) {
            uint32_t v[kH][16];
#pragma unroll
            for (int h = 0; h < kH; h++) {
                const int gl = (c_sin << gl_shift) + gl_base[h];  // group inside the 8-group slot
#ifdef GBXQ_TS_DIRECT
                const uint32_t sraw = d_s[h], braw = d_b[h];
                (void)gl;
#else
                const uint32_t sraw = pick16(sreg, gl), braw = pick16(breg, gl);
#endif
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    uint32_t o[4];
                    dequant8<BITS, BITS>(w[h], c, sraw, braw, o);
                    v[h][4 * c] = o[0]; v[h][4 * c + 1] = o[1]; v[h][4 * c + 2] = o[2]; v[h][4 * c + 3] = o[3];
                }
            }
            if (s > 0) {  // stage s-1: its store has had the whole dequantisation above to complete
                tmem_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_u32(fa_bar + 8u * (uint32_t)((c_sa + AS - 1) & (AS - 1)));
            }
            mbar_wait_u32(ea_bar + 8u * c_sa, c_aph);        // the MMAs that read this stage have retired
            tc_fence_after();
#pragma unroll
            for (int h = 0; h < kH; h++) tmem_st16(a_lane + (uint32_t)(c_sa * (kStageK / 2) + h * (kHalfK / 2)), v[h]);
            __syncwarp();
            if (lane == 0) {
                mbar_arrive_u32(we_bar + 8u * c_ws);         // the packed words of stage s were consumed above
#ifndef GBXQ_TS_DIRECT
                if (c_sin == sps_mask || s == nst - 1) mbar_arrive_u32(se_bar + 8u * c_ss);  // ... and the slot's scales
#endif
            }
            if (c_sin == sps_mask) { if (++c_ss == SS) c_ss = 0; }
            c_sin = (c_sin + 1) & sps_mask;
            if (++c_ws == WS) c_ws = 0;
            if (++c_sa == AS) { c_sa = 0; c_aph ^= 1u; }
            if (s + 1 < nst) fetch();
        }
        if (nst > 0) {
            tmem_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_u32(fa_bar + 8u * (uint32_t)((c_sa + AS - 1) & (AS - 1)));
        }

        // ---- epilogue: TMEM -> registers -> bf16 -> y[m, n]; warp drains its lane quarter and column quarter
        mbar_wait(tmem_full, 0);
        if (threadIdx.x == 32) TS_STAMP(2);
        tc_fence_after();
        griddep_wait();  // y may still be read by an earlier kernel of the stream
        const int er = rq * 32 + lane;
        const int64_t n = (int64_t)n0 + er;
        const bool row_ok = n < P_N;
        const float bias_f = (P_BIAS != nullptr && row_ok) ? __bfloat162float(P_BIAS[n]) : 0.f;
        constexpr int QCOLS = BN / 4;
        constexpr int STEP = QCOLS >= 32 ? 32 : (QCOLS >= 16 ? 16 : (QCOLS >= 8 ? 8 : 4));
        const int cq = dw >> 2;
#pragma unroll 1
        for (int c0 = cq * QCOLS; c0 < (cq + 1) * QCOLS; c0 += STEP) {
            uint32_t v[32];
            tmem_ld<STEP>(tmem_base + ((uint32_t)(rq * 32) << 16) + (uint32_t)c0, v);
#pragma unroll
            for (int j = 1; j < C::NACC; j++) {  // fixed order: deterministic
                uint32_t u[32];
                tmem_ld<STEP>(tmem_base + ((uint32_t)(rq * 32) << 16) + (uint32_t)(j * BN + c0), u);
#pragma unroll
                for (int i = 0; i < STEP; i++) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(u[i]));
            }
            if (row_ok) {
#pragma unroll
                for (int j = 0; j < STEP; j++) {
                    const int64_t m = (int64_t)m0 + c0 + j;
                    if (m < p.M) {
                        if (p.splits > 1) {
                            P_WS[((size_t)blockIdx.z * p.M + m) * P_N + n] = __uint_as_float(v[j]);
                        } else {
                            float f = __bfloat162float(__float2bfloat16_rn(__uint_as_float(v[j])));
                            if (P_BIAS != nullptr) f = __fadd_rn(f, bias_f);
                            P_Y[(size_t)m * P_N + n] = __float2bfloat16_rn(f);
                        }
                    }
                }
            }
        }
        tc_fence_before();
        if (p.splits > 1) {
            // the last split to arrive at this tile's counter adds the partial tiles in split order and writes y
            __threadfence();
            asm volatile("bar.sync 2, %0;" ::"n"(kDqWarps * 32) : "memory");
            uint32_t* flag = tmem_slot + 1;
            const uint32_t tile = blockIdx.y * gridDim.x + blockIdx.x;
            if (warp == 1 && lane == 0) *flag = atomicAdd(p.cnt + tile, 1u) == (uint32_t)p.splits - 1u ? 1u : 0u;
            asm volatile("bar.sync 2, %0;" ::"n"(kDqWarps * 32) : "memory");
            if (*flag != 0u) {
                __threadfence();
                if (row_ok) {
                    for (int c = cq * QCOLS; c < (cq + 1) * QCOLS; c++) {
                        const int64_t m = (int64_t)m0 + c;
                        if (m < p.M) {
                            float acc = 0.f;
                            for (int z = 0; z < p.splits; z++) acc += __ldcg(P_WS + ((size_t)z * p.M + m) * P_N + n);
                            float f = __bfloat162float(__float2bfloat16_rn(acc));
                            if (P_BIAS != nullptr) f = __fadd_rn(f, bias_f);
                            P_Y[(size_t)m * P_N + n] = __float2bfloat16_rn(f);
                        }
                    }
                }
                if (warp == 1 && lane == 0) p.cnt[tile] = 0u;  // left zero for the next launch
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) TS_STAMP(3);
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

#ifndef GBXQ_TS_GROUPED
struct Maps {
    CUtensorMap x, w, s, b;
};

template <int BITS, int BN>
int launch_inst(const Maps& mp, const TsParams& p, cudaStream_t st) {
    constexpr size_t smem = Cfg<BITS, BN>::SMEM;
    static_assert(smem <= 227 * 1024, "shared memory budget");
    constexpr auto kern = TS_KERNEL<BITS, BN>;
    const int rc = allow_dynamic_smem<kern>((int)smem);
    if (rc != GBXQ_OK) return rc;
    const dim3 grid((unsigned)((p.N + kTileN - 1) / kTileN), (unsigned)((p.M + BN - 1) / BN), (unsigned)(p.splits > 1 ? p.splits : 1));
    return launch(kern, grid, dim3(kThreads), smem, st, true, mp.x, mp.w, mp.s, mp.b, p);
}

template <int BITS>
int launch_bn(int bn, const Maps& mp, const TsParams& p, cudaStream_t st) {
    switch (bn) {
        case 16: return launch_inst<BITS, 16>(mp, p, st);
        case 32: return launch_inst<BITS, 32>(mp, p, st);
        case 64: return launch_inst<BITS, 64>(mp, p, st);
        case 128: return launch_inst<BITS, 128>(mp, p, st);
        default: return launch_inst<BITS, 256>(mp, p, st);
    }
}

unsigned long long* g_ts_dbg = nullptr;

int pick_bn(int64_t M) { return M <= 16 ? 16 : (M <= 32 ? 32 : (M <= 64 ? 64 : (M <= 128 ? 128 : 256))); }

}  // namespace

#ifndef GBXQ_TS_DIRECT
void gemm_ts_debug_timeline(unsigned long long* buf) { g_ts_dbg = buf; }

bool gemm_ts_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                       const void* y) {
    if (dtype != GBXQ_BF16 || M < 1 || N < 1) return false;
    if (K % kStageK) return false;              // whole 256-k stages
    if ((K * bits / 8) % 16) return false;      // TMA: packed row pitch must be a multiple of 16 bytes
    if (((uintptr_t)x | (uintptr_t)w) & 15) return false;
    if ((uintptr_t)y & 1) return false;
    if (M > (int64_t)1 << 24 || (N + kTileN - 1) / kTileN > 65535 * 32) return false;
    return tma_encode_available();
}

#endif

int TS_LAUNCH(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M, int64_t N,
              int64_t K, int bits, int gs, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    if (!tma_encode_available()) return GBXQ_EUNSUPPORTED;
#ifndef GBXQ_TS_DIRECT
    // a row of scales that is no legal TMA row pitch (or unaligned scale tensors): the direct-scale variant
    if (((((uintptr_t)s | (uintptr_t)b) & 15) != 0) || (((K / gs) * 2) % 16 != 0))
        return launch_gemm_ts_direct(x, w, s, b, bias, y, M, N, K, bits, gs, workspace, workspace_bytes, st);
#endif
    const int bn = pick_bn(M);
    if ((M + bn - 1) / bn > 65535) return GBXQ_EUNSUPPORTED;
    Maps mp;
    const uint64_t words = (uint64_t)(K * bits / 32), G = (uint64_t)(K / gs);
    const int swz = bits == 4 ? 64 : (bits == 2 ? 32 : (bits == 8 ? 128 : 0));
    bool ok = encode_tensor_map_2d_sw(&mp.x, 0, x, (uint64_t)K, (uint64_t)M, (uint64_t)K * 2, kAtomK, (uint32_t)bn, 128);
    ok = ok && encode_tensor_map_2d_sw(&mp.w, 1, w, words, (uint64_t)N, words * 4, (uint32_t)(4 * bits), kTileN, swz);
#ifdef GBXQ_TS_DIRECT
    mp.s = mp.w;  // never used
    mp.b = mp.w;
    (void)G;
#else
    ok = ok && encode_tensor_map_2d_sw(&mp.s, 0, s, G, (uint64_t)N, G * 2, 8, kTileN, 0);
    ok = ok && encode_tensor_map_2d_sw(&mp.b, 0, b, G, (uint64_t)N, G * 2, 8, kTileN, 0);
#endif
    if (!ok) return GBXQ_EUNSUPPORTED;
    TsParams p{};
    p.bias = reinterpret_cast<const __nv_bfloat16*>(bias);
    p.y = reinterpret_cast<__nv_bfloat16*>(y);
    p.M = M;
    p.N = N;
    p.K = K;
    p.gs_shift = gs == 32 ? 5 : (gs == 64 ? 6 : 7);
    p.splits = 1;
    p.early_w = pdl_early_weights();
    p.w_raw = reinterpret_cast<const uint8_t*>(w);
    p.row_bytes = K * bits / 8;
    static const int rotate = env_int("GBXQ_TS_ROTATE", 0);
    p.rotate = rotate;
#ifdef GBXQ_TS_DIRECT
    p.s_raw = reinterpret_cast<const uint16_t*>(s);
    p.b_raw = reinterpret_cast<const uint16_t*>(b);
    p.G = (int64_t)(K / gs);
#endif
    p.dbg = g_ts_dbg;
    g_ts_dbg = nullptr;  // one launch
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

#else  // GBXQ_TS_GROUPED: host side of the grouped launch

template <int BITS, int BN>
int launch_inst(const TsMaps& mp, const TsParams& p, int tiles, cudaStream_t st) {
    constexpr size_t smem = Cfg<BITS, BN>::SMEM;
    constexpr auto kern = TS_KERNEL<BITS, BN>;
    const int rc = allow_dynamic_smem<kern>((int)smem);
    if (rc != GBXQ_OK) return rc;
    const dim3 grid((unsigned)tiles, (unsigned)((p.M + BN - 1) / BN), (unsigned)(p.splits > 1 ? p.splits : 1));
    return launch(kern, grid, dim3(kThreads), smem, st, true, mp, p);
}

template <int BITS>
int launch_bn(int bn, const TsMaps& mp, const TsParams& p, int tiles, cudaStream_t st) {
    switch (bn) {
        case 16: return launch_inst<BITS, 16>(mp, p, tiles, st);
        case 32: return launch_inst<BITS, 32>(mp, p, tiles, st);
        case 64: return launch_inst<BITS, 64>(mp, p, tiles, st);
        case 128: return launch_inst<BITS, 128>(mp, p, tiles, st);
        default: return launch_inst<BITS, 256>(mp, p, tiles, st);
    }
}
}  // namespace

// The padded output width the split-K plan and the workspace of a grouped launch are sized for.
int64_t gemm_ts_grouped_npad(const gbxq_segment* segs, int nseg) {
    int64_t tiles = 0;
    for (int i = 0; i < nseg; i++) tiles += (segs[i].N + kTileN - 1) / kTileN;
    return tiles * kTileN;
}

// Returns GBXQ_EUNSUPPORTED (nothing enqueued) when the segments cannot share one launch.
int launch_gemm_ts_grouped(const gbxq_segment* segs, int nseg, const void* x, int64_t M, int64_t K, void* workspace,
                           size_t workspace_bytes, cudaStream_t st) {
    if (nseg < 2 || nseg > 3 || M < 1 || !tma_encode_available()) return GBXQ_EUNSUPPORTED;
    const int bits = segs[0].bits, gs = segs[0].group_size;
    if (K % kStageK || (K * bits / 8) % 16 || ((K / gs) * 2) % 16 || ((uintptr_t)x & 15)) return GBXQ_EUNSUPPORTED;
    const int bn = M <= 16 ? 16 : (M <= 32 ? 32 : (M <= 64 ? 64 : (M <= 128 ? 128 : 256)));
    if ((M + bn - 1) / bn > 65535) return GBXQ_EUNSUPPORTED;
    TsMaps mp;
    TsParams p{};
    const uint64_t words = (uint64_t)(K * bits / 32), G = (uint64_t)(K / gs);
    const int swz = bits == 4 ? 64 : (bits == 2 ? 32 : (bits == 8 ? 128 : 0));
    bool ok = encode_tensor_map_2d_sw(&mp.x, 0, x, (uint64_t)K, (uint64_t)M, (uint64_t)K * 2, kAtomK, (uint32_t)bn, 128);
    int tiles = 0;
    int64_t nsum = 0;
    for (int i = 0; i < nseg; i++) {
        const gbxq_segment& sg = segs[i];
        if (sg.bits != bits || sg.group_size != gs || sg.N < 1) return GBXQ_EUNSUPPORTED;
        if (((uintptr_t)sg.qweight | (uintptr_t)sg.scales | (uintptr_t)sg.biases) & 15) return GBXQ_EUNSUPPORTED;
        if ((uintptr_t)sg.y & 1) return GBXQ_EUNSUPPORTED;
        ok = ok && encode_tensor_map_2d_sw(&mp.w[i], 1, sg.qweight, words, (uint64_t)sg.N, words * 4, (uint32_t)(4 * bits), kTileN, swz);
        ok = ok && encode_tensor_map_2d_sw(&mp.s[i], 0, sg.scales, G, (uint64_t)sg.N, G * 2, 8, kTileN, 0);
        ok = ok && encode_tensor_map_2d_sw(&mp.b[i], 0, sg.biases, G, (uint64_t)sg.N, G * 2, 8, kTileN, 0);
        p.tile0[i] = tiles;
        p.seg_n[i] = sg.N;
        p.seg_bias[i] = reinterpret_cast<const __nv_bfloat16*>(sg.bias);
        p.seg_y[i] = reinterpret_cast<__nv_bfloat16*>(sg.y);
        tiles += (int)((sg.N + kTileN - 1) / kTileN);
        nsum += sg.N;
    }
    for (int i = nseg; i < 3; i++) {
        mp.w[i] = mp.w[0];
        mp.s[i] = mp.s[0];
        mp.b[i] = mp.b[0];
    }
    p.tile0[nseg] = tiles;
    if (!ok || tiles > 65535 * 32) return GBXQ_EUNSUPPORTED;
    p.nseg = nseg;
    p.M = M;
    p.N = nsum;
    p.K = K;
    p.gs_shift = gs == 32 ? 5 : (gs == 64 ? 6 : 7);
    p.splits = 1;
    p.early_w = pdl_early_weights();
    p.rotate = 0;
    p.dbg = nullptr;
    {
        int sp, per;
        size_t need;
        gemm_split_plan(M, (int64_t)tiles * kTileN, K, &sp, &per, &need);
        if (sp > 1 && workspace != nullptr && workspace_bytes >= need && !((uintptr_t)workspace & 15)) {
            p.splits = sp;
            p.kb_per_split = per;
            p.cnt = reinterpret_cast<uint32_t*>(workspace);
            p.ws = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + kCntBytes);
            int64_t off = 0;
            for (int i = 0; i < nseg; i++) {
                p.seg_ws_off[i] = off;
                off += (int64_t)sp * M * segs[i].N;
            }
        }
    }
    switch (bits) {
        case 2: return launch_bn<2>(bn, mp, p, tiles, st);
        case 3: return launch_bn<3>(bn, mp, p, tiles, st);
        case 4: return launch_bn<4>(bn, mp, p, tiles, st);
        case 6: return launch_bn<6>(bn, mp, p, tiles, st);
        case 8: return launch_bn<8>(bn, mp, p, tiles, st);
    }
    return GBXQ_EINVAL_BITS;
}

#endif  // GBXQ_TS_GROUPED

}  // namespace gbxq
