// gbxq_mmv8_body.cuh -- device body of the integer tensor-pipe decode kernel, shared by the single-layer launch
// (gbxq_mmv8.cu) and the grouped q|k|v / gate|up launch (gbxq_mmv8_grouped.cu).  See gbxq_mmv8.cu for the design.
#pragma once
#include "gbxq_common.cuh"


namespace gbxq {
namespace mmv8 {

#ifndef GBXQ_MMV8_CW
#define GBXQ_MMV8_CW 16
#endif
// consumer warps: 16 = one CTA per SM (default since r02p/r02q: the x -> digit conversion is done once per SM instead of
// once per co-resident CTA: down_proj K = 14336 10.1 -> 9.0 us, 70B step 0.69 -> 0.72, bpw-2.2 0.31 -> 0.35), 8 = two
// CTAs per SM (-DGBXQ_MMV8_CW=8: the round-1 geometry, 0.8 us faster on a lone 14336 x 4096 launch)
constexpr int kCW = GBXQ_MMV8_CW;
constexpr int kWide = kCW / 8;                // shared memory, stage and ring budgets scale with the CTA
constexpr int kSmemCap = 110 * 1024 * kWide;
constexpr int kThreads = (kCW + 1) * 32;      // + producer warp
constexpr int kMaxStages = 8;                // barrier slots; one-call launches plan at most kPlanStages
constexpr int kPlanStages = GBXQ_MMV8_CW == 16 ? 3 : 4;  // r03s/r03t: three (larger-share) stages 0.526 vs 0.522 on the 8B step
constexpr int kArMaxCtas = GBXQ_RP_MAX_CTAS;
#ifndef GBXQ_MMV8_MINCTAS
#define GBXQ_MMV8_MINCTAS (GBXQ_MMV8_CW == 8 ? 2 : 1)
#endif
constexpr int kMinCtas = GBXQ_MMV8_MINCTAS;    // register cap 112; a cap of 72 (3 CTAs / SM) measured 15 % slower
constexpr int S = 4;                          // group slices per chunk column (= 8 columns / 2 digits)
constexpr int W = 4;                          // weight rows per MMA set (= 16 A rows / S)

__device__ __forceinline__ void imma16832(int (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                          uint32_t b1, const int (&c)[4]) {
    asm("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%12,%13};"
        : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "r"(c[0]), "r"(c[1]), "r"(c[2]), "r"(c[3]));
}
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// timeline stamps (development aid): CTA 0 only, or every CTA (dbg_all: 8 slots per CTA, slot 5 = %smid)
#define STAMP(i)                                                                                   \
    do {                                                                                           \
        if (p.dbg != nullptr && threadIdx.x == 0 && (p.dbg_all != 0 || blockIdx.x == 0))           \
            p.dbg[(p.dbg_all != 0 ? (size_t)blockIdx.x * 8 : 0) + (i)] = gtime();                  \
    } while (0)

template <int NWORD> __device__ __forceinline__ void lds_words(const uint8_t* addr, uint32_t (&w)[NWORD]) {
    if constexpr (NWORD == 1) {
        w[0] = *reinterpret_cast<const uint32_t*>(addr);
    } else if constexpr (NWORD == 2) {
        const uint2 v = *reinterpret_cast<const uint2*>(addr);
        w[0] = v.x; w[1] = v.y;
    } else {
#pragma unroll
        for (int i = 0; i < NWORD / 4; i++) {
            const uint4 v = *reinterpret_cast<const uint4*>(addr + 16 * i);
            w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w;
        }
    }
}
__device__ __forceinline__ float lds_bf16(const uint8_t* addr) {
    return __uint_as_float((uint32_t)(*reinterpret_cast<const uint16_t*>(addr)) << 16);
}

// ---- packing geometry.  A thread chunk = CQ = group_size/4 codes of one (row, group).  NMMA MMAs per chunk and
//      accumulator class; MMA u of class c takes A registers areg(c, u, 0) [k-slots 4t..4t+3] and areg(c, u, 1)
//      [k-slots 16+4t..]; byte i of such a register is code code_of(c, u, half, i) of the chunk.
//      The 3- and 6-bit packings (codes straddle bytes and words: quantized_linear_gba.py:61, 8 codes / 3 bytes and
//      4 codes / 3 bytes) are realigned to one byte per code right after the shared-memory load (load_chunk) and run
//      through the 8-bit geometry from there: EB = the width of a code once it sits in registers.
template <int BITS, int CQ> struct Geo {
    static constexpr int EB = (BITS == 3 || BITS == 6) ? 8 : BITS;
    static constexpr int NWORD = CQ * EB / 32;
    static constexpr int NCLASS = EB == 8 ? 1 : 2;
    static constexpr int NREG = CQ / 4;                    // A registers (4 codes each) per chunk
    static constexpr int NMMA = (NREG / NCLASS + 1) / 2;   // k32 MMAs per class (a lone register pairs with zero)
    static constexpr bool HALF = (NREG / NCLASS) % 2 == 1; // last MMA of a class has no second register
    static constexpr int CMUL = EB == 8 ? 1 : (EB == 4 ? 16 : 4);  // T = CMUL * D0 + D1; scale / CMUL
    __host__ __device__ static constexpr int code_of(int c, int u, int half, int i) {
        if (EB == 8) return 8 * u + 4 * half + i;                         // word 2u+half, byte i
        if (EB == 4) return 16 * u + 8 * half + 2 * i + c;                // word 2u+half, nibble 2i+c
        return 16 * u + 4 * i + 2 * half + c;                             // 2-bit: word u, field 4i + 2*half + c
    }
};

template <int BITS, int CQ>
__device__ __forceinline__ uint32_t areg(const uint32_t (&w)[Geo<BITS, CQ>::NWORD], int c, int u, int half) {
    if constexpr (Geo<BITS, CQ>::EB == 8) {
        return w[2 * u + half];
    } else if constexpr (BITS == 4) {
        const uint32_t word = w[2 * u + half];
        return c == 0 ? (word & 0x0f0f0f0fu) : (word & 0xf0f0f0f0u);
    } else {
        const uint32_t word = half == 0 ? w[u] : (w[u] >> 4);
        return c == 0 ? (word & 0x03030303u) : (word & 0x0c0c0c0cu);
    }
}

// bits [pos, pos + 32) of a little-endian word stream (only as many as the caller masks are meaningful)
template <int NR> __device__ __forceinline__ uint32_t bit_window(const uint32_t (&r)[NR], int pos) {
    const int i = pos >> 5, off = pos & 31;
    if (off == 0) return r[i];
    if (i + 1 < NR) return __funnelshift_r(r[i], r[i + 1], off);
    return r[i] >> off;
}
// four 3-bit fields (bits 0..11 of x) -> one byte each.  Even and odd fields are spread by one multiply each (the
// shifted copies do not overlap, so the adds inside the multiply carry nothing) and masked into place.
__device__ __forceinline__ uint32_t spread3(uint32_t x) {
    const uint32_t e = (x & 0x1c7u) * 0x401u;    // f0 @0, f2 @6 | f0 @10, f2 @16
    const uint32_t o = (x & 0xe38u) * 0x8020u;   // f1 @8, f3 @14 | f1 @18, f3 @24
    return (e & 0x00070007u) | (o & 0x07000700u);
}
// four 6-bit fields (bits 0..23 of x) -> one byte each
__device__ __forceinline__ uint32_t spread6(uint32_t x) {
    return (x & 0x3fu) | ((x << 2) & 0x3f00u) | ((x << 4) & 0x3f0000u) | ((x << 6) & 0x3f000000u);
}

// The thread chunk at shared-memory address `addr` as A-operand words: packed words as they are for 2/4/8-bit,
// one byte per code for 3/6-bit.  3-bit chunks of 16 codes are 6 bytes long and only 2-byte aligned.
template <int BITS, int CQ>
__device__ __forceinline__ void load_chunk(const uint8_t* addr, uint32_t (&w)[Geo<BITS, CQ>::NWORD]) {
    if constexpr (BITS == 3 || BITS == 6) {
        constexpr int RAWB = CQ * BITS / 8;           // 6, 12 (3-bit) or 12, 24 (6-bit) bytes
        constexpr int NR = (RAWB + 3) / 4 + (RAWB % 4 ? 0 : 0);
        uint32_t r[RAWB == 6 ? 2 : NR];
        if constexpr (RAWB == 6) {
            const uintptr_t a = reinterpret_cast<uintptr_t>(addr);
            const uint32_t* al = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
            const uint32_t r0 = al[0], r1 = al[1];
            const uint32_t sh = (uint32_t)(a & 3) * 8u;  // 0 or 16
            r[0] = __funnelshift_r(r0, r1, sh);
            r[1] = r1 >> sh;
        } else {
#pragma unroll
            for (int i = 0; i < NR; i++) r[i] = reinterpret_cast<const uint32_t*>(addr)[i];
        }
#pragma unroll
        for (int j = 0; j < CQ / 4; j++) {
            if constexpr (BITS == 3) w[j] = spread3(bit_window(r, 12 * j));
            else w[j] = spread6(bit_window(r, 24 * j));
        }
    } else {
        lds_words<Geo<BITS, CQ>::NWORD>(addr, w);
    }
}

struct Mmv8Params {
    const __nv_bfloat16* x;
    const uint8_t* w;
    const uint16_t* scales;
    const uint16_t* biases;
    const __nv_bfloat16* bias;
    __nv_bfloat16* y;
    int64_t N, K;
    int M;                // rows of x in this launch (<= MT)
    int G;                // groups per row
    uint32_t row_bytes;
    int nch;              // chunk columns per row (a chunk column = S groups)
    int cw, rg;           // warp grid: cw chunk columns x rg row groups (cw * rg <= 8)
    int tr;               // rows per ring stage (= rg * R)
    int stages;
    uint32_t slot_bytes;  // ring slot size
    uint32_t sb_off;      // offset of the scales inside a slot (biases follow at sb_off + tr*G*2)
    int early_weights;    // 1: weights are immutable while the call is in flight -> stream them before griddepcontrol.wait
    int row_unit;         // rows are shared out in units of 1 row, or of 4 rows when a row of scales is only 8-byte aligned
    unsigned long long* dbg;  // optional timeline (gbxq_debug_timeline): 8 globaltimer stamps per launch, CTA 0 / warp 0
    int dbg_all;              // 1: every CTA stamps (8 slots per CTA)
    int pre_stages;           // > 0: the producer issues only this many stages until the activations have been read
    int rows_base, rows_rem;  // CTA b owns rows_base + (b < rows_rem) rows starting at b*rows_base + min(b, rows_rem)
    int spr0, spr1;           // rows per stage for CTAs with rows_base / rows_base+1 rows (balanced, whole MMA sets)
};

// Fused row-parallel all-reduce (world > 1, one-call launches only): every CTA pushes the fp32 partial sums of ITS rows
// into every peer's staging buffer over NVLink and adds the `world` partials of its rows in rank order (bitwise identical
// on all ranks).  Low-latency protocol: a partial travels as ONE 8-byte store {fp32 bits, epoch}; the receiver polls the
// word itself until the epoch matches -- no fence, no separate flag, one NVLink one-way latency per exchange.
// Staging of rank d: [2 halves (epoch parity)][world][M][N] 8-byte words, zeroed once; `flags` of the own rank: control
// words {epoch, CTAs done, error} at [world * kArMaxCtas] (device-resident epoch: CUDA-graph replayable).
struct ArParams {
    unsigned long long* stage[8];
    uint32_t* flags[8];
    int64_t half_elems;
    int world, rank;
};

// State a persistent chain launch (gbxq_stream.cu) carries from one call to the next: the ring position and the
// device-wide completion counters that order the calls (x of a call may be the y of any earlier one).
struct StreamCtx {
    int s;                      // ring slot of the next stage
    uint32_t phase;             // its parity
    const unsigned* wait_cnt;   // counter that must reach wait_target before x is read / y is written (nullptr: none)
    unsigned wait_target;
    unsigned* done_cnt;         // incremented once by this CTA when its part of y is in global memory
    unsigned* err;              // set to 1 when a wait timed out (the launch then runs to its end unordered)
    bool dead;                  // thread 0: a wait has timed out, stop waiting
};

__device__ __forceinline__ void consumer_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kCW * 32) : "memory"); }
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// BITS, GS = group size, MT = tokens (1, 2, 4), CPW = chunk columns per warp, R = rows per warp and stage (4 or 8).
// STREAM = false: the whole CTA of a one-call launch (barrier set-up, producer warp, consumers, epilogue).
// STREAM = true: one call of a persistent chain, entered by the kCW consumer warps only; barriers (empty barriers
// initialised to kCW arrivals) and the producer live in the caller, `sc` carries the ring position.
// PARTIAL: the row ends in the middle of a chunk column (G % 4 == 2; tensor-parallel K shards).  A separate instantiation:
// compiled into the common kernels the three extra predicates cost the 8B step 1.7 % (r03i: 0.5221 -> 0.5134).
template <int BITS, int GS, int MT, int CPW, int R, bool STREAM = false, bool PARTIAL = false>
__device__ __forceinline__ void mmv8_body(const Mmv8Params& p, const int bid, uint8_t* smem, StreamCtx* sc = nullptr,
                                          const ArParams* ar = nullptr) {
    const bool ar_on = !STREAM && ar != nullptr && ar->world > 1;
    constexpr int CQ = GS / 4;
    using GE = Geo<BITS, CQ>;
    constexpr int NWORD = GE::NWORD, NCLASS = GE::NCLASS, NMMA = GE::NMMA;
    constexpr int TB = CQ * BITS / 8;        // bytes per thread chunk
    constexpr int NSET = R / W;
    constexpr int KSTEP_B = S * 4 * TB;      // bytes of one weight row inside a chunk column
    constexpr int LPR = 32 / R;              // lanes per row in the bias dot product
    constexpr int NGL = (CPW * S + LPR - 1) / LPR;
    static_assert(R % W == 0 && NWORD >= 1, "geometry");

    // layout: [ring stages * slot][full/empty barriers (2*kMaxStages)][xsc kCW * CPW*S*MT f32][ysum rows * 2cw * MT f32]
    uint8_t* ring = smem;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(ring + (size_t)p.stages * p.slot_bytes);
    uint64_t* empty_bar = full_bar + kMaxStages;
    float* xsc = reinterpret_cast<float*>(empty_bar + kMaxStages);
    uint32_t* ar_epoch_s = reinterpret_cast<uint32_t*>(&empty_bar[kMaxStages - 1]);  // scratch (one-call plans use < kMaxStages stages)
    float* ysum = xsc + kCW * (CPW * S * MT);

    STAMP(0);
    const bool extra = bid < p.rows_rem;
    const int64_t r0 = (int64_t)bid * p.rows_base + (int64_t)(extra ? bid : p.rows_rem) * p.row_unit;
    const int rows = p.rows_base + (extra ? p.row_unit : 0);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int nstg = p.stages;
    const int spr = extra ? p.spr1 : p.spr0;
    const int active_warps = p.cw * p.rg;
    const int slots = 2 * p.cw;

    if constexpr (!STREAM) {
        if (threadIdx.x == 0) {
            for (int s = 0; s < nstg; s++) {
                mbar_init(&full_bar[s], 1);
                mbar_init(&empty_bar[s], active_warps);
            }
            mbar_init(&full_bar[kMaxStages - 1], active_warps);  // "activations read" (plans use < kMaxStages stages)
            fence_mbar_init();
        }
        __syncthreads();
        if (threadIdx.x == 0) griddep_launch_dependents();  // the next kernel of the stream may become resident now
    } else {
        // every earlier call this one depends on must be complete on ALL CTAs before x is read or y overwritten
        if (threadIdx.x == 0 && sc->wait_cnt != nullptr && !sc->dead) {
            const unsigned long long t0 = gtime();
            while (ld_acquire_gpu(sc->wait_cnt) < sc->wait_target) {
                if (gtime() - t0 > 2000000000ull) {  // 2 s: a CTA of the grid is not resident; never hang the device
                    atomicExch(sc->err, 1u);
                    sc->dead = true;
                    break;
                }
            }
            __threadfence();
        }
        consumer_bar();
        STAMP(5);
    }
    int s = 0;
    uint32_t phase = 0;
    if constexpr (STREAM) {
        s = sc->s;
        phase = sc->phase;
    }

    if (!STREAM && warp == kCW) {
        // ===================== producer warp: one elected lane drives the TMA engine =====================
        if (lane == 0 && rows > 0) {
            if (!p.early_weights) griddep_wait();
            const uint8_t* wsrc = p.w + (uint64_t)r0 * p.row_bytes;
            const uint32_t g2 = (uint32_t)p.G * 2u;
            int issued = 0;
            for (int ra = 0; ra < rows; ra += spr) {
                // hold the stream back while the consumers fetch the activations: with every SM's ring filling, a load
                // that hits in L2 takes ~1 us instead of ~0.3 us (profiles/r02a_timeline_allcta.txt: waited -> x)
                if (p.pre_stages > 0 && issued++ == p.pre_stages) mbar_wait(&full_bar[kMaxStages - 1], 0u);
                mbar_wait(&empty_bar[s], phase ^ 1u);
                int nr = rows - ra;
                if (nr > spr) nr = spr;
                const uint32_t wbytes = (uint32_t)nr * p.row_bytes;
                const uint32_t sbytes = (uint32_t)nr * g2;
                uint8_t* slot = ring + (size_t)s * p.slot_bytes;
                mbar_arrive_expect_tx(&full_bar[s], wbytes + 2u * sbytes);
                bulk_g2s(slot, wsrc + (uint64_t)ra * p.row_bytes, wbytes, &full_bar[s]);
                const uint64_t soff = (uint64_t)(r0 + ra) * g2;
                bulk_g2s(slot + p.sb_off, reinterpret_cast<const uint8_t*>(p.scales) + soff, sbytes, &full_bar[s]);
                bulk_g2s(slot + p.sb_off + (uint32_t)p.tr * g2, reinterpret_cast<const uint8_t*>(p.biases) + soff, sbytes,
                         &full_bar[s]);
                if (++s == nstg) {
                    s = 0;
                    phase ^= 1u;
                }
            }
        }
    } else if (warp < active_warps && rows > 0) {
        // ===================== consumer warps =====================
        const int cwi = warp % p.cw;  // chunk column
        const int rgi = warp / p.cw;  // row group
        const int g = lane >> 2, t = lane & 3;
        // lane -> (weight row inside the set, group slice) of the two A-row parts (MMA rows g and g+8).  The slices are
        // rotated with the weight row so that the 16 lanes of one LDS.64 wavefront read ONE contiguous 128-byte piece:
        // rows 2i / 2i+1 of a set take slices {0,1} / {2,3} for part A and the other pair for part B.  Rows of a stage are
        // row_bytes apart (a multiple of 128: the same banks); with slices {0,1} for every row the two rows of a wavefront
        // collided (r01i ncu: 4.3 wavefronts per useful one).  4-byte chunks (2-bit, gs 64) stay 2-way conflicting: a
        // chunk column of theirs is only 64 bytes wide.
        const int wrow = g >> 1;
        const int sA = g & 3;
        const int sB = sA ^ 2;
        // lane as B-column holder: column g = (slice g>>1, digit g&1)
        const int bsl = g >> 1, bdig = g & 1;
        // accumulators c0,c1 (c2,c3) = columns 2t, 2t+1 = (slice t, digits 0/1): meaningful for part A iff t == sA,
        // for part B iff t == sB; this lane's meaningful part (if any) multiplies group slice t
        const bool mean = ((t ^ sA) & 1) == 0;
        const bool partA = t == sA;

        if constexpr (!STREAM) griddep_wait();  // x (and y) belong to the previous kernels of the stream
        STAMP(1);
        if constexpr (!STREAM) {
            // epoch of a fused all-reduce: advanced by the last CTA of the previous such launch, complete by now
            if (ar_on && threadIdx.x == 0)
                *ar_epoch_s = *reinterpret_cast<volatile uint32_t*>(ar->flags[ar->rank] + ar->world * kArMaxCtas) + 1u;
        }

        // ---- stationary operands: digit fragments of the activations, per-group power-of-two factors, group sums
        uint32_t bfr[MT][CPW][NCLASS][NMMA][2];
        float pw[MT][CPW];  // 2^(e-13) / CMUL of group slice t of chunk column j (the slice this lane's accumulators need)
        float* myx = xsc + warp * (CPW * S * MT);
        // activations of up to JB chunk columns are requested together: one L2 round trip per batch instead of one per
        // column (K = 14336 has 8 columns per warp; fetched one by one the prologue was 4 us, profiles/r01h_*)
        constexpr int JBmax = 64 / CQ;  // at most 8 uint4 (32 registers) in flight per lane
        constexpr int JB = CPW < JBmax ? CPW : JBmax;
#pragma unroll
        for (int m = 0; m < MT; m++) {
#pragma unroll
            for (int j0 = 0; j0 < CPW; j0 += JB) {
            uint4 raw[JB][CQ / 8];
#pragma unroll
            for (int jj = 0; jj < JB; jj++) {
                const int c = cwi + (j0 + jj) * p.cw;
                // groups past the end of the row (G % 4 == 2: the last chunk column holds two live slices) read zeros
                const bool ld = (c < p.nch) && (!PARTIAL || c * S + bsl < p.G) && (m < p.M);
                const int64_t k0 = ((int64_t)c * S + bsl) * GS + t * CQ;
                const uint4* src = reinterpret_cast<const uint4*>(p.x + (size_t)m * p.K + k0);
#pragma unroll
                for (int v = 0; v < CQ / 8; v++)
                    // chain launches read activations another SM wrote during this launch: L2-coherent loads there
                    raw[jj][v] = ld ? (STREAM ? __ldcg(src + v) : __ldg(src + v)) : make_uint4(0u, 0u, 0u, 0u);
            }
#pragma unroll
            for (int jj = 0; jj < JB; jj++) {
                const int j = j0 + jj;
                uint32_t n32[CQ / 2];  // n32[i] = codes (2i, 2i+1) of the chunk, natural order
#pragma unroll
                for (int v = 0; v < CQ / 8; v++) {
                    const uint4 q = raw[jj][v];
                    n32[4 * v + 0] = q.x; n32[4 * v + 1] = q.y; n32[4 * v + 2] = q.z; n32[4 * v + 3] = q.w;
                }
                // |x| maximum of the chunk as packed 16-bit lanes; sum of x in fp32
                uint32_t amax2 = 0;
                float sx = 0.f;
                float xf[CQ];
#pragma unroll
                for (int i = 0; i < CQ / 2; i++) {
                    amax2 = __vmaxu2(amax2, n32[i] & 0x7fff7fffu);
                    xf[2 * i] = __uint_as_float(n32[i] << 16);
                    xf[2 * i + 1] = __uint_as_float(n32[i] & 0xffff0000u);
                    sx += xf[2 * i];
                    sx += xf[2 * i + 1];
                }
                uint32_t amax = max(amax2 & 0xffffu, amax2 >> 16);  // bf16 bits of the largest |x|
                sx += __shfl_xor_sync(0xffffffffu, sx, 1);
                sx += __shfl_xor_sync(0xffffffffu, sx, 2);
                amax = max(amax, __shfl_xor_sync(0xffffffffu, amax, 1));
                amax = max(amax, __shfl_xor_sync(0xffffffffu, amax, 2));
                if (m == 0 && j == 0 && amax != 0xffffffffu) STAMP(7);  // the first activations have arrived
                if (t == 0 && bdig == 0) myx[(j * S + bsl) * MT + m] = sx;  // true sum of x over (group, token)
                // block exponent of the group: |x| < 2^(e+1); m = round(x * 2^(13-e)), |m| < 2^14
                int e = (int)(amax >> 7) - 127;
                if (e < -100) e = -100;  // zeros / denormal groups: any finite scale works
                const bool bad = (amax >> 7) == 255u;  // inf / nan in the group: poison the group's factor
                const float up = __uint_as_float((uint32_t)(127 + 13 - e) << 23);        // 2^(13-e)
                const float dn = __uint_as_float((uint32_t)(127 - 13 + e) << 23);        // 2^(e-13)
                // the factor this lane needs is the one of slice t, held by the lanes with g>>1 == t
                const float dn_t = __shfl_sync(0xffffffffu, bad ? __uint_as_float(0x7fc00000u) : dn, t << 3);
                pw[m][j] = dn_t * (1.0f / GE::CMUL);
                // balanced base-256 digits: lo = low byte of m (as s8), hi = (m + 128) >> 8.  1.5*2^23 + m has m's two's
                // complement in its low mantissa bits; adding 128 there puts hi into byte 1: each lane takes byte `bdig`.
                const float magic = bdig ? 12583040.0f : 12582912.0f;  // 1.5*2^23 (+ 128)
                const uint32_t sel2 = bdig ? 0x0051u : 0x0040u;        // PRMT: byte bdig of two words -> low half
                uint32_t pr[CQ / 2];  // pr[i] = digit bytes of codes (2i, 2i+1) in the low half
#pragma unroll
                for (int i = 0; i < CQ / 2; i++) {
                    const uint32_t m0 = __float_as_uint(fmaf(xf[2 * i], up, magic));
                    const uint32_t m1 = __float_as_uint(fmaf(xf[2 * i + 1], up, magic));
                    pr[i] = __byte_perm(m0, m1, sel2);
                }
#pragma unroll
                for (int c2 = 0; c2 < NCLASS; c2++)
#pragma unroll
                    for (int u = 0; u < NMMA; u++)
#pragma unroll
                        for (int h = 0; h < 2; h++) {
                            uint32_t r = 0;
                            if (!(GE::HALF && u == NMMA - 1 && h == 1)) {
                                // bytes i = 0..3 <- codes code_of(c2,u,h,i); code k sits in byte (k&1) of pr[k>>1]
                                const int k0c = GE::code_of(c2, u, h, 0), k1c = GE::code_of(c2, u, h, 1);
                                const int k2c = GE::code_of(c2, u, h, 2), k3c = GE::code_of(c2, u, h, 3);
                                const uint32_t lo2 = __byte_perm(pr[k0c >> 1], pr[k1c >> 1], (k0c & 1) | ((4 + (k1c & 1)) << 4));
                                const uint32_t hi2 = __byte_perm(pr[k2c >> 1], pr[k3c >> 1], (k2c & 1) | ((4 + (k3c & 1)) << 4));
                                r = __byte_perm(lo2, hi2, 0x5410);
                            }
                            bfr[m][j][c2][u][h] = r;
                        }
            }
            }
        }
        __syncwarp();
        if constexpr (!STREAM) {
            if (lane == 0) mbar_arrive(&full_bar[kMaxStages - 1]);  // activations are in registers: the stream may flood
        }
        const int brow = lane / LPR, bq = lane % LPR;
        const uint32_t g2 = (uint32_t)p.G * 2u;
        const int lrow0 = rgi * R;
        int ncl = 0;  // live chunk columns of this warp (warp-uniform)
#pragma unroll
        for (int j = 0; j < CPW; j++) ncl += (cwi + j * p.cw < p.nch) ? 1 : 0;
        float xg[NGL][MT];
        uint32_t bofs[NGL];  // byte offset of the lane's bias entries inside a stage (dead entries: x sum = 0, offset 0)
#pragma unroll
        for (int i = 0; i < NGL; i++) {
            // R = 16 (two lanes per row): strided groups and separately rounded products below reproduce the summation
            // tree of the R = 8 geometry bit for bit (single, grouped and chain launches must agree)
            const int idx = R == 16 ? bq + i * LPR : bq * NGL + i;
            const int c = cwi + (idx / S) * p.cw;
            const bool on = idx < CPW * S && c < p.nch && (!PARTIAL || c * S + idx % S < p.G);
#pragma unroll
            for (int m = 0; m < MT; m++) xg[i][m] = on ? myx[idx * MT + m] : 0.f;
            bofs[i] = (uint32_t)(p.tr + lrow0 + brow) * g2 + (on ? (uint32_t)(c * S + idx % S) * 2u : 0u);
        }

        const uint32_t colstride = (uint32_t)p.cw * KSTEP_B;
        const uint32_t offA = (uint32_t)wrow * p.row_bytes + (uint32_t)cwi * KSTEP_B + (uint32_t)(sA * 4 + t) * TB;
        const uint32_t offB = (uint32_t)wrow * p.row_bytes + (uint32_t)cwi * KSTEP_B + (uint32_t)(sB * 4 + t) * TB;
        // scale of the slice this lane's accumulators belong to (slice t of the chunk column), row = wrow
        const uint32_t sofT = (uint32_t)wrow * g2 + (uint32_t)(cwi * S + t) * 2u;
        const uint32_t sstride = (uint32_t)p.cw * S * 2u;
        // Scale offset per chunk column.  Where this lane's slice t of column j lies past the row's last group (G % 4 == 2)
        // its weight reads run into the next row -- exact zeros once multiplied with the zero activations of a dead slice,
        // in the integer domain -- and the scale read is redirected to live slice t - 2 of the same column: always a real
        // scale, never stale shared memory (a NaN there would survive the multiplication by zero).  No cost in the loop.
        uint32_t sof[PARTIAL ? CPW : 1];
        if constexpr (PARTIAL) {
#pragma unroll
            for (int j = 0; j < CPW; j++)
                sof[j] = (uint32_t)j * sstride + sofT - (((cwi + j * p.cw) * S + t >= p.G && t >= 2) ? 4u : 0u);
        }

        STAMP(2);
        for (int ra = 0; ra < rows; ra += spr) {
            int nr = rows - ra;
            if (nr > spr) nr = spr;
            mbar_wait(&full_bar[s], phase);
            if (ra == 0) STAMP(3);
            const uint8_t* slot = ring + (size_t)s * p.slot_bytes;
            const uint8_t* sslot = slot + p.sb_off;

            float yacc[NSET][MT];
            // one (set, chunk column) unit: 2 LDS of packed words, mask into u8 A registers, NCLASS*NMMA IMMAs per token on the
            // group's accumulators, recombine classes and digits in int32, one I2F, fold with scale * 2^(e-13).
            // Sets past `nr` read stale shared memory; their rows are dropped at the write.
            auto unit = [&](int q, int j) {
                const uint8_t* rbase = slot + (uint32_t)(lrow0 + q * W) * p.row_bytes + j * colstride;
                uint32_t wa[NWORD], wb[NWORD];
                load_chunk<BITS, CQ>(rbase + offA, wa);
                load_chunk<BITS, CQ>(rbase + offB, wb);
                const float sc = lds_bf16(sslot + (uint32_t)(lrow0 + q * W) * g2 + (PARTIAL ? sof[PARTIAL ? j : 0] : j * sstride + sofT));
                const int kZero4[4] = {0, 0, 0, 0};
                int T[MT][2];  // [token][part]: 256 * hi + lo of the meaningful part's group
#pragma unroll
                for (int m = 0; m < MT; m++) {
                    int d[NCLASS][4];
#pragma unroll
                    for (int c = 0; c < NCLASS; c++) {
#pragma unroll
                        for (int u = 0; u < NMMA; u++) {
                            const bool lone = GE::HALF && u == NMMA - 1;
                            const uint32_t a0 = areg<BITS, CQ>(wa, c, u, 0), a1 = areg<BITS, CQ>(wb, c, u, 0);
                            const uint32_t a2 = lone ? 0u : areg<BITS, CQ>(wa, c, u, 1), a3 = lone ? 0u : areg<BITS, CQ>(wb, c, u, 1);
                            if (u == 0) imma16832(d[c], a0, a1, a2, a3, bfr[m][j][c][u][0], bfr[m][j][c][u][1], kZero4);
                            else imma16832(d[c], a0, a1, a2, a3, bfr[m][j][c][u][0], bfr[m][j][c][u][1], d[c]);
                        }
                    }
#pragma unroll
                    for (int e = 0; e < 4; e++)
                        if constexpr (NCLASS == 2) d[0][e] = d[0][e] * GE::CMUL + d[1][e];
                    T[m][0] = d[0][1] * 256 + d[0][0];
                    T[m][1] = d[0][3] * 256 + d[0][2];
                }
#pragma unroll
                for (int m = 0; m < MT; m++) {
                    const int tt = partA ? T[m][0] : T[m][1];  // the part whose slice is t (garbage where !mean: dropped below)
                    yacc[q][m] = fmaf(sc * pw[m][j], (float)tt, yacc[q][m]);
                }
            };
#pragma unroll
            for (int q = 0; q < NSET; q++)
#pragma unroll
                for (int m = 0; m < MT; m++) yacc[q][m] = 0.f;
            if (ncl == CPW) {
                // fast path: straight-line code, the NSET * CPW units are independent chains the scheduler interleaves
#pragma unroll
                for (int q = 0; q < NSET; q++)
#pragma unroll
                    for (int j = 0; j < CPW; j++) unit(q, j);
            } else {
#pragma unroll
                for (int q = 0; q < NSET; q++)
#pragma unroll
                    for (int j = 0; j < CPW; j++)
                        if (j < ncl) unit(q, j);
            }
            // ---- biases: sum_g bias * sum(x over g), a rows x groups dot product against per-lane stationary group sums
            float bacc[MT];
#pragma unroll
            for (int m = 0; m < MT; m++) bacc[m] = 0.f;
#pragma unroll
            for (int i = 0; i < NGL; i++) {
                const float bv = lds_bf16(sslot + bofs[i]);
#pragma unroll
                for (int m = 0; m < MT; m++)
                    bacc[m] = R == 16 ? __fadd_rn(bacc[m], __fmul_rn(bv, xg[i][m])) : fmaf(bv, xg[i][m], bacc[m]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[s]);  // slot free: all of this warp's shared-memory reads are done
            if (++s == nstg) {
                s = 0;
                phase ^= 1u;
            }
#pragma unroll
            for (int m = 0; m < MT; m++) {
#pragma unroll
                for (int o = LPR / 2; o > 0; o >>= 1) bacc[m] += __shfl_xor_sync(0xffffffffu, bacc[m], o);
            }
            if (bq == 0 && lrow0 + brow < nr) {
#pragma unroll
                for (int m = 0; m < MT; m++) ysum[((ra + lrow0 + brow) * slots + p.cw + cwi) * MT + m] = bacc[m];
            }
            // ---- keep the meaningful accumulators; the 8 lanes (g&1, t) of a weight row are folded by a butterfly
#pragma unroll
            for (int q = 0; q < NSET; q++) {
#pragma unroll
                for (int m = 0; m < MT; m++) {
                    float v = mean ? yacc[q][m] : 0.f;
                    v += __shfl_xor_sync(0xffffffffu, v, 4);
                    v += __shfl_xor_sync(0xffffffffu, v, 2);
                    v += __shfl_xor_sync(0xffffffffu, v, 1);
                    const int lr = lrow0 + q * W + (lane >> 3);
                    if ((lane & 7) == 0 && lr < nr) ysum[((ra + lr) * slots + cwi) * MT + m] = v;
                }
            }
        }
    }
    else if (STREAM && rows > 0) {
        // idle warps of a narrow call keep the ring's arrival counts whole
        for (int ra = 0; ra < rows; ra += spr) {
            mbar_wait(&full_bar[s], phase);
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[s]);
            if (++s == nstg) {
                s = 0;
                phase ^= 1u;
            }
        }
    }
    STAMP(4);
    if constexpr (STREAM) {
        consumer_bar();
        sc->s = s;
        sc->phase = phase;
    } else {
        __syncthreads();
        STAMP(5);
        if (p.dbg != nullptr && p.dbg_all != 0 && threadIdx.x == 0) {
            unsigned smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            p.dbg[(size_t)blockIdx.x * 8 + 5] = smid;
        }
        griddep_wait();  // every thread stores y below (returns at once when a consumer warp has already waited)
    }
    // ---- epilogue: 4 lanes per output row sum a quarter of the partial slots each (fixed order: deterministic), two
    // shuffles, one rounding to bf16, optional bias as a second rounded add
    {
        constexpr int kNT = STREAM ? kCW * 32 : kThreads;
        const int q4 = threadIdx.x & 3;
#pragma unroll
        for (int m = 0; m < MT; m++) {
            for (int rb = 0; rb < rows; rb += kNT / 4) {  // trip count uniform over the CTA: full-mask shuffles
                const int r = rb + ((int)threadIdx.x >> 2);
                float tot = 0.f;
                if (r < rows) {
                    const float* src = ysum + ((size_t)r * slots) * MT + m;
                    for (int c = q4; c < slots; c += 4) tot += src[c * MT];
                }
                tot += __shfl_xor_sync(0xffffffffu, tot, 1);
                tot += __shfl_xor_sync(0xffffffffu, tot, 2);
                if (q4 == 0 && r < rows && m < p.M) {
                    if (ar_on) {
                        // row-parallel shard: the fp32 partial (+ this rank's bias share) goes to every peer
                        if (p.bias != nullptr) tot += __bfloat162float(p.bias[r0 + r]);
                        const uint32_t epoch = *ar_epoch_s;
                        const size_t at = (size_t)(epoch & 1u) * ar->half_elems + ((size_t)ar->rank * p.M + m) * p.N + r0 + r;
                        const unsigned long long word = ((unsigned long long)epoch << 32) | (unsigned long long)__float_as_uint(tot);
                        for (int d = 0; d < ar->world; d++)
                            asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(ar->stage[d] + at), "l"(word) : "memory");
                    } else {
                        float v = __bfloat162float(__float2bfloat16_rn(tot));
                        if (p.bias != nullptr) v = __fadd_rn(v, __bfloat162float(p.bias[r0 + r]));
                        p.y[(size_t)m * p.N + r0 + r] = __float2bfloat16_rn(v);
                    }
                }
            }
        }
    }
    if constexpr (!STREAM) {
        if (ar_on) {
            const uint32_t epoch = *ar_epoch_s;
            uint32_t* ctl = ar->flags[ar->rank] + ar->world * kArMaxCtas;
            const unsigned long long* st = ar->stage[ar->rank] + (size_t)(epoch & 1u) * ar->half_elems;
            const unsigned long long t0 = gtime();
            for (int i = threadIdx.x; i < rows * p.M; i += kThreads) {
                const int m = i / rows, r = i - m * rows;
                float acc = 0.f;
                for (int w = 0; w < ar->world; w++) {
                    const unsigned long long* src = st + ((size_t)w * p.M + m) * p.N + r0 + r;
                    unsigned long long v;
                    for (;;) {
                        asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(src) : "memory");
                        if ((uint32_t)(v >> 32) == epoch) break;
                        if (gtime() - t0 > 4000000000ull) {  // 4 s: a peer is gone; flag the error, never hang the device
                            atomicExch(ctl + 2, 1u);
                            break;
                        }
                    }
                    acc += __uint_as_float((uint32_t)v);
                }
                p.y[(size_t)m * p.N + r0 + r] = __float2bfloat16_rn(acc);
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                if (atomicAdd(ctl + 1, 1u) == gridDim.x - 1u) {  // last CTA of the launch: advance the epoch
                    ctl[1] = 0u;
                    __threadfence();
                    *reinterpret_cast<volatile uint32_t*>(ctl) = epoch;
                }
            }
        }
    }
    STAMP(6);
    if constexpr (STREAM) {
        consumer_bar();  // all of this CTA's y stores are issued (and ysum / the call descriptor may be reused)
        if (threadIdx.x == 0) {
            __threadfence();
            atomicAdd(sc->done_cnt, 1u);
        }
    }
}


// ------------------------------------------------------------------------------------------ host side
struct Plan {
    bool ok;
    int mt, cpw, R, nch, cw, rg, tr, stages, grid, row_unit;
    bool partial;  // G % 4 == 2: the last chunk column is half full (PARTIAL instantiation)
    uint32_t slot_bytes, sb_off;
    size_t smem;
};

// grid_want > 0: the number of CTAs this layer may use (a segment of a grouped launch); 0: the whole device
inline Plan make_plan(int64_t M, int64_t N, int64_t K, int bits, int gs, int grid_want = 0, bool allow_r16 = true,
                      bool allow_partial = false) {
    Plan pl{};
    if (!(bits == 2 || bits == 3 || bits == 4 || bits == 6 || bits == 8) || M < 1 || M > 4 || N < 1) return pl;
    if ((bits == 2 || bits == 3 || bits == 6) && gs == 32) return pl;  // a thread chunk would be a fraction of a word
    const int64_t G = K / gs;
    // S | G.  The scales / biases of a stage travel as ONE bulk copy (the rows of a stage are contiguous), which needs a
    // 16-byte aligned start: any row when G % 8 == 0; with G % 8 == 4 (tensor-parallel K shards: Qwen2.5-32B down_proj
    // K/2 = 13824 at gs 128) every CTA range and stage must start on an even row -> rows are shared out in units of 4
    // G % 4 == 2 (tensor-parallel K shards: Qwen2.5-32B at tp4, o_proj 1280 = 10 and down_proj 6912 = 54 groups of 128):
    // the last chunk column is half full; its dead slices multiply zero activations
    pl.partial = (G % 4) != 0;
    // served by the one-call launches at group size 128 and <= 2 rows of x only (the instantiations that exist)
    if (G % 2 || G < 2 || (pl.partial && !(allow_partial && gs == 128 && M <= 2))) return pl;
    pl.row_unit = (G % 8) ? 4 : 1;
    if (pl.row_unit == 4 && (N % 4)) return pl;
    const int64_t row_bytes = K * bits / 8;
    pl.mt = M == 1 ? 1 : (M == 2 ? 2 : 4);
    pl.nch = (int)((G + S - 1) / S);
    static const int force_cpw = env_int("GBXQ_MMV8_CPW", 0);
    static const int grid_mult = env_int("GBXQ_MMV8_GRID_MULT", 2 / kWide);
    static const int stage_kb = env_int("GBXQ_MMV8_STAGE_KB", 32 * kWide);
    static const int ring_kb = env_int("GBXQ_MMV8_RING_KB", 96 * kWide);
    // r03a sweep (16 warps): two columns per warp from 16 columns (K = 4096 at gs 64: 0.52 of HBM on the 8B step against
    // 0.46 with one column and 16-row stages), one column and 16-row stages below (K = 3072: 3B step 0.40 against 0.37)
    static const int two_cols_from = env_int("GBXQ_MMV8_TWOCOLS", kCW == 8 ? 8 : 16);
    static const int r16 = env_int("GBXQ_MMV8_R16", kCW == 16 ? 1 : 0);
    // chunk columns per warp: the smallest power of two that covers the row with 8 warps, but at least 2 (two
    // independent MMA chains per set) when the row has 8 columns or more
    pl.cpw = pl.nch >= two_cols_from ? 2 : 1;
    while ((pl.nch + pl.cpw - 1) / pl.cpw > kCW && pl.cpw < 8) pl.cpw *= 2;
    if (force_cpw) pl.cpw = force_cpw;
    if (!(pl.cpw == 1 || pl.cpw == 2 || pl.cpw == 4 || pl.cpw == 8)) return pl;
    pl.cw = (pl.nch + pl.cpw - 1) / pl.cpw;
    if (pl.cw > kCW) return pl;
    pl.rg = kCW / pl.cw;
    pl.R = pl.cpw <= 2 ? 8 : 4;
    // one chunk column per warp and 16 warps: 16 rows per warp and stage keep a stage at 2 x 16 rows of a 2/4 KB row
    if (r16 && allow_r16 && pl.cpw == 1 && pl.nch > kCW / 2 && M <= 2 && 16 * row_bytes <= (int64_t)stage_kb * 1024) pl.R = 16;
    if (pl.R == 8 && (int64_t)pl.R * row_bytes > (int64_t)stage_kb * 1024) pl.R = 4;
    if ((int64_t)pl.R * row_bytes > (int64_t)stage_kb * 1024) return pl;
    while (pl.rg > 1 && (int64_t)pl.rg * pl.R * row_bytes > (int64_t)stage_kb * 1024 / 2) pl.rg--;
    pl.tr = pl.rg * pl.R;
    const uint32_t wpart = (uint32_t)(((int64_t)pl.tr * row_bytes + 127) & ~(int64_t)127);
    pl.sb_off = wpart;
    pl.slot_bytes = wpart + (uint32_t)((2 * (int64_t)pl.tr * G * 2 + 127) & ~(int64_t)127);
    static const int plan_stages = env_int("GBXQ_MMV8_STAGES", kPlanStages);
    pl.stages = plan_stages < 2 ? 2 : (plan_stages > kMaxStages - 1 ? kMaxStages - 1 : plan_stages);
    while (pl.stages > 2 && (size_t)pl.stages * pl.slot_bytes > (size_t)ring_kb * 1024) pl.stages--;
    int grid = grid_want > 0 ? grid_want : device_sm_count() * grid_mult;
    const int64_t min_rows = pl.tr;
    if ((int64_t)grid * min_rows > N) grid = (int)((N + min_rows - 1) / min_rows);
    if (grid < 1) grid = 1;
    pl.grid = grid;
    const int64_t rows_max = ((N / pl.row_unit + grid - 1) / grid) * pl.row_unit;
    pl.smem = (size_t)pl.stages * pl.slot_bytes + 2 * kMaxStages * 8 + (size_t)kCW * pl.cpw * S * pl.mt * 4 +
              (size_t)rows_max * 2 * pl.cw * pl.mt * 4 + 16;
    if (pl.smem > (size_t)kSmemCap) return pl;
    pl.ok = true;
    return pl;
}

// Relative cost of a segment when CTAs are shared out between the segments of one call.  Measured steady state
// (profiles/r01b_big.txt): 4-bit rows stream at 0.90 of HBM, 2-bit rows at 0.50 -- both 10.5e12 codes/s, the kernel's
// unpack/IMMA ceiling -- so a row costs max(its bytes, K codes at that ceiling = 0.5625 byte-equivalents per code).
inline double segment_cost(int64_t N, int64_t K, int bits, int gs) {
    const double bytes_per_code = bits / 8.0 + 4.0 / gs;
    return (double)N * (double)K * (bytes_per_code > 0.5625 ? bytes_per_code : 0.5625);
}

inline int mmv8_total_ctas() {
    static const int grid_mult = env_int("GBXQ_MMV8_GRID_MULT", 2 / kWide);
    return device_sm_count() * grid_mult;
}

// Kernel parameters of one layer from its plan (everything but the debug pointer).
inline Mmv8Params make_params(const Plan& pl, const void* x, const uint32_t* w, const void* s, const void* b,
                              const void* bias, void* y, int64_t M, int64_t N, int64_t K, int bits, int gs, int early) {
    Mmv8Params p{};
    p.x = reinterpret_cast<const __nv_bfloat16*>(x);
    p.w = reinterpret_cast<const uint8_t*>(w);
    p.scales = reinterpret_cast<const uint16_t*>(s);
    p.biases = reinterpret_cast<const uint16_t*>(b);
    p.bias = reinterpret_cast<const __nv_bfloat16*>(bias);
    p.y = reinterpret_cast<__nv_bfloat16*>(y);
    p.N = N;
    p.K = K;
    p.M = (int)M;
    p.G = (int)(K / gs);
    p.row_bytes = (uint32_t)(K * bits / 8);
    p.nch = pl.nch;
    p.cw = pl.cw;
    p.rg = pl.rg;
    p.tr = pl.tr;
    p.stages = pl.stages;
    p.slot_bytes = pl.slot_bytes;
    p.sb_off = pl.sb_off;
    p.early_weights = early;
    static const int pre_stages = env_int("GBXQ_MMV8_PRE_STAGES", 2);
    p.pre_stages = pre_stages;
    p.row_unit = pl.row_unit;
    p.rows_base = (int)((N / pl.row_unit) / pl.grid) * pl.row_unit;
    p.rows_rem = (int)((N / pl.row_unit) % pl.grid);
    auto spr_of = [&](int rows) {
        if (rows <= 0) return W;
        const int ns = (rows + pl.tr - 1) / pl.tr;
        return (((rows + ns - 1) / ns + W - 1) / W) * W;  // balanced stages, whole MMA sets
    };
    p.spr0 = spr_of(p.rows_base);
    p.spr1 = spr_of(p.rows_base + pl.row_unit);
    return p;
}


}  // namespace mmv8
}  // namespace gbxq
