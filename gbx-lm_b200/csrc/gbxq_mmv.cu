// gbxq_mmv.cu -- decode matrix-vector kernel on the tensor pipe ("mmv"): 1..4 rows of x per pass,
// bf16 activations, 2-/4-/8-bit packings.  The headline kernel of the path:
// QuantizedLinear.__call__ -> mx.quantized_matmul(transpose=True)
// (gbx_lm/models/quantized_linear_gba.py:195-203) at decode batch sizes.
//
// Why: at 4 bits a B200 SM has to retire ~45 weights per clock to keep up with its share of HBM.
// One FMA per weight on the CUDA cores (gbxq_gemv.cu) measured 3.0 issued instructions per weight
// (profiles/r01a_ncu_gemv_summary.txt) -- issue bound at 40 % of the HBM roofline.  Here the
// multiply-accumulate is `mma.sync.m16n8k16` and everything else is trimmed to ~1.6 instructions
// per weight.
//
//   * Streaming is the GEMV's: the packed rows a CTA owns are one contiguous byte range; a producer
//     warp moves `tr` whole rows + their scales + their biases per stage with 1-D bulk copies
//     (cp.async.bulk, SASS UBLKCP) through a 4-stage mbarrier ring.  Shared memory per CTA stays
//     under 76 KB and registers under 112, so 2-3 CTAs are co-resident per SM; kernels are launched
//     with programmatic dependent launch (PDL): the next projection's CTAs become resident and
//     prefetch their (immutable) weights while this one drains, and only wait
//     (`griddepcontrol.wait`) before they touch x / y.
//   * "Slice" trick: an m16n8k16 MMA wants 16 A rows that share one B operand.  With M <= 4 tokens
//     the 8 B columns are used as (quantisation group s, token m): column j holds the activations
//     of group j / MP for token j % MP (MP = 1, 2 or 4).  The 16 A rows are then W = 2*MP weight
//     rows x S = 8/MP consecutive groups of each -- for M = 1 two weight rows x 8 groups -- so a
//     warp-wide shared-memory load reads long contiguous pieces of few rows, the tile granularity
//     is 2 rows instead of 16, and every MMA still does 256 useful multiply-adds per thread-octet.
//     Only the accumulators whose column group equals their row group are meaningful; the others
//     are dropped at the end of the stage.
//   * The k order inside a group is free, so the pair one LOP3 extracts -- (w >> s) & mask |
//     0x4300 = two bf16 values 128 + q -- IS an A register; the activations are permuted (and, for
//     the shift-free 2-bit fields at bits 2 and 4, pre-divided by 4 and 16) once per kernel into
//     stationary B fragments.  All 16 k-slots of an MMA belong to one group, so the group's partial
//     product sits alone in the accumulator and is folded as y += scale * D.
//   * biases and the 128 offset of the code images: y += sum_g (bias[n,g] * sum(x over g) - 128 * scale[n,g] *
//     sum(B column of g)) is a [rows x groups] dot product against per-lane stationary group sums, a handful of
//     FMAs per row and stage.
//   * per stage every warp reduces its rows with a transposing shuffle butterfly; every (chunk
//     column, part) owns a shared-memory slot per row (no atomics: bitwise reproducible); the
//     epilogue sums the slots in fixed order, rounds once to bf16 (+ optional bias as a second
//     rounded add) and stores coalesced.
#include "gbxq_common.cuh"

namespace gbxq {

namespace {

constexpr int kCW = 8;                        // consumer warps
constexpr int kThreads = (kCW + 1) * 32;      // + producer warp
constexpr int kMaxStages = 4;
constexpr int kMinCtasPerSm = 2;              // register cap 112 (72 measured 35% slower: the MMA chains serialise)
constexpr uint32_t kMagic = 0x43004300u;      // bf16x2 (128, 128)

__device__ __forceinline__ void mma16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1, const float (&c)[4]) {
    // not volatile: a pure function of its operands, so independent chains can be interleaved by the scheduler
    asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%12,%13};"
        : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "f"(c[0]), "f"(c[1]), "f"(c[2]), "f"(c[3]));
}
__device__ __forceinline__ uint32_t hmul2_bf16(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}

// ---- packing geometry.  A thread chunk = TB bytes = CQ codes = NP pairs; pair p = codes (pa, pb) that one LOP3
//      extracts together (same position in the low / high half of a 32-bit word).
template <int BITS> __host__ __device__ constexpr int pair_a(int p) {
    if (BITS == 4) return 8 * (p >> 2) + (p & 3);
    if (BITS == 2) return 16 * (p >> 3) + (p & 7);
    return 4 * (p >> 1) + (p & 1);  // 8-bit
}
template <int BITS> __host__ __device__ constexpr int pair_b(int p) {
    return pair_a<BITS>(p) + (BITS == 4 ? 4 : (BITS == 2 ? 8 : 2));
}
// 2-bit: field i of a half-word is used in place at bit 2*(i%3) after a shift by 6*(i/3): value 128 + 4^cexp * q
__host__ __device__ constexpr int cexp2(int i) { return i < 6 ? i % 3 : i - 6; }

template <int BITS, int NWORD>
__device__ __forceinline__ uint32_t unpack_pair(const uint32_t (&w)[NWORD], int p) {
    if constexpr (BITS == 4) {
        return lop3_and_or(w[p >> 2] >> (4 * (p & 3)), 0x000f000fu, kMagic);
    } else if constexpr (BITS == 2) {
        const int i = p & 7;
        const uint32_t base = w[p >> 3] >> (6 * (i / 3));
        return lop3_and_or(base, 0x00030003u << (2 * cexp2(i)), kMagic);
    } else {
        return lop3_and_or(w[p >> 1] >> (8 * (p & 1)), 0x007f007fu, kMagic);
    }
}
// 8-bit second image: 128 + 128 * (top bit)
template <int NWORD> __device__ __forceinline__ uint32_t unpack_pair_top(const uint32_t (&w)[NWORD], int p) {
    return lop3_and_or(w[p >> 1] >> (8 * (p & 1)), 0x00800080u, kMagic);
}

// plain C++ loads from the ring (ordered by the "memory" clobber of the mbarrier wait, freely scheduled otherwise)
template <int NWORD> __device__ __forceinline__ void lds_words(const uint8_t* addr, uint32_t (&w)[NWORD]) {
    if constexpr (NWORD == 1) {
        w[0] = *reinterpret_cast<const uint32_t*>(addr);
    } else if constexpr (NWORD == 2) {
        const uint2 v = *reinterpret_cast<const uint2*>(addr);
        w[0] = v.x; w[1] = v.y;
    } else {
        const uint4 v = *reinterpret_cast<const uint4*>(addr);
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    }
}
__device__ __forceinline__ float lds_bf16(const uint8_t* addr) {
    return __uint_as_float((uint32_t)(*reinterpret_cast<const uint16_t*>(addr)) << 16);
}

struct MmvParams {
    const __nv_bfloat16* x;
    const uint8_t* w;
    const uint16_t* scales;
    const uint16_t* biases;
    const __nv_bfloat16* bias;
    __nv_bfloat16* y;
    int64_t N, K;
    int M;                // rows of x in this launch (<= MP)
    int G;                // groups per row
    uint32_t row_bytes;
    int nch;              // chunk columns per row (a chunk column = S groups)
    int cw, rg;           // warp grid: cw chunk columns x rg row groups (cw * rg <= 8)
    int tr;               // rows per ring stage (= rg * R)
    int stages;
    uint32_t slot_bytes;  // ring slot size
    uint32_t sb_off;      // offset of the scales inside a slot (biases follow at sb_off + tr*G*2)
    int early_weights;    // 1: weights are immutable while the call is in flight -> stream them before griddepcontrol.wait
};

// BITS, TB = bytes per thread chunk (= group_size*BITS/32), MP = token columns per group (1, 2, 4),
// CPW = chunk columns per warp, R = rows per warp and stage (multiple of W = 2*MP)
template <int BITS, int TB, int MP, int CPW, int R>
__global__ void __launch_bounds__(kThreads, kMinCtasPerSm) mmv_kernel(const MmvParams p) {
    constexpr int NWORD = TB / 4;
    constexpr int CQ = TB * 8 / BITS;        // codes per thread chunk (= group_size / 4)
    constexpr int NP = CQ / 2;               // pairs per chunk
    constexpr int NH = NP / 2;               // MMA k16 steps per group
    constexpr int GS = CQ * 4;
    constexpr int S = 8 / MP;                // groups (slices) per weight row and MMA set
    constexpr int W = 2 * MP;                // weight rows per MMA set
    constexpr int NSET = R / W;
    constexpr int KSTEP_B = S * 4 * TB;      // bytes of one weight row inside a chunk column
    constexpr int LPR = 32 / R;              // lanes per row in the bias dot product
    constexpr int NGL = (CPW * S + LPR - 1) / LPR;  // groups per lane there
    constexpr float OFF = BITS == 8 ? 256.f : 128.f;  // additive offset carried by the bf16 images of the codes
    static_assert(R % W == 0 && NH >= 1 && (NWORD == 1 || NWORD == 2 || NWORD == 4), "geometry");

    extern __shared__ __align__(1024) uint8_t smem[];
    // layout: [ring stages * slot][full/empty barriers (2*kMaxStages)][xsc kCW*128 f32][ysum rows * 2cw * MP f32]
    uint8_t* ring = smem;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(ring + (size_t)p.stages * p.slot_bytes);
    uint64_t* empty_bar = full_bar + kMaxStages;
    float* xsc = reinterpret_cast<float*>(empty_bar + kMaxStages);
    float* ysum = xsc + kCW * 128;

    const int grid = gridDim.x;
    const int64_t r0 = ((int64_t)blockIdx.x * p.N) / grid;
    const int64_t r1 = ((int64_t)(blockIdx.x + 1) * p.N) / grid;
    const int rows = (int)(r1 - r0);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int nstg = p.stages;
    const int ns = rows > 0 ? (rows + p.tr - 1) / p.tr : 0;
    const int spr = ns > 0 ? (rows + ns - 1) / ns : 0;
    const int active_warps = p.cw * p.rg;
    const int slots = 2 * p.cw;

    if (threadIdx.x == 0) {
        for (int s = 0; s < nstg; s++) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], active_warps);
        }
        fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) griddep_launch_dependents();  // the next kernel of the stream may become resident now

    if (warp == kCW) {
        // ===================== producer warp: one elected lane drives the TMA engine =====================
        if (lane == 0 && rows > 0) {
            if (!p.early_weights) griddep_wait();
            const uint8_t* wsrc = p.w + (uint64_t)r0 * p.row_bytes;
            const uint32_t g2 = (uint32_t)p.G * 2u;
            int s = 0;
            uint32_t phase = 0;
            for (int it = 0; it < ns; it++) {
                mbar_wait(&empty_bar[s], phase ^ 1u);
                const int ra = it * spr;
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
        // lane -> (weight row inside the set, group slice) of the two A-row parts (rows g and g+8 of the MMA)
        const int wrow = MP == 1 ? (g >> 2) : (MP == 2 ? (g >> 1) : g);
        const int sA = MP == 1 ? (g & 3) : (g & 1);
        const int sB = MP == 1 ? 4 + (g & 3) : (MP == 2 ? 2 + (g & 1) : (sA ^ 1));
        // lane as B-column holder: column g = (slice, token)
        const int bsl = g / MP, btok = g % MP;

        griddep_wait();  // x (and y) belong to the previous kernels of the stream

        // ---- stationary operands: B fragments (activations in LOP3 pair order), accumulator init, group sums
        uint32_t bfr[CPW][NP];
        float* myx = xsc + warp * 128;  // [64] sum of x per (group, token); [64] same, weighted like the B fragments
#pragma unroll
        for (int j = 0; j < CPW; j++) {
            const int c = cwi + j * p.cw;
            const bool ld = (c < p.nch) && (btok < p.M);
            const int64_t k0 = ((int64_t)c * S + bsl) * GS + t * CQ;
            uint32_t n32[NP];  // n32[i] = codes (2i, 2i+1) of the chunk, natural order
            if constexpr (CQ >= 8) {
                const uint4* src = reinterpret_cast<const uint4*>(p.x + (size_t)btok * p.K + k0);
#pragma unroll
                for (int v = 0; v < CQ / 8; v++) {
                    const uint4 q = ld ? __ldg(src + v) : make_uint4(0u, 0u, 0u, 0u);
                    n32[4 * v + 0] = q.x; n32[4 * v + 1] = q.y; n32[4 * v + 2] = q.z; n32[4 * v + 3] = q.w;
                }
            } else {  // CQ == 4
                const uint2 q = ld ? __ldg(reinterpret_cast<const uint2*>(p.x + (size_t)btok * p.K + k0)) : make_uint2(0u, 0u);
                n32[0] = q.x; n32[1] = q.y;
            }
            float sx = 0.f;
#pragma unroll
            for (int i = 0; i < NP; i++) {
                sx += __uint_as_float(n32[i] << 16);
                sx += __uint_as_float(n32[i] & 0xffff0000u);
            }
            sx += __shfl_xor_sync(0xffffffffu, sx, 1);
            sx += __shfl_xor_sync(0xffffffffu, sx, 2);
            float sw = 0.f;  // sum of the B column as the MMA sees it (2-bit: x / 4^ce): the offset term is -OFF * scale * sw
#pragma unroll
            for (int q = 0; q < NP; q++) {
                const int ia = pair_a<BITS>(q), ib = pair_b<BITS>(q);
                const uint32_t sel = ((ia & 1) ? 0x32u : 0x10u) | (((ib & 1) ? 0x76u : 0x54u) << 8);
                uint32_t v = __byte_perm(n32[ia >> 1], n32[ib >> 1], sel);
                if constexpr (BITS == 2) {
                    const int ce = cexp2(q & 7);  // field used in place: value 128 + 4^ce * q -> x / 4^ce (exact)
                    if (ce == 1) v = hmul2_bf16(v, 0x3E803E80u);       // 0.25
                    else if (ce == 2) v = hmul2_bf16(v, 0x3D803D80u);  // 0.0625
                }
                bfr[j][q] = v;
                if constexpr (BITS == 2) {
                    sw += __uint_as_float(v << 16);
                    sw += __uint_as_float(v & 0xffff0000u);
                }
            }
            if constexpr (BITS == 2) {
                sw += __shfl_xor_sync(0xffffffffu, sw, 1);
                sw += __shfl_xor_sync(0xffffffffu, sw, 2);
            } else {
                sw = sx;
            }
            if (t == 0) {
                myx[(j * S + bsl) * MP + btok] = sx;
                myx[64 + (j * S + bsl) * MP + btok] = -OFF * sw;
            }
        }
        __syncwarp();
        const int brow = lane / LPR, bq = lane % LPR;
        const uint32_t g2 = (uint32_t)p.G * 2u;
        const int lrow0 = rgi * R;
        int ncl = 0;  // live chunk columns of this warp (warp-uniform)
#pragma unroll
        for (int j = 0; j < CPW; j++) ncl += (cwi + j * p.cw < p.nch) ? 1 : 0;
        float xg[NGL][MP], xo[NGL][MP];
        uint32_t bofs[NGL];  // byte offset of the lane's bias entries inside a stage (dead entries: x sum = 0, offset 0)
#pragma unroll
        for (int i = 0; i < NGL; i++) {
            const int idx = bq * NGL + i;
            const int c = cwi + (idx / S) * p.cw;
            const bool on = idx < CPW * S && c < p.nch;
#pragma unroll
            for (int m = 0; m < MP; m++) {
                xg[i][m] = on ? myx[idx * MP + m] : 0.f;
                xo[i][m] = on ? myx[64 + idx * MP + m] : 0.f;
            }
            bofs[i] = (uint32_t)(p.tr + lrow0 + brow) * g2 + (on ? (uint32_t)(c * S + idx % S) * 2u : 0u);
        }

        const uint32_t colstride = (uint32_t)p.cw * KSTEP_B;
        const uint32_t offA = (uint32_t)wrow * p.row_bytes + (uint32_t)cwi * KSTEP_B + (uint32_t)(sA * 4 + t) * TB;
        const uint32_t offB = (uint32_t)wrow * p.row_bytes + (uint32_t)cwi * KSTEP_B + (uint32_t)(sB * 4 + t) * TB;
        const uint32_t sofA = (uint32_t)wrow * g2 + (uint32_t)(cwi * S + sA) * 2u;
        const uint32_t sofB = (uint32_t)wrow * g2 + (uint32_t)(cwi * S + sB) * 2u;
        const uint32_t sstride = (uint32_t)p.cw * S * 2u;

        int s = 0;
        uint32_t phase = 0;
        for (int it = 0; it < ns; it++) {
            const int ra = it * spr;
            int nr = rows - ra;
            if (nr > spr) nr = spr;
            mbar_wait(&full_bar[s], phase);
            const uint8_t* slot = ring + (size_t)s * p.slot_bytes;
            const uint8_t* sslot = slot + p.sb_off;

            float yacc[NSET][4];
            // one (set, chunk column) unit: 2 LDS of packed words, unpack, NH MMAs chained on the group's accumulator, fold
            // with the two group scales.  Sets past `nr` read stale shared memory; their rows are dropped at the write.
            auto unit = [&](int q, int j) {
                const uint8_t* rbase = slot + (uint32_t)(lrow0 + q * W) * p.row_bytes + j * colstride;
                const uint8_t* sbase = sslot + (uint32_t)(lrow0 + q * W) * g2 + j * sstride;
                uint32_t wa[NWORD], wb[NWORD];
                lds_words<NWORD>(rbase + offA, wa);
                lds_words<NWORD>(rbase + offB, wb);
                const float scA = lds_bf16(sbase + sofA);
                const float scB = lds_bf16(sbase + sofB);
                float d[4];
                const float kZero4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int h = 0; h < NH; h++) {
                    const uint32_t a0 = unpack_pair<BITS, NWORD>(wa, 2 * h), a2 = unpack_pair<BITS, NWORD>(wa, 2 * h + 1);
                    const uint32_t a1 = unpack_pair<BITS, NWORD>(wb, 2 * h), a3 = unpack_pair<BITS, NWORD>(wb, 2 * h + 1);
                    if (h == 0) mma16816(d, a0, a1, a2, a3, bfr[j][0], bfr[j][1], kZero4);
                    else mma16816(d, a0, a1, a2, a3, bfr[j][2 * h], bfr[j][2 * h + 1], d);
                    if constexpr (BITS == 8) {
                        const uint32_t t0 = unpack_pair_top<NWORD>(wa, 2 * h), t2 = unpack_pair_top<NWORD>(wa, 2 * h + 1);
                        const uint32_t t1 = unpack_pair_top<NWORD>(wb, 2 * h), t3 = unpack_pair_top<NWORD>(wb, 2 * h + 1);
                        mma16816(d, t0, t1, t2, t3, bfr[j][2 * h], bfr[j][2 * h + 1], d);
                    }
                }
                yacc[q][0] = fmaf(scA, d[0], yacc[q][0]);
                yacc[q][1] = fmaf(scA, d[1], yacc[q][1]);
                yacc[q][2] = fmaf(scB, d[2], yacc[q][2]);
                yacc[q][3] = fmaf(scB, d[3], yacc[q][3]);
            };
#pragma unroll
            for (int q = 0; q < NSET; q++)
#pragma unroll
                for (int e = 0; e < 4; e++) yacc[q][e] = 0.f;
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
            // ---- biases and the code offset: sum_g (bias * sum(x) - OFF * scale * sum(B column)), a rows x groups dot product
            //      against per-lane stationary group sums
            float bacc[MP];
#pragma unroll
            for (int m = 0; m < MP; m++) bacc[m] = 0.f;
#pragma unroll
            for (int i = 0; i < NGL; i++) {
                const float bv = lds_bf16(sslot + bofs[i]);
                const float sv = lds_bf16(sslot + bofs[i] - (uint32_t)p.tr * g2);  // the same entry of the scales
#pragma unroll
                for (int m = 0; m < MP; m++) bacc[m] = fmaf(bv, xg[i][m], fmaf(sv, xo[i][m], bacc[m]));
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[s]);  // slot free: all of this warp's shared-memory reads are done
            if (++s == nstg) {
                s = 0;
                phase ^= 1u;
            }

#pragma unroll
            for (int m = 0; m < MP; m++) {
#pragma unroll
                for (int o = LPR / 2; o > 0; o >>= 1) bacc[m] += __shfl_xor_sync(0xffffffffu, bacc[m], o);
            }
            if (bq == 0 && lrow0 + brow < nr) {
#pragma unroll
                for (int m = 0; m < MP; m++) ysum[((ra + lrow0 + brow) * slots + p.cw + cwi) * MP + m] = bacc[m];
            }
            // ---- keep the meaningful accumulators, fold the lanes of a row with a transposing butterfly
            if constexpr (MP == 1) {
                // part A (c0/c1) meaningful on t == (g>>1)&1, part B (c2/c3) on t == 2 + ((g>>1)&1); element = g&1
                float v[NSET];
#pragma unroll
                for (int q = 0; q < NSET; q++) {
                    const float lo = (g & 1) ? yacc[q][1] : yacc[q][0];
                    const float hi = (g & 1) ? yacc[q][3] : yacc[q][2];
                    const float u = (t & 2) ? hi : lo;
                    v[q] = ((t & 1) == ((g >> 1) & 1)) ? u : 0.f;
                }
                float keep;
                if constexpr (NSET == 2) {
                    keep = (lane & 8) ? v[1] : v[0];
                    const float send = (lane & 8) ? v[0] : v[1];
                    keep += __shfl_xor_sync(0xffffffffu, send, 8);
                } else {
                    keep = v[0] + __shfl_xor_sync(0xffffffffu, v[0], 8);
                }
                keep += __shfl_xor_sync(0xffffffffu, keep, 4);
                keep += __shfl_xor_sync(0xffffffffu, keep, 2);
                keep += __shfl_xor_sync(0xffffffffu, keep, 1);
                const int lr = lrow0 + (NSET == 2 ? 2 * ((lane >> 3) & 1) : 0) + (lane >> 4);
                const bool writer = NSET == 2 ? (lane & 7) == 0 : (lane & 15) == 0;
                if (writer && lr < nr) ysum[((ra + lr) * slots + cwi) * MP] = keep;
            } else if constexpr (MP == 2) {
                // meaningful on (t&1) == (g&1); part = t>>1; c0/c1 (c2/c3) = tokens 0/1; weight row = g>>1
                const bool ok = (t & 1) == (g & 1);
                const float v0 = ok ? ((t & 2) ? yacc[0][2] : yacc[0][0]) : 0.f;
                const float v1 = ok ? ((t & 2) ? yacc[0][3] : yacc[0][1]) : 0.f;
                float keep = (lane & 4) ? v1 : v0;
                const float send = (lane & 4) ? v0 : v1;
                keep += __shfl_xor_sync(0xffffffffu, send, 4);
                keep += __shfl_xor_sync(0xffffffffu, keep, 2);
                keep += __shfl_xor_sync(0xffffffffu, keep, 1);
                const int lr = lrow0 + (lane >> 3);
                if ((lane & 3) == 0 && lr < nr) ysum[((ra + lr) * slots + cwi) * MP + ((lane >> 2) & 1)] = keep;
            } else {
                // MP == 4: columns 2t, 2t+1 = slice t>>1, tokens 2(t&1), 2(t&1)+1; part A meaningful iff (t>>1) == (g&1)
                const bool pa = (t >> 1) == (g & 1);
                const float v0 = pa ? yacc[0][0] : yacc[0][2];
                const float v1 = pa ? yacc[0][1] : yacc[0][3];
                float keep = (lane & 2) ? v1 : v0;
                const float send = (lane & 2) ? v0 : v1;
                keep += __shfl_xor_sync(0xffffffffu, send, 2);
                const int lr = lrow0 + g;
                if (lr < nr) ysum[((ra + lr) * slots + cwi) * MP + 2 * (t & 1) + ((t >> 1) & 1)] = keep;
            }
        }
    } else {
        griddep_wait();
    }
    __syncthreads();
    griddep_wait();  // every thread stores y below (returns at once when a consumer warp has already waited)
    // ---- epilogue: one rounding to bf16, optional bias as a second rounded add, coalesced store
    for (int i = threadIdx.x; i < rows * MP; i += kThreads) {
        const int m = i / rows, r = i - m * rows;
        if (m < p.M) {
            float tot = 0.f;
            for (int c = 0; c < slots; c++) tot += ysum[(r * slots + c) * MP + m];
            float v = __bfloat162float(__float2bfloat16_rn(tot));
            if (p.bias != nullptr) v = __fadd_rn(v, __bfloat162float(p.bias[r0 + r]));
            p.y[(size_t)m * p.N + r0 + r] = __float2bfloat16_rn(v);
        }
    }
}

// ------------------------------------------------------------------------------------------ host side
struct Plan {
    bool ok;
    int mp, tb, cpw, R, nch, cw, rg, tr, stages, grid;
    uint32_t slot_bytes, sb_off;
    size_t smem;
};

Plan make_plan(int64_t M, int64_t N, int64_t K, int bits, int gs) {
    Plan pl{};
    if (!(bits == 2 || bits == 4 || bits == 8) || M < 1 || M > 4 || N < 1) return pl;
    pl.tb = gs * bits / 32;
    if (!(pl.tb == 4 || pl.tb == 8 || pl.tb == 16) || (gs * bits) % 32) return pl;
    const int64_t G = K / gs;
    if (G % 8) return pl;  // S | G for every MP, and 16-byte rows of scales for the bulk copies
    const int64_t row_bytes = K * bits / 8;
    pl.mp = M == 1 ? 1 : (M == 2 ? 2 : 4);
    const int S = 8 / pl.mp, W = 2 * pl.mp;
    pl.nch = (int)(G / S);
    pl.R = W < 4 ? 4 : W;
    static const int force_cpw = env_int("GBXQ_MMV_CPW", 0);
    static const int grid_mult = env_int("GBXQ_MMV_GRID_MULT", 2);
    static const int stage_kb = env_int("GBXQ_MMV_STAGE_KB", 20);
    // chunk columns per warp: 2 when the row is long enough (two independent MMA chains per set), more for long rows
    pl.cpw = pl.nch >= 8 ? 2 : 1;
    while ((pl.nch + pl.cpw - 1) / pl.cpw > kCW && pl.cpw < 4) pl.cpw *= 2;
    if (force_cpw) pl.cpw = force_cpw;
    if (!(pl.cpw == 1 || pl.cpw == 2 || pl.cpw == 4)) return pl;
    pl.cw = (pl.nch + pl.cpw - 1) / pl.cpw;
    if (pl.cw > kCW) return pl;
    if (pl.mp == 1 && (int64_t)pl.R * row_bytes > (int64_t)stage_kb * 1024) pl.R = 2;  // long rows: one set per stage
    pl.rg = kCW / pl.cw;
    while (pl.rg > 1 && (int64_t)pl.rg * pl.R * row_bytes > (int64_t)stage_kb * 1024) pl.rg--;
    pl.tr = pl.rg * pl.R;
    const uint32_t wpart = (uint32_t)(((int64_t)pl.tr * row_bytes + 127) & ~(int64_t)127);
    pl.sb_off = wpart;
    pl.slot_bytes = wpart + (uint32_t)((2 * (int64_t)pl.tr * G * 2 + 127) & ~(int64_t)127);
    static const int ring_kb = env_int("GBXQ_MMV_RING_KB", 64);
    pl.stages = kMaxStages;
    while (pl.stages > 2 && (size_t)pl.stages * pl.slot_bytes > (size_t)ring_kb * 1024) pl.stages--;
    int grid = device_sm_count() * grid_mult;
    // at least ~2 stages of rows per CTA, never more CTAs than rows
    const int64_t min_rows = pl.tr;
    if ((int64_t)grid * min_rows > N) grid = (int)((N + min_rows - 1) / min_rows);
    if (grid < 1) grid = 1;
    pl.grid = grid;
    const int64_t rows_max = (N + grid - 1) / grid;
    pl.smem = (size_t)pl.stages * pl.slot_bytes + 2 * kMaxStages * 8 + (size_t)kCW * 128 * 4 +
              (size_t)rows_max * 2 * pl.cw * pl.mp * 4 + 16;
    if (pl.smem > 110 * 1024) return pl;
    pl.ok = true;
    return pl;
}

template <int BITS, int TB, int MP, int CPW, int R>
int launch_inst(const MmvParams& p, const Plan& pl, cudaStream_t st) {
    constexpr auto kern = mmv_kernel<BITS, TB, MP, CPW, R>;
    const int rc = allow_dynamic_smem<kern>(110 * 1024);
    if (rc != GBXQ_OK) return rc;
    return launch(kern, dim3((unsigned)pl.grid), dim3(kThreads), pl.smem, st, true, p);
}

template <int BITS, int TB, int MP, int CPW>
int launch_r(const MmvParams& p, const Plan& pl, cudaStream_t st) {
    constexpr int W = 2 * MP;
    constexpr int RDEF = W < 4 ? 4 : W;
    if (pl.R == RDEF) return launch_inst<BITS, TB, MP, CPW, RDEF>(p, pl, st);
    if constexpr (MP == 1) {
        if (pl.R == 2) return launch_inst<BITS, TB, MP, CPW, 2>(p, pl, st);
    }
    return GBXQ_EUNSUPPORTED;
}

template <int BITS, int TB, int MP>
int launch_cpw(const MmvParams& p, const Plan& pl, cudaStream_t st) {
    switch (pl.cpw) {
        case 1: return launch_r<BITS, TB, MP, 1>(p, pl, st);
        case 2: return launch_r<BITS, TB, MP, 2>(p, pl, st);
        case 4: return launch_r<BITS, TB, MP, 4>(p, pl, st);
    }
    return GBXQ_EUNSUPPORTED;
}

template <int BITS, int TB>
int launch_mp(const MmvParams& p, const Plan& pl, cudaStream_t st) {
    switch (pl.mp) {
        case 1: return launch_cpw<BITS, TB, 1>(p, pl, st);
        case 2: return launch_cpw<BITS, TB, 2>(p, pl, st);
        case 4: return launch_cpw<BITS, TB, 4>(p, pl, st);
    }
    return GBXQ_EUNSUPPORTED;
}

template <int BITS>
int launch_tb(const MmvParams& p, const Plan& pl, cudaStream_t st) {
    if constexpr (BITS != 8) {
        if (pl.tb == 4) return launch_mp<BITS, 4>(p, pl, st);
    }
    if (pl.tb == 8) return launch_mp<BITS, 8>(p, pl, st);
    if constexpr (BITS != 2) {
        if (pl.tb == 16) return launch_mp<BITS, 16>(p, pl, st);
    }
    return GBXQ_EUNSUPPORTED;
}

}  // namespace

bool mmv_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                   const void* y) {
    if (dtype != GBXQ_BF16 || M < 1 || N < 1) return false;
    if (((uintptr_t)x | (uintptr_t)w) & 15) return false;
    if ((uintptr_t)y & 1) return false;
    if ((K * 2) % 16) return false;
    return make_plan(M, N, K, bits, gs).ok;
}

int launch_mmv(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
               int64_t N, int64_t K, int bits, int gs, cudaStream_t st) {
    if (((uintptr_t)s | (uintptr_t)b) & 15) return GBXQ_EUNSUPPORTED;
    const Plan pl = make_plan(M, N, K, bits, gs);
    if (!pl.ok) return GBXQ_EUNSUPPORTED;
    MmvParams p{};
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
    p.early_weights = pdl_early_weights();
    switch (bits) {
        case 2: return launch_tb<2>(p, pl, st);
        case 4: return launch_tb<4>(p, pl, st);
        case 8: return launch_tb<8>(p, pl, st);
    }
    return GBXQ_EINVAL_BITS;
}

}  // namespace gbxq
