// gbxq_skinny.cu -- decode GEMV / skinny matmul for 1..8 rows of x per pass on the tensor pipe
// (bf16 activations; 2-, 4- and 8-bit packings).
//
// Hot path of gbx-lm decode: QuantizedLinear.__call__ -> mx.quantized_matmul(transpose=True)
// (gbx_lm/models/quantized_linear_gba.py:195-203) with M = batch rows of x ("decode batch 1-16").
//
// Why tensor cores for an HBM-bound GEMV: at 4 bits a B200 SM must retire ~46 weights per clock to
// keep up with its share of HBM; one FMA per weight on the CUDA cores (gbxq_gemv.cu) already spends
// the whole issue budget.  Here the multiply-accumulate goes to `mma.sync.m16n8k16` (A = 16 weight
// rows x 16 k, B = 16 k x 8 tokens): 0.125 issue slots per weight instead of 1, so the kernel is
// bounded by the packed-byte stream again, and 8 tokens cost the same as one.
//
//   * Work split: a CTA owns a contiguous range of weight rows (balanced at single-row granularity).
//     It walks row-blocks (<= 64 rows) x k-tiles (16 quantisation groups, one per consumer warp).
//     Stage = (row-block, k-tile): the producer issues one 2-D TMA box [rows x 128 B] per 128 bytes of
//     row piece (cp.async.bulk.tensor.2d, SWIZZLE_128B so that the fragment loads of 8 different rows
//     hit different banks) into a 4-deep shared-memory ring, completion counted in bytes on an
//     mbarrier.  (Per-row 1-D bulk copies were measured at ~85 cycles per request -- 6 B/clk/SM --
//     which is why the tile goes through tensor maps.)
//   * Consumer warp w owns group (16*kt + w): thread (g, t) of the warp holds the t-th quarter of
//     the group's codes of rows g and g+8 -- exactly the m16n8k16 A fragment.  The k order inside a
//     group is free, so the pair one LOP3 extracts ((w >> s) & mask | 0x4300 = two bf16 values
//     128+q) IS an A register; the matching activations are permuted once per stage into the B
//     fragment.  All 16 k-slots of every MMA belong to one quantisation group, so the group's partial
//     product sits alone in the accumulator and is folded as
//         y += scale * D + (bias - OFF*scale) * sum(x over the group)
//     in fp32 (OFF = 128 carried by the bf16 images of the codes; 256 for the two 8-bit images).
//   * the stage's scales and biases ride the same ring (one 2-D TMA box [rows x 16 groups] each), the x
//     B-fragments are prefetched one stage ahead from L2 into registers, and sum(x) per group comes
//     out of one extra MMA against an all-ones A fragment; the 16 per-warp partial sums of a row-block meet in shared memory and are added in
//     fixed order (bitwise reproducible), rounded once to bf16 (+ optional bias as a second rounded
//     add) and stored coalesced.
#include <cuda.h>
#include <string.h>

#include "gbxq_common.cuh"

namespace gbxq {

namespace {

constexpr int kWarps = 16;                   // consumer warps == groups per k-tile
constexpr int kThreads = (kWarps + 1) * 32;  // + producer warp
constexpr int kStages = 4;
constexpr int kMaxRS = 64;                   // rows per stage (multiple of 16)
constexpr uint32_t kMagic = 0x43004300u;

__device__ __forceinline__ void mma16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// pair p of a thread's quarter = codes (pa, pb) that one LOP3 extracts together
template <int BITS> __host__ __device__ constexpr int pair_a(int p) {
    if (BITS == 4) return 8 * (p >> 2) + (p & 3);
    if (BITS == 2) return 16 * (p >> 3) + (p & 7);
    return 4 * (p >> 1) + (p & 1);  // 8-bit
}
template <int BITS> __host__ __device__ constexpr int pair_b(int p) {
    return pair_a<BITS>(p) + (BITS == 4 ? 4 : (BITS == 2 ? 8 : 2));
}

struct SkinnyParams {
    const __nv_bfloat16* x;
    const uint8_t* w;
    const uint16_t* scales;
    const uint16_t* biases;
    const __nv_bfloat16* bias;
    __nv_bfloat16* y;
    int64_t N, K;
    int M;            // tokens in this pass (1..8)
    int G;            // groups per row
    int n_kt;         // k-tiles (16 groups each)
    int rs;           // rows per stage (multiple of 16, <= kMaxRS)
    uint32_t row_bytes;
    uint32_t piece_words;  // 32-bit words of one row inside a full k-tile (16 groups)
    int nbox;              // 128-byte-wide TMA boxes per row piece
    uint32_t sb_off;       // offset of the scale box inside a ring slot (bias box follows at + rs*32)
    uint32_t slot_bytes;
    int early_weights;     // 1: parameters are frozen -> the producer streams them before griddepcontrol.wait (GBXQ_OPT_PDL 2)
};

__device__ __forceinline__ void tma_load_2d(void* dst, const void* tmap, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}

// BITS in {2,4,8}; QW = 32-bit words per thread-quarter of a group (= group_size * BITS / 128)
// NT = token octets per pass (1: up to 8 tokens, 2: up to 16): the second octet reuses the unpacked A registers, so
// 9..16 tokens cost two more MMAs and folds per tile instead of a second pass over the weights.
template <int BITS, int QW, bool SB_TMA, int NT>
__global__ void __launch_bounds__(kThreads, 1)
skinny_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_s,
              const __grid_constant__ CUtensorMap tmap_b, const SkinnyParams p) {
    constexpr int CQ = QW * 32 / BITS;       // codes per quarter
    constexpr int P = CQ / 2;                // pairs (= A/B registers) per quarter
    constexpr int S = P / 2;                 // MMA k16 steps per group
    constexpr int GS = CQ * 4;               // group size
    constexpr int RT = kMaxRS / 16;          // row tiles per stage (upper bound)
    constexpr float OFF = BITS == 8 ? 256.f : 128.f;
    static_assert(S >= 1 && (QW == 1 || QW == 2 || QW == 4 || QW == 8), "unsupported quarter");

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // layout: [ring kStages * slot][barriers][red kWarps * rs * 8 f32]; slot = [nbox boxes of rs rows x 128 B,
    // 128B-swizzled][scales rs x 16 bf16][biases rs x 16 bf16]
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const uint32_t slot_bytes = p.slot_bytes;
    uint8_t* ring = smem;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(ring + (size_t)kStages * slot_bytes);
    uint64_t* empty_bar = full_bar + kStages;
    float* red = reinterpret_cast<float*>(empty_bar + kStages);

    const int grid = gridDim.x;
    const int64_t r0 = ((int64_t)blockIdx.x * p.N) / grid;
    const int64_t r1 = ((int64_t)(blockIdx.x + 1) * p.N) / grid;
    const int rows = (int)(r1 - r0);
    if (rows <= 0) return;
    const int n_rb = (rows + p.rs - 1) / p.rs;
    const int rb_rows = ((rows + n_rb - 1) / n_rb + 15) & ~15;  // balanced row-blocks, multiple of 16
    const int ns = n_rb * p.n_kt;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < kStages; s++) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], kWarps);
        }
        fence_mbar_init();
    }
    __syncthreads();
    // programmatic dependent launch, as in the mmv8 kernels: the next kernel of the stream may become resident now;
    // x and y are touched only after griddepcontrol.wait (a no-op for plain launches)
    if (threadIdx.x == 0) griddep_launch_dependents();

    if (warp == kWarps) {
        // ===================== producer: a handful of TMA boxes per stage =====================
        if (lane == 0) {
            if (!p.early_weights) griddep_wait();
            const uint32_t box_bytes = (uint32_t)p.rs * 128u;
            for (int it = 0; it < ns; it++) {
                const int s = it % kStages;
                const uint32_t phase = (uint32_t)(it / kStages) & 1u;
                const int rb = it / p.n_kt, kt = it - rb * p.n_kt;
                const int row = (int)(r0 + rb * rb_rows);
                mbar_wait(&empty_bar[s], phase ^ 1u);
                uint8_t* dst = ring + (size_t)s * slot_bytes;
                // boxes always count full bytes: rows past N and words past the row end are zero-filled by the TMA unit
                mbar_arrive_expect_tx(&full_bar[s], (uint32_t)p.nbox * box_bytes + (SB_TMA ? 2u * (uint32_t)p.rs * 32u : 0u));
                for (int b = 0; b < p.nbox; b++)
                    tma_load_2d(dst + (size_t)b * box_bytes, &tmap_w, kt * (int)p.piece_words + b * 32, row, &full_bar[s]);
                if constexpr (SB_TMA) {
                    tma_load_2d(dst + p.sb_off, &tmap_s, kt * kWarps, row, &full_bar[s]);
                    tma_load_2d(dst + p.sb_off + (uint32_t)p.rs * 32u, &tmap_b, kt * kWarps, row, &full_bar[s]);
                }
            }
        }
    } else {
        // ===================== consumer warps =====================
        const int g = lane >> 2, t = lane & 3;
        const uint32_t ring_u32 = smem_u32(ring);
        griddep_wait();  // x (and y) belong to the previous kernels of the stream

        struct Pre {            // per-stage operands fetched one stage ahead
            uint4 xn[NT][(CQ * 2 + 15) / 16];  // this thread's quarter of tokens g (+8), natural order (CQ bf16)
            uint32_t sc[RT][2], bi[RT][2];  // raw bf16 scale / bias of rows (16q+g, 16q+g+8)
        };
        constexpr int XV = (CQ * 2 + 15) / 16;

        auto prefetch = [&](int it, Pre& pre) {
            const int rb = it / p.n_kt, kt = it - rb * p.n_kt;
            const int grp = kt * kWarps + warp;
            const bool gv = it < ns && grp < p.G;
            const int ra = rb * rb_rows;
            int nr = rows - ra;
            if (nr > rb_rows) nr = rb_rows;
            const int64_t k0 = (int64_t)grp * GS + t * CQ;
            if constexpr (CQ * 2 >= 16) {
#pragma unroll
                for (int nt = 0; nt < NT; nt++) {
                    const int tk = g + 8 * nt;
                    const uint4* src = reinterpret_cast<const uint4*>(p.x + (size_t)tk * p.K + k0);
#pragma unroll
                    for (int v = 0; v < XV; v++) pre.xn[nt][v] = (gv && tk < p.M) ? __ldg(src + v) : make_uint4(0u, 0u, 0u, 0u);
                }
            } else {  // CQ == 4 codes (8-bit, gs 32... not instantiated) -- kept for completeness
#pragma unroll
                for (int nt = 0; nt < NT; nt++) pre.xn[nt][0] = make_uint4(0u, 0u, 0u, 0u);
            }
            if constexpr (!SB_TMA) {
#pragma unroll
                for (int q = 0; q < RT; q++) {
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        const int lr = 16 * q + g + 8 * h;
                        const bool ok = gv && lr < nr;
                        const int64_t gi = (r0 + ra + lr) * (int64_t)p.G + grp;
                        pre.sc[q][h] = ok ? (uint32_t)__ldg(p.scales + gi) : 0u;
                        pre.bi[q][h] = ok ? (uint32_t)__ldg(p.biases + gi) : 0u;
                    }
                }
            }
        };

        float yacc[NT][RT][4];
#pragma unroll
        for (int nt = 0; nt < NT; nt++)
#pragma unroll
            for (int q = 0; q < RT; q++)
#pragma unroll
                for (int e = 0; e < 4; e++) yacc[nt][q][e] = 0.f;

        auto consume = [&](int it, const Pre& pre) {
            const int s = it % kStages;
            const uint32_t phase = (uint32_t)(it / kStages) & 1u;
            const int rb = it / p.n_kt, kt = it - rb * p.n_kt;
            const int grp = kt * kWarps + warp;
            const int ra = rb * rb_rows;
            int nr = rows - ra;
            if (nr > rb_rows) nr = rb_rows;
            const int nrt = (nr + 15) >> 4;

            // ---- B fragments: permute this thread's quarter of x into LOP3 pair order.  sum(x) over the group
            //      for tokens (2t, 2t+1) = one more MMA chain against an all-ones A fragment (exact: 1.0 * x)
            uint32_t bfrag[NT][P];
            float xs0[NT], xs1[NT];
#pragma unroll
            for (int nt = 0; nt < NT; nt++) {
                const uint32_t* n32 = reinterpret_cast<const uint32_t*>(pre.xn[nt]);  // n32[i] = codes (2i, 2i+1)
#pragma unroll
                for (int q = 0; q < P; q++) {
                    const int ia = pair_a<BITS>(q), ib = pair_b<BITS>(q);
                    const uint32_t sel = ((ia & 1) ? 0x32u : 0x10u) | (((ib & 1) ? 0x76u : 0x54u) << 8);
                    bfrag[nt][q] = __byte_perm(n32[ia >> 1], n32[ib >> 1], sel);
                }
                float d1[4] = {0.f, 0.f, 0.f, 0.f};
                constexpr uint32_t kOnes = 0x3F803F80u;
#pragma unroll
                for (int st = 0; st < S; st++) mma16816(d1, kOnes, kOnes, kOnes, kOnes, bfrag[nt][2 * st], bfrag[nt][2 * st + 1]);
                xs0[nt] = d1[0];
                xs1[nt] = d1[1];
            }

            mbar_wait(&full_bar[s], phase);
            if (grp < p.G) {  // warp-uniform: the last k-tile may hold fewer than 16 groups
                // this thread's quarter inside the stage: byte `off` of the row piece -> TMA box off/128, 16-byte chunk
                // (off%128)/16 XOR (row & 7) (SWIZZLE_128B; rows 16q+g and 16q+g+8 share row&7 == g)
                constexpr int NPC = QW == 8 ? 2 : 1;  // 16-byte pieces per quarter
                uint32_t toff[NPC];
#pragma unroll
                for (int v = 0; v < NPC; v++) {
                    const uint32_t off = (uint32_t)warp * (QW * 16) + (uint32_t)t * (QW * 4) + 16u * v;
                    toff[v] = (off >> 7) * ((uint32_t)p.rs * 128u) + ((((off & 127u) >> 4) ^ (uint32_t)g) << 4) + (off & 15u) +
                              (uint32_t)g * 128u;
                }
                const uint32_t base = ring_u32 + (uint32_t)s * slot_bytes;
                const uint32_t sbase = ring_u32 + (uint32_t)s * slot_bytes + p.sb_off + (uint32_t)warp * 2u;
                (void)sbase;
#pragma unroll
                for (int q = 0; q < RT; q++) {
                    if (q < nrt) {  // warp-uniform
                        uint32_t wl[QW], wh[QW];
                        const uint32_t al = base + toff[0] + (uint32_t)q * 2048u;
                        const uint32_t ah = al + 1024u;
                        if constexpr (QW == 1) {
                            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(wl[0]) : "r"(al));
                            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(wh[0]) : "r"(ah));
                        } else if constexpr (QW == 2) {
                            asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(wl[0]), "=r"(wl[1]) : "r"(al));
                            asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(wh[0]), "=r"(wh[1]) : "r"(ah));
                        } else {
#pragma unroll
                            for (int v = 0; v < QW / 4; v++) {
                                const uint32_t dv = toff[v < NPC ? v : 0] - toff[0];
                                const uint4 a = lds128(al + dv), b = lds128(ah + dv);
                                wl[4 * v] = a.x; wl[4 * v + 1] = a.y; wl[4 * v + 2] = a.z; wl[4 * v + 3] = a.w;
                                wh[4 * v] = b.x; wh[4 * v + 1] = b.y; wh[4 * v + 2] = b.z; wh[4 * v + 3] = b.w;
                            }
                        }
                        float d[NT][4];
#pragma unroll
                        for (int nt = 0; nt < NT; nt++)
#pragma unroll
                            for (int e = 0; e < 4; e++) d[nt][e] = 0.f;
#pragma unroll
                        for (int st = 0; st < S; st++) {
                            // pairs 2st, 2st+1 of the quarter -> (a0,a1) and (a2,a3)
                            uint32_t al2[2], ah2[2], al2b[2], ah2b[2];
#pragma unroll
                            for (int e = 0; e < 2; e++) {
                                const int pr = 2 * st + e;
                                if constexpr (BITS == 4) {
                                    const int wi = pr >> 2, sh = 4 * (pr & 3);
                                    al2[e] = lop3_and_or(wl[wi] >> sh, 0x000f000fu, kMagic);
                                    ah2[e] = lop3_and_or(wh[wi] >> sh, 0x000f000fu, kMagic);
                                } else if constexpr (BITS == 2) {
                                    const int wi = pr >> 3, sh = 2 * (pr & 7);
                                    al2[e] = lop3_and_or(wl[wi] >> sh, 0x00030003u, kMagic);
                                    ah2[e] = lop3_and_or(wh[wi] >> sh, 0x00030003u, kMagic);
                                } else {
                                    const int wi = pr >> 1, sh = 8 * (pr & 1);
                                    al2[e] = lop3_and_or(wl[wi] >> sh, 0x007f007fu, kMagic);
                                    ah2[e] = lop3_and_or(wh[wi] >> sh, 0x007f007fu, kMagic);
                                    al2b[e] = lop3_and_or(wl[wi] >> sh, 0x00800080u, kMagic);
                                    ah2b[e] = lop3_and_or(wh[wi] >> sh, 0x00800080u, kMagic);
                                }
                            }
#pragma unroll
                            for (int nt = 0; nt < NT; nt++) {
                                mma16816(d[nt], al2[0], ah2[0], al2[1], ah2[1], bfrag[nt][2 * st], bfrag[nt][2 * st + 1]);
                                if constexpr (BITS == 8)
                                    mma16816(d[nt], al2b[0], ah2b[0], al2b[1], ah2b[1], bfrag[nt][2 * st], bfrag[nt][2 * st + 1]);
                            }
                        }
                        uint32_t s0, s1, b0, b1;
                        if constexpr (SB_TMA) {
                            // [rs][16] bf16 boxes: (row, this warp's group); rows beyond the tensor are zero-filled
                            const uint32_t sa = sbase + (uint32_t)(16 * q + g) * 32u;
                            asm volatile("ld.shared.u16 %0, [%1];" : "=r"(s0) : "r"(sa));
                            asm volatile("ld.shared.u16 %0, [%1];" : "=r"(s1) : "r"(sa + 256u));
                            asm volatile("ld.shared.u16 %0, [%1];" : "=r"(b0) : "r"(sa + (uint32_t)p.rs * 32u));
                            asm volatile("ld.shared.u16 %0, [%1];" : "=r"(b1) : "r"(sa + (uint32_t)p.rs * 32u + 256u));
                        } else {
                            s0 = pre.sc[q][0]; s1 = pre.sc[q][1]; b0 = pre.bi[q][0]; b1 = pre.bi[q][1];
                        }
                        const float sl = __uint_as_float(s0 << 16), sh_ = __uint_as_float(s1 << 16);
                        const float cl = fmaf(-OFF, sl, __uint_as_float(b0 << 16));
                        const float ch = fmaf(-OFF, sh_, __uint_as_float(b1 << 16));
#pragma unroll
                        for (int nt = 0; nt < NT; nt++) {
                            yacc[nt][q][0] = fmaf(sl, d[nt][0], fmaf(cl, xs0[nt], yacc[nt][q][0]));
                            yacc[nt][q][1] = fmaf(sl, d[nt][1], fmaf(cl, xs1[nt], yacc[nt][q][1]));
                            yacc[nt][q][2] = fmaf(sh_, d[nt][2], fmaf(ch, xs0[nt], yacc[nt][q][2]));
                            yacc[nt][q][3] = fmaf(sh_, d[nt][3], fmaf(ch, xs1[nt], yacc[nt][q][3]));
                        }
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[s]);

            if (kt == p.n_kt - 1) {
                // ---- row-block done: 16 per-warp partials -> shared memory -> fixed-order sum -> y
                float* mine = red + (size_t)warp * (p.rs * 8 * NT);
#pragma unroll
                for (int q = 0; q < RT; q++) {
#pragma unroll
                    for (int nt = 0; nt < NT; nt++) {
                        if (q < nrt) {
                            const int rl = 16 * q + g;
                            *reinterpret_cast<float2*>(mine + rl * (8 * NT) + 8 * nt + 2 * t) = make_float2(yacc[nt][q][0], yacc[nt][q][1]);
                            *reinterpret_cast<float2*>(mine + (rl + 8) * (8 * NT) + 8 * nt + 2 * t) = make_float2(yacc[nt][q][2], yacc[nt][q][3]);
                        }
#pragma unroll
                        for (int e = 0; e < 4; e++) yacc[nt][q][e] = 0.f;
                    }
                }
                asm volatile("bar.sync 1, %0;" ::"n"(kWarps * 32) : "memory");
                const int ctid = threadIdx.x;
                for (int i = ctid; i < nr * p.M; i += kWarps * 32) {
                    const int m = i / nr, r = i - m * nr;
                    float tot = 0.f;
#pragma unroll
                    for (int w2 = 0; w2 < kWarps; w2++) tot += red[(size_t)w2 * (p.rs * 8 * NT) + r * (8 * NT) + m];
                    float v = __bfloat162float(__float2bfloat16_rn(tot));
                    if (p.bias != nullptr) v = __fadd_rn(v, __bfloat162float(p.bias[r0 + ra + r]));
                    p.y[(size_t)m * p.N + r0 + ra + r] = __float2bfloat16_rn(v);
                }
                asm volatile("bar.sync 1, %0;" ::"n"(kWarps * 32) : "memory");
            }
        };

        Pre pa, pb;
        prefetch(0, pa);
        for (int it = 0; it < ns;) {
            prefetch(it + 1, pb);
            consume(it, pa);
            if (++it >= ns) break;
            prefetch(it + 1, pa);
            consume(it, pb);
            ++it;
        }
    }
}

struct Plan {
    bool ok, sb_tma;
    int qw, rs, n_kt;
    uint32_t piece, sb_off, slot;
    int nbox;
    size_t smem;
};

Plan make_plan(int64_t N, int64_t K, int bits, int gs, int nt = 1) {
    Plan pl{};
    if (!(bits == 2 || bits == 4 || bits == 8)) return pl;
    if ((gs * bits) % 128) return pl;
    pl.qw = gs * bits / 128;
    if (!(pl.qw == 1 || pl.qw == 2 || pl.qw == 4 || pl.qw == 8)) return pl;
    if (gs / 4 * 2 < 16) return pl;  // a quarter of x must be at least one 16-byte vector (gs >= 32)
    const int64_t row_bytes = K * bits / 8;
    if (row_bytes % 16) return pl;
    const int64_t G = K / gs;
    pl.piece = (uint32_t)(kWarps * gs * bits / 8);
    if (pl.piece % 16) return pl;
    pl.n_kt = (int)((G + kWarps - 1) / kWarps);
    if (pl.piece % 128) return pl;
    pl.nbox = (int)(pl.piece / 128);
    int rs = (int)((32 * 1024) / pl.piece) & ~15;
    if (rs > kMaxRS) rs = kMaxRS;
    if (rs < 16) return pl;
    pl.rs = rs;
    pl.sb_tma = (G * 2) % 16 == 0;  // TMA needs a 16-byte row pitch for the scale / bias matrices
    pl.sb_off = (uint32_t)rs * pl.piece;
    pl.slot = pl.sb_off + 2u * (uint32_t)rs * 32u;  // multiple of 1024: every slot keeps the swizzle alignment
    pl.smem = (size_t)kStages * pl.slot + 2 * kStages * 8 + (size_t)kWarps * rs * 8 * 4 * nt + 16 + 1024;
    if (pl.smem > 227 * 1024) return pl;
    (void)N;
    pl.ok = true;
    return pl;
}

template <int BITS, int QW, bool SB_TMA, int NT>
int launch_inst3(const CUtensorMap& tw, const CUtensorMap& ts, const CUtensorMap& tb, const SkinnyParams& p, size_t smem, int grid,
                 cudaStream_t st) {
    constexpr auto kern = skinny_kernel<BITS, QW, SB_TMA, NT>;
    const int rc = allow_dynamic_smem<kern>(227 * 1024);
    if (rc != GBXQ_OK) return rc;
    return launch(kern, dim3((unsigned)grid), dim3(kThreads), smem, st, true, tw, ts, tb, p);
}

template <int BITS, int QW, bool SB_TMA>
int launch_inst2(const CUtensorMap& tw, const CUtensorMap& ts, const CUtensorMap& tb, const SkinnyParams& p, size_t smem, int grid,
                 cudaStream_t st) {
    return p.M > 8 ? launch_inst3<BITS, QW, SB_TMA, 2>(tw, ts, tb, p, smem, grid, st)
                   : launch_inst3<BITS, QW, SB_TMA, 1>(tw, ts, tb, p, smem, grid, st);
}

template <int BITS, int QW>
int launch_inst(bool sb_tma, const CUtensorMap& tw, const CUtensorMap& ts, const CUtensorMap& tb, const SkinnyParams& p,
                size_t smem, int grid, cudaStream_t st) {
    return sb_tma ? launch_inst2<BITS, QW, true>(tw, ts, tb, p, smem, grid, st)
                  : launch_inst2<BITS, QW, false>(tw, ts, tb, p, smem, grid, st);
}

}  // namespace

bool skinny_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                      const void* y) {
    if (dtype != GBXQ_BF16 || M < 1 || N < 1) return false;
    if (((uintptr_t)x | (uintptr_t)w) & 15) return false;
    if ((uintptr_t)y & 1) return false;
    if ((K * 2) % 16) return false;
    return make_plan(N, K, bits, gs).ok && tma_encode_available();
}

int launch_skinny(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                  int64_t N, int64_t K, int bits, int gs, cudaStream_t st) {
    const Plan pl = make_plan(N, K, bits, gs);
    if (!pl.ok) return GBXQ_EUNSUPPORTED;
    SkinnyParams p{};
    p.w = reinterpret_cast<const uint8_t*>(w);
    p.scales = reinterpret_cast<const uint16_t*>(s);
    p.biases = reinterpret_cast<const uint16_t*>(b);
    p.bias = reinterpret_cast<const __nv_bfloat16*>(bias);
    p.N = N;
    p.K = K;
    p.G = (int)(K / gs);
    p.n_kt = pl.n_kt;
    p.rs = pl.rs;
    p.row_bytes = (uint32_t)(K * bits / 8);
    p.piece_words = pl.piece / 4;
    p.nbox = pl.nbox;
    p.sb_off = pl.sb_off;
    p.slot_bytes = pl.slot;
    p.early_weights = pdl_early_weights();
    CUtensorMap tw, ts, tb;
    memset(&ts, 0, sizeof(ts));
    memset(&tb, 0, sizeof(tb));
    {
        const uint64_t words = (uint64_t)(K * bits / 32);
        if (!encode_tensor_map_2d(&tw, /*uint32*/ 1, w, words, (uint64_t)N, words * 4, 32, (uint32_t)pl.rs, true))
            return GBXQ_EUNSUPPORTED;
    }
    bool sb_tma = pl.sb_tma && !(((uintptr_t)s | (uintptr_t)b) & 15);
    if (sb_tma) {
        const uint64_t G = (uint64_t)(K / gs);
        sb_tma = encode_tensor_map_2d(&ts, /*bf16*/ 0, s, G, (uint64_t)N, G * 2, kWarps, (uint32_t)pl.rs, false) &&
                 encode_tensor_map_2d(&tb, 0, b, G, (uint64_t)N, G * 2, kWarps, (uint32_t)pl.rs, false);
    }
    int grid = device_sm_count();
    if (grid > N) grid = (int)N;
    // 16 tokens per pass when more than 8 remain and the 16-token reduction buffer fits (else octets)
    const Plan pl2 = make_plan(N, K, bits, gs, 2);
    for (int64_t m0 = 0; m0 < M;) {
        const int64_t left = M - m0;
        const int take = (left > 8 && pl2.ok) ? (int)(left < 16 ? left : 16) : (int)(left < 8 ? left : 8);
        p.x = reinterpret_cast<const __nv_bfloat16*>(x) + m0 * K;
        p.y = reinterpret_cast<__nv_bfloat16*>(y) + m0 * N;
        p.M = take;
        const size_t smem_now = take > 8 ? pl2.smem : pl.smem;
        m0 += take;
        int rc = GBXQ_EUNSUPPORTED;
        switch (bits * 16 + pl.qw) {
            case 4 * 16 + 1: rc = launch_inst<4, 1>(sb_tma, tw, ts, tb, p, smem_now, grid, st); break;
            case 4 * 16 + 2: rc = launch_inst<4, 2>(sb_tma, tw, ts, tb, p, smem_now, grid, st); break;
            case 4 * 16 + 4: rc = launch_inst<4, 4>(sb_tma, tw, ts, tb, p, smem_now, grid, st); break;
            case 2 * 16 + 1: rc = launch_inst<2, 1>(sb_tma, tw, ts, tb, p, smem_now, grid, st); break;
            case 2 * 16 + 2: rc = launch_inst<2, 2>(sb_tma, tw, ts, tb, p, smem_now, grid, st); break;
            case 8 * 16 + 2: rc = launch_inst<8, 2>(sb_tma, tw, ts, tb, p, smem_now, grid, st); break;
            case 8 * 16 + 4: rc = launch_inst<8, 4>(sb_tma, tw, ts, tb, p, smem_now, grid, st); break;
            case 8 * 16 + 8: rc = launch_inst<8, 8>(sb_tma, tw, ts, tb, p, smem_now, grid, st); break;
        }
        if (rc != GBXQ_OK) return rc;
    }
    return GBXQ_OK;
}

}  // namespace gbxq
