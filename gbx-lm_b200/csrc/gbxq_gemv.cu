// gbxq_gemv.cu -- decode GEMV / skinny matmul (M tiles of 1 or 2 tokens) for bf16 activations.
//
// Hot path of gbx-lm decode: QuantizedLinear.__call__ -> mx.quantized_matmul(transpose=True)
// (gbx_lm/models/quantized_linear_gba.py:195-203) with M = batch rows of x.
//
// HBM-bound by design: every packed weight byte is read from HBM exactly once per M tile and the
// only shared-memory traffic of the main loop is that same byte stream (one TMA write + one LDS).
//
//   * qweight is row-major [N, K*bits/32]: the packed rows owned by one CTA are ONE contiguous byte
//     range, and so are their scales and biases.  A dedicated producer warp streams them through a
//     4-stage shared-memory ring with the TMA engine: per stage one `cp.async.bulk` (SASS UBLKCP) of
//     up to 32 KB of whole rows plus one each for the rows' scales and biases, completion counted in
//     bytes on an mbarrier (full/empty pair per stage).  ~128 KB in flight per SM, independent of
//     occupancy.  Rows are balanced over the grid at single-row granularity.
//   * The activations are STATIONARY IN REGISTERS: the 16 consumer warps form a (chunk-column x
//     row-group) grid; a warp owns one 32-lane x 16 B (48 B for 3/6-bit) column of every row and
//     keeps the matching slice of x, pre-permuted into packed bf16 pairs, in registers for the whole
//     kernel.  Per row a lane issues one conflict-free LDS.128 (three for 3/6-bit) and unpacks in
//     registers: (w >> s) & mask | 0x4300 builds two bf16 values (128 + q) per LOP3, FHFMA.BF16
//     (fma.rn.f32.bf16) multiplies them with the packed activations into fp32 accumulators: no
//     int->float conversion, no activation unpacking.  3-/6-bit codes that straddle a 32-bit word
//     are fetched with one funnel shift.
//   * group affine:  y += scale * sum(x*(q+OFF)) + (bias - OFF*scale) * sum(x) per (row, group
//     fragment); sum(x) per fragment is a register constant.
//   * per stage a warp reduces its <=4 row partials with a transposing shuffle butterfly
//     (6 shuffles for 4 rows), every chunk column owns a shared-memory slot per row (no atomics: results are
//     bitwise reproducible), and the epilogue sums the columns in fixed order, rounds
//     once to bf16 (+ optional bias as a second rounded add) and stores coalesced.
#include "gbxq_common.cuh"

namespace gbxq {

namespace {

constexpr int kConsumerWarps = 16;
constexpr int kThreads = (kConsumerWarps + 1) * 32;
constexpr int kStages = 4;
constexpr int kRowsPerWarp = 4;               // R: rows a warp handles per ring stage
constexpr int kStageWBytes = 32 * 1024;       // packed-weight bytes per ring stage (upper bound)
constexpr int kMaxRowsPerCta = 2048;
constexpr uint32_t kMagic = 0x43004300u;      // bf16x2 (128, 128): OR-ing a code < 128 into the mantissa gives 128+q

template <int BITS> struct Fmt;
// UB: bytes per lane-unit, CPU: codes per lane-unit, ATOMS: processing atoms per unit,
// OFF: additive offset carried by the unpacked codes.
template <> struct Fmt<2> { static constexpr int UB = 16, CPU = 64, ATOMS = 4, OFF = 128; };
template <> struct Fmt<3> { static constexpr int UB = 48, CPU = 128, ATOMS = 4, OFF = 128; };
template <> struct Fmt<4> { static constexpr int UB = 16, CPU = 32, ATOMS = 4, OFF = 128; };
template <> struct Fmt<6> { static constexpr int UB = 48, CPU = 64, ATOMS = 4, OFF = 128; };
template <> struct Fmt<8> { static constexpr int UB = 16, CPU = 16, ATOMS = 2, OFF = 256; };

// Pair p of a lane-unit multiplies codes (pair_a, pair_b): the two codes one LOP3 extracts together.
template <int BITS> __host__ __device__ constexpr int pair_a(int p) {
    if (BITS == 4) return 8 * (p >> 2) + (p & 3);        // word j = p/4: nibble t with nibble t+4
    if (BITS == 2) return 16 * (p >> 3) + (p & 7);       // word j = p/8: field t with field t+8
    if (BITS == 8) return 4 * (p >> 1) + (p & 1);        // word j = p/2: byte t with byte t+2
    return 2 * p;                                        // 3/6-bit: natural order
}
template <int BITS> __host__ __device__ constexpr int pair_b(int p) {
    if (BITS == 4) return pair_a<4>(p) + 4;
    if (BITS == 2) return pair_a<2>(p) + 8;
    if (BITS == 8) return pair_a<8>(p) + 2;
    return 2 * p + 1;
}

__device__ __forceinline__ uint16_t lo16(uint32_t v) { return (uint16_t)(v & 0xffffu); }
__device__ __forceinline__ uint16_t hi16(uint32_t v) { return (uint16_t)(v >> 16); }

// One atom: accumulate sum_k x[k] * (q[k] + OFF) for the atom's codes into acc[m].
// `w` = the unit's words, `a` = atom index, xr[m] = the unit's activation pairs (pair order above).
template <int BITS, int MT, int NP>
__device__ __forceinline__ void atom_dot(const uint32_t* w, int a, const uint32_t (&xr)[MT][NP], float (&acc)[MT]) {
    if constexpr (BITS == 4) {
        const uint32_t word = w[a];
#pragma unroll
        for (int t = 0; t < 4; t++) {
            const uint32_t v = lop3_and_or(word >> (4 * t), 0x000f000fu, kMagic);
#pragma unroll
            for (int m = 0; m < MT; m++) {
                const uint32_t x2 = xr[m][4 * a + t];
                acc[m] = fma_bf16_f32(lo16(v), lo16(x2), acc[m]);
                acc[m] = fma_bf16_f32(hi16(v), hi16(x2), acc[m]);
            }
        }
    } else if constexpr (BITS == 2) {
        const uint32_t word = w[a];
#pragma unroll
        for (int t = 0; t < 8; t++) {
            const uint32_t v = lop3_and_or(word >> (2 * t), 0x00030003u, kMagic);
#pragma unroll
            for (int m = 0; m < MT; m++) {
                const uint32_t x2 = xr[m][8 * a + t];
                acc[m] = fma_bf16_f32(lo16(v), lo16(x2), acc[m]);
                acc[m] = fma_bf16_f32(hi16(v), hi16(x2), acc[m]);
            }
        }
    } else if constexpr (BITS == 8) {
        // byte = low7 + 128*top: two bf16 images, (128 + low7) and (128 + 128*top) -> OFF = 256
#pragma unroll
        for (int j = 0; j < 2; j++) {
            const uint32_t word = w[2 * a + j];
#pragma unroll
            for (int t = 0; t < 2; t++) {
                const uint32_t sh = word >> (8 * t);
                const uint32_t v1 = lop3_and_or(sh, 0x007f007fu, kMagic);
                const uint32_t v2 = lop3_and_or(sh, 0x00800080u, kMagic);
#pragma unroll
                for (int m = 0; m < MT; m++) {
                    const uint32_t x2 = xr[m][4 * a + 2 * j + t];
                    acc[m] = fma_bf16_f32(lo16(v1), lo16(x2), acc[m]);
                    acc[m] = fma_bf16_f32(hi16(v1), hi16(x2), acc[m]);
                    acc[m] = fma_bf16_f32(lo16(v2), lo16(x2), acc[m]);
                    acc[m] = fma_bf16_f32(hi16(v2), hi16(x2), acc[m]);
                }
            }
        }
    } else {
        // 3-bit: atom = 3 words = 32 codes; 6-bit: atom = 3 words = 16 codes.  Natural k order.
        constexpr int NC = 96 / BITS;
        constexpr uint32_t MASK = (1u << BITS) - 1u;
        const uint32_t* g = w + 3 * a;
#pragma unroll
        for (int t = 0; t < NC; t++) {
            const int bit = t * BITS;
            const int wi = bit >> 5, off = bit & 31;
            uint32_t sh;
            if (off + BITS <= 32) sh = g[wi] >> off;
            else sh = __funnelshift_r(g[wi], g[wi + 1], off);
            const uint32_t v = lop3_and_or(sh, MASK, 0x4300u);
#pragma unroll
            for (int m = 0; m < MT; m++) {
                const uint32_t x2 = xr[m][(a * NC + t) >> 1];
                acc[m] = fma_bf16_f32(lo16(v), (t & 1) ? hi16(x2) : lo16(x2), acc[m]);
            }
        }
    }
}

struct GemvParams {
    const __nv_bfloat16* x;
    const uint8_t* w;  // packed rows as bytes
    const uint16_t* scales;
    const uint16_t* biases;
    const __nv_bfloat16* bias;
    __nv_bfloat16* y;
    int64_t N, K;
    int M;          // rows of x in this launch (<= MT)
    int gs_shift;   // log2(group_size)
    int G;          // K / group_size
    uint32_t row_bytes;
    int nch;        // 32-lane chunk columns per row
    int cw, rg;     // warp grid: cw chunk columns x rg row groups (cw * rg <= 16)
    int tr;         // rows per ring stage (<= rg * kRowsPerWarp)
    uint32_t slot_bytes;  // ring slot size
    uint32_t sb_off;      // offset of the scales inside a slot (biases follow at sb_off + tr*G*2)
};

// Transposing butterfly: R per-lane partial sums -> lane 8*i of the warp holds the full sum of row i
// (valid where (lane & 7) == 0, row index = lane >> 3).
template <int R> __device__ __forceinline__ float reduce_rows(const float (&v)[R], int lane) {
    static_assert(R == 4, "kRowsPerWarp");
    const bool h16 = lane & 16, h8 = lane & 8;
    float k0 = h16 ? v[2] : v[0], k1 = h16 ? v[3] : v[1];
    const float s0 = h16 ? v[0] : v[2], s1 = h16 ? v[1] : v[3];
    k0 += __shfl_xor_sync(0xffffffffu, s0, 16);
    k1 += __shfl_xor_sync(0xffffffffu, s1, 16);
    float b = h8 ? k1 : k0;
    const float snd = h8 ? k0 : k1;
    b += __shfl_xor_sync(0xffffffffu, snd, 8);
    b += __shfl_xor_sync(0xffffffffu, b, 4);
    b += __shfl_xor_sync(0xffffffffu, b, 2);
    b += __shfl_xor_sync(0xffffffffu, b, 1);
    return b;
}

template <int BITS, int NSB, int MT, int CPW, bool SB_TMA>
__global__ void __launch_bounds__(kThreads, 1) gemv_kernel(const GemvParams p) {
    using F = Fmt<BITS>;
    constexpr int UB = F::UB, CPU = F::CPU;
    constexpr int CHUNK_B = 32 * UB;         // bytes one warp sweep covers in a row
    constexpr int SBC = CPU / NSB;           // codes per scale fragment (== min(CPU, group_size))
    constexpr int APS = F::ATOMS / NSB;      // atoms per fragment
    constexpr int NW = UB / 4;               // words per unit
    constexpr int NP = CPU / 2;              // activation pairs per unit
    constexpr int NV = CPU / 8;              // 16-byte activation vectors per unit
    constexpr int R = kRowsPerWarp;

    extern __shared__ __align__(1024) uint8_t smem[];
    // layout: [ring kStages * slot_bytes][barriers][ypart rows*cw*MT f32: one slot per (row, chunk column, token)]
    uint8_t* ring = smem;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(ring + (size_t)kStages * p.slot_bytes);
    uint64_t* empty_bar = full_bar + kStages;
    float* ysum = reinterpret_cast<float*>(empty_bar + kStages);

    const int grid = gridDim.x;
    const int64_t r0 = ((int64_t)blockIdx.x * p.N) / grid;
    const int64_t r1 = ((int64_t)(blockIdx.x + 1) * p.N) / grid;
    const int rows = (int)(r1 - r0);
    if (rows <= 0) return;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    // balanced stage sizing: ns stages of `spr` (<= tr) rows
    const int ns = (rows + p.tr - 1) / p.tr;
    const int spr = (rows + ns - 1) / ns;
    const int active_warps = p.cw * p.rg;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < kStages; s++) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], active_warps);
        }
        fence_mbar_init();
    }
    __syncthreads();

    if (warp == kConsumerWarps) {
        // ===================== producer warp: one elected lane drives the TMA engine =====================
        if (lane == 0) {
            const uint8_t* wsrc = p.w + (uint64_t)r0 * p.row_bytes;
            const uint32_t g2 = (uint32_t)p.G * 2u;  // bytes of one row of scales (or biases)
            for (int it = 0; it < ns; it++) {
                const int s = it % kStages;
                const uint32_t phase = (uint32_t)(it / kStages) & 1u;
                mbar_wait(&empty_bar[s], phase ^ 1u);
                const int ra = it * spr;
                int nr = rows - ra;
                if (nr > spr) nr = spr;
                const uint32_t wbytes = (uint32_t)nr * p.row_bytes;
                uint8_t* slot = ring + (size_t)s * p.slot_bytes;
                if constexpr (SB_TMA) {
                    const uint32_t sbytes = (uint32_t)nr * g2;
                    mbar_arrive_expect_tx(&full_bar[s], wbytes + 2u * sbytes);
                    bulk_g2s(slot, wsrc + (uint64_t)ra * p.row_bytes, wbytes, &full_bar[s]);
                    const uint64_t soff = (uint64_t)(r0 + ra) * g2;
                    bulk_g2s(slot + p.sb_off, reinterpret_cast<const uint8_t*>(p.scales) + soff, sbytes, &full_bar[s]);
                    bulk_g2s(slot + p.sb_off + (uint32_t)p.tr * g2, reinterpret_cast<const uint8_t*>(p.biases) + soff,
                             sbytes, &full_bar[s]);
                } else {
                    mbar_arrive_expect_tx(&full_bar[s], wbytes);
                    bulk_g2s(slot, wsrc + (uint64_t)ra * p.row_bytes, wbytes, &full_bar[s]);
                }
            }
        }
    } else if (warp < active_warps) {
        // ===================== consumer warps =====================
        const int cwi = warp % p.cw;  // chunk column
        const int rgi = warp / p.cw;  // row group
        // ---- stationary activations: this lane's slice of x for each of its chunk columns, as packed
        //      bf16 pairs in LOP3 pairing order; sum(x) per scale fragment; group index of the unit
        uint32_t xr[CPW][MT][NP];
        float xsum[CPW][MT][NSB];
        int gidx[CPW];
        bool live[CPW];
#pragma unroll
        for (int j = 0; j < CPW; j++) {
            const int c = cwi + j * p.cw;
            const uint32_t ubyte = (uint32_t)c * CHUNK_B + (uint32_t)lane * UB;
            live[j] = (c < p.nch) && (ubyte < p.row_bytes);
            const int k0 = (c * 32 + lane) * CPU;
            gidx[j] = k0 >> p.gs_shift;
#pragma unroll
            for (int m = 0; m < MT; m++) {
                uint4 nat[NV];
                const bool ld = live[j] && (m < p.M);
                const uint4* src = reinterpret_cast<const uint4*>(p.x + (size_t)m * p.K + k0);
#pragma unroll
                for (int v = 0; v < NV; v++) nat[v] = ld ? __ldg(src + v) : make_uint4(0u, 0u, 0u, 0u);
                uint32_t n32[NP];  // n32[i] = codes (2i, 2i+1) in natural order
#pragma unroll
                for (int v = 0; v < NV; v++) {
                    n32[4 * v + 0] = nat[v].x; n32[4 * v + 1] = nat[v].y; n32[4 * v + 2] = nat[v].z; n32[4 * v + 3] = nat[v].w;
                }
#pragma unroll
                for (int f = 0; f < NSB; f++) {
                    float sx = 0.f;
#pragma unroll
                    for (int i = 0; i < SBC / 2; i++) {
                        const uint32_t w32 = n32[f * (SBC / 2) + i];
                        sx += __uint_as_float(w32 << 16);
                        sx += __uint_as_float(w32 & 0xffff0000u);
                    }
                    xsum[j][m][f] = sx;
                }
#pragma unroll
                for (int q = 0; q < NP; q++) {
                    const int ia = pair_a<BITS>(q), ib = pair_b<BITS>(q);
                    const uint32_t sel = ((ia & 1) ? 0x32u : 0x10u) | (((ib & 1) ? 0x76u : 0x54u) << 8);
                    xr[j][m][q] = __byte_perm(n32[ia >> 1], n32[ib >> 1], sel);
                }
            }
        }

        const uint32_t ring_u32 = smem_u32(ring);
        const uint32_t g2 = (uint32_t)p.G * 2u;
        const int lrow0 = rgi * R;  // first stage-local row of this warp
        bool all_live = true;       // warp-uniform: every lane of every owned chunk column is inside the row
#pragma unroll
        for (int j = 0; j < CPW; j++) {
            const int c = cwi + j * p.cw;
            all_live = all_live && (c < p.nch) && ((uint32_t)(c + 1) * CHUNK_B <= p.row_bytes);
        }

        // one (row, chunk column) unit: LDS the packed words + scale/bias, unpack, FMA, apply the group affine
        auto unit = [&](uint32_t slot, int lr, int j, int64_t grow, float (&yrow)[MT]) {
            const int c = cwi + j * p.cw;
            const uint32_t waddr = slot + (uint32_t)lr * p.row_bytes + (uint32_t)c * CHUNK_B + (uint32_t)lane * UB;
            uint32_t w[NW];
#pragma unroll
            for (int v = 0; v < NW / 4; v++) {
                const uint4 t = lds128(waddr + 16 * v);
                w[4 * v + 0] = t.x; w[4 * v + 1] = t.y; w[4 * v + 2] = t.z; w[4 * v + 3] = t.w;
            }
#pragma unroll
            for (int f = 0; f < NSB; f++) {
                uint32_t sraw, braw;
                if constexpr (SB_TMA) {
                    const uint32_t sa = slot + p.sb_off + (uint32_t)lr * g2 + (uint32_t)(gidx[j] + f) * 2u;
                    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(sraw) : "r"(sa));
                    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(braw) : "r"(sa + (uint32_t)p.tr * g2));
                } else {
                    const int64_t gi = grow * (int64_t)p.G + gidx[j] + f;
                    sraw = __ldg(p.scales + gi);
                    braw = __ldg(p.biases + gi);
                }
                float dot[MT];
#pragma unroll
                for (int m = 0; m < MT; m++) dot[m] = 0.f;
#pragma unroll
                for (int aa = 0; aa < APS; aa++) {
                    float acc[MT];
#pragma unroll
                    for (int m = 0; m < MT; m++) acc[m] = 0.f;
                    atom_dot<BITS, MT, NP>(w, f * APS + aa, xr[j], acc);
#pragma unroll
                    for (int m = 0; m < MT; m++) dot[m] += acc[m];
                }
                const float sc = __uint_as_float(sraw << 16);
                const float bi = __uint_as_float(braw << 16);
                const float cc = fmaf(-(float)F::OFF, sc, bi);
#pragma unroll
                for (int m = 0; m < MT; m++) {
                    yrow[m] = fmaf(sc, dot[m], yrow[m]);
                    yrow[m] = fmaf(cc, xsum[j][m][f], yrow[m]);
                }
            }
        };

        for (int it = 0; it < ns; it++) {
            const int s = it % kStages;
            const uint32_t phase = (uint32_t)(it / kStages) & 1u;
            const int ra = it * spr;
            int nr = rows - ra;
            if (nr > spr) nr = spr;
            float yacc[R][MT];
#pragma unroll
            for (int i = 0; i < R; i++)
#pragma unroll
                for (int m = 0; m < MT; m++) yacc[i][m] = 0.f;

            mbar_wait(&full_bar[s], phase);
            const uint32_t slot = ring_u32 + (uint32_t)s * p.slot_bytes;
            if (all_live && lrow0 + R <= nr) {
                // fast path: no predicates, the R rows are independent instruction streams the compiler interleaves
#pragma unroll
                for (int i = 0; i < R; i++)
#pragma unroll
                    for (int j = 0; j < CPW; j++) unit(slot, lrow0 + i, j, r0 + ra + lrow0 + i, yacc[i]);
            } else {
#pragma unroll
                for (int i = 0; i < R; i++) {
                    const int lr = lrow0 + i;
                    if (lr < nr) {  // warp-uniform
#pragma unroll
                        for (int j = 0; j < CPW; j++)
                            if (live[j]) unit(slot, lr, j, r0 + ra + lr, yacc[i]);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[s]);  // slot free: all of this warp's reads are done
            // ---- fold the warp's row partials with the butterfly; lane 8*i then owns row i.  Each chunk
            //      column writes its own slot of ypart (no atomics -> bitwise reproducible results)
            if (lrow0 < nr) {
#pragma unroll
                for (int m = 0; m < MT; m++) {
                    float v4[R];
#pragma unroll
                    for (int i = 0; i < R; i++) v4[i] = yacc[i][m];
                    const float tot = reduce_rows<R>(v4, lane);
                    const int lr = lrow0 + (lane >> 3);
                    if ((lane & 7) == 0 && lr < nr) ysum[((ra + lr) * p.cw + cwi) * MT + m] = tot;
                }
            }
        }
    }
    __syncthreads();
    // ---- epilogue: one rounding to bf16, optional bias as a second rounded add, coalesced store
    for (int i = threadIdx.x; i < rows * MT; i += kThreads) {
        const int m = i / rows, r = i - m * rows;
        if (m < p.M) {
            float tot = 0.f;
            for (int c = 0; c < p.cw; c++) tot += ysum[(r * p.cw + c) * MT + m];
            float v = __bfloat162float(__float2bfloat16_rn(tot));
            if (p.bias != nullptr) v = __fadd_rn(v, __bfloat162float(p.bias[r0 + r]));
            p.y[(size_t)m * p.N + r0 + r] = __float2bfloat16_rn(v);
        }
    }
}

template <int BITS, int NSB, int MT, int CPW, bool SB_TMA>
int launch_inst(const GemvParams& p, size_t smem_bytes, int grid, cudaStream_t st) {
    constexpr auto kern = gemv_kernel<BITS, NSB, MT, CPW, SB_TMA>;
    const int rc = allow_dynamic_smem<kern>(227 * 1024);
    if (rc != GBXQ_OK) return rc;
    return launch(kern, dim3(grid), dim3(kThreads), smem_bytes, st, false, p);
}

template <int BITS> constexpr int nsb_for(int gs) { return Fmt<BITS>::CPU > gs ? Fmt<BITS>::CPU / gs : 1; }
template <int BITS> constexpr int max_cpw() { return BITS == 8 ? 4 : (BITS == 4 ? 2 : 1); }

struct Plan {
    bool ok;
    int mt, cpw, nch, cw, rg, tr;
    bool sb_tma;
    uint32_t slot_bytes, sb_off;
    size_t smem;
};

template <int BITS> Plan make_plan(int64_t M, int64_t N, int64_t K, int gs) {
    using F = Fmt<BITS>;
    Plan pl{};
    const int64_t row_bytes = K * BITS / 8;
    if (row_bytes % F::UB || row_bytes % 16 || row_bytes > kStageWBytes) return pl;
    const int chunk_b = 32 * F::UB;
    pl.nch = (int)((row_bytes + chunk_b - 1) / chunk_b);
    // warp grid: as many chunk columns as fit in 16 warps (each warp owning cpw columns), the rest row groups
    pl.cpw = (pl.nch + kConsumerWarps - 1) / kConsumerWarps;
    if (pl.cpw == 3) pl.cpw = 4;
    if (pl.cpw > max_cpw<BITS>()) return pl;
    pl.cw = (pl.nch + pl.cpw - 1) / pl.cpw;
    pl.rg = kConsumerWarps / pl.cw;
    const int64_t tr_fit = kStageWBytes / row_bytes;  // >= 1
    if ((int64_t)pl.rg * kRowsPerWarp > tr_fit) pl.rg = (int)((tr_fit + kRowsPerWarp - 1) / kRowsPerWarp);
    if (pl.rg < 1) pl.rg = 1;
    pl.tr = (int)(tr_fit < (int64_t)pl.rg * kRowsPerWarp ? tr_fit : (int64_t)pl.rg * kRowsPerWarp);
    const int grid = device_sm_count();
    if ((N + grid - 1) / grid > kMaxRowsPerCta) return pl;
    const int64_t G = K / gs;
    pl.sb_tma = (G * 2) % 16 == 0;
    const uint32_t wpart = (uint32_t)(((int64_t)pl.tr * row_bytes + 127) & ~(int64_t)127);
    pl.sb_off = wpart;
    pl.slot_bytes = wpart + (pl.sb_tma ? (uint32_t)((2 * (int64_t)pl.tr * G * 2 + 127) & ~(int64_t)127) : 0u);
    pl.mt = (M >= 2 && BITS != 3) ? 2 : 1;  // 3-bit units hold 64 activation registers per token
    const int64_t rows_max = (N + grid - 1) / grid;
    pl.smem = (size_t)kStages * pl.slot_bytes + 2 * kStages * 8 + (size_t)rows_max * pl.cw * pl.mt * 4 + 16;
    if (pl.smem > 227 * 1024) return pl;
    pl.ok = true;
    return pl;
}

template <int BITS, int NSB, int MT, int CPW>
int launch_sb(const GemvParams& p, const Plan& pl, int grid, cudaStream_t st) {
    return pl.sb_tma ? launch_inst<BITS, NSB, MT, CPW, true>(p, pl.smem, grid, st)
                     : launch_inst<BITS, NSB, MT, CPW, false>(p, pl.smem, grid, st);
}

template <int BITS, int NSB, int MT>
int launch_cpw(const GemvParams& p, const Plan& pl, int grid, cudaStream_t st) {
    if (pl.cpw == 1) return launch_sb<BITS, NSB, MT, 1>(p, pl, grid, st);
    if constexpr (max_cpw<BITS>() >= 2) {
        if (pl.cpw == 2) return launch_sb<BITS, NSB, MT, 2>(p, pl, grid, st);
    }
    if constexpr (max_cpw<BITS>() >= 4) {
        if (pl.cpw == 4) return launch_sb<BITS, NSB, MT, 4>(p, pl, grid, st);
    }
    return GBXQ_EUNSUPPORTED;
}

template <int BITS, int NSB>
int launch_mt(const GemvParams& p, const Plan& pl, int grid, cudaStream_t st) {
    if constexpr (BITS != 3) {
        if (pl.mt == 2) return launch_cpw<BITS, NSB, 2>(p, pl, grid, st);
    }
    return launch_cpw<BITS, NSB, 1>(p, pl, grid, st);
}

template <int BITS>
int launch_bits(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                int64_t N, int64_t K, int gs, cudaStream_t st) {
    const Plan pl = make_plan<BITS>(M, N, K, gs);
    if (!pl.ok) return GBXQ_EUNSUPPORTED;
    GemvParams p{};
    p.w = reinterpret_cast<const uint8_t*>(w);
    p.scales = reinterpret_cast<const uint16_t*>(s);
    p.biases = reinterpret_cast<const uint16_t*>(b);
    p.bias = reinterpret_cast<const __nv_bfloat16*>(bias);
    p.N = N;
    p.K = K;
    p.gs_shift = gs == 32 ? 5 : (gs == 64 ? 6 : 7);
    p.G = (int)(K / gs);
    p.row_bytes = (uint32_t)(K * BITS / 8);
    p.nch = pl.nch;
    p.cw = pl.cw;
    p.rg = pl.rg;
    p.tr = pl.tr;
    p.slot_bytes = pl.slot_bytes;
    p.sb_off = pl.sb_off;
    const int nsb = nsb_for<BITS>(gs);
    int grid = device_sm_count();
    if (grid > N) grid = (int)N;
    for (int64_t m0 = 0; m0 < M; m0 += pl.mt) {
        p.x = reinterpret_cast<const __nv_bfloat16*>(x) + m0 * K;
        p.y = reinterpret_cast<__nv_bfloat16*>(y) + m0 * N;
        p.M = (int)((M - m0) < pl.mt ? (M - m0) : pl.mt);
        int rc = GBXQ_EUNSUPPORTED;
        if (nsb == 1) rc = launch_mt<BITS, 1>(p, pl, grid, st);
        if constexpr (Fmt<BITS>::CPU >= 64) {
            if (nsb == 2) rc = launch_mt<BITS, 2>(p, pl, grid, st);
        }
        if constexpr (Fmt<BITS>::CPU >= 128) {
            if (nsb == 4) rc = launch_mt<BITS, 4>(p, pl, grid, st);
        }
        if (rc != GBXQ_OK) return rc;
    }
    return GBXQ_OK;
}

}  // namespace

bool gemv_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                    const void* y) {
    if (dtype != GBXQ_BF16 || M < 1 || N < 1) return false;
    if (((uintptr_t)x | (uintptr_t)w) & 15) return false;
    if ((uintptr_t)y & 1) return false;
    if ((K * 2) % 16) return false;
    Plan pl{};
    switch (bits) {
        case 2: pl = make_plan<2>(M, N, K, gs); break;
        case 3: pl = make_plan<3>(M, N, K, gs); break;
        case 4: pl = make_plan<4>(M, N, K, gs); break;
        case 6: pl = make_plan<6>(M, N, K, gs); break;
        case 8: pl = make_plan<8>(M, N, K, gs); break;
        default: return false;
    }
    return pl.ok;
}

int launch_gemv(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                int64_t N, int64_t K, int bits, int gs, cudaStream_t st) {
    switch (bits) {
        case 2: return launch_bits<2>(x, w, s, b, bias, y, M, N, K, gs, st);
        case 3: return launch_bits<3>(x, w, s, b, bias, y, M, N, K, gs, st);
        case 4: return launch_bits<4>(x, w, s, b, bias, y, M, N, K, gs, st);
        case 6: return launch_bits<6>(x, w, s, b, bias, y, M, N, K, gs, st);
        case 8: return launch_bits<8>(x, w, s, b, bias, y, M, N, K, gs, st);
    }
    return GBXQ_EINVAL_BITS;
}

}  // namespace gbxq
