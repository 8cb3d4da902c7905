// gbxq_mmv8.cu -- decode matrix-vector kernel on the INTEGER tensor pipe ("mmv8"): 1..4 rows of x,
// bf16 activations, 2-/4-/8-bit packings.  The headline kernel of the path:
// QuantizedLinear.__call__ -> mx.quantized_matmul(transpose=True)
// (gbx_lm/models/quantized_linear_gba.py:195-203) at decode batch sizes.
//
// Why integers: measured on B200 (tools/ubench/ub_pipes.cu, profiles/) LOP3/SHF/PRMT issue at one warp
// instruction per 2 clocks per SM sub-partition, and the bf16 kernels (gbxq_gemv.cu, gbxq_mmv.cu) spend
// 0.9 of them per weight turning codes into bf16 (shift, mask, or-in a magic exponent) -- ALU-pipe bound at
// ~70 % of HBM.  `mma.sync.m16n8k32.s32.u8.s8` (SASS IMMA.16832.U8.S8) issues as fast as the bf16 HMMA, does
// twice the multiply-adds, and takes the codes AS THEY ARE: a u8 A-operand byte is just a masked field of the
// packed word, even in place (w & 0xf0f0f0f0 = 16*q), so unpacking costs 0.25 plain ANDs per 4-bit weight and
// nothing at all for 8-bit weights.
//
//   * Activations: per (token, quantisation group) block fixed point.  m = round(x * 2^(13 - e)), e = exponent
//     of the group's largest |x|, |m| < 2^14, split into two balanced s8 digits m = 256*hi + lo (lo = low byte as s8).
//     Elements within 2^-6 of the group maximum are represented exactly (bf16 carries 8 significant bits), the
//     others to 2^-14 of the maximum.  Products and sums are exact in int32; one fp32 conversion per group.
//   * "Slice" layout as in gbxq_mmv.cu: the 8 B columns are (group slice s, digit d): column j = (j>>1, j&1);
//     the 16 A rows are W = 4 weight rows x S = 4 consecutive groups of each.  Only the accumulators whose
//     column slice equals their row slice are meaningful -- the two digits of one (row, group) land in the same
//     thread (c0, c1) and are recombined with one IMAD (256*hi + lo).  More tokens = more MMAs on the same A registers.
//   * In-place fields are compensated exactly in the integer domain: 4-bit T = 16*D(even codes) + D(odd codes
//     in place, 16*q), folded scale/16; 2-bit T = 4*D(fields 0,2) + D(fields 1,3 in place, 4*q), scale/4.
//   * y += scale[n,g] * 2^(e-13) * T(n,g)  per group, in fp32;  biases: y += sum_g bias[n,g] * sum(x over g),
//     a [rows x groups] dot product against per-lane stationary group sums.
//   * Streaming, ring, PDL, deterministic shared-memory reduction and epilogue are those of gbxq_mmv.cu.
#include "gbxq_mmv8_body.cuh"

namespace gbxq {

using namespace mmv8;

namespace {

// BITS, GS = group size, MT = tokens (1, 2, 4), CPW = chunk columns per warp, R = rows per warp and stage (4 or 8)
template <int BITS, int GS, int MT, int CPW, int R, bool PARTIAL>
__global__ void __launch_bounds__(kThreads, kMinCtas) mmv8_kernel(const Mmv8Params p, const __grid_constant__ ArParams ar) {
    extern __shared__ __align__(1024) uint8_t smem[];
    mmv8_body<BITS, GS, MT, CPW, R, false, PARTIAL>(p, (int)blockIdx.x, smem, nullptr, &ar);
}

template <int BITS, int GS, int MT, int CPW, int R, bool PARTIAL>
int launch_inst2(const Mmv8Params& p, const ArParams& ar, const Plan& pl, cudaStream_t st) {
    constexpr auto kern = mmv8_kernel<BITS, GS, MT, CPW, R, PARTIAL>;
    const int rc = allow_dynamic_smem<kern>(kSmemCap);
    if (rc != GBXQ_OK) return rc;
    return launch(kern, dim3((unsigned)pl.grid), dim3(kThreads), pl.smem, st, true, p, ar);
}

template <int BITS, int GS, int MT, int CPW, int R>
int launch_inst(const Mmv8Params& p, const ArParams& ar, const Plan& pl, cudaStream_t st) {
    if constexpr (GS == 128 && MT <= 2) {  // the half-full-column instantiations (make_plan admits nothing else)
        if (pl.partial) return launch_inst2<BITS, GS, MT, CPW, R, true>(p, ar, pl, st);
    }
    if (pl.partial) return GBXQ_EUNSUPPORTED;
    return launch_inst2<BITS, GS, MT, CPW, R, false>(p, ar, pl, st);
}

template <int BITS, int GS, int MT>
int launch_cpw(const Mmv8Params& p, const ArParams& ar, const Plan& pl, cudaStream_t st) {
    if (pl.R == 16) {
        if constexpr (MT <= 2)
            if (pl.cpw == 1) return launch_inst<BITS, GS, MT, 1, 16>(p, ar, pl, st);
    } else if (pl.R == 8) {
        if (pl.cpw == 1) return launch_inst<BITS, GS, MT, 1, 8>(p, ar, pl, st);
        if (pl.cpw == 2) return launch_inst<BITS, GS, MT, 2, 8>(p, ar, pl, st);
    } else if (pl.R == 4) {
        switch (pl.cpw) {
            case 1: return launch_inst<BITS, GS, MT, 1, 4>(p, ar, pl, st);
            case 2: return launch_inst<BITS, GS, MT, 2, 4>(p, ar, pl, st);
            case 4:
                if constexpr (MT <= 2) return launch_inst<BITS, GS, MT, 4, 4>(p, ar, pl, st);
                break;
            case 8:
                if constexpr (MT == 1) return launch_inst<BITS, GS, MT, 8, 4>(p, ar, pl, st);
                break;
        }
    }
    return GBXQ_EUNSUPPORTED;
}

template <int BITS, int GS>
int launch_mt(const Mmv8Params& p, const ArParams& ar, const Plan& pl, cudaStream_t st) {
    switch (pl.mt) {
        case 1: return launch_cpw<BITS, GS, 1>(p, ar, pl, st);
        case 2: return launch_cpw<BITS, GS, 2>(p, ar, pl, st);
        case 4: return launch_cpw<BITS, GS, 4>(p, ar, pl, st);
    }
    return GBXQ_EUNSUPPORTED;
}

unsigned long long* g_dbg = nullptr;
int g_dbg_left = 0;
int g_dbg_stride = 0;  // > 0: all-CTA timeline, CTAs per launch region
}  // namespace

void mmv8_debug_timeline(unsigned long long* buf, int launches) {
    g_dbg = buf;
    g_dbg_left = launches;
    g_dbg_stride = 0;
}
// every CTA stamps: launch i writes 8 slots per CTA at buf + i * 8 * stride_ctas
void mmv8_debug_timeline_all(unsigned long long* buf, int launches, int stride_ctas) {
    g_dbg = buf;
    g_dbg_left = launches;
    g_dbg_stride = stride_ctas;
}

bool mmv8_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                    const void* y) {
    if (dtype != GBXQ_BF16 || M < 1 || N < 1) return false;
    if (((uintptr_t)x | (uintptr_t)w) & 15) return false;
    if ((uintptr_t)y & 1) return false;
    if ((K * 2) % 16) return false;
    const Plan pl = make_plan(M, N, K, bits, gs, 0, true, true);
    if (!pl.ok) return false;
    return pl.cpw * pl.mt <= 8;  // register budget of the stationary digit fragments
}

int launch_mmv8(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                int64_t N, int64_t K, int bits, int gs, cudaStream_t st) {
    return launch_mmv8_ar(x, w, s, b, bias, y, M, N, K, bits, gs, nullptr, st);
}

// comm != nullptr: row-parallel shard with the all-reduce fused into the epilogue (gbxq_qmm_rowpar_allreduce)
int launch_mmv8_ar(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                   int64_t N, int64_t K, int bits, int gs, const gbxq_comm* comm, cudaStream_t st) {
    if (((uintptr_t)s | (uintptr_t)b) & 15) return GBXQ_EUNSUPPORTED;
    const Plan pl = make_plan(M, N, K, bits, gs, 0, true, true);
    if (!pl.ok || pl.cpw * pl.mt > 8) return GBXQ_EUNSUPPORTED;
    Mmv8Params p = make_params(pl, x, w, s, b, bias, y, M, N, K, bits, gs, pdl_early_weights());
    ArParams ar{};
    if (comm != nullptr && comm->world > 1) {
        if (comm->world > 8 || comm->rank < 0 || comm->rank >= comm->world) return GBXQ_ESHAPE;
        if (pl.grid > GBXQ_RP_MAX_CTAS) return GBXQ_EUNSUPPORTED;
        if (comm->stage_elems < 2 * (int64_t)comm->world * M * N) return GBXQ_EWORKSPACE;
        for (int r = 0; r < comm->world; r++) {
            if (comm->peer_stage_host[r] == nullptr || comm->peer_flags_host[r] == nullptr) return GBXQ_ENULL;
            if ((uintptr_t)comm->peer_stage_host[r] & 7) return GBXQ_EALIGN;
            ar.stage[r] = reinterpret_cast<unsigned long long*>(comm->peer_stage_host[r]);
            ar.flags[r] = comm->peer_flags_host[r];
        }
        ar.half_elems = comm->stage_elems / 2;
        ar.world = comm->world;
        ar.rank = comm->rank;
    }
    if (g_dbg != nullptr && g_dbg_left > 0) {
        p.dbg = g_dbg;
        p.dbg_all = g_dbg_stride > 0 && pl.grid <= g_dbg_stride ? 1 : 0;
        g_dbg += g_dbg_stride > 0 ? (size_t)8 * g_dbg_stride : 8;
        g_dbg_left--;
    }
    switch (bits * 1000 + gs) {
        case 4064: return launch_mt<4, 64>(p, ar, pl, st);
        case 4128: return launch_mt<4, 128>(p, ar, pl, st);
        case 4032: return launch_mt<4, 32>(p, ar, pl, st);
        case 3064: return launch_mt<3, 64>(p, ar, pl, st);
        case 3128: return launch_mt<3, 128>(p, ar, pl, st);
        case 6064: return launch_mt<6, 64>(p, ar, pl, st);
        case 6128: return launch_mt<6, 128>(p, ar, pl, st);
        case 2064: return launch_mt<2, 64>(p, ar, pl, st);
        case 2128: return launch_mt<2, 128>(p, ar, pl, st);
        case 8064: return launch_mt<8, 64>(p, ar, pl, st);
        case 8128: return launch_mt<8, 128>(p, ar, pl, st);
        case 8032: return launch_mt<8, 32>(p, ar, pl, st);
    }
    return GBXQ_EUNSUPPORTED;
}

}  // namespace gbxq
