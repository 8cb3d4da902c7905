// gbxq_mmv8_grouped.cu -- ONE launch for the projections that read the same activations:
// q_proj | k_proj | v_proj (gbx_lm/models/qllama.py:76, qqwen2.py:66) and gate_proj | up_proj (qllama.py:115,
// qqwen2.py:94), each with its own bit width as in the layer-mix checkpoints (quantized_linear_gba.py:258-272).
//
// Why: at decode sizes a projection is shorter than the dependent-launch chain around it (k_proj of Llama-3-8B is
// 2.4 MB = 0.36 us of HBM time against ~3 us from the previous kernel's last store to this kernel's first MMA), so
// the number of dependent launches per transformer block bounds the step.  A grouped launch turns 7 dependent
// launches per block into 4 and lets the wide segments hide the narrow ones.
//
// How: the CTAs of the grid are divided among the segments in proportion to their packed bytes; a CTA looks up its
// segment, then runs the unchanged mmv8 body (gbxq_mmv8_body.cuh) instantiated for that segment's bit width.
// Segments must agree on K, group size and the derived warp geometry (CPW, R); otherwise the caller
// (gbxq_qmm_grouped, gbxq_api.cu) falls back to one launch per segment.
#include "gbxq_mmv8_body.cuh"

namespace gbxq {

using namespace mmv8;

namespace {

struct GroupParams {
    Mmv8Params seg[GBXQ_MAX_SEGMENTS];
    int cta0[GBXQ_MAX_SEGMENTS + 1];  // segment s owns CTAs [cta0[s], cta0[s+1])
    int bits[GBXQ_MAX_SEGMENTS];
    int nseg;
};

// ODD: the launch holds a 3- or 6-bit segment.  Those bodies (register realignment of the straddling codes) live in a
// kernel of their own: with five bodies in one kernel the common 2/4/8-bit launches of the 8B step ran 10 % slower
// (profiles/r02g_variants.txt: instruction footprint), although a CTA only ever executes one body.
template <int GS, int MT, int CPW, int R, bool ODD>
__global__ void __launch_bounds__(kThreads, kMinCtas) mmv8_grouped_kernel(const __grid_constant__ GroupParams gp) {
    extern __shared__ __align__(1024) uint8_t smem[];
    int bid = (int)blockIdx.x;
    int s = 0;
#pragma unroll
    for (int i = 1; i < GBXQ_MAX_SEGMENTS; i++)
        if (i < gp.nseg && bid >= gp.cta0[i]) s = i;
    bid -= gp.cta0[s];
    // one copy of the body per bit width; the switch is CTA-uniform
    const int bits = gp.bits[s];
    if constexpr (ODD) {
        if (bits == 3) {
            mmv8_body<3, GS, MT, CPW, R>(gp.seg[s], bid, smem);
            return;
        }
        if (bits == 6) {
            mmv8_body<6, GS, MT, CPW, R>(gp.seg[s], bid, smem);
            return;
        }
    }
    switch (bits) {
        case 2: mmv8_body<2, GS, MT, CPW, R>(gp.seg[s], bid, smem); break;
        case 4: mmv8_body<4, GS, MT, CPW, R>(gp.seg[s], bid, smem); break;
        default: mmv8_body<8, GS, MT, CPW, R>(gp.seg[s], bid, smem); break;
    }
}

template <int GS, int MT, int CPW, int R, bool ODD>
int launch_inst2(const GroupParams& gp, int grid, size_t smem, cudaStream_t st) {
    constexpr auto kern = mmv8_grouped_kernel<GS, MT, CPW, R, ODD>;
    const int rc = allow_dynamic_smem<kern>(kSmemCap);
    if (rc != GBXQ_OK) return rc;
    return launch(kern, dim3((unsigned)grid), dim3(kThreads), smem, st, true, gp);
}

template <int GS, int MT, int CPW, int R>
int launch_inst(const GroupParams& gp, int grid, size_t smem, cudaStream_t st) {
    bool odd = false;
    for (int i = 0; i < gp.nseg; i++) odd |= gp.bits[i] == 3 || gp.bits[i] == 6;
    return odd ? launch_inst2<GS, MT, CPW, R, true>(gp, grid, smem, st) : launch_inst2<GS, MT, CPW, R, false>(gp, grid, smem, st);
}

template <int GS, int MT>
int launch_cpw(const GroupParams& gp, int cpw, int R, int grid, size_t smem, cudaStream_t st) {
    if (R == 16) {
        if constexpr (MT <= 2)
            if (cpw == 1) return launch_inst<GS, MT, 1, 16>(gp, grid, smem, st);
    } else if (R == 8) {
        if (cpw == 1) return launch_inst<GS, MT, 1, 8>(gp, grid, smem, st);
        if (cpw == 2) return launch_inst<GS, MT, 2, 8>(gp, grid, smem, st);
    } else if (R == 4) {
        switch (cpw) {
            case 1: return launch_inst<GS, MT, 1, 4>(gp, grid, smem, st);
            case 2: return launch_inst<GS, MT, 2, 4>(gp, grid, smem, st);
            case 4:
                if constexpr (MT <= 2) return launch_inst<GS, MT, 4, 4>(gp, grid, smem, st);
                break;
            case 8:
                if constexpr (MT == 1) return launch_inst<GS, MT, 8, 4>(gp, grid, smem, st);
                break;
        }
    }
    return GBXQ_EUNSUPPORTED;
}

template <int GS>
int launch_mt(const GroupParams& gp, int mt, int cpw, int R, int grid, size_t smem, cudaStream_t st) {
    switch (mt) {
        case 1: return launch_cpw<GS, 1>(gp, cpw, R, grid, smem, st);
        case 2: return launch_cpw<GS, 2>(gp, cpw, R, grid, smem, st);
        case 4: return launch_cpw<GS, 4>(gp, cpw, R, grid, smem, st);
    }
    return GBXQ_EUNSUPPORTED;
}

}  // namespace

// Returns GBXQ_EUNSUPPORTED (nothing enqueued) when the segments cannot share one launch.
int launch_mmv8_grouped(const gbxq_segment* segs, int nseg, const void* x, int64_t M, int64_t K, cudaStream_t st) {
    if (nseg < 2 || nseg > GBXQ_MAX_SEGMENTS || M < 1 || M > 4) return GBXQ_EUNSUPPORTED;
    if (((uintptr_t)x & 15) || (K * 2) % 16) return GBXQ_EUNSUPPORTED;
    const int gs = segs[0].group_size;
    if (gs == 32) return GBXQ_EUNSUPPORTED;
    double bytes[GBXQ_MAX_SEGMENTS], total = 0;
    for (int i = 0; i < nseg; i++) {
        const gbxq_segment& sg = segs[i];
        if (sg.group_size != gs || !(sg.bits == 2 || sg.bits == 3 || sg.bits == 4 || sg.bits == 6 || sg.bits == 8) || sg.N < 1) return GBXQ_EUNSUPPORTED;
        if (((uintptr_t)sg.qweight | (uintptr_t)sg.scales | (uintptr_t)sg.biases) & 15) return GBXQ_EUNSUPPORTED;
        if ((uintptr_t)sg.y & 1) return GBXQ_EUNSUPPORTED;
        bytes[i] = segment_cost(sg.N, K, sg.bits, gs);
        total += bytes[i];
    }
    // CTAs per segment in proportion to its bytes (largest-remainder rounding, at least one each)
    const int total_ctas = mmv8_total_ctas();
    int ctas[GBXQ_MAX_SEGMENTS], given = 0;
    for (int i = 0; i < nseg; i++) {
        ctas[i] = (int)(total_ctas * bytes[i] / total);
        if (ctas[i] < 1) ctas[i] = 1;
        given += ctas[i];
    }
    for (int i = 0; given < total_ctas; i = (i + 1) % nseg, given++) ctas[i]++;
    GroupParams gp{};
    gp.nseg = nseg;
    Plan first{};
    size_t smem = 0;
    int grid = 0;
    const int early = pdl_early_weights();
    for (int i = 0; i < nseg; i++) {
        const gbxq_segment& sg = segs[i];
        const Plan pl = make_plan(M, sg.N, K, sg.bits, gs, ctas[i]);
        if (!pl.ok || pl.cpw * pl.mt > 8) return GBXQ_EUNSUPPORTED;
        if (i == 0) first = pl;
        if (pl.cpw != first.cpw || pl.R != first.R || pl.mt != first.mt) return GBXQ_EUNSUPPORTED;
        gp.seg[i] = make_params(pl, x, sg.qweight, sg.scales, sg.biases, sg.bias, sg.y, M, sg.N, K, sg.bits, gs, early);
        gp.bits[i] = sg.bits;
        gp.cta0[i] = grid;
        grid += pl.grid;
        if (pl.smem > smem) smem = pl.smem;
    }
    gp.cta0[nseg] = grid;
    switch (gs) {
        case 64: return launch_mt<64>(gp, first.mt, first.cpw, first.R, grid, smem, st);
        case 128: return launch_mt<128>(gp, first.mt, first.cpw, first.R, grid, smem, st);
    }
    return GBXQ_EUNSUPPORTED;
}

}  // namespace gbxq
