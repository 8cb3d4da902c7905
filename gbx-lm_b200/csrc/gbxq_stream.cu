// gbxq_stream.cu -- a whole chain of decode-sized quantized matmuls in ONE persistent launch (gbxq_qmm_stream).
//
// Replaces: the back-to-back QuantizedLinear forwards of a decode step (gbx_lm/models/qllama.py:76-115 -- q|k|v,
// o_proj, gate|up, down_proj of every block; each is mx.quantized_matmul, quantized_linear_gba.py:195-203).
//
// Why (profiles/r01e_*): inside one call the stage loop of the mmv8 kernel already runs at the HBM rate (33 MB in
// 5.0 us), but a call is only 2-66 MB, so the ~4 us around the loop (dependent launch, barrier set-up, activations ->
// digit fragments, ring fill = one HBM round trip, epilogue, drain) keep the step at 0.42 of the HBM roofline even
// with programmatic dependent launch.  Weights never depend on activations, so the weight stream does not have to
// stop where a call ends:
//   * grid = 2 CTAs per SM, all co-resident for the whole chain; each CTA owns a row range of EVERY call;
//   * the producer warp walks the chain on its own, bounded only by the ring's empty barriers: while the consumer
//     warps finish call i (reduction, y store, completion counter) and prepare call i+1 (wait for the counter, x ->
//     fragments), the packed rows, scales and biases of calls i+1, i+2 ... are already landing in shared memory
//     (2 x ~100 KB per SM = ~29 MB device-wide = 4.4 us of HBM time of look-ahead);
//   * calls are ordered by device-wide completion counters (one atomic per CTA and call, one polling thread per
//     CTA), which gives exactly the semantics of issuing the calls one after another on a stream;
//   * the per-call maths is the unchanged mmv8 body (gbxq_mmv8_body.cuh, STREAM = true): results are bitwise equal
//     to gbxq_qmm / gbxq_qmm_grouped.
//   * call descriptors travel to shared memory by bulk copies issued two (consumers) / three (producer) calls ahead.
// Deadlock safety: the launch is refused unless the occupancy query says the whole grid is co-resident, and every
// spin has a 2 s globaltimer bail-out that flags the error instead of hanging the device.
// Measured (profiles/r01h_stream_timeline.txt, DESIGN.md 3.1): the hand-over between two calls (counter, wait, x,
// fragments, epilogue) costs ~4.2 us, as much as a dependent launch, and the consumers cannot drain a full ring faster
// than HBM fills it, so the chain runs the 8B step at 0.43 of the HBM roofline against 0.45 for launch-per-call: it is
// an API and `bench.py --stream 1`, not the default path, until the consumer loop is faster than the stream.
#include <cstring>
#include <vector>

#include "gbxq_mmv8_body.cuh"

namespace gbxq {

using namespace mmv8;

namespace {

constexpr int kDescBytes = 4096;          // shared-memory descriptor rings (consumers 2, producer 4) in front of the weight ring
constexpr size_t kStreamSmemMax = 112 * 1024 * kWide;

inline int variant_of(int cpw, int R) {  // (CPW, R): (1,8) (2,8) (1,4) (2,4) (4,4) (8,4)
    if (R == 8) return cpw == 1 ? 0 : (cpw == 2 ? 1 : -1);
    if (R == 4) return cpw == 1 ? 2 : (cpw == 2 ? 3 : (cpw == 4 ? 4 : (cpw == 8 ? 5 : -1)));
    return -1;
}

// one call of the chain as the device reads it (array in global memory, immutable while launches are in flight)
struct StreamCallDev {
    Mmv8Params seg[GBXQ_MAX_SEGMENTS];
    int cta0[GBXQ_MAX_SEGMENTS + 1];  // segment s owns CTAs [cta0[s], cta0[s+1]); CTAs >= cta0[MAX] idle in this call
    int bits[GBXQ_MAX_SEGMENTS];
    int nseg;
    int variant;
    int dep;                          // completion counter this call waits for (-1: none)
    int pad[4];
};
constexpr int kCallBytes = (int)sizeof(StreamCallDev);
constexpr int kCallSlot = 640;
constexpr int kConsDesc = 2, kProdDesc = 4;
static_assert(kCallBytes % 16 == 0 && kCallBytes <= kCallSlot, "descriptors travel by bulk copy");
static_assert((kConsDesc + kProdDesc) * kCallSlot + (kConsDesc + kProdDesc) * 8 <= kDescBytes, "descriptor area");

// segment of CTA `bid` in a call (descriptor already in shared memory): -1 = no rows of this call
__device__ __forceinline__ int find_segment(const StreamCallDev* d, int bid, int& lbid) {
    int s = 0, base = 0;
#pragma unroll
    for (int i = 1; i < GBXQ_MAX_SEGMENTS; i++) {
        const int c0 = d->cta0[i];
        if (i < d->nseg && bid >= c0) {
            s = i;
            base = c0;
        }
    }
    lbid = bid - base;
    return bid >= d->cta0[GBXQ_MAX_SEGMENTS] ? -1 : s;
}

template <int GS, int MT, int CPW, int R>
__device__ __forceinline__ void run_bits(const Mmv8Params& p, int bits, int lbid, uint8_t* ring, StreamCtx* sc) {
    // one copy of the body per bit width; the switch is CTA-uniform
    switch (bits) {
        case 2: mmv8_body<2, GS, MT, CPW, R, true>(p, lbid, ring, sc); break;
        case 4: mmv8_body<4, GS, MT, CPW, R, true>(p, lbid, ring, sc); break;
        default: mmv8_body<8, GS, MT, CPW, R, true>(p, lbid, ring, sc); break;
    }
}

template <int GS, int MT>
__global__ void __launch_bounds__(kThreads, kMinCtas)
    stream_kernel(const StreamCallDev* __restrict__ calls, const int ncalls, unsigned* __restrict__ cnt, const int stages,
                  const uint32_t slot_bytes) {
    extern __shared__ __align__(1024) uint8_t smem[];
    // descriptors of the calls reach shared memory by bulk copies issued well ahead of their use (cold reads from
    // DRAM: ~1 us each, kept off the critical path between calls); nothing of a descriptor lives in registers
    uint64_t* cbar = reinterpret_cast<uint64_t*>(smem + (kConsDesc + kProdDesc) * kCallSlot);
    uint64_t* pbar = cbar + kConsDesc;
    uint8_t* ring = smem + kDescBytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(ring + (size_t)stages * slot_bytes);
    uint64_t* empty_bar = full_bar + kMaxStages;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int bid = (int)blockIdx.x;
    const unsigned grid = gridDim.x;

    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; s++) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], kCW);  // idle warps of a narrow call arrive too
        }
        for (int i = 0; i < kConsDesc + kProdDesc; i++) mbar_init(&cbar[i], 1);
        fence_mbar_init();
    }
    __syncthreads();

    if (warp == kCW) {
        // ===================== producer: walks the whole chain, held back only by the ring =====================
        if (lane == 0) {
            auto pdesc = [&](int c) { return reinterpret_cast<StreamCallDev*>(smem + (kConsDesc + (c % kProdDesc)) * kCallSlot); };
            auto pfetch = [&](int c) {
                mbar_arrive_expect_tx(&pbar[c % kProdDesc], kCallBytes);
                bulk_g2s(pdesc(c), calls + c, kCallBytes, &pbar[c % kProdDesc]);
            };
            for (int c = 0; c < kProdDesc - 1 && c < ncalls; c++) pfetch(c);
            int s = 0;
            uint32_t phase = 0;
            for (int c = 0; c < ncalls; c++) {
                if (c + kProdDesc - 1 < ncalls) pfetch(c + kProdDesc - 1);  // its slot held call c-1: fully issued
                mbar_wait(&pbar[c % kProdDesc], (uint32_t)(c / kProdDesc) & 1u);
                const StreamCallDev* d = pdesc(c);
                int lbid;
                const int sg = find_segment(d, bid, lbid);
                if (sg < 0) continue;
                const Mmv8Params& q = d->seg[sg];
                const bool extra = lbid < q.rows_rem;
                const int rows = q.rows_base + (extra ? q.row_unit : 0);
                const int64_t r0 = (int64_t)lbid * q.rows_base + (int64_t)(extra ? lbid : q.rows_rem) * q.row_unit;
                const int spr = extra ? q.spr1 : q.spr0;
                const uint32_t row_bytes = q.row_bytes, g2 = (uint32_t)q.G * 2u, sb_off = q.sb_off;
                const uint32_t bi_off = sb_off + (uint32_t)q.tr * g2;
                const uint8_t* wsrc = q.w;
                const uint8_t* ssrc = reinterpret_cast<const uint8_t*>(q.scales);
                const uint8_t* bsrc = reinterpret_cast<const uint8_t*>(q.biases);
                for (int ra = 0; ra < rows; ra += spr) {
                    mbar_wait(&empty_bar[s], phase ^ 1u);
                    int nr = rows - ra;
                    if (nr > spr) nr = spr;
                    const uint32_t wbytes = (uint32_t)nr * row_bytes;
                    const uint32_t sbytes = (uint32_t)nr * g2;
                    uint8_t* slot = ring + (size_t)s * slot_bytes;
                    mbar_arrive_expect_tx(&full_bar[s], wbytes + 2u * sbytes);
                    bulk_g2s(slot, wsrc + (uint64_t)(r0 + ra) * row_bytes, wbytes, &full_bar[s]);
                    const uint64_t soff = (uint64_t)(r0 + ra) * g2;
                    bulk_g2s(slot + sb_off, ssrc + soff, sbytes, &full_bar[s]);
                    bulk_g2s(slot + bi_off, bsrc + soff, sbytes, &full_bar[s]);
                    if (++s == stages) {
                        s = 0;
                        phase ^= 1u;
                    }
                }
            }
        }
    } else {
        // ===================== consumers: one call after the other =====================
        StreamCtx sc{};
        sc.err = cnt + ncalls + 1;
        auto cdesc = [&](int c) { return reinterpret_cast<StreamCallDev*>(smem + (c % kConsDesc) * kCallSlot); };
        auto cfetch = [&](int c) {
            mbar_arrive_expect_tx(&cbar[c % kConsDesc], kCallBytes);
            bulk_g2s(cdesc(c), calls + c, kCallBytes, &cbar[c % kConsDesc]);
        };
        if (threadIdx.x == 0)
            for (int c = 0; c < kConsDesc && c < ncalls; c++) cfetch(c);
        for (int c = 0; c < ncalls; c++) {
            mbar_wait(&cbar[c % kConsDesc], (uint32_t)(c / kConsDesc) & 1u);
            const StreamCallDev* d = cdesc(c);
            int lbid;
            const int seg = find_segment(d, bid, lbid);
            if (seg < 0) {
                // no rows of this call: only report it complete (this CTA neither reads x nor writes y)
                consumer_bar();  // every warp has read the descriptor before its slot is refilled
                if (threadIdx.x == 0) atomicAdd(cnt + c, 1u);
            } else {
                const int dep = d->dep;
                sc.wait_cnt = dep >= 0 ? cnt + dep : nullptr;
                sc.wait_target = grid;
                sc.done_cnt = cnt + c;
                const Mmv8Params& p = d->seg[seg];
                const int bits = d->bits[seg];
                switch (d->variant) {
                    case 0: run_bits<GS, MT, 1, 8>(p, bits, lbid, ring, &sc); break;
                    case 1: run_bits<GS, MT, 2, 8>(p, bits, lbid, ring, &sc); break;
                    case 2: run_bits<GS, MT, 1, 4>(p, bits, lbid, ring, &sc); break;
                    case 3: run_bits<GS, MT, 2, 4>(p, bits, lbid, ring, &sc); break;
                    case 4:
                        if constexpr (MT <= 2) run_bits<GS, MT, 4, 4>(p, bits, lbid, ring, &sc);
                        break;
                    default:
                        if constexpr (MT == 1) run_bits<GS, MT, 8, 4>(p, bits, lbid, ring, &sc);
                        break;
                }
            }
            // the call ended with a barrier of the consumer warps: its descriptor slot is free for call c + 2
            if (threadIdx.x == 0 && c + kConsDesc < ncalls) cfetch(c + kConsDesc);
        }
    }
    // ---- exit: the last CTA to leave puts the counters back to zero for the next launch
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned old = atomicAdd(cnt + ncalls, 1u);
        if (old == grid - 1u) {
            for (int i = 0; i <= ncalls; i++) cnt[i] = 0u;
            __threadfence();
        }
    }
}

template <int GS, int MT> int launch_inst(const gbxq_stream_info* info, const void* blob, void* counters, cudaStream_t st) {
    constexpr auto kern = stream_kernel<GS, MT>;
    static DeviceOnce configured;            // per device: occupancy is a per-device property
    static std::atomic<int> max_grid_of[64];  // resident CTAs of this kernel per device
    const int dev = DeviceOnce::dev();
    if (dev < 0) return GBXQ_ECUDA;
    if (configured.need()) {
        const int rc = allow_dynamic_smem<kern>((int)kStreamSmemMax);
        if (rc != GBXQ_OK) return rc;
        int per_sm = 0;
        const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, kStreamSmemMax);
        if (e != cudaSuccess) return check_cuda(e);
        max_grid_of[dev].store(per_sm * device_sm_count(), std::memory_order_relaxed);
        configured.done();
    }
    if (info->grid > max_grid_of[dev].load(std::memory_order_relaxed)) return GBXQ_EUNSUPPORTED;  // every CTA must be resident
    // no PDL: the chain reads its first x without griddep_wait() (mmv8_body with STREAM = true)
    return launch(kern, dim3(info->grid), dim3(kThreads), (size_t)info->smem_bytes, st, false,
                  reinterpret_cast<const StreamCallDev*>(blob), info->ncalls, reinterpret_cast<unsigned*>(counters), info->stages,
                  info->slot_bytes);
}

}  // namespace

int stream_plan(const gbxq_stream_call* calls, int ncalls, int64_t M, int dtype, void* host_blob, size_t cap,
                gbxq_stream_info* info) {
    if (info == nullptr || calls == nullptr) return GBXQ_ENULL;
    if (ncalls < 1 || ncalls > 4096) return GBXQ_ESHAPE;
    if (dtype != GBXQ_BF16 || M < 1 || M > 4) return GBXQ_EUNSUPPORTED;
    const int mt = M == 1 ? 1 : (M == 2 ? 2 : 4);
    const int total_ctas = mmv8_total_ctas();
    std::memset(info, 0, sizeof(*info));
    info->ncalls = ncalls;
    info->grid = total_ctas;
    info->mt = mt;
    info->blob_bytes = (uint64_t)ncalls * sizeof(StreamCallDev);
    info->counter_bytes = (uint64_t)(ncalls + 2) * 4u;

    // pass 1: per-segment plans (geometry, CTA shares), the largest slot and reduction buffer of the chain
    struct SegPlan { Plan pl; };
    std::vector<SegPlan> plans((size_t)ncalls * GBXQ_MAX_SEGMENTS);
    uint32_t slot_max = 0;
    size_t tail_max = 0;
    int gs = 0;
    for (int c = 0; c < ncalls; c++) {
        const gbxq_stream_call& cl = calls[c];
        if (cl.nseg < 1 || cl.nseg > GBXQ_MAX_SEGMENTS || cl.x == nullptr) return GBXQ_ENULL;
        if (((uintptr_t)cl.x & 15) || (cl.K * 2) % 16) return GBXQ_EUNSUPPORTED;
        if (!(cl.dep == GBXQ_DEP_PREV || cl.dep == GBXQ_DEP_NONE || (cl.dep >= 0 && cl.dep < c))) return GBXQ_ESHAPE;
        double bytes[GBXQ_MAX_SEGMENTS], total = 0;
        for (int i = 0; i < cl.nseg; i++) {
            const gbxq_segment& sg = cl.segs[i];
            if (sg.qweight == nullptr || sg.scales == nullptr || sg.biases == nullptr || sg.y == nullptr) return GBXQ_ENULL;
            const int v = validate(M, sg.N, cl.K, sg.bits, sg.group_size, dtype);
            if (v != GBXQ_OK) return v;
            if (gs == 0) gs = sg.group_size;
            if (sg.group_size != gs || !(gs == 64 || gs == 128)) return GBXQ_EUNSUPPORTED;
            if (!(sg.bits == 2 || sg.bits == 4 || sg.bits == 8) || sg.N < 1) return GBXQ_EUNSUPPORTED;
            if (((uintptr_t)sg.qweight | (uintptr_t)sg.scales | (uintptr_t)sg.biases) & 15) return GBXQ_EUNSUPPORTED;
            if ((uintptr_t)sg.y & 1) return GBXQ_EUNSUPPORTED;
            bytes[i] = segment_cost(sg.N, cl.K, sg.bits, gs);
            total += bytes[i];
        }
        int ctas[GBXQ_MAX_SEGMENTS], given = 0;
        for (int i = 0; i < cl.nseg; i++) {
            ctas[i] = (int)(total_ctas * bytes[i] / total);
            if (ctas[i] < 1) ctas[i] = 1;
            given += ctas[i];
        }
        if (given > total_ctas) return GBXQ_EUNSUPPORTED;
        for (int i = 0; given < total_ctas; i = (i + 1) % cl.nseg, given++) ctas[i]++;
        for (int i = 0; i < cl.nseg; i++) {
            const gbxq_segment& sg = cl.segs[i];
            const Plan pl = make_plan(M, sg.N, cl.K, sg.bits, gs, ctas[i], false);
            if (!pl.ok || pl.cpw * pl.mt > 8 || variant_of(pl.cpw, pl.R) < 0) return GBXQ_EUNSUPPORTED;
            const Plan& first = plans[(size_t)c * GBXQ_MAX_SEGMENTS].pl;
            if (i > 0 && (pl.cpw != first.cpw || pl.R != first.R)) return GBXQ_EUNSUPPORTED;
            plans[(size_t)c * GBXQ_MAX_SEGMENTS + i].pl = pl;
            if (pl.slot_bytes > slot_max) slot_max = pl.slot_bytes;
            const int64_t rows_max = ((sg.N / pl.row_unit + pl.grid - 1) / pl.grid) * pl.row_unit;
            const size_t tail = (size_t)kCW * pl.cpw * S * mt * 4 + (size_t)rows_max * 2 * pl.cw * mt * 4 + 16;
            if (tail > tail_max) tail_max = tail;
        }
    }
    const size_t fixed = kDescBytes + 2 * kMaxStages * 8 + tail_max;
    static const int force_stages = env_int("GBXQ_STREAM_STAGES", 0);
    int stages = kMaxStages;
    while (stages > 2 && fixed + (size_t)stages * slot_max > kStreamSmemMax) stages--;
    if (force_stages >= 2 && force_stages < stages) stages = force_stages;
    if (fixed + (size_t)stages * slot_max > kStreamSmemMax) return GBXQ_EUNSUPPORTED;
    info->group_size = gs;
    info->stages = stages;
    info->slot_bytes = slot_max;
    info->smem_bytes = (int32_t)(fixed + (size_t)stages * slot_max);
    if (host_blob == nullptr) return GBXQ_OK;
    if (cap < info->blob_bytes) return GBXQ_EWORKSPACE;

    // pass 2: descriptors with the chain's ring geometry
    StreamCallDev* out = reinterpret_cast<StreamCallDev*>(host_blob);
    std::memset(out, 0, (size_t)info->blob_bytes);
    for (int c = 0; c < ncalls; c++) {
        const gbxq_stream_call& cl = calls[c];
        StreamCallDev& d = out[c];
        d.nseg = cl.nseg;
        d.dep = cl.dep == GBXQ_DEP_PREV ? c - 1 : cl.dep;
        int grid = 0;
        for (int i = 0; i < cl.nseg; i++) {
            const gbxq_segment& sg = cl.segs[i];
            const Plan& pl = plans[(size_t)c * GBXQ_MAX_SEGMENTS + i].pl;
            Mmv8Params p = make_params(pl, cl.x, sg.qweight, sg.scales, sg.biases, sg.bias, sg.y, M, sg.N, cl.K, sg.bits, gs, 1);
            p.stages = stages;
            p.slot_bytes = slot_max;
            d.seg[i] = p;
            d.bits[i] = sg.bits;
            d.cta0[i] = grid;
            grid += pl.grid;
            if (i == 0) d.variant = variant_of(pl.cpw, pl.R);
        }
        for (int i = cl.nseg; i <= GBXQ_MAX_SEGMENTS; i++) d.cta0[i] = grid;
    }
    return GBXQ_OK;
}

// Development aid (not in gbxq.h): patch a HOST blob so that call c writes its 8 %globaltimer stamps (CTA 0, thread 0)
// to dbg_dev + 8 c: [0] call entered, [5] ordered after the calls before it, [7] activations arrived, [2] fragments
// built, [3] first stage landed, [4] last stage consumed, [6] y stored.
void stream_debug_patch(void* host_blob, int ncalls, unsigned long long* dbg_dev) {
    StreamCallDev* d = reinterpret_cast<StreamCallDev*>(host_blob);
    for (int c = 0; c < ncalls; c++)
        for (int i = 0; i < GBXQ_MAX_SEGMENTS; i++) d[c].seg[i].dbg = dbg_dev ? dbg_dev + 8 * c : nullptr;
}

int launch_stream(const gbxq_stream_info* info, const void* blob, void* counters, cudaStream_t st) {
    if (info == nullptr || blob == nullptr || counters == nullptr) return GBXQ_ENULL;
    if (((uintptr_t)blob & 15) || ((uintptr_t)counters & 3)) return GBXQ_EALIGN;
    if (info->ncalls < 1 || info->stages < 2 || info->stages > kMaxStages || (size_t)info->smem_bytes > kStreamSmemMax)
        return GBXQ_ESHAPE;
    switch (info->group_size * 10 + info->mt) {
        case 641: return launch_inst<64, 1>(info, blob, counters, st);
        case 1281: return launch_inst<128, 1>(info, blob, counters, st);
        case 642: return launch_inst<64, 2>(info, blob, counters, st);
        case 1282: return launch_inst<128, 2>(info, blob, counters, st);
        case 644: return launch_inst<64, 4>(info, blob, counters, st);
        case 1284: return launch_inst<128, 4>(info, blob, counters, st);
    }
    return GBXQ_EUNSUPPORTED;
}

}  // namespace gbxq
