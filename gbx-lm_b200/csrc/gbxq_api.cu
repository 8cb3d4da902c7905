// gbxq_api.cu -- extern "C" entry points of libgbxq.so (include/gbxq.h): validation + dispatch.
// Replaces the reference's calls into the MLX extension at
// gbx_lm/models/quantized_linear_gba.py:195-205 (quantized_matmul + bias) and
// gbx_lm/tuner/lora.py:62-68 (dequantize).
#include <atomic>

#include "gbxq_common.cuh"

namespace gbxq {

thread_local cudaError_t g_last_cuda_error = cudaSuccess;
static std::atomic<uint64_t> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

// GBXQ_OPT_PDL: written by gbxq_set_option, read by every launching thread
static std::atomic<int> g_pdl{2};
int pdl_mode() { return g_pdl.load(std::memory_order_relaxed); }

int device_sm_count() {
    // per-device cache (the library may be used from several devices of one process)
    static std::atomic<int> cache[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    int v = cache[dev].load(std::memory_order_relaxed);
    if (v == 0) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        cache[dev].store(v, std::memory_order_relaxed);
    }
    return v;
}

// M above which the tensor-core kernel takes over from the streaming GEMV.  The GEMV re-streams
// the weights once per 2 tokens, the GEMM dequantises each weight once per <=256 tokens.
static constexpr int64_t kMmvMaxM = 2;
static constexpr int64_t kSkinnyMaxM = 16;  // 2 passes of 8 tokens; above that the tcgen05 GEMM amortises better

// Rows of x from which the TMEM-operand GEMM (gbxq_gemm_ts_sm100.cu) takes over (GBXQ_TS_MIN_M overrides; 0 = never).
// Measured on the 8B decode step (profiles/r02y_*): 8 rows 2.09 ms on the skinny kernel against 3.22 ms, 16 rows 3.9
// against 3.28 ms, 32 rows 5.9 (shared-memory-operand GEMM) against 3.76 ms -> from 9 rows.
static int ts_min_m() {
    static const int v = env_int("GBXQ_TS_MIN_M", 9);
    return v;
}

static int select(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                  const void* y) {
    if (ts_min_m() > 0 && M >= ts_min_m() && gemm_ts_supported(M, N, K, bits, gs, dtype, x, w, y)) return GBXQ_KERNEL_GEMM_TS;
    const bool skinny_ok = skinny_supported(M, N, K, bits, gs, dtype, x, w, y);
    const bool gemv_ok = gemv_supported(M, N, K, bits, gs, dtype, x, w, y);
    const bool gemm_ok = gemm_supported(M, N, K, bits, gs, dtype, x, w, y);
    // tensor-pipe matrix-vector kernels: their IMMA/HMMA work grows with the token count, so they win at 1-2 tokens
    // only (profiles/r01g_micro_m234.txt: q/o M=3 9.6 us against 7.1 us for the 8-token skinny kernel; M=2 6.2 vs 7.1)
    if (M <= kMmvMaxM && mmv8_supported(M, N, K, bits, gs, dtype, x, w, y)) return GBXQ_KERNEL_MMV8;
    if (M <= kMmvMaxM && mmv_supported(M, N, K, bits, gs, dtype, x, w, y)) return GBXQ_KERNEL_MMV;
    if (M > kMmvMaxM && M <= 4 && !skinny_ok && mmv8_supported(M, N, K, bits, gs, dtype, x, w, y)) return GBXQ_KERNEL_MMV8;
    // measured on B200 (profiles/): the FMA-pipe GEMV wins at M <= 2, the tensor-pipe skinny kernel costs the
    // same for 1..8 tokens and wins from M = 3
    if (gemv_ok && M <= 2) return GBXQ_KERNEL_GEMV;
    if (skinny_ok && (M <= kSkinnyMaxM || !gemm_ok)) return GBXQ_KERNEL_SKINNY;
    if (gemv_ok && (M <= 4 || !gemm_ok)) return GBXQ_KERNEL_GEMV;  // 3-/6-bit packings and odd shapes
    if (gemm_ok) return GBXQ_KERNEL_GEMM;
    if (gemv_ok) return GBXQ_KERNEL_GEMV;
    return GBXQ_KERNEL_GENERIC;
}

}  // namespace gbxq

using namespace gbxq;

extern "C" {

int gbxq_abi_version(void) { return GBXQ_ABI_VERSION; }

const char* gbxq_status_string(int status) {
    switch (status) {
        case GBXQ_OK: return "ok";
        case GBXQ_EINVAL_BITS: return "bits must be one of 2, 3, 4, 6, 8";
        case GBXQ_EINVAL_GROUP: return "group_size must be 32, 64 or 128";
        case GBXQ_ESHAPE: return "inconsistent shapes (need K % 32 == 0, K % group_size == 0, sizes >= 0)";
        case GBXQ_EDTYPE: return "dtype must be 0 (bf16), 1 (f16) or 2 (f32)";
        case GBXQ_EALIGN: return "pointer alignment (x, y, qweight, w_out need 16 bytes)";
        case GBXQ_ENULL: return "required pointer is NULL";
        case GBXQ_ECUDA: return "CUDA runtime error (see gbxq_last_cuda_error_string)";
        case GBXQ_EWORKSPACE: return "workspace too small";
        case GBXQ_EUNSUPPORTED: return "kernel family does not support these arguments";
    }
    return "unknown status";
}

int gbxq_last_cuda_error(void) { return (int)g_last_cuda_error; }
const char* gbxq_last_cuda_error_string(void) { return cudaGetErrorString(g_last_cuda_error); }
uint64_t gbxq_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

// Development aid (not in gbxq.h): the next `launches` mmv8 launches write 8 %globaltimer stamps each (CTA 0, thread 0)
// to `buf_dev`: entry, after griddepcontrol.wait, after the prologue, first stage landed, main loop done, CTA barrier,
// exit.  tools/timeline.py prints them.
void gbxq_debug_timeline(unsigned long long* buf_dev, int launches) { mmv8_debug_timeline(buf_dev, launches); }
void gbxq_debug_timeline_all(unsigned long long* buf_dev, int launches, int stride_ctas) {
    mmv8_debug_timeline_all(buf_dev, launches, stride_ctas);
}

// Development aid: the NEXT GBXQ_KERNEL_GEMM_TS launch writes its CTA-0 timeline (8 + 4 * 64 slots) to buf_dev.
void gbxq_debug_ts_timeline(unsigned long long* buf_dev) { gemm_ts_debug_timeline(buf_dev); }

void gbxq_debug_stream_timeline(void* host_blob, int ncalls, unsigned long long* dbg_dev) {
    stream_debug_patch(host_blob, ncalls, dbg_dev);
}

int gbxq_set_option(int key, int value) {
    if (key == GBXQ_OPT_PDL) {
        g_pdl.store(value < 0 ? 0 : (value > 2 ? 2 : value), std::memory_order_relaxed);
        return GBXQ_OK;
    }
    return GBXQ_EUNSUPPORTED;
}
int gbxq_get_option(int key) {
    if (key == GBXQ_OPT_PDL) return pdl_mode();
    return GBXQ_EUNSUPPORTED;
}

size_t gbxq_workspace_bytes(int64_t M, int64_t N, int64_t K, int bits, int group_size, int dtype) {
    // only the split-K path of the tensor-core GEMM (17..256 rows of x on a layer with few output tiles) uses scratch
    if (validate(M, N, K, bits, group_size, dtype) != GBXQ_OK || dtype != GBXQ_BF16) return 0;
    // sized for either tensor-core kernel whichever AUTO would pick (an explicit GBXQ_KERNEL_GEMM* request uses it too)
    if (M <= 4) return 0;
    const void* al = (const void*)16;
    if (!gemm_supported(M, N, K, bits, group_size, dtype, al, al, al) && !gemm_ts_supported(M, N, K, bits, group_size, dtype, al, al, al))
        return 0;
    return gemm_workspace_bytes(M, N, K);
}

int gbxq_select_kernel(int64_t M, int64_t N, int64_t K, int bits, int group_size, int dtype) {
    const int rc = validate(M, N, K, bits, group_size, dtype);
    if (rc != GBXQ_OK) return rc;
    // alignment-agnostic answer: assume 16-byte aligned tensors
    return select(M, N, K, bits, group_size, dtype, (const void*)16, (const void*)16, (const void*)16);
}

int gbxq_qmm_ex(const void* x, const uint32_t* qweight, const void* scales, const void* biases, const void* bias,
                void* y, int64_t M, int64_t N, int64_t K, int bits, int group_size, int dtype, int kernel,
                void* workspace, size_t workspace_bytes, void* stream) {
    const int rc = validate(M, N, K, bits, group_size, dtype);
    if (rc != GBXQ_OK) return rc;
    if (M == 0 || N == 0) return GBXQ_OK;
    if (!x || !qweight || !scales || !biases || !y) return GBXQ_ENULL;
    const size_t esz = dtype == GBXQ_F32 ? 4 : 2;
    if (((uintptr_t)x | (uintptr_t)y | (uintptr_t)scales | (uintptr_t)biases | (uintptr_t)bias) & (esz - 1))
        return GBXQ_EALIGN;
    if ((uintptr_t)qweight & 3) return GBXQ_EALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    int k = kernel;
    if (k == GBXQ_KERNEL_AUTO) k = select(M, N, K, bits, group_size, dtype, x, qweight, y);
    switch (k) {
        case GBXQ_KERNEL_GENERIC:
            return launch_generic(x, qweight, scales, biases, bias, y, M, N, K, bits, group_size, dtype, st);
        case GBXQ_KERNEL_GEMV:
            if (!gemv_supported(M, N, K, bits, group_size, dtype, x, qweight, y)) return GBXQ_EUNSUPPORTED;
            return launch_gemv(x, qweight, scales, biases, bias, y, M, N, K, bits, group_size, st);
        case GBXQ_KERNEL_SKINNY:
            if (!skinny_supported(M, N, K, bits, group_size, dtype, x, qweight, y)) return GBXQ_EUNSUPPORTED;
            return launch_skinny(x, qweight, scales, biases, bias, y, M, N, K, bits, group_size, st);
        case GBXQ_KERNEL_MMV8:
            if (!mmv8_supported(M, N, K, bits, group_size, dtype, x, qweight, y)) return GBXQ_EUNSUPPORTED;
            return launch_mmv8(x, qweight, scales, biases, bias, y, M, N, K, bits, group_size, st);
        case GBXQ_KERNEL_MMV:
            if (!mmv_supported(M, N, K, bits, group_size, dtype, x, qweight, y)) return GBXQ_EUNSUPPORTED;
            return launch_mmv(x, qweight, scales, biases, bias, y, M, N, K, bits, group_size, st);
        case GBXQ_KERNEL_GEMM:
            if (!gemm_supported(M, N, K, bits, group_size, dtype, x, qweight, y)) return GBXQ_EUNSUPPORTED;
            return launch_gemm(x, qweight, scales, biases, bias, y, M, N, K, bits, group_size, workspace, workspace_bytes, st);
        case GBXQ_KERNEL_GEMM_TS:
            if (!gemm_ts_supported(M, N, K, bits, group_size, dtype, x, qweight, y)) return GBXQ_EUNSUPPORTED;
            return launch_gemm_ts(x, qweight, scales, biases, bias, y, M, N, K, bits, group_size, workspace, workspace_bytes, st);
    }
    return GBXQ_EUNSUPPORTED;
}

int gbxq_qmm(const void* x, const uint32_t* qweight, const void* scales, const void* biases, const void* bias,
             void* y, int64_t M, int64_t N, int64_t K, int bits, int group_size, int dtype, void* workspace,
             size_t workspace_bytes, void* stream) {
    return gbxq_qmm_ex(x, qweight, scales, biases, bias, y, M, N, K, bits, group_size, dtype, GBXQ_KERNEL_AUTO,
                       workspace, workspace_bytes, stream);
}

int gbxq_qmm_rowpar_allreduce(const void* x, const uint32_t* qweight, const void* scales, const void* biases,
                              const void* bias, void* y, int64_t M, int64_t N, int64_t K, int bits, int group_size,
                              int dtype, const gbxq_comm* comm, void* stream) {
    const int rc = validate(M, N, K, bits, group_size, dtype);
    if (rc != GBXQ_OK) return rc;
    if (!comm || !comm->peer_stage_host || !comm->peer_flags_host) return GBXQ_ENULL;
    if (comm->world < 1 || comm->world > 8 || comm->rank < 0 || comm->rank >= comm->world) return GBXQ_ESHAPE;
    if (M == 0 || N == 0) return GBXQ_OK;
    if (!x || !qweight || !scales || !biases || !y) return GBXQ_ENULL;
    if (((uintptr_t)x | (uintptr_t)y | (uintptr_t)scales | (uintptr_t)biases | (uintptr_t)bias) & 1) return GBXQ_EALIGN;
    if ((uintptr_t)qweight & 3) return GBXQ_EALIGN;
    if (dtype != GBXQ_BF16 || M > 4 || !mmv8_supported(M, N, K, bits, group_size, dtype, x, qweight, y))
        return GBXQ_EUNSUPPORTED;
    return launch_mmv8_ar(x, qweight, scales, biases, bias, y, M, N, K, bits, group_size, comm, (cudaStream_t)stream);
}

int gbxq_qmm_grouped(const gbxq_segment* segs, int nseg, const void* x, int64_t M, int64_t K, int dtype, void* stream) {
    return gbxq_qmm_grouped_ws(segs, nseg, x, M, K, dtype, nullptr, 0, stream);
}

size_t gbxq_grouped_workspace_bytes(const gbxq_segment* segs, int nseg, int64_t M, int64_t K, int dtype) {
    if (!segs || nseg < 1 || dtype != GBXQ_BF16 || M <= 4) return 0;
    size_t need = 0;
    for (int i = 0; i < nseg; i++) {  // the per-segment fallback uses the same scratch, one call after the other
        const size_t b = gbxq_workspace_bytes(M, segs[i].N, K, segs[i].bits, segs[i].group_size, dtype);
        if (b > need) need = b;
    }
    if (nseg >= 2 && nseg <= 3) {
        const size_t b = gemm_workspace_bytes(M, gemm_ts_grouped_npad(segs, nseg), K);
        if (b > need) need = b;
    }
    return need;
}

int gbxq_qmm_grouped_ws(const gbxq_segment* segs, int nseg, const void* x, int64_t M, int64_t K, int dtype, void* workspace,
                        size_t workspace_bytes, void* stream) {
    if (nseg < 0) return GBXQ_ESHAPE;
    if (nseg == 0) return GBXQ_OK;
    if (!segs) return GBXQ_ENULL;
    const size_t esz = dtype == GBXQ_F32 ? 4 : 2;
    for (int i = 0; i < nseg; i++) {
        const gbxq_segment& s = segs[i];
        const int rc = validate(M, s.N, K, s.bits, s.group_size, dtype);
        if (rc != GBXQ_OK) return rc;
        if (M == 0 || s.N == 0) continue;
        if (!x || !s.qweight || !s.scales || !s.biases || !s.y) return GBXQ_ENULL;
        if (((uintptr_t)x | (uintptr_t)s.y | (uintptr_t)s.scales | (uintptr_t)s.biases | (uintptr_t)s.bias) & (esz - 1))
            return GBXQ_EALIGN;
        if ((uintptr_t)s.qweight & 3) return GBXQ_EALIGN;
    }
    if (M == 0) return GBXQ_OK;
    if (dtype == GBXQ_BF16 && nseg >= 2 && nseg <= GBXQ_MAX_SEGMENTS && M <= kMmvMaxM) {
        const int rc = launch_mmv8_grouped(segs, nseg, x, M, K, (cudaStream_t)stream);
        if (rc != GBXQ_EUNSUPPORTED) return rc;
    }
    // decode batches / prefill: segments of one bit width and group size share ONE launch of the TMEM-operand GEMM
    if (dtype == GBXQ_BF16 && nseg >= 2 && nseg <= 3 && ts_min_m() > 0 && M >= ts_min_m()) {
        const int rc = launch_gemm_ts_grouped(segs, nseg, x, M, K, workspace, workspace_bytes, (cudaStream_t)stream);
        if (rc != GBXQ_EUNSUPPORTED) return rc;
    }
    for (int i = 0; i < nseg; i++) {
        const gbxq_segment& s = segs[i];
        const int rc = gbxq_qmm_ex(x, s.qweight, s.scales, s.biases, s.bias, s.y, M, s.N, K, s.bits, s.group_size, dtype,
                                   GBXQ_KERNEL_AUTO, workspace, workspace_bytes, stream);
        if (rc != GBXQ_OK) return rc;
    }
    return GBXQ_OK;
}

int gbxq_head_gemv(const void* x, const void* weight, void* y, int64_t M, int64_t V, int64_t K, int dtype, void* stream) {
    if (dtype != GBXQ_BF16) return GBXQ_EUNSUPPORTED;
    if (M < 0 || V < 0 || K <= 0) return GBXQ_ESHAPE;
    if (M == 0 || V == 0) return GBXQ_OK;
    if (!x || !weight || !y) return GBXQ_ENULL;
    return launch_head_gemv(x, weight, y, M, V, K, (cudaStream_t)stream);
}

int gbxq_gather_qmm(const void* x, const uint32_t* qweight, const void* scales, const void* biases, const void* bias,
                    const int32_t* lhs_indices, const int32_t* rhs_indices, void* y, int64_t R, int64_t XB, int64_t E,
                    int64_t M, int64_t N, int64_t K, int transpose, int bits, int group_size, int dtype, void* stream) {
    // the quantized axis is K for transpose = 1 (rows of an [N, K] matrix) and N for transpose = 0 (rows of a [K, N] one)
    const int rc = transpose ? validate(M, N, K, bits, group_size, dtype) : validate(M, K, N, bits, group_size, dtype);
    if (rc != GBXQ_OK) return rc;
    if (R < 0 || XB < 0 || E < 0 || K <= 0 || N < 0) return GBXQ_ESHAPE;
    if (R == 0 || M == 0 || N == 0) return GBXQ_OK;
    if (XB == 0 || E == 0) return GBXQ_ESHAPE;
    if (lhs_indices == nullptr && R > XB) return GBXQ_ESHAPE;
    if (rhs_indices == nullptr && R > E) return GBXQ_ESHAPE;
    if (!x || !qweight || !scales || !biases || !y) return GBXQ_ENULL;
    if (!transpose && bias != nullptr) return GBXQ_EUNSUPPORTED;
    const size_t esz = dtype == GBXQ_F32 ? 4 : 2;
    if (((uintptr_t)x | (uintptr_t)y | (uintptr_t)scales | (uintptr_t)biases | (uintptr_t)bias) & (esz - 1)) return GBXQ_EALIGN;
    if (((uintptr_t)qweight | (uintptr_t)lhs_indices | (uintptr_t)rhs_indices) & 3) return GBXQ_EALIGN;
    return launch_gather_qmm(x, qweight, scales, biases, bias, lhs_indices, rhs_indices, y, R, XB, E, M, N, K, transpose ? 1 : 0,
                             bits, group_size, dtype, (cudaStream_t)stream);
}

int gbxq_stream_plan(const gbxq_stream_call* calls_host, int ncalls, int64_t M, int dtype, void* host_blob,
                     size_t blob_capacity, gbxq_stream_info* info) {
    return stream_plan(calls_host, ncalls, M, dtype, host_blob, blob_capacity, info);
}

int gbxq_qmm_stream(const gbxq_stream_info* info, const void* blob_dev, void* counters_dev, void* stream) {
    return launch_stream(info, blob_dev, counters_dev, (cudaStream_t)stream);
}

int gbxq_dequantize(const uint32_t* qweight, const void* scales, const void* biases, void* w_out, int64_t N,
                    int64_t K, int bits, int group_size, int dtype, void* stream) {
    const int rc = validate(0, N, K, bits, group_size, dtype);
    if (rc != GBXQ_OK) return rc;
    if (N == 0) return GBXQ_OK;
    if (!qweight || !scales || !biases || !w_out) return GBXQ_ENULL;
    if (((uintptr_t)w_out & 15) || ((uintptr_t)qweight & 3)) return GBXQ_EALIGN;
    return launch_dequantize(qweight, scales, biases, w_out, N, K, bits, group_size, dtype, (cudaStream_t)stream);
}

int gbxq_rope_cache(void* q, const void* k, const void* v, const int64_t* pos_dev, int pos_stride,
                    const float* inv_freq_dev, void* k_cache, void* v_cache, int B, int Hq, int Hkv, int D,
                    int64_t max_len, int64_t keep, void* stream) {
    return launch_rope_cache(q, k, v, pos_dev, pos_stride, inv_freq_dev, k_cache, v_cache, B, 1, Hq, Hkv, D, max_len, keep,
                             (cudaStream_t)stream);
}

int gbxq_rope_cache_multi(void* q, const void* k, const void* v, const int64_t* pos_dev, int pos_stride,
                          const float* inv_freq_dev, void* k_cache, void* v_cache, int B, int T, int Hq, int Hkv, int D,
                          int64_t max_len, void* stream) {
    return launch_rope_cache(q, k, v, pos_dev, pos_stride, inv_freq_dev, k_cache, v_cache, B, T, Hq, Hkv, D, max_len, -1,
                             (cudaStream_t)stream);
}

int gbxq_decode_attention(const void* q, const void* k_cache, const void* v_cache, const int64_t* pos_dev,
                          int pos_stride, void* out, int B, int Hq, int Hkv, int D, int64_t max_len,
                          int64_t attend_len, float scale, void* stream) {
    return launch_decode_attention(q, k_cache, v_cache, pos_dev, pos_stride, out, B, 1, Hq, Hkv, D, max_len, attend_len,
                                   scale, (cudaStream_t)stream);
}

int gbxq_decode_attention_multi(const void* q, const void* k_cache, const void* v_cache, const int64_t* pos_dev,
                                int pos_stride, void* out, int B, int T, int Hq, int Hkv, int D, int64_t max_len,
                                int64_t attend_len, float scale, void* stream) {
    return launch_decode_attention(q, k_cache, v_cache, pos_dev, pos_stride, out, B, T, Hq, Hkv, D, max_len, attend_len,
                                   scale, (cudaStream_t)stream);
}

int gbxq_rope_cache_quantized(void* q, const void* k, const void* v, const int64_t* pos_dev, int pos_stride,
                              const float* inv_freq_dev, uint32_t* k_codes, void* k_scales, void* k_biases,
                              uint32_t* v_codes, void* v_scales, void* v_biases, int B, int Hq, int Hkv, int D,
                              int64_t max_len, int64_t keep, int bits, int group_size, void* stream) {
    return launch_rope_cache_quantized({q, k, v, pos_dev, pos_stride, inv_freq_dev, k_codes, k_scales, k_biases, v_codes,
                                        v_scales, v_biases, B, 1, Hq, Hkv, D, max_len, keep, bits, group_size},
                                       (cudaStream_t)stream);
}

int gbxq_rope_cache_quantized_multi(void* q, const void* k, const void* v, const int64_t* pos_dev, int pos_stride,
                                    const float* inv_freq_dev, uint32_t* k_codes, void* k_scales, void* k_biases,
                                    uint32_t* v_codes, void* v_scales, void* v_biases, int B, int T, int Hq, int Hkv,
                                    int D, int64_t max_len, int bits, int group_size, void* stream) {
    return launch_rope_cache_quantized({q, k, v, pos_dev, pos_stride, inv_freq_dev, k_codes, k_scales, k_biases, v_codes,
                                        v_scales, v_biases, B, T, Hq, Hkv, D, max_len, -1, bits, group_size},
                                       (cudaStream_t)stream);
}

size_t gbxq_decode_attention_quantized_workspace_bytes(int B, int Hq, int Hkv, int D, int64_t attend_len) {
    return qattn_workspace_bytes(B, Hq, Hkv, D, attend_len);
}

int gbxq_decode_attention_quantized(const void* q, const uint32_t* k_codes, const void* k_scales,
                                    const void* k_biases, const uint32_t* v_codes, const void* v_scales,
                                    const void* v_biases, const int64_t* pos_dev, int pos_stride, void* out, int B,
                                    int Hq, int Hkv, int D, int64_t max_len, int64_t attend_len, float scale,
                                    int bits, int group_size, void* workspace, size_t workspace_bytes, void* stream) {
    return launch_decode_attention_quantized({q, k_codes, k_scales, k_biases, v_codes, v_scales, v_biases, pos_dev,
                                              pos_stride, out, B, 1, Hq, Hkv, D, max_len, attend_len, scale, bits,
                                              group_size, workspace, workspace_bytes},
                                             (cudaStream_t)stream);
}

int gbxq_decode_attention_quantized_multi(const void* q, const uint32_t* k_codes, const void* k_scales,
                                          const void* k_biases, const uint32_t* v_codes, const void* v_scales,
                                          const void* v_biases, const int64_t* pos_dev, int pos_stride, void* out, int B,
                                          int T, int Hq, int Hkv, int D, int64_t max_len, int64_t attend_len,
                                          float scale, int bits, int group_size, void* workspace,
                                          size_t workspace_bytes, void* stream) {
    return launch_decode_attention_quantized({q, k_codes, k_scales, k_biases, v_codes, v_scales, v_biases, pos_dev,
                                              pos_stride, out, B, T, Hq, Hkv, D, max_len, attend_len, scale, bits,
                                              group_size, workspace, workspace_bytes},
                                             (cudaStream_t)stream);
}

int gbxq_add_rmsnorm(const void* x, const void* r, const void* w, float eps, void* h_out, void* y_out, int64_t rows, int H,
                     void* stream) {
    if (!x || !w || !y_out) return GBXQ_ENULL;
    if (((uintptr_t)x | (uintptr_t)r | (uintptr_t)w | (uintptr_t)h_out | (uintptr_t)y_out) & 15) return GBXQ_EALIGN;
    return launch_add_rmsnorm(x, r, w, eps, h_out, y_out, rows, H, (cudaStream_t)stream);
}

int gbxq_silu_mul(const void* gate, const void* up, void* out, int64_t n, void* stream) {
    if (!gate || !up || !out) return GBXQ_ENULL;
    if (((uintptr_t)gate | (uintptr_t)up | (uintptr_t)out) & 15) return GBXQ_EALIGN;
    return launch_silu_mul(gate, up, out, n, (cudaStream_t)stream);
}

int gbxq_allreduce_oneshot(const void* in, void* out, int64_t count, int dtype, void* const* peer_bufs_dev,
                           uint32_t* const* peer_flags_dev, int64_t capacity, int rank, int world, uint32_t seq,
                           void* stream) {
    if (dtype < 0 || dtype > 2) return GBXQ_EDTYPE;
    if (count < 0 || world < 1 || world > 8 || rank < 0 || rank >= world || capacity < 2 * count) return GBXQ_ESHAPE;
    if (count == 0) return GBXQ_OK;
    if (!in || !out || !peer_bufs_dev || !peer_flags_dev) return GBXQ_ENULL;
    if (((uintptr_t)in | (uintptr_t)out) & 15) return GBXQ_EALIGN;
    const size_t esz = dtype == GBXQ_F32 ? 4 : 2;
    if (((capacity / 2) * esz) % 16) return GBXQ_EALIGN;
    return launch_allreduce_oneshot(in, out, count, dtype, peer_bufs_dev, peer_flags_dev, capacity, rank, world, seq,
                                    (cudaStream_t)stream);
}

}  // extern "C"
