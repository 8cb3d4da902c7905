// gbxq_common.cuh -- shared device/host helpers for libgbxq (sm_100a only).
//
// Numerical contract (restating MLX affine quantisation as used by the reference at
// gbx_lm/models/quantized_linear_gba.py:195-203; see include/gbxq.h):
//   code k of row n = bits [k*bits,(k+1)*bits) of the row's LSB-first bitstream (uint32 LE words).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <atomic>

#include "../../include/gbxq.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libgbxq is written for sm_100a (B200) only"
#endif

namespace gbxq {

// ------------------------------------------------------------------ error plumbing (host)
extern thread_local cudaError_t g_last_cuda_error;
void count_launch();

inline int check_cuda(cudaError_t e) {
    if (e != cudaSuccess) {
        g_last_cuda_error = e;
        return GBXQ_ECUDA;
    }
    return GBXQ_OK;
}

// GBXQ_OPT_PDL (include/gbxq.h), set by gbxq_set_option: 0 plain launches; 1 PDL, every global read after
// griddepcontrol.wait; 2 (default) PDL, frozen weights streamed before the wait.
int pdl_mode();
inline int pdl_early_weights() { return pdl_mode() >= 2 ? 1 : 0; }

// an integer tuning knob from the environment, `dflt` when unset
inline int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v ? atoi(v) : dflt;
}

// Per-DEVICE one-time configuration of a kernel (cudaFuncSetAttribute is a per-device property: a process that drives
// several GPUs must set it on each).  `need()` is true until `done()` was called on the current device.
struct DeviceOnce {
    std::atomic<uint64_t> mask{0};
    static int dev() {
        int d = 0;
        return (cudaGetDevice(&d) == cudaSuccess && d >= 0 && d < 64) ? d : -1;
    }
    bool need() const {
        const int d = dev();
        return d < 0 || !((mask.load(std::memory_order_relaxed) >> d) & 1u);
    }
    void done() {
        const int d = dev();
        if (d >= 0) mask.fetch_or(uint64_t(1) << d, std::memory_order_relaxed);
    }
};

// Lets kernel Kern take up to `bytes` of dynamic shared memory, once per device.  The state is keyed on the kernel
// itself: every instantiation of a kernel template is configured on its own.
template <auto Kern>
int allow_dynamic_smem(int bytes) {
    static DeviceOnce configured;
    if (configured.need()) {
        const cudaError_t e = cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) return check_cuda(e);
        configured.done();
    }
    return GBXQ_OK;
}

// Every kernel launch of the library: enqueues kern(args...) on st with `smem` bytes of dynamic shared memory, counts
// it and returns its status.  pdl: the launch carries the programmatic-stream-serialization attribute while
// pdl_mode() > 0, so the kernel may start before the previous kernel of the stream has ended.  Such a kernel must
// execute griddep_wait() before it reads what an earlier kernel wrote (or writes what one may still read).
template <typename... KArgs, typename... Args>
int launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, const Args&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl && pdl_mode() > 0 ? 1 : 0;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
    count_launch();
    return check_cuda(e);
}

// ------------------------------------------------------------------ element types
template <int DT> struct TypeOf;
template <> struct TypeOf<GBXQ_BF16> { using T = __nv_bfloat16; };
template <> struct TypeOf<GBXQ_F16> { using T = __half; };
template <> struct TypeOf<GBXQ_F32> { using T = float; };

__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(float v) { return v; }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }

// round an fp32 value to T and widen back (one rounding step of T-typed arithmetic)
template <typename T> __device__ __forceinline__ float round_to(float v) { return to_f32(from_f32<T>(v)); }

// ------------------------------------------------------------------ code extraction
// 8 consecutive codes starting at code index k8*8 of a row (k8 = index of the 8-code octet).
// Octets never need more than a 64-bit window: bit offset of octet = 8*bits*k8; within its first
// word the offset is in {0,8,16,24} and 8*bits <= 64 - offset for every supported width
// (3-bit: 24 bits, offset<=24; 6-bit: 48 bits, offset in {0,16}).
template <int BITS>
__device__ __forceinline__ void extract_octet(const uint32_t* __restrict__ row, int64_t k8, int64_t words_per_row,
                                              uint32_t (&q)[8]) {
    const int64_t bit = k8 * (8 * BITS);
    const int64_t wi = bit >> 5;
    const int off = (int)(bit & 31);
    uint64_t win = row[wi];
    if (off + 8 * BITS > 32) {
        // second word exists whenever the octet crosses a word border (K % 32 == 0 keeps rows whole)
        win |= (uint64_t)row[wi + 1] << 32;
    }
    (void)words_per_row;
    win >>= off;
#pragma unroll
    for (int i = 0; i < 8; i++) q[i] = (uint32_t)((win >> (i * BITS)) & ((1u << BITS) - 1u));
}

// Row of a static KV cache of max_len rows that receives absolute position pos, or -1 for none (the decode-step cache
// writes of gbxq_glue.cu / gbxq_qattn.cu).  keep < 0: a flat cache, row = pos, nothing outside [0, max_len).
// keep in [0, max_len): a rotating cache of window max_len whose first keep rows are attention sinks; the rule of
// cache.py's ring_slot: pos below max_len, keep + (pos - keep) mod (max_len - keep) from there.
__device__ __forceinline__ int64_t kv_cache_row(int64_t pos, int64_t max_len, int64_t keep) {
    if (pos < 0) return -1;
    if (pos < max_len) return pos;
    return keep < 0 ? -1 : keep + (pos - keep) % (max_len - keep);
}

// ------------------------------------------------------------------ small PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Programmatic dependent launch (both are no-ops in a launch without the attribute): wait until the kernels before this
// one in the stream have completed and their writes are visible; let the next kernel of the stream start launching.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// The small decode-step kernels (gbxq_glue.cu, gbxq_qattn.cu): wait for the producers of the inputs FIRST, then let the
// next kernel of the stream (a QuantizedLinear forward) become resident and stream its frozen weights while this one
// runs.  The order matters: triggering before the wait would let the next matmul's CTAs fill the SMs while this grid is
// not yet scheduled, and they would wait for it forever.
__device__ __forceinline__ void pdl_wait_then_trigger() {
    griddep_wait();
    griddep_launch_dependents();
}

// d = a(bf16) * b(bf16) + c(f32): one FHFMA.BF16 on sm_100 (PTX ISA 8.6 mixed-precision fma).
__device__ __forceinline__ float fma_bf16_f32(uint16_t a, uint16_t b, float c) {
    float d;
    asm("fma.rn.f32.bf16 %0, %1, %2, %3;" : "=f"(d) : "h"(a), "h"(b), "f"(c));
    return d;
}

// (a & b) | c in one LOP3
__device__ __forceinline__ uint32_t lop3_and_or(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------ mbarrier / bulk-copy (TMA engine)
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra.uni WAIT_DONE;\n"
        "bra.uni WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// the same on 32-bit shared-memory addresses (loops that step ring positions by increments)
__device__ __forceinline__ void mbar_arrive_u32(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra.uni WAIT_DONE;\n"
        "bra.uni WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// 1-D bulk async copy global -> shared, completion counted in bytes on `bar` (SASS: UBLKCP).
// dst/src 16-byte aligned, bytes % 16 == 0.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}

// ------------------------------------------------------------------ host-side argument validation
inline int validate(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype) {
    if (!(bits == 2 || bits == 3 || bits == 4 || bits == 6 || bits == 8)) return GBXQ_EINVAL_BITS;
    if (!(gs == 32 || gs == 64 || gs == 128)) return GBXQ_EINVAL_GROUP;
    if (dtype < 0 || dtype > 2) return GBXQ_EDTYPE;
    if (M < 0 || N < 0 || K <= 0 || (K % 32) || (K % gs)) return GBXQ_ESHAPE;
    if (M > (int64_t)1 << 30 || N > (int64_t)1 << 30 || K > (int64_t)1 << 30) return GBXQ_ESHAPE;
    return GBXQ_OK;
}

// launchers implemented in the per-kernel translation units
int launch_dequantize(const uint32_t* w, const void* s, const void* b, void* out, int64_t N, int64_t K, int bits,
                      int gs, int dtype, cudaStream_t st);
int launch_generic(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y,
                   int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, cudaStream_t st);
bool gemv_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                    const void* y);
int launch_gemv(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                int64_t N, int64_t K, int bits, int gs, cudaStream_t st);
bool skinny_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                      const void* y);
int launch_skinny(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                  int64_t N, int64_t K, int bits, int gs, cudaStream_t st);
bool mmv_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                   const void* y);
int launch_mmv(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
               int64_t N, int64_t K, int bits, int gs, cudaStream_t st);
bool mmv8_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                    const void* y);
int launch_mmv8(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                int64_t N, int64_t K, int bits, int gs, cudaStream_t st);
int launch_mmv8_ar(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                   int64_t N, int64_t K, int bits, int gs, const gbxq_comm* comm, cudaStream_t st);
void mmv8_debug_timeline(unsigned long long* buf, int launches);
void mmv8_debug_timeline_all(unsigned long long* buf, int launches, int stride_ctas);
int launch_mmv8_grouped(const gbxq_segment* segs, int nseg, const void* x, int64_t M, int64_t K, cudaStream_t st);
int stream_plan(const gbxq_stream_call* calls, int ncalls, int64_t M, int dtype, void* host_blob, size_t cap,
                gbxq_stream_info* info);
void stream_debug_patch(void* host_blob, int ncalls, unsigned long long* dbg_dev);
int launch_stream(const gbxq_stream_info* info, const void* blob, void* counters, cudaStream_t st);
// The decode-step cache write and attention (gbxq_glue.cu / gbxq_qattn.cu).  pos_stride 0: pos[0] is the position of
// every batch row; 1: pos[b] is row b's; else GBXQ_ESHAPE.  keep < 0: a flat cache; keep in [0, max_len): a rotating
// cache with keep sink rows (kv_cache_row); else GBXQ_ESHAPE.  T in [1, kMaxBlockTokens]: T consecutive tokens per
// batch row at pos .. pos + T - 1 (a verify block; the `_multi` entry points pass keep = -1).  The launchers check
// every argument.
constexpr int kMaxBlockTokens = 8;
int launch_rope_cache(void* q, const void* k, const void* v, const int64_t* pos, int pos_stride, const float* inv_freq,
                      void* kc, void* vc, int B, int T, int Hq, int Hkv, int D, int64_t max_len, int64_t keep,
                      cudaStream_t st);
int launch_decode_attention(const void* q, const void* kc, const void* vc, const int64_t* pos, int pos_stride, void* out,
                            int B, int T, int Hq, int Hkv, int D, int64_t max_len, int64_t attend_len, float scale,
                            cudaStream_t st);
// arguments of the quantized-cache decode step (gbxq_qattn.cu): one (codes, scales, biases) triple per side, bf16
struct QCacheWrite {
    void* q;
    const void* k;
    const void* v;
    const int64_t* pos;
    int pos_stride;
    const float* inv_freq;
    uint32_t* kq;
    void *ks, *kb;
    uint32_t* vq;
    void *vs, *vb;
    int B, T, Hq, Hkv, D;
    int64_t max_len, keep;
    int bits, gs;
};
struct QAttn {
    const void* q;
    const uint32_t* kq;
    const void *ks, *kb;
    const uint32_t* vq;
    const void *vs, *vb;
    const int64_t* pos;
    int pos_stride;
    void* out;
    int B, T, Hq, Hkv, D;
    int64_t max_len, attend_len;
    float scale;
    int bits, gs;
    void* ws;
    size_t ws_bytes;
};
int launch_rope_cache_quantized(const QCacheWrite& a, cudaStream_t st);
int launch_decode_attention_quantized(const QAttn& a, cudaStream_t st);
size_t qattn_workspace_bytes(int B, int Hq, int Hkv, int D, int64_t attend_len);
int launch_add_rmsnorm(const void* x, const void* r, const void* w, float eps, void* h_out, void* y_out, int64_t rows, int H,
                       cudaStream_t st);
int launch_silu_mul(const void* g, const void* u, void* out, int64_t n, cudaStream_t st);
int launch_head_gemv(const void* x, const void* w, void* y, int64_t M, int64_t V, int64_t K, cudaStream_t st);
int launch_gather_qmm(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, const int32_t* lhs,
                      const int32_t* rhs, void* y, int64_t R, int64_t XB, int64_t E, int64_t M, int64_t N, int64_t K,
                      int transpose, int bits, int gs, int dtype, cudaStream_t st);
bool gemm_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                    const void* y);
int launch_gemm(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                int64_t N, int64_t K, int bits, int gs, void* workspace, size_t workspace_bytes, cudaStream_t st);
size_t gemm_workspace_bytes(int64_t M, int64_t N, int64_t K);
void gemm_ts_debug_timeline(unsigned long long* buf);
int64_t gemm_ts_grouped_npad(const gbxq_segment* segs, int nseg);
int launch_gemm_ts_grouped(const gbxq_segment* segs, int nseg, const void* x, int64_t M, int64_t K, void* workspace,
                           size_t workspace_bytes, cudaStream_t st);
bool gemm_ts_supported(int64_t M, int64_t N, int64_t K, int bits, int gs, int dtype, const void* x, const void* w,
                       const void* y);
int launch_gemm_ts(const void* x, const uint32_t* w, const void* s, const void* b, const void* bias, void* y, int64_t M,
                   int64_t N, int64_t K, int bits, int gs, void* workspace, size_t workspace_bytes, cudaStream_t st);
int launch_allreduce_oneshot(const void* in, void* out, int64_t count, int dtype, void* const* peer_bufs,
                             uint32_t* const* peer_flags, int64_t capacity, int rank, int world, uint32_t seq,
                             cudaStream_t st);

int device_sm_count();

// Host: encode a 2-D tiled TMA descriptor (dtype 0 = bf16, 1 = uint32) through the driver entry point obtained with
// cudaGetDriverEntryPoint (no libcuda link).  `tm` points at a CUtensorMap.  Returns false if unavailable.
bool tma_encode_available();
bool encode_tensor_map_2d(void* tm, int dtype, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                          uint32_t box_inner, uint32_t box_outer, bool swizzle128);
// the same with the swizzle span in bytes (0 = none, 32, 64, 128)
bool encode_tensor_map_2d_sw(void* tm, int dtype, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                             uint32_t box_inner, uint32_t box_outer, int swizzle_bytes);

}  // namespace gbxq
