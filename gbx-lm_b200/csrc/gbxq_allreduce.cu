// gbxq_allreduce.cu -- one-shot NVLink sum all-reduce for the row-parallel QuantizedLinear
// epilogue (o_proj / down_proj under tensor parallelism; new work, SURVEY.md 8e).
//
// Every rank owns a staging buffer and a flag array that are mapped into every peer
// (symmetric memory).  Per call and per CTA slice:
//   1. copy this rank's partial slice into its own staging half (seq parity)
//   2. __threadfence_system(); publish `seq` into slot [rank][cta] of every peer's flag array
//   3. spin until all peers have published `seq` for this slice (bounded: 4 s, then the error word
//      [world*GBXQ_AR_MAX_CTAS + 2] of the own flag array is set and the call runs to its end)
//   4. read the slice from every peer's staging half over NVLink, add in rank order in fp32,
//      round once to T and store.
// Rank-order summation makes the result bitwise identical on all ranks.  Double buffering by
// seq parity is sufficient: a rank can only start call s after every peer signalled call s-1,
// i.e. after every peer finished reading call s-2.
// The launch carries the programmatic-dependent-launch attribute: it becomes resident while the matmul before it
// drains (griddepcontrol.wait before the first read of `in`), and lets the kernel after it do the same.
// For o_proj / down_proj at decode sizes the all-reduce inside the matmul kernel (gbxq_qmm_rowpar_allreduce,
// gbxq_mmv8_body.cuh) replaces this kernel; it stays for the shapes that kernel does not serve.
#include "gbxq_common.cuh"

namespace gbxq {

namespace {

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

template <typename T, int WORLD_MAX>
__global__ void __launch_bounds__(256) allreduce_oneshot_kernel(const T* in, T* out,  // may alias
                                                                int64_t count, void* const* peer_bufs,
                                                                uint32_t* const* peer_flags, int64_t half_elems,
                                                                int rank, int world, uint32_t seq) {
    constexpr int VEC = 16 / sizeof(T);
    const int64_t nvec = count / VEC;  // count % VEC == 0 (checked on the host)
    const int64_t per_cta = (nvec + gridDim.x - 1) / gridDim.x;
    const int64_t v0 = (int64_t)blockIdx.x * per_cta;
    int64_t v1 = v0 + per_cta;
    if (v1 > nvec) v1 = nvec;
    // seq == 0: the sequence number lives on the device (own flag array, entry world*GBXQ_AR_MAX_CTAS; entry +1 counts
    // the CTAs that are done), so that a CUDA graph can replay the call: every CTA reads it at entry, the last CTA to
    // finish advances it.  The launch is plain stream-ordered, so the next call sees the advanced value.
    uint32_t* local = peer_flags[rank] + world * GBXQ_AR_MAX_CTAS;
    griddep_launch_dependents();
    griddep_wait();  // `in` (and the device-resident sequence number) belong to earlier kernels
    const bool dev_seq = seq == 0u;
    if (dev_seq) seq = *reinterpret_cast<volatile uint32_t*>(local) + 1u;
    const int64_t half = (int64_t)(seq & 1u) * half_elems;

    // 1. stage own slice
    uint4* mine = reinterpret_cast<uint4*>(reinterpret_cast<T*>(peer_bufs[rank]) + half);
    const uint4* src = reinterpret_cast<const uint4*>(in);
    for (int64_t v = v0 + threadIdx.x; v < v1; v += blockDim.x) mine[v] = src[v];
    __threadfence_system();
    __syncthreads();
    // 2. publish
    if (threadIdx.x < world) st_release_sys(peer_flags[threadIdx.x] + rank * GBXQ_AR_MAX_CTAS + blockIdx.x, seq);
    // 3. wait for all peers (flags are monotonic: >= seq means published)
    if (threadIdx.x < world) {
        const uint32_t* f = peer_flags[rank] + threadIdx.x * GBXQ_AR_MAX_CTAS + blockIdx.x;
        unsigned long long t0, t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        while ((int32_t)(ld_acquire_sys(f) - seq) < 0) {
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > 4000000000ull) {  // a peer is gone or out of step: flag it, never hang the device
                atomicExch(local + 2, 1u);
                break;
            }
        }
    }
    __syncthreads();
    // 4. reduce in rank order
    for (int64_t v = v0 + threadIdx.x; v < v1; v += blockDim.x) {
        float acc[VEC];
#pragma unroll
        for (int e = 0; e < VEC; e++) acc[e] = 0.f;
        for (int r = 0; r < world; r++) {
            const uint4 t = reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(peer_bufs[r]) + half)[v];
            const T* tv = reinterpret_cast<const T*>(&t);
#pragma unroll
            for (int e = 0; e < VEC; e++) acc[e] += to_f32(tv[e]);
        }
        uint4 o;
        T* ov = reinterpret_cast<T*>(&o);
#pragma unroll
        for (int e = 0; e < VEC; e++) ov[e] = from_f32<T>(acc[e]);
        reinterpret_cast<uint4*>(out)[v] = o;
    }
    if (dev_seq) {
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t old = atomicAdd(local + 1, 1u);
            if (old == gridDim.x - 1u) {
                local[1] = 0u;
                *reinterpret_cast<volatile uint32_t*>(local) = seq;
            }
        }
    }
}

template <typename T>
int launch_t(const void* in, void* out, int64_t count, void* const* peer_bufs, uint32_t* const* peer_flags,
             int64_t capacity, int rank, int world, uint32_t seq, cudaStream_t st) {
    constexpr int VEC = 16 / sizeof(T);
    if (count % VEC) return GBXQ_ESHAPE;
    const int64_t nvec = count / VEC;
    int ctas = (int)((nvec + 255) / 256);
    if (ctas < 1) ctas = 1;
    if (ctas > GBXQ_AR_MAX_CTAS) ctas = GBXQ_AR_MAX_CTAS;
    return launch(allreduce_oneshot_kernel<T, 8>, dim3((unsigned)ctas), dim3(256), 0, st, true, (const T*)in, (T*)out, count,
                  peer_bufs, peer_flags, capacity / 2, rank, world, seq);
}

}  // namespace

int launch_allreduce_oneshot(const void* in, void* out, int64_t count, int dtype, void* const* peer_bufs,
                             uint32_t* const* peer_flags, int64_t capacity, int rank, int world, uint32_t seq,
                             cudaStream_t st) {
    switch (dtype) {
        case GBXQ_BF16: return launch_t<__nv_bfloat16>(in, out, count, peer_bufs, peer_flags, capacity, rank, world, seq, st);
        case GBXQ_F16: return launch_t<__half>(in, out, count, peer_bufs, peer_flags, capacity, rank, world, seq, st);
        case GBXQ_F32: return launch_t<float>(in, out, count, peer_bufs, peer_flags, capacity, rank, world, seq, st);
    }
    return GBXQ_EDTYPE;
}

}  // namespace gbxq
