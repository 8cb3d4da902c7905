/*
 * gbxq.h -- C ABI of libgbxq.so: B200 (sm_100a) group-affine low-bit quantized matmul.
 *
 * Drop-in boundary for ONE hot path of GreenBitAI/gbx-lm: the call that
 * `QuantizedLinear.__call__` makes into the MLX extension module,
 *
 *     mx.quantized_matmul(x, qweight, scales=scales, biases=zeros, transpose=True,
 *                         group_size=gs, bits=b)   gbx_lm/models/quantized_linear_gba.py:195-203
 *     (+ bias)                                      gbx_lm/models/quantized_linear_gba.py:204-205
 *     mx.dequantize(w, scales, biases, gs, bits)    gbx_lm/tuner/lora.py:62-68
 *                                                   gbx_lm/tuner/utils.py:214-220
 *
 * The reference has no FFI layer of its own (it is pure Python over the `mlx` wheel); these
 * entry points are what a ctypes/nanobind binding placed at that seam would call
 * (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer owned by the caller unless the name ends in `_host`.
 *     Inputs are never written.  Outputs are fully overwritten.
 *   - Calls only ENQUEUE work on `stream` (a cudaStream_t passed as void*; NULL = legacy default
 *     stream) and return; they never synchronise, never allocate device memory and keep no
 *     global mutable state besides the options of gbxq_set_option, so they are CUDA-graph capturable
 *     and thread-safe across streams.
 *   - Return value: GBXQ_OK (0) or a negative gbxq_status.  Nothing throws.
 *   - Tensor layout = MLX affine quantisation as emitted by gba2mlx (gbx_lm/gba2mlx.py:47-65,
 *     gbx_lm/utils.py:828-843):
 *        qweight  uint32 [N, K*bits/32]  row-major; row n is the LSB-first bitstream of the K codes
 *                                         of output feature n, cut into little-endian words
 *        scales   T      [N, K/group_size]
 *        biases   T      [N, K/group_size]   (the checkpoint's `zeros`: already the ADDITIVE term,
 *                                            quantized_linear_gba.py:151-155)
 *        x        T      [M, K]  row-major (M = product of the leading dims)
 *        y        T      [M, N]  row-major
 *        bias     T      [N]     optional (Qwen2 q/k/v: gbx_lm/models/qqwen2.py:44-46)
 *     W[n,k] = scales[n,k/gs] * q[n,k] + biases[n,k/gs];  y = x . W^T (+ bias)
 *   - T is selected by `dtype` (gbxq_dtype).  bits in {2,3,4,6,8}; group_size in {32,64,128}
 *     (asserted by the reference at quantized_linear_gba.py:250,272 and utils.py:819-821).
 */
#ifndef GBXQ_H_
#define GBXQ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GBXQ_ABI_VERSION 2

typedef enum gbxq_status {
    GBXQ_OK = 0,
    GBXQ_EINVAL_BITS = -1,   /* bits not in {2,3,4,6,8} */
    GBXQ_EINVAL_GROUP = -2,  /* group_size not in {32,64,128} */
    GBXQ_ESHAPE = -3,        /* M,N,K inconsistent (K % 32, K % group_size, negative, ...) */
    GBXQ_EDTYPE = -4,        /* unknown dtype code */
    GBXQ_EALIGN = -5,        /* a pointer is not aligned as required (16 B for x/y/qweight rows) */
    GBXQ_ENULL = -6,         /* a required pointer is NULL */
    GBXQ_ECUDA = -7,         /* a CUDA runtime call failed; see gbxq_last_cuda_error() */
    GBXQ_EWORKSPACE = -8,    /* workspace too small (gbxq_workspace_bytes) */
    GBXQ_EUNSUPPORTED = -9   /* feature not available for this argument combination */
} gbxq_status;

typedef enum gbxq_dtype { GBXQ_BF16 = 0, GBXQ_F16 = 1, GBXQ_F32 = 2 } gbxq_dtype;

/* Kernel selection for gbxq_qmm_ex (tests / benchmarks); gbxq_qmm uses GBXQ_KERNEL_AUTO. */
typedef enum gbxq_kernel {
    GBXQ_KERNEL_AUTO = 0,
    GBXQ_KERNEL_GENERIC = 1, /* shape-agnostic warp-per-row kernel (all dtypes)            */
    GBXQ_KERNEL_GEMV = 2,    /* TMA-bulk ring streaming GEMV on the FMA pipe, M tiles of 1/2 */
    GBXQ_KERNEL_GEMM = 3,    /* tcgen05/TMEM tensor-core GEMM with in-kernel dequant (bf16) */
    GBXQ_KERNEL_SKINNY = 4,  /* mma.sync skinny matmul, 8 tokens per pass, 2/4/8-bit (bf16)  */
    GBXQ_KERNEL_MMV = 5,     /* bf16 tensor-pipe decode matrix-vector kernel, 1..4 tokens, 2/4/8-bit, PDL */
    GBXQ_KERNEL_MMV8 = 6,    /* integer tensor-pipe (IMMA u8 x s8) decode kernel: codes used in place, activations as
                                per-group 15-bit block fixed point; 1..4 tokens, every width (bf16 in/out), PDL.
                                GBXQ_KERNEL_AUTO picks it for M <= 2 and the skinny kernel from M = 3 */
    GBXQ_KERNEL_GEMM_TS = 7  /* tcgen05 GEMM with the dequantised weights as the TMEM ("TS") operand: one weight row
                                per thread, no shared-memory round trip of the bf16 tile; K % 128 == 0 (bf16), PDL */
} gbxq_kernel;

/* Process-wide options (gbxq_set_option / gbxq_get_option). */
typedef enum gbxq_option {
    /* Programmatic dependent launch of the decode kernels:
     *   0  plain stream-ordered launches
     *   1  PDL launch attribute; every global read waits for the preceding kernels of the stream
     *   2  (default) as 1, but qweight/scales/biases are streamed BEFORE that wait: the caller guarantees
     *      that no kernel still in flight on the stream writes them (true for QuantizedLinear: its
     *      parameters are frozen, quantized_linear_gba.py:57-58,162-166).  x, bias and y are always
     *      touched after the wait. */
    GBXQ_OPT_PDL = 1
} gbxq_option;

/* Library / ABI identification. */
int gbxq_abi_version(void);
const char* gbxq_status_string(int status);
/* Last cudaError_t seen by the calling thread inside libgbxq (0 if none), and its text. */
int gbxq_last_cuda_error(void);
const char* gbxq_last_cuda_error_string(void);

/*
 * y[M,N] = x[M,K] . dequant(qweight)[N,K]^T (+ bias)
 * Replaces mx.quantized_matmul(..., transpose=True) + the bias add of QuantizedLinear.__call__
 * (quantized_linear_gba.py:195-205).  Output is rounded once to T; the optional bias is a second,
 * separately rounded add, as in the reference.  M == 0 or N == 0 is a no-op returning GBXQ_OK.
 * `workspace` may be NULL when gbxq_workspace_bytes(...) == 0.
 */
int gbxq_qmm(const void* x, const uint32_t* qweight, const void* scales, const void* biases,
             const void* bias /* nullable */, void* y, int64_t M, int64_t N, int64_t K, int bits,
             int group_size, int dtype, void* workspace, size_t workspace_bytes, void* stream);

/* Same, forcing one kernel family (returns GBXQ_EUNSUPPORTED if it cannot serve the arguments). */
int gbxq_qmm_ex(const void* x, const uint32_t* qweight, const void* scales, const void* biases,
                const void* bias, void* y, int64_t M, int64_t N, int64_t K, int bits,
                int group_size, int dtype, int kernel, void* workspace, size_t workspace_bytes,
                void* stream);

/*
 * Grouped launch: nseg (<= GBXQ_MAX_SEGMENTS) quantized projections that read the SAME activations x[M,K], each
 * with its own weights, bit width, optional bias and output -- the back-to-back q_proj/k_proj/v_proj and
 * gate_proj/up_proj calls of the reference (gbx_lm/models/qllama.py:76,115; gbx_lm/models/qqwen2.py:66,94), whose
 * bit widths differ per projection in layer-mix checkpoints (quantized_linear_gba.py:258-272).
 * Semantics are exactly those of nseg gbxq_qmm calls (y_s[M,N_s] = x . dequant(W_s)^T (+ bias_s)), results are
 * identical to them; when M <= 2 and the segments share K and group_size the work is ONE kernel launch, otherwise
 * the call enqueues one launch per segment.  `segs` is a HOST array read before the call returns.
 */
#define GBXQ_MAX_SEGMENTS 4
typedef struct gbxq_segment {
    const uint32_t* qweight; /* [N, K*bits/32] */
    const void* scales;      /* [N, K/group_size] */
    const void* biases;      /* [N, K/group_size] */
    const void* bias;        /* [N] or NULL */
    void* y;                 /* [M, N] row-major, fully overwritten */
    int64_t N;
    int bits;
    int group_size;
} gbxq_segment;
int gbxq_qmm_grouped(const gbxq_segment* segs_host, int nseg, const void* x, int64_t M, int64_t K, int dtype,
                     void* stream);
/*
 * The same with scratch for the rows-of-x regime above the decode kernel (M > 4): segments that share bit width and
 * group size then run as ONE launch of the tensor-core GEMM (gbxq_gemm_ts_grouped_sm100.cu), splitting K where the
 * segments leave SMs idle; without a workspace (or with gbxq_qmm_grouped) such launches run unsplit.
 * gbxq_grouped_workspace_bytes sizes the scratch; the rules of gbxq_qmm's workspace apply (first 16 KB zero once,
 * owned by the stream).
 */
size_t gbxq_grouped_workspace_bytes(const gbxq_segment* segs_host, int nseg, int64_t M, int64_t K, int dtype);
int gbxq_qmm_grouped_ws(const gbxq_segment* segs_host, int nseg, const void* x, int64_t M, int64_t K, int dtype,
                        void* workspace, size_t workspace_bytes, void* stream);

/*
 * Chain launch: an ordered list of decode-sized (M <= 4, bf16) quantized matmuls -- the QuantizedLinear forwards of
 * one decode step in the order the reference's blocks issue them (gbx_lm/models/qllama.py:76-115: q|k|v, o_proj,
 * gate|up, down_proj per block) -- executed by ONE persistent kernel launch.  Semantics are those of issuing the
 * calls one after another on a stream: call i reads its x and writes its y only after every call <= dep_i is
 * complete (dep_i = i-1 by default: plain stream order), and results are bitwise identical to gbxq_qmm /
 * gbxq_qmm_grouped on the same arguments.  What changes is that the packed weights, scales and biases of LATER calls
 * keep streaming into the shared-memory rings while earlier calls finish, so HBM does not idle at call borders
 * (QuantizedLinear parameters are frozen: quantized_linear_gba.py:57-58,162-166).
 *
 * Two steps, because weights and activation buffers of a decode loop are fixed: gbxq_stream_plan (host only) checks
 * the chain and writes a descriptor blob into HOST memory; the caller copies the blob to the device once and then
 * calls gbxq_qmm_stream any number of times (CUDA-graph capturable, no allocation, no synchronisation).
 *   dep : index of the last earlier call whose output this call's x may alias; GBXQ_DEP_PREV = the call before it
 *         (stream order), GBXQ_DEP_NONE = x is not produced inside the chain.
 *   counters_dev : (ncalls + 2) uint32, zeroed ONCE by the caller before the first launch; the kernel leaves them
 *         zero again.  Entry ncalls+1 is set to 1 if a CTA ever gave up waiting (grid not co-resident): results
 *         of that launch are then undefined; the kernel never hangs.
 * gbxq_stream_plan returns GBXQ_EUNSUPPORTED when a call cannot be served by the chain kernel (M > 4, 3-/6-bit,
 * fp16/fp32, mixed group sizes): issue such steps as individual gbxq_qmm calls.
 */
#define GBXQ_DEP_PREV (-2)
#define GBXQ_DEP_NONE (-1)
typedef struct gbxq_stream_call {
    const void* x;       /* [M, K] */
    int64_t K;
    int nseg;            /* 1 .. GBXQ_MAX_SEGMENTS projections reading this x */
    int dep;
    gbxq_segment segs[GBXQ_MAX_SEGMENTS];
} gbxq_stream_call;
typedef struct gbxq_stream_info {
    int32_t ncalls, grid, smem_bytes, group_size, mt, stages;
    uint32_t slot_bytes;
    uint32_t reserved;
    uint64_t blob_bytes;     /* size of the descriptor blob */
    uint64_t counter_bytes;  /* size of the counter array */
} gbxq_stream_info;
/* host_blob == NULL: only fills `info` (sizes).  Otherwise writes info->blob_bytes bytes (blob_capacity checked). */
int gbxq_stream_plan(const gbxq_stream_call* calls_host, int ncalls, int64_t M, int dtype, void* host_blob,
                     size_t blob_capacity, gbxq_stream_info* info);
int gbxq_qmm_stream(const gbxq_stream_info* info, const void* blob_dev, void* counters_dev, void* stream);

/* Scratch bytes gbxq_qmm can use for these arguments: non-zero only where the tensor-core GEMM splits K (17..256 rows of x
 * on a layer with fewer output tiles than SMs).  The first 16 KB of the workspace must be zero before the first call
 * and are left zero by every call; one workspace may serve all calls of a stream.  With workspace == NULL (or too
 * small) the call runs unsplit -- same result up to fp32 summation order, fewer SMs busy. */
size_t gbxq_workspace_bytes(int64_t M, int64_t N, int64_t K, int bits, int group_size, int dtype);

/*
 * w_out[N,K] (T) = T( T(scales * T(q)) + biases )      -- bit-exact with mx.dequantize
 * Replaces mx.dequantize(w, scales, biases, group_size, bits) (tuner/lora.py:62-68).
 */
int gbxq_dequantize(const uint32_t* qweight, const void* scales, const void* biases, void* w_out,
                    int64_t N, int64_t K, int bits, int group_size, int dtype, void* stream);

/*
 * (qweight, scales, biases) = quantize(w): group-affine quantisation of a T matrix w[rows, K] into the layout above
 * (codes uint32 [rows, K*bits/32], scales / biases T [rows, K/group_size]).
 * Replaces mx.quantize(x, group_size=, bits=) where the reference quantises on the fly: the new keys / values of every
 * step in QuantizedKVCache.update_and_fetch (gbx_lm/models/cache.py:176-177) and a whole dense cache in
 * KVCache.to_quantized (cache.py:251-263); the consumers are the quantized_matmul calls of
 * quantized_scaled_dot_product_attention (gbx_lm/models/base.py:85-93, gbxq_gather_qmm here).
 * Per group, in fp32:  scale = max((max - min) / (2^bits - 1), 1e-7), signed so that the edge of larger magnitude is
 * hit exactly (scale = edge / rint(edge / scale), bias = edge; bias = 0 when that rint is 0),
 * code = clamp(rint((w - bias) / scale), 0, 2^bits - 1) from the unrounded scale / bias, which are then stored as T.
 * K % group_size == 0; w 16-byte aligned.  rows == 0 is a no-op.
 *
 * gbxq_quantize_rows: the same with destination rows remapped -- source row r lands in row
 *     (r / inner_rows) * out_outer_stride_rows + out_row_offset + r % inner_rows
 * of the three outputs, i.e. the `inner_rows` new positions of every (batch, head) go to positions
 * [out_row_offset, out_row_offset + inner_rows) of a cache of capacity out_outer_stride_rows
 * (`self.keys[i][..., prev : self.offset, :] = keys[i]`, cache.py:178-180) without a staging copy.
 * rows % inner_rows == 0 and out_row_offset + inner_rows <= out_outer_stride_rows, else GBXQ_ESHAPE.
 */
int gbxq_quantize(const void* w, uint32_t* qweight, void* scales, void* biases, int64_t rows, int64_t K, int bits,
                  int group_size, int dtype, void* stream);
int gbxq_quantize_rows(const void* w, uint32_t* qweight, void* scales, void* biases, int64_t rows, int64_t K, int bits,
                       int group_size, int dtype, int64_t inner_rows, int64_t out_outer_stride_rows,
                       int64_t out_row_offset, void* stream);

/* Which kernel family GBXQ_KERNEL_AUTO picks for these arguments (a gbxq_kernel value, or <0). */
int gbxq_select_kernel(int64_t M, int64_t N, int64_t K, int bits, int group_size, int dtype);

/* Set / read a gbxq_option.  Returns GBXQ_OK / the value, or GBXQ_EUNSUPPORTED for an unknown key. */
int gbxq_set_option(int key, int value);
int gbxq_get_option(int key);

/* Number of kernel launches libgbxq has enqueued from this process (monotonic; for benches). */
uint64_t gbxq_launch_count(void);

/*
 * Decode-step glue (SURVEY.md 8f rank 2: the fusions either side of the path).  What the reference's callers do
 * between the QuantizedLinear forwards of a block at decode (one new token per sequence), as four launches instead of
 * ~45 framework launches; bf16 tensors, fp32 arithmetic, the step's positions read from DEVICE memory so that a CUDA
 * graph can replay the step.
 *
 * Positions: pos_dev is int64 on the device and row b of the batch is at p_b = pos_dev[b * pos_stride].
 *   pos_stride 0: pos_dev[0] is the position of every row; 1: pos_dev[b] is row b's (B sequences at different
 *   positions, e.g. prompts of different lengths; no counterpart in the reference, whose generate_step is batch-1).
 *   Other values return GBXQ_ESHAPE.  At B = 1 the two are the same call, and with all B positions equal stride 1 is
 *   bitwise stride 0 and enqueues the same launches.
 * Cache rows: the cache writes take `keep`, the layout of a cache of max_len rows.
 *   keep < 0: a flat cache; position p goes to row p, and nothing is written for p outside [0, max_len).
 *   0 <= keep < max_len: a ROTATING cache (the reference's RotatingKVCache, gbx_lm/models/cache.py:280-420): window
 *     W = max_len rows, of which the first `keep` are attention sinks; position p goes to row
 *         ring_slot(p) = p                                   if p < W
 *                      = keep + (p - keep) mod (W - keep)    otherwise
 *     computed on the device, so a captured decode step wraps without the host.  Below W it is the flat cache's row.
 *   keep >= max_len: GBXQ_ESHAPE.
 *   The RoPE angle is the absolute position, q is rotated in place, and nothing outside row b's slot is written (the
 *   other rows of the batch are unaffected).
 * The attention calls attend keys [0, min(p_b, attend_len-1)] of row b's cache.  Over a ring, with max_len = W and
 * attend_len = min(tokens so far, W) (a replayed graph: W), those rows are exactly the ring's contents -- the sinks and
 * the last W - keep positions.  Softmax does not depend on the order of the rows, so the result is the windowed
 * attention up to the order of summation.
 *
 *   gbxq_rope_cache       q[B,Hq,D] rotated in place, k[B,Hkv,D] rotated into k_cache[B,Hkv,max_len,D] and v copied
 *                         into v_cache, each at row b's cache row (mx.fast.rope traditional=False +
 *                         cache.update_and_fetch, gbx_lm/models/qllama.py:83-88); inv_freq f32 [D/2] already carries
 *                         the rope scaling
 *   gbxq_decode_attention out[B,Hq,D] = softmax(scale * q . K[0..min(p_b, attend_len-1)]) . V, GQA by Hq/Hkv
 *                         (scaled_dot_product_attention, qllama.py:90-93); D = 64 or 128
 *   gbxq_add_rmsnorm      h = x + r (r NULL: h = x), y = RMSNorm(h) * w; h_out may be NULL or alias x
 *                         (residual + nn.RMSNorm, qllama.py:137-141)
 *   gbxq_silu_mul         out = silu(gate) * up (qllama.py:115), n elements, n % 8 == 0
 */
int gbxq_rope_cache(void* q, const void* k, const void* v, const int64_t* pos_dev, int pos_stride,
                    const float* inv_freq_dev, void* k_cache, void* v_cache, int B, int Hq, int Hkv, int D,
                    int64_t max_len, int64_t keep, void* stream);
int gbxq_decode_attention(const void* q, const void* k_cache, const void* v_cache, const int64_t* pos_dev,
                          int pos_stride, void* out, int B, int Hq, int Hkv, int D, int64_t max_len,
                          int64_t attend_len, float scale, void* stream);
/*
 * Verify blocks (speculative decoding): T consecutive tokens per batch row, 1 <= T <= 8, token t of row b at position
 * p_b + t (p_b from pos_dev / pos_stride as above), on a flat cache (no keep argument).  q is [B,T,Hq,D], k / v
 * [B,T,Hkv,D], out [B,T,Hq,D].  T outside 1..8 returns GBXQ_ESHAPE, before any CUDA call.
 *   gbxq_rope_cache_multi       bitwise T calls of gbxq_rope_cache at p_b .. p_b + T - 1; positions >= max_len are not
 *                               written (q is not rotated there either)
 *   gbxq_decode_attention_multi query t of row b attends keys [0, min(p_b + t, attend_len-1)] of row b's cache, bitwise
 *                               the gbxq_decode_attention call for that query at p_b + t.  The block's own keys are
 *                               written before the call, so this is the causal mask inside the block.
 */
int gbxq_rope_cache_multi(void* q, const void* k, const void* v, const int64_t* pos_dev, int pos_stride,
                          const float* inv_freq_dev, void* k_cache, void* v_cache, int B, int T, int Hq, int Hkv, int D,
                          int64_t max_len, void* stream);
int gbxq_decode_attention_multi(const void* q, const void* k_cache, const void* v_cache, const int64_t* pos_dev,
                                int pos_stride, void* out, int B, int T, int Hq, int Hkv, int D, int64_t max_len,
                                int64_t attend_len, float scale, void* stream);
int gbxq_add_rmsnorm(const void* x, const void* r, const void* w, float eps, void* h_out, void* y_out, int64_t rows,
                     int H, void* stream);
int gbxq_silu_mul(const void* gate, const void* up, void* out, int64_t n, void* stream);

/*
 * The same two steps of a decode step over a group-quantized KV cache (the reference's kv_bits path:
 * QuantizedKVCache.update_and_fetch, gbx_lm/models/cache.py:172-185, and quantized_scaled_dot_product_attention,
 * gbx_lm/models/base.py:65-98).  Each side of the cache is a triple in the layout of gbxq_quantize, position-major:
 *     codes uint32 [B, Hkv, max_len, D*bits/32],  scales / biases bf16 [B, Hkv, max_len, D/group_size]
 * bits in {2,3,4,6,8}, group_size in {32,64,128} with group_size <= D, D in {64, 128}, Hq/Hkv <= 8; other shapes return
 * GBXQ_EUNSUPPORTED (nothing enqueued).  pos_dev / pos_stride and keep are as for gbxq_rope_cache /
 * gbxq_decode_attention above.
 *   gbxq_rope_cache_quantized       q rotated in place as gbxq_rope_cache does; k rotated and v copied, each quantized
 *                                   into row b's cache row of its triple.  Codes, scales and biases are bit-identical
 *                                   to gbxq_rope_cache into a bf16 row followed by gbxq_quantize_rows of that row.
 *                                   Nothing outside that row is written (nothing at all for a position outside a flat
 *                                   cache).
 *   gbxq_decode_attention_quantized out[B,Hq,D] = softmax(scale * q . K[0..min(p_b, attend_len-1)]) . V over the
 *                                   triples, fp32 inside.  Keys are split into chunks of 256 positions, one CTA per
 *                                   (chunk, kv head, batch) for all query heads of the group, and the partial results
 *                                   are combined by a second launch in chunk order; the chunks past a row's own
 *                                   position are empty partials.  So each row's result does not depend on attend_len,
 *                                   max_len or the other rows (bitwise), and there is no context limit.  `workspace`
 *                                   holds the partials: at least gbxq_decode_attention_quantized_workspace_bytes(B, Hq,
 *                                   Hkv, D, attend_len) bytes, 16-byte aligned, no initialisation needed; a workspace
 *                                   serves the calls of one stream one after another.  Returns 0 from the size query
 *                                   for unsupported arguments.
 */
int gbxq_rope_cache_quantized(void* q, const void* k, const void* v, const int64_t* pos_dev, int pos_stride,
                              const float* inv_freq_dev, uint32_t* k_codes, void* k_scales, void* k_biases,
                              uint32_t* v_codes, void* v_scales, void* v_biases, int B, int Hq, int Hkv, int D,
                              int64_t max_len, int64_t keep, int bits, int group_size, void* stream);
size_t gbxq_decode_attention_quantized_workspace_bytes(int B, int Hq, int Hkv, int D, int64_t attend_len);
int gbxq_decode_attention_quantized(const void* q, const uint32_t* k_codes, const void* k_scales,
                                    const void* k_biases, const uint32_t* v_codes, const void* v_scales,
                                    const void* v_biases, const int64_t* pos_dev, int pos_stride, void* out, int B,
                                    int Hq, int Hkv, int D, int64_t max_len, int64_t attend_len, float scale,
                                    int bits, int group_size, void* workspace, size_t workspace_bytes, void* stream);
/*
 * Their verify-block forms, as gbxq_rope_cache_multi / gbxq_decode_attention_multi (T consecutive tokens per row, flat
 * cache): the write is bitwise T calls of gbxq_rope_cache_quantized; each query of the attention is bitwise the
 * gbxq_decode_attention_quantized call at its position, while one CTA reads each chunk's codes once for the T queries
 * of its row.  The workspace holds B*T rows of partials: gbxq_decode_attention_quantized_workspace_bytes(B*T, Hq, Hkv,
 * D, attend_len) bytes.
 */
int gbxq_rope_cache_quantized_multi(void* q, const void* k, const void* v, const int64_t* pos_dev, int pos_stride,
                                    const float* inv_freq_dev, uint32_t* k_codes, void* k_scales, void* k_biases,
                                    uint32_t* v_codes, void* v_scales, void* v_biases, int B, int T, int Hq, int Hkv,
                                    int D, int64_t max_len, int bits, int group_size, void* stream);
int gbxq_decode_attention_quantized_multi(const void* q, const uint32_t* k_codes, const void* k_scales,
                                          const void* k_biases, const uint32_t* v_codes, const void* v_scales,
                                          const void* v_biases, const int64_t* pos_dev, int pos_stride, void* out, int B,
                                          int T, int Hq, int Hkv, int D, int64_t max_len, int64_t attend_len,
                                          float scale, int bits, int group_size, void* workspace,
                                          size_t workspace_bytes, void* stream);

/*
 * Vocabulary projection of the decode step (SURVEY.md 8f rank 1): y[M,V] = x[M,K] . weight[V,K]^T with UNQUANTIZED bf16
 * weights -- `self.lm_head(out)` / `self.model.embed_tokens.as_linear(out)` (gbx_lm/models/qllama.py:183-184,194-198).
 * A streaming GEMV for M <= 8 rows (K % 256 == 0, 16-byte aligned x / weight): fp32 accumulation, one rounding to bf16.
 * Returns GBXQ_EUNSUPPORTED (nothing enqueued) for other arguments: use the framework's dense matmul then.
 */
int gbxq_head_gemv(const void* x, const void* weight, void* y, int64_t M, int64_t V, int64_t K, int dtype, void* stream);

/*
 * Index-batched quantized matmul (SURVEY.md 8f ranks 3 and 4), the two forms either side of the QuantizedLinear path:
 *   transpose = 1:  y[r] = x[lhs[r]] . dequant(qweight[rhs[r]])^T (+ bias[rhs[r]])      -- mx.gather_qmm(x, w, scales,
 *                   biases, rhs_indices=indices, transpose=True) of QuantizedSwitchLinear.__call__
 *                   (gbx_lm/models/switch_layers.py:78-92); qweight [E, N, K*bits/32], scales / biases [E, N, K/gs],
 *                   bias [E, N] or NULL.
 *   transpose = 0:  y[r] = x[lhs[r]] . dequant(qweight[rhs[r]])                          -- mx.quantized_matmul(scores,
 *                   *q_values, transpose=False) of the quantized KV cache attention (gbx_lm/models/base.py:90-92);
 *                   qweight [E, K, N*bits/32] quantized along N, scales / biases [E, K, N/gs]; bias must be NULL.
 * x is [XB, M, K], y is [R, M, N]; lhs_indices / rhs_indices are DEVICE int32 arrays of R entries (NULL = the identity
 * r -> r); out-of-range indices are clamped into [0, XB) / [0, E).  transpose = 1 needs K % 32 == 0 and
 * K % group_size == 0, transpose = 0 needs the same of N.  All dtypes (0 bf16, 1 f16, 2 f32), every width.
 */
int gbxq_gather_qmm(const void* x, const uint32_t* qweight, const void* scales, const void* biases, const void* bias,
                    const int32_t* lhs_indices, const int32_t* rhs_indices, void* y, int64_t R, int64_t XB, int64_t E,
                    int64_t M, int64_t N, int64_t K, int transpose, int bits, int group_size, int dtype, void* stream);
/*
 * Tensor-parallel row-parallel epilogue (new work; the reference has no TP -- SURVEY.md 2.2):
 * one-shot sum all-reduce of a small [count] T vector over peer-mapped buffers on NVLink
 * (P2P loads/stores, no NCCL call).  Meant for the latency-bound decode messages
 * (M*hidden*2 bytes: 16 KB .. 1 MB) that follow o_proj / down_proj.
 *   peer_bufs_dev  : device array of `world` pointers; entry r = rank r's staging buffer of
 *                    `capacity` elements of T, mapped into THIS process (symmetric memory).
 *                    The buffer is used as two halves (seq parity), so count <= capacity/2.
 *   peer_flags_dev : device array of `world` pointers; entry r = rank r's uint32 flag array of
 *                    world * GBXQ_AR_MAX_CTAS entries, zero-initialised once.
 *   in  : this rank's partial sums          out: reduced result (rank-order sum, identical on
 *                                                every rank), may alias `in`
 *   seq : starts at 1, increases by exactly 1 per call, same on every rank; or 0 on every call: the sequence
 *         number is then kept on the device in entry world*GBXQ_AR_MAX_CTAS of this rank's flag array (flag arrays
 *         need world*GBXQ_AR_MAX_CTAS + 3 entries), which makes the call replayable from a CUDA graph.  Entry
 *         world*GBXQ_AR_MAX_CTAS + 2 is set to 1 if a wait for a peer ever timed out (4 s): results are then undefined,
 *         the device never hangs.
 * Every rank must enqueue the call with the same count/dtype/seq on a stream of its own device.
 */
#define GBXQ_AR_MAX_CTAS 32
int gbxq_allreduce_oneshot(const void* in, void* out, int64_t count, int dtype,
                           void* const* peer_bufs_dev, uint32_t* const* peer_flags_dev,
                           int64_t capacity, int rank, int world, uint32_t seq, void* stream);

/*
 * Row-parallel QuantizedLinear with the all-reduce INSIDE the matmul kernel (o_proj / down_proj under tensor
 * parallelism: gbx_lm/models/qllama.py:96,115 are the call sites that get K-sharded; new work, SURVEY.md 8e).
 * Rank r holds the K-slice [r*K/world, (r+1)*K/world) of the layer (`K` below is that LOCAL size) and a slice of x;
 * the result y[M,N] = sum over ranks of x_r . dequant(W_r)^T (+ bias) is identical on every rank.
 * One launch per rank: each CTA of the decode kernel pushes the fp32 partial sums of the output rows it owns into
 * every peer's staging buffer (P2P stores over NVLink) and adds the `world` partials of those rows in rank order,
 * rounding once to T.  A partial travels as one 8-byte word {fp32 bits, epoch} and the receiver polls the word itself
 * (no fence, no flag: one NVLink one-way latency).  No second kernel, no NCCL call; the exchange of a CTA overlaps the
 * matmul of the others.
 *   comm->peer_stage_host : HOST array [world]; entry r = rank r's staging buffer of `stage_elems` 8-byte words,
 *                           8-byte aligned, ZEROED ONCE, mapped into this process (symmetric memory).
 *                           Needs stage_elems >= 2 * world * M * N.
 *   comm->peer_flags_host : HOST array [world]; entry r = rank r's uint32 array of world * GBXQ_RP_MAX_CTAS + 4
 *                           entries, zeroed once (only the control words at [world*GBXQ_RP_MAX_CTAS ..] of the own
 *                           rank are used: epoch, CTAs done, error).  Entry +2 becomes 1 if a wait timed out (4 s).
 * Every rank must enqueue the same call (same M, N, bits, group_size) in the same order.  `bias`, if given, is added
 * by the rank that holds it (pass NULL on the others).  CUDA-graph capturable (the epoch lives in the flag array).
 * Returns GBXQ_EUNSUPPORTED (nothing enqueued) when the decode kernel cannot serve the arguments (M > 4, 3-/6-bit,
 * non-bf16): use gbxq_qmm followed by gbxq_allreduce_oneshot then.
 */
#define GBXQ_RP_MAX_CTAS 512
typedef struct gbxq_comm {
    void* const* peer_stage_host;
    uint32_t* const* peer_flags_host;
    int64_t stage_elems;
    int rank, world;
} gbxq_comm;
int gbxq_qmm_rowpar_allreduce(const void* x, const uint32_t* qweight, const void* scales, const void* biases,
                              const void* bias /* nullable */, void* y, int64_t M, int64_t N, int64_t K, int bits,
                              int group_size, int dtype, const gbxq_comm* comm, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GBXQ_H_ */
