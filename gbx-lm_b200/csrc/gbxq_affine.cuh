// gbxq_affine.cuh -- the per-group recipe of mx.quantize (oracle/MLX_SPEC.md R6), shared by every kernel that writes
// group-affine codes: gbxq_quantize.cu (whole matrices, cache rows) and gbxq_qattn.cu (the fused RoPE + quantized cache
// write of a decode step).  One implementation, so that both produce bit-identical codes, scales and biases.
//
// Arithmetic (fp32, every operation separately rounded):
//     mask = |w_min| > |w_max|
//     scale = max((w_max - w_min) / (2^bits - 1), 1e-7);  scale = mask ? scale : -scale;  edge = mask ? w_min : w_max
//     q0 = rint(edge / scale);  if (q0 != 0) { scale = edge / q0;  bias = edge; } else bias = 0
//     code = clamp(rint((w - bias) / scale), 0, 2^bits - 1)         <- from the UNROUNDED fp32 scale / bias
#pragma once

#include <stdint.h>

namespace gbxq {

struct AffineGroup {
    float scale, bias;  // unrounded fp32 statistics (stored rounded to the element type by the caller)
    float r, nscale;    // RN(1 / scale) and -scale, for the division-free quotient of affine_code
};

// statistics of one group from its maximum and minimum (reduced by the caller over the group's elements)
template <int BITS>
__device__ __forceinline__ AffineGroup affine_group(float mx, float mn) {
    const float nb = (float)((1 << BITS) - 1);
    const bool mask = fabsf(mn) > fabsf(mx);
    float scale = fmaxf(__fdiv_rn(__fsub_rn(mx, mn), nb), 1e-7f);
    scale = mask ? scale : -scale;
    const float edge = mask ? mn : mx;
    const float q0 = rintf(__fdiv_rn(edge, scale));
    float bias = 0.f;
    if (q0 != 0.f) {
        scale = __fdiv_rn(edge, q0);
        bias = edge;
    }
    return AffineGroup{scale, bias, __frcp_rn(scale), -scale};
}

// (w - bias) / scale, correctly rounded, without a division per element: with r = RN(1 / scale),
// q1 = RN(d * r), rem = d - q1 * scale (exact in one FMA), q = RN(q1 + rem * r) is the IEEE quotient (Markstein;
// |scale| >= ~5e-8 keeps r and the quotients that can reach a rounding boundary of rint() in the normal range).
// rint() and the float -> int conversion are one add of 1.5 * 2^23 (ulp 1, ties to even; |q| < 2^22 always:
// every |w - bias| <= max - min <= (2^bits) * |scale|), the clamp is an integer min / max.
template <int BITS>
__device__ __forceinline__ uint32_t affine_code(float w, const AffineGroup& g) {
    const float d = __fsub_rn(w, g.bias);
    const float q1 = __fmul_rn(d, g.r);
    const float rem = __fmaf_rn(q1, g.nscale, d);
    const float qq = __fmaf_rn(rem, g.r, q1);
    int code = (int)__float_as_uint(__fadd_rn(qq, 12582912.0f)) - 0x4B400000;
    return (uint32_t)min(max(code, 0), (1 << BITS) - 1);
}

// 8 codes as the BITS bytes of the row's LSB-first stream that hold them (first code in the lowest bits)
template <int BITS>
__device__ __forceinline__ uint64_t pack_octet(const uint32_t (&c)[8]) {
    uint64_t pack = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) pack |= (uint64_t)c[i] << (i * BITS);
    return pack;
}

}  // namespace gbxq
