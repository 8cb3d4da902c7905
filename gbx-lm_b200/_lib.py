"""ctypes binding of libgbxq.so (include/gbxq.h).  There is NO fallback: if the CUDA library is
missing or fails to load, importing the ops raises."""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# GBXQ_LIB: development aid (A/B builds of the same library); still a CUDA build of this tree, never a fallback
LIB_PATH = os.environ.get("GBXQ_LIB") or os.path.join(HERE, "libgbxq.so")

BF16, F16, F32 = 0, 1, 2
KERNEL_AUTO, KERNEL_GENERIC, KERNEL_GEMV, KERNEL_GEMM, KERNEL_SKINNY, KERNEL_MMV, KERNEL_MMV8, KERNEL_GEMM_TS = 0, 1, 2, 3, 4, 5, 6, 7
OPT_PDL = 1
AR_MAX_CTAS = 32
RP_MAX_CTAS = 512

EXPORTS = (
    "gbxq_abi_version",
    "gbxq_status_string",
    "gbxq_last_cuda_error",
    "gbxq_last_cuda_error_string",
    "gbxq_qmm",
    "gbxq_qmm_ex",
    "gbxq_qmm_grouped",
    "gbxq_qmm_grouped_ws",
    "gbxq_grouped_workspace_bytes",
    "gbxq_stream_plan",
    "gbxq_qmm_stream",
    "gbxq_workspace_bytes",
    "gbxq_dequantize",
    "gbxq_quantize",
    "gbxq_quantize_rows",
    "gbxq_select_kernel",
    "gbxq_launch_count",
    "gbxq_set_option",
    "gbxq_get_option",
    "gbxq_allreduce_oneshot",
    "gbxq_qmm_rowpar_allreduce",
    "gbxq_rope_cache",
    "gbxq_decode_attention",
    "gbxq_rope_cache_quantized",
    "gbxq_decode_attention_quantized",
    "gbxq_decode_attention_quantized_workspace_bytes",
    "gbxq_rope_cache_multi",
    "gbxq_decode_attention_multi",
    "gbxq_rope_cache_quantized_multi",
    "gbxq_decode_attention_quantized_multi",
    "gbxq_add_rmsnorm",
    "gbxq_silu_mul",
    "gbxq_head_gemv",
    "gbxq_gather_qmm",
)


MAX_SEGMENTS = 4


class Segment(ctypes.Structure):
    """struct gbxq_segment (include/gbxq.h)."""

    _fields_ = [
        ("qweight", ctypes.c_void_p), ("scales", ctypes.c_void_p), ("biases", ctypes.c_void_p), ("bias", ctypes.c_void_p),
        ("y", ctypes.c_void_p), ("N", ctypes.c_int64), ("bits", ctypes.c_int), ("group_size", ctypes.c_int),
    ]


DEP_PREV, DEP_NONE = -2, -1


class Comm(ctypes.Structure):
    """struct gbxq_comm (include/gbxq.h): peer staging buffers / flag arrays of a tensor-parallel group."""

    _fields_ = [("peer_stage_host", ctypes.POINTER(ctypes.c_void_p)), ("peer_flags_host", ctypes.POINTER(ctypes.c_void_p)),
                ("stage_elems", ctypes.c_int64), ("rank", ctypes.c_int), ("world", ctypes.c_int)]


class StreamCall(ctypes.Structure):
    """struct gbxq_stream_call (include/gbxq.h)."""

    _fields_ = [("x", ctypes.c_void_p), ("K", ctypes.c_int64), ("nseg", ctypes.c_int), ("dep", ctypes.c_int),
                ("segs", Segment * MAX_SEGMENTS)]


class StreamInfo(ctypes.Structure):
    """struct gbxq_stream_info (include/gbxq.h)."""

    _fields_ = [("ncalls", ctypes.c_int32), ("grid", ctypes.c_int32), ("smem_bytes", ctypes.c_int32),
                ("group_size", ctypes.c_int32), ("mt", ctypes.c_int32), ("stages", ctypes.c_int32),
                ("slot_bytes", ctypes.c_uint32), ("reserved", ctypes.c_uint32), ("blob_bytes", ctypes.c_uint64),
                ("counter_bytes", ctypes.c_uint64)]


class GbxqError(RuntimeError):
    def __init__(self, status: int, where: str):
        lib = get()
        msg = lib.gbxq_status_string(status).decode()
        if status == -7:
            msg += ": " + lib.gbxq_last_cuda_error_string().decode()
        super().__init__(f"{where}: {msg} (status {status})")
        self.status = status


class GbxqValueError(GbxqError, ValueError):
    """Argument errors surface as ValueError, like MLX's quantized_matmul/dequantize."""


_lib = None


def get() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m gbx_lm_b200.build` (needs nvcc). "
            "gbx_lm_b200 has no CPU or PyTorch fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    vp, i64, ci, u32, sz = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_uint32, ctypes.c_size_t
    lib.gbxq_abi_version.restype = ci
    lib.gbxq_status_string.restype = ctypes.c_char_p
    lib.gbxq_status_string.argtypes = [ci]
    lib.gbxq_last_cuda_error.restype = ci
    lib.gbxq_last_cuda_error_string.restype = ctypes.c_char_p
    lib.gbxq_qmm.restype = ci
    lib.gbxq_qmm.argtypes = [vp, vp, vp, vp, vp, vp, i64, i64, i64, ci, ci, ci, vp, sz, vp]
    lib.gbxq_qmm_ex.restype = ci
    lib.gbxq_qmm_ex.argtypes = [vp, vp, vp, vp, vp, vp, i64, i64, i64, ci, ci, ci, ci, vp, sz, vp]
    lib.gbxq_qmm_grouped.restype = ci
    lib.gbxq_qmm_grouped.argtypes = [ctypes.POINTER(Segment), ci, vp, i64, i64, ci, vp]
    lib.gbxq_qmm_grouped_ws.restype = ci
    lib.gbxq_qmm_grouped_ws.argtypes = [ctypes.POINTER(Segment), ci, vp, i64, i64, ci, vp, sz, vp]
    lib.gbxq_grouped_workspace_bytes.restype = sz
    lib.gbxq_grouped_workspace_bytes.argtypes = [ctypes.POINTER(Segment), ci, i64, i64, ci]
    lib.gbxq_stream_plan.restype = ci
    lib.gbxq_stream_plan.argtypes = [ctypes.POINTER(StreamCall), ci, i64, ci, vp, sz, ctypes.POINTER(StreamInfo)]
    lib.gbxq_qmm_stream.restype = ci
    lib.gbxq_qmm_stream.argtypes = [ctypes.POINTER(StreamInfo), vp, vp, vp]
    lib.gbxq_workspace_bytes.restype = sz
    lib.gbxq_workspace_bytes.argtypes = [i64, i64, i64, ci, ci, ci]
    lib.gbxq_dequantize.restype = ci
    lib.gbxq_dequantize.argtypes = [vp, vp, vp, vp, i64, i64, ci, ci, ci, vp]
    lib.gbxq_quantize.restype = ci
    lib.gbxq_quantize.argtypes = [vp, vp, vp, vp, i64, i64, ci, ci, ci, vp]
    lib.gbxq_quantize_rows.restype = ci
    lib.gbxq_quantize_rows.argtypes = [vp, vp, vp, vp, i64, i64, ci, ci, ci, i64, i64, i64, vp]
    lib.gbxq_select_kernel.restype = ci
    lib.gbxq_select_kernel.argtypes = [i64, i64, i64, ci, ci, ci]
    lib.gbxq_launch_count.restype = ctypes.c_uint64
    lib.gbxq_set_option.restype = ci
    lib.gbxq_set_option.argtypes = [ci, ci]
    lib.gbxq_get_option.restype = ci
    lib.gbxq_get_option.argtypes = [ci]
    cf = ctypes.c_float
    lib.gbxq_rope_cache.restype = ci
    lib.gbxq_rope_cache.argtypes = [vp, vp, vp, vp, ci, vp, vp, vp, ci, ci, ci, ci, i64, i64, vp]
    lib.gbxq_decode_attention.restype = ci
    lib.gbxq_decode_attention.argtypes = [vp, vp, vp, vp, ci, vp, ci, ci, ci, ci, i64, i64, cf, vp]
    lib.gbxq_rope_cache_quantized.restype = ci
    lib.gbxq_rope_cache_quantized.argtypes = [vp] * 4 + [ci] + [vp] * 7 + [ci, ci, ci, ci, i64, i64, ci, ci, vp]
    lib.gbxq_decode_attention_quantized_workspace_bytes.restype = sz
    lib.gbxq_decode_attention_quantized_workspace_bytes.argtypes = [ci, ci, ci, ci, i64]
    lib.gbxq_decode_attention_quantized.restype = ci
    lib.gbxq_decode_attention_quantized.argtypes = [vp] * 8 + [ci, vp, ci, ci, ci, ci, i64, i64, cf, ci, ci, vp, sz, vp]
    # the `_multi` forms: T after B, no keep
    lib.gbxq_rope_cache_multi.restype = ci
    lib.gbxq_rope_cache_multi.argtypes = [vp, vp, vp, vp, ci, vp, vp, vp, ci, ci, ci, ci, ci, i64, vp]
    lib.gbxq_decode_attention_multi.restype = ci
    lib.gbxq_decode_attention_multi.argtypes = [vp, vp, vp, vp, ci, vp, ci, ci, ci, ci, ci, i64, i64, cf, vp]
    lib.gbxq_rope_cache_quantized_multi.restype = ci
    lib.gbxq_rope_cache_quantized_multi.argtypes = [vp] * 4 + [ci] + [vp] * 7 + [ci, ci, ci, ci, ci, i64, ci, ci, vp]
    lib.gbxq_decode_attention_quantized_multi.restype = ci
    lib.gbxq_decode_attention_quantized_multi.argtypes = ([vp] * 8 + [ci, vp, ci, ci, ci, ci, ci, i64, i64, cf, ci, ci, vp,
                                                          sz, vp])
    lib.gbxq_add_rmsnorm.restype = ci
    lib.gbxq_add_rmsnorm.argtypes = [vp, vp, vp, cf, vp, vp, i64, ci, vp]
    lib.gbxq_silu_mul.restype = ci
    lib.gbxq_silu_mul.argtypes = [vp, vp, vp, i64, vp]
    lib.gbxq_head_gemv.restype = ci
    lib.gbxq_head_gemv.argtypes = [vp, vp, vp, i64, i64, i64, ci, vp]
    lib.gbxq_gather_qmm.restype = ci
    lib.gbxq_gather_qmm.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, i64, i64, i64, ci, ci, ci, ci, vp]
    lib.gbxq_allreduce_oneshot.restype = ci
    lib.gbxq_allreduce_oneshot.argtypes = [vp, vp, i64, ci, vp, vp, i64, ci, ci, u32, vp]
    lib.gbxq_qmm_rowpar_allreduce.restype = ci
    lib.gbxq_qmm_rowpar_allreduce.argtypes = [vp, vp, vp, vp, vp, vp, i64, i64, i64, ci, ci, ci, ctypes.POINTER(Comm), vp]
    if lib.gbxq_abi_version() != 2:
        raise ImportError("libgbxq.so ABI version mismatch; rebuild with `python -m gbx_lm_b200.build --force`")
    _lib = lib
    return lib


def check(status: int, where: str) -> None:
    if status == 0:
        return
    if status in (-1, -2, -3, -4, -5, -6):
        raise GbxqValueError(status, where)
    raise GbxqError(status, where)
