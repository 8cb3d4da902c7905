"""PyTorch operators over the C ABI: `quantized_matmul` and `dequantize` with the signatures of
the MLX calls they replace.

    mx.quantized_matmul(x, w, scales, biases, transpose=True, group_size=64, bits=4)
        -- gbx_lm/models/quantized_linear_gba.py:195-203
    mx.dequantize(w, scales, biases, group_size=64, bits=4)
        -- gbx_lm/tuner/lora.py:62-68, gbx_lm/tuner/utils.py:214-220

Registered as torch custom ops `gbxq::qmm` / `gbxq::dequantize` (fake kernels for shape
propagation, CUDA-graph capturable: the library only enqueues on the current stream).
CUDA only -- there is deliberately no CPU implementation."""
from __future__ import annotations

import os

from typing import List, Optional, Sequence

import torch

from . import _lib

_DT = {torch.bfloat16: _lib.BF16, torch.float16: _lib.F16, torch.float32: _lib.F32}
_KERNELS = {"auto": 0, "generic": 1, "gemv": 2, "gemm": 3, "skinny": 4, "mmv": 5, "mmv8": 6, "gemm_ts": 7}


def _dt(t: torch.Tensor) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise ValueError(f"[quantized_matmul] activations/scales must be bf16, f16 or f32, got {t.dtype}") from None


def _as_u32_ptr_tensor(w: torch.Tensor) -> torch.Tensor:
    # checkpoints hold uint32; torch kernels are sparse for uint32, so int32 views are accepted too
    if w.dtype not in (torch.uint32, torch.int32):
        raise ValueError(f"[quantized_matmul] qweight must be uint32, got {w.dtype}")
    return w


def _require_cuda(*ts: Optional[torch.Tensor]) -> torch.device:
    dev = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(
                "gbx_lm_b200 ops run on CUDA (sm_100a) only; there is no CPU fallback. Got a tensor on "
                f"{t.device}."
            )
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError("all tensors must live on the same CUDA device")
    return dev


def _check_shapes(w, scales, biases, group_size: int, bits: int, k_x: Optional[int]) -> tuple[int, int]:
    if bits not in (2, 3, 4, 6, 8):
        raise ValueError(f"[quantized_matmul] bits must be one of 2, 3, 4, 6, 8; got {bits}")
    if group_size not in (32, 64, 128):
        raise ValueError(f"[quantized_matmul] group_size must be 32, 64 or 128; got {group_size}")
    if w.dim() != 2 or scales.dim() != 2 or scales.shape != biases.shape:
        raise ValueError("[quantized_matmul] qweight/scales/biases must be 2-D, scales.shape == biases.shape")
    n = w.shape[0]
    if (w.shape[1] * 32) % bits:
        raise ValueError("[quantized_matmul] qweight last dim incompatible with bits")
    k = w.shape[1] * 32 // bits
    if scales.shape[0] != n or scales.shape[1] * group_size != k:
        raise ValueError(
            f"[quantized_matmul] shapes disagree: qweight {tuple(w.shape)} (bits={bits}) implies K={k}, "
            f"scales {tuple(scales.shape)} (group_size={group_size})"
        )
    if k_x is not None and k_x != k:
        raise ValueError(f"[quantized_matmul] x last dim {k_x} != K {k}")
    if scales.dtype != biases.dtype:
        raise ValueError("[quantized_matmul] scales and biases must share a dtype")
    return n, k


_WORKSPACES: dict = {}


def _workspace(device: torch.device, stream: int, m: int, n: int, k: int, bits: int, group_size: int, dt: int):
    """Scratch for the split-K path of the tensor-core GEMM (gbxq_workspace_bytes): one zero-initialised buffer per
    (device, stream), grown on demand and reused by every call of that stream (calls of one stream are ordered; the kernel
    leaves the counter header zero)."""
    need = int(_lib.get().gbxq_workspace_bytes(m, n, k, bits, group_size, dt))
    if need == 0 or os.environ.get("GBXQ_NO_SPLITK") == "1":  # the switch exists for A/B measurements and tests
        return None, 0
    key = (device.index, stream)
    buf = _WORKSPACES.get(key)
    if buf is None or buf.numel() < need:
        buf = torch.zeros((max(need, 8 << 20),), dtype=torch.uint8, device=device)
        _WORKSPACES[key] = buf
    return buf, buf.numel()


def _qmm_impl(x, w, scales, biases, bias, group_size: int, bits: int, kernel: int) -> torch.Tensor:
    _require_cuda(x, w, scales, biases, bias)
    _as_u32_ptr_tensor(w)
    n, k = _check_shapes(w, scales, biases, group_size, bits, x.shape[-1])
    if x.dtype != scales.dtype:
        raise ValueError(
            f"[quantized_matmul] x ({x.dtype}) and scales ({scales.dtype}) must share a dtype; cast the "
            "activations like the reference loader casts scales/zeros to bf16 (gbx_lm/utils.py:841-843)"
        )
    dt = _dt(x)
    lead = x.shape[:-1]
    x2 = x.reshape(-1, k)
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    w = w.contiguous()
    scales = scales.contiguous()
    biases = biases.contiguous()
    if bias is not None:
        if bias.dtype != x.dtype or bias.numel() != n:
            raise ValueError("[quantized_matmul] bias must be [N] in the activation dtype")
        bias = bias.contiguous()
    m = x2.shape[0]
    y = torch.empty((m, n), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device):
        st = torch.cuda.current_stream().cuda_stream
        ws, ws_bytes = _workspace(x.device, st, m, n, k, bits, group_size, dt) if m > 4 else (None, 0)
        rc = _lib.get().gbxq_qmm_ex(
            x2.data_ptr(), w.data_ptr(), scales.data_ptr(), biases.data_ptr(),
            bias.data_ptr() if bias is not None else None, y.data_ptr(),
            m, n, k, bits, group_size, dt, kernel, ws.data_ptr() if ws is not None else None, ws_bytes, st,
        )
    _lib.check(rc, "gbxq_qmm")
    return y.reshape(*lead, n)


@torch.library.custom_op("gbxq::qmm", mutates_args=(), device_types="cuda")
def _qmm_op(
    x: torch.Tensor,
    w: torch.Tensor,
    scales: torch.Tensor,
    biases: torch.Tensor,
    bias: Optional[torch.Tensor],
    group_size: int,
    bits: int,
    kernel: int,
) -> torch.Tensor:
    return _qmm_impl(x, w, scales, biases, bias, group_size, bits, kernel)


@_qmm_op.register_fake
def _(x, w, scales, biases, bias, group_size, bits, kernel):
    return x.new_empty((*x.shape[:-1], w.shape[0]))


@torch.library.custom_op("gbxq::qmm_grouped", mutates_args=(), device_types="cuda")
def _qmm_grouped_op(
    x: torch.Tensor,
    ws: List[torch.Tensor],
    scales: List[torch.Tensor],
    biases: List[torch.Tensor],
    bias: List[Optional[torch.Tensor]],
    group_sizes: List[int],
    bits: List[int],
) -> List[torch.Tensor]:
    nseg = len(ws)
    if not (len(scales) == len(biases) == len(bias) == len(group_sizes) == len(bits) == nseg):
        raise ValueError("[quantized_matmul_grouped] per-segment lists must have the same length")
    _require_cuda(x, *ws, *scales, *biases, *bias)
    dt = _dt(x)
    k = x.shape[-1]
    lead = x.shape[:-1]
    x2 = x.reshape(-1, k)
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    m = x2.shape[0]
    segs = (_lib.Segment * max(nseg, 1))()
    outs, keep = [], []
    for i in range(nseg):
        _as_u32_ptr_tensor(ws[i])
        n, _ = _check_shapes(ws[i], scales[i], biases[i], group_sizes[i], bits[i], k)
        if x.dtype != scales[i].dtype:
            raise ValueError(f"[quantized_matmul_grouped] x ({x.dtype}) and scales ({scales[i].dtype}) must share a dtype")
        w, s, b = ws[i].contiguous(), scales[i].contiguous(), biases[i].contiguous()
        bi = bias[i]
        if bi is not None:
            if bi.dtype != x.dtype or bi.numel() != n:
                raise ValueError("[quantized_matmul_grouped] bias must be [N] in the activation dtype")
            bi = bi.contiguous()
        y = torch.empty((m, n), dtype=x.dtype, device=x.device)
        keep.append((w, s, b, bi))
        outs.append(y)
        segs[i] = _lib.Segment(w.data_ptr(), s.data_ptr(), b.data_ptr(), bi.data_ptr() if bi is not None else None,
                               y.data_ptr(), n, bits[i], group_sizes[i])
    with torch.cuda.device(x.device):
        st = torch.cuda.current_stream().cuda_stream
        wsb, wsn = None, 0
        if m > 4:  # decode batches / prefill: split-K scratch for the tensor-core GEMM (one grouped launch or per segment)
            need = int(_lib.get().gbxq_grouped_workspace_bytes(segs, nseg, m, k, dt))
            if need and os.environ.get("GBXQ_NO_SPLITK") != "1":
                key = (x.device.index, st)
                wsb = _WORKSPACES.get(key)
                if wsb is None or wsb.numel() < need:
                    wsb = torch.zeros((max(need, 8 << 20),), dtype=torch.uint8, device=x.device)
                    _WORKSPACES[key] = wsb
                wsn = wsb.numel()
        rc = _lib.get().gbxq_qmm_grouped_ws(segs, nseg, x2.data_ptr(), m, k, dt, wsb.data_ptr() if wsb is not None else None, wsn, st)
    _lib.check(rc, "gbxq_qmm_grouped")
    return [y.reshape(*lead, y.shape[-1]) for y in outs]


@_qmm_grouped_op.register_fake
def _(x, ws, scales, biases, bias, group_sizes, bits):
    return [x.new_empty((*x.shape[:-1], w.shape[0])) for w in ws]


@torch.library.custom_op("gbxq::dequantize", mutates_args=(), device_types="cuda")
def _dequantize_op(w: torch.Tensor, scales: torch.Tensor, biases: torch.Tensor, group_size: int, bits: int) -> torch.Tensor:
    _require_cuda(w, scales, biases)
    _as_u32_ptr_tensor(w)
    n, k = _check_shapes(w, scales, biases, group_size, bits, None)
    dt = _dt(scales)
    w = w.contiguous()
    scales = scales.contiguous()
    biases = biases.contiguous()
    out = torch.empty((n, k), dtype=scales.dtype, device=w.device)
    with torch.cuda.device(w.device):
        st = torch.cuda.current_stream().cuda_stream
        rc = _lib.get().gbxq_dequantize(w.data_ptr(), scales.data_ptr(), biases.data_ptr(), out.data_ptr(), n, k, bits, group_size, dt, st)
    _lib.check(rc, "gbxq_dequantize")
    return out


@_dequantize_op.register_fake
def _(w, scales, biases, group_size, bits):
    return scales.new_empty((w.shape[0], w.shape[1] * 32 // bits))


def quantized_matmul(
    x: torch.Tensor,
    w: torch.Tensor,
    scales: torch.Tensor,
    biases: torch.Tensor,
    transpose: bool = True,
    group_size: int = 64,
    bits: int = 4,
    *,
    bias: Optional[torch.Tensor] = None,
    kernel: str = "auto",
) -> torch.Tensor:
    """Drop-in for `mx.quantized_matmul`.  2-D weights with transpose=True are the QuantizedLinear call
    (quantized_linear_gba.py:195-203; `bias` fuses its `x + bias`, :204-205).  transpose=False (weights [.., K, N*bits/32]
    quantized along N) and weights with leading batch dimensions are the quantized-KV attention forms
    (gbx_lm/models/base.py:85-93): batch dimensions broadcast like a matmul's and run through `gbxq_gather_qmm`."""
    if transpose and w.dim() == 2:
        return _qmm_op(x, w, scales, biases, bias, int(group_size), int(bits), _KERNELS[kernel])
    if bias is not None:
        raise ValueError("[quantized_matmul] bias is fused for the 2-D transpose=True form only")
    return _qmm_batched(x, w, scales, biases, bool(transpose), int(group_size), int(bits))


def _gather_call(x3, w3, s3, b3, bias2, lhs, rhs, r: int, transpose: bool, group_size: int, bits: int) -> torch.Tensor:
    """x3 [XB, M, K]; w3 [E, N, K*bits/32] (transpose) or [E, K, N*bits/32]; lhs / rhs int32 device tensors of r entries or
    None (identity); returns [r, M, N]."""
    _require_cuda(x3, w3, s3, b3, bias2, lhs, rhs)
    _as_u32_ptr_tensor(w3)
    if bits not in (2, 3, 4, 6, 8):
        raise ValueError(f"[gather_qmm] bits must be one of 2, 3, 4, 6, 8; got {bits}")
    if group_size not in (32, 64, 128):
        raise ValueError(f"[gather_qmm] group_size must be 32, 64 or 128; got {group_size}")
    if x3.dtype != s3.dtype or s3.dtype != b3.dtype or s3.shape != b3.shape:
        raise ValueError("[gather_qmm] x, scales and biases must share a dtype; scales.shape == biases.shape")
    xb, m, k = x3.shape
    e = w3.shape[0]
    quant = w3.shape[2] * 32 // bits          # length of the quantized (last) axis
    if (w3.shape[2] * 32) % bits or s3.shape[0] != e or s3.shape[1] != w3.shape[1] or s3.shape[2] * group_size != quant:
        raise ValueError(f"[gather_qmm] shapes disagree: qweight {tuple(w3.shape)} bits={bits}, scales {tuple(s3.shape)} group_size={group_size}")
    if transpose:
        n = w3.shape[1]
        if quant != k:
            raise ValueError(f"[gather_qmm] x last dim {k} != K {quant}")
    else:
        n = quant
        if w3.shape[1] != k:
            raise ValueError(f"[gather_qmm] x last dim {k} != K {w3.shape[1]}")
    if bias2 is not None and (not transpose or bias2.shape != (e, n) or bias2.dtype != x3.dtype):
        raise ValueError("[gather_qmm] bias must be [E, N] in the activation dtype (transpose=True only)")
    x3, w3, s3, b3 = x3.contiguous(), w3.contiguous(), s3.contiguous(), b3.contiguous()
    y = torch.empty((r, m, n), dtype=x3.dtype, device=x3.device)
    with torch.cuda.device(x3.device):
        st = torch.cuda.current_stream().cuda_stream
        rc = _lib.get().gbxq_gather_qmm(
            x3.data_ptr(), w3.data_ptr(), s3.data_ptr(), b3.data_ptr(), bias2.contiguous().data_ptr() if bias2 is not None else None,
            lhs.data_ptr() if lhs is not None else None, rhs.data_ptr() if rhs is not None else None, y.data_ptr(),
            r, xb, e, m, n, k, 1 if transpose else 0, bits, group_size, _dt(x3), st,
        )
    _lib.check(rc, "gbxq_gather_qmm")
    return y


def _batch_index(shape, out_shape, device) -> Optional[torch.Tensor]:
    """int32 map from the flattened broadcast batch `out_shape` to the flattened batch `shape` (None = identity)."""
    n = 1
    for d in shape:
        n *= d
    if tuple(shape) == tuple(out_shape):
        return None
    idx = torch.arange(n, dtype=torch.int32, device=device).reshape(shape)
    return idx.expand(out_shape).reshape(-1).contiguous()


def _qmm_batched(x, w, scales, biases, transpose: bool, group_size: int, bits: int) -> torch.Tensor:
    if w.dim() < 2 or x.dim() < 1 or scales.dim() != w.dim() or biases.shape != scales.shape:
        raise ValueError("[quantized_matmul] qweight / scales / biases rank mismatch")
    squeeze = x.dim() == 1
    if squeeze:
        x = x.unsqueeze(0)
    xbat, wbat = tuple(x.shape[:-2]), tuple(w.shape[:-2])
    if tuple(scales.shape[:-2]) != wbat:
        raise ValueError("[quantized_matmul] scales batch dimensions differ from qweight's")
    out_bat = tuple(torch.broadcast_shapes(xbat, wbat))
    r = 1
    for d in out_bat:
        r *= d
    x3 = x.reshape(-1, x.shape[-2], x.shape[-1])
    w3 = w.reshape(-1, w.shape[-2], w.shape[-1])
    s3 = scales.reshape(-1, scales.shape[-2], scales.shape[-1])
    b3 = biases.reshape(-1, biases.shape[-2], biases.shape[-1])
    # align the batch ranks before broadcasting the index maps
    pad = lambda b: (1,) * (len(out_bat) - len(b)) + b  # noqa: E731
    lhs = _batch_index(pad(xbat), out_bat, x.device)
    rhs = _batch_index(pad(wbat), out_bat, x.device)
    y = _gather_call(x3, w3, s3, b3, None, lhs, rhs, r, transpose, group_size, bits)
    y = y.reshape(*out_bat, y.shape[-2], y.shape[-1])
    return y.squeeze(-2) if squeeze else y


def gather_qmm(
    x: torch.Tensor,
    w: torch.Tensor,
    scales: torch.Tensor,
    biases: torch.Tensor,
    lhs_indices: Optional[torch.Tensor] = None,
    rhs_indices: Optional[torch.Tensor] = None,
    transpose: bool = True,
    group_size: int = 64,
    bits: int = 4,
    *,
    sorted_indices: bool = False,
    bias: Optional[torch.Tensor] = None,
) -> torch.Tensor:
    """Drop-in for `mx.gather_qmm` as QuantizedSwitchLinear calls it (gbx_lm/models/switch_layers.py:78-92):
    x [..., M, K], w [E, N, K*bits/32] (a stack of experts; any leading batch shape), indices select the batch item of x
    (lhs, default: x's own batch broadcast against the indices) and the expert (rhs) per output batch item.  The result
    has shape broadcast(lhs_indices, rhs_indices).shape + [M, N].  `sorted_indices` is a scheduling hint in MLX; results
    do not depend on it.  `bias` ([E, N]) fuses the layer's `x + bias[indices]` (switch_layers.py:89-90)."""
    if w.dim() < 3:
        raise ValueError("[gather_qmm] qweight must be a stack of matrices [..., E, N, K*bits/32]")
    dev = x.device
    xbat, wbat = tuple(x.shape[:-2]), tuple(w.shape[:-2])
    nx = 1
    for d in xbat:
        nx *= d
    ne = 1
    for d in wbat:
        ne *= d
    if rhs_indices is None:
        rhs_indices = torch.arange(ne, dtype=torch.int32, device=dev).reshape(wbat)
    if lhs_indices is None:
        lhs_indices = torch.arange(nx, dtype=torch.int32, device=dev).reshape(xbat)
    out_bat = tuple(torch.broadcast_shapes(tuple(lhs_indices.shape), tuple(rhs_indices.shape)))
    lhs = lhs_indices.to(device=dev, dtype=torch.int32).expand(out_bat).reshape(-1).contiguous()
    rhs = rhs_indices.to(device=dev, dtype=torch.int32).expand(out_bat).reshape(-1).contiguous()
    x3 = x.reshape(-1, x.shape[-2], x.shape[-1])
    w3 = w.reshape(-1, w.shape[-2], w.shape[-1])
    s3 = scales.reshape(-1, scales.shape[-2], scales.shape[-1])
    b3 = biases.reshape(-1, biases.shape[-2], biases.shape[-1])
    bias2 = bias.reshape(-1, bias.shape[-1]) if bias is not None else None
    y = _gather_call(x3, w3, s3, b3, bias2, lhs, rhs, lhs.numel(), bool(transpose), int(group_size), int(bits))
    return y.reshape(*out_bat, y.shape[-2], y.shape[-1])


def quantized_matmul_grouped(x: torch.Tensor, layers: Sequence) -> List[torch.Tensor]:
    """The projections that read the same activations -- q_proj|k_proj|v_proj (gbx_lm/models/qllama.py:76) and
    gate_proj|up_proj (qllama.py:115) -- as ONE call: `layers` are QuantizedLinear-like objects (attributes
    qweight/scales/zeros/bias/group_size/bits).  Results are identical to calling each layer on x; at decode
    batch sizes (M <= 2) with a common group size the work is a single kernel launch (gbxq_qmm_grouped)."""
    layers = list(layers)
    if len(layers) > _lib.MAX_SEGMENTS:
        raise ValueError(f"[quantized_matmul_grouped] at most {_lib.MAX_SEGMENTS} projections per call")
    return _qmm_grouped_op(
        x, [l.qweight for l in layers], [l.scales for l in layers], [l.zeros for l in layers],
        [getattr(l, "bias", None) for l in layers], [int(l.group_size) for l in layers], [int(l.bits) for l in layers],
    )


class StreamChain:
    """An ordered chain of decode-sized QuantizedLinear forwards executed by ONE persistent kernel launch
    (gbxq_stream_plan / gbxq_qmm_stream, include/gbxq.h): the q|k|v, o_proj, gate|up, down_proj calls of the blocks
    (gbx_lm/models/qllama.py:76-115) in issue order.  Semantics and results are those of issuing the calls one after
    another (bitwise equal to `quantized_matmul` / `quantized_matmul_grouped`); later calls' weights stream into
    shared memory while earlier calls finish.

        chain = StreamChain(M)
        ys = chain.add(x_buf, [q, k, v])          # x_buf: persistent [M, K] bf16 buffer; returns the output buffers
        (o,) = chain.add(attn_buf, [o_proj])      # dep="prev" (stream order) by default, dep=None: x is external
        chain.finalize()
        chain.run()                               # enqueue on the current stream (CUDA-graph capturable)

    Buffers are fixed at plan time (as in a CUDA graph): write new activations INTO x_buf, read results from ys."""

    def __init__(self, m: int):
        self.m = int(m)
        self._calls = []
        self._keep = []
        self._info = None
        self._blob = None
        self._counters = None
        self.device = None

    def add(self, x: torch.Tensor, layers: Sequence, dep="prev", out: Optional[Sequence[torch.Tensor]] = None) -> List[torch.Tensor]:
        if self._info is not None:
            raise RuntimeError("StreamChain is finalized")
        layers = list(layers)
        if not 1 <= len(layers) <= _lib.MAX_SEGMENTS:
            raise ValueError(f"[StreamChain] 1..{_lib.MAX_SEGMENTS} projections per call")
        dev = _require_cuda(x, *[l.qweight for l in layers])
        if self.device is None:
            self.device = dev
        elif dev != self.device:
            raise RuntimeError("all tensors of a chain must live on the same CUDA device")
        if x.dim() != 2 or x.shape[0] != self.m or not x.is_contiguous() or x.dtype != torch.bfloat16:
            raise ValueError("[StreamChain] x must be a contiguous [M, K] bf16 buffer")
        k = x.shape[1]
        call = _lib.StreamCall()
        call.x, call.K, call.nseg = x.data_ptr(), k, len(layers)
        if dep == "prev":
            call.dep = _lib.DEP_PREV
        elif dep is None:
            call.dep = _lib.DEP_NONE
        else:
            call.dep = int(dep)
        outs = []
        for i, l in enumerate(layers):
            _as_u32_ptr_tensor(l.qweight)
            n, _ = _check_shapes(l.qweight, l.scales, l.zeros, int(l.group_size), int(l.bits), k)
            if l.scales.dtype != torch.bfloat16:
                raise ValueError("[StreamChain] scales/biases must be bf16")
            w, sc, b = l.qweight.contiguous(), l.scales.contiguous(), l.zeros.contiguous()
            bi = getattr(l, "bias", None)
            if bi is not None:
                if bi.dtype != x.dtype or bi.numel() != n:
                    raise ValueError("[StreamChain] bias must be [N] in the activation dtype")
                bi = bi.contiguous()
            y = out[i] if out is not None else torch.empty((self.m, n), dtype=x.dtype, device=x.device)
            if y.shape != (self.m, n) or y.dtype != x.dtype or not y.is_contiguous():
                raise ValueError("[StreamChain] out buffers must be contiguous [M, N] in the activation dtype")
            self._keep.append((x, w, sc, b, bi, y))
            outs.append(y)
            call.segs[i] = _lib.Segment(w.data_ptr(), sc.data_ptr(), b.data_ptr(), bi.data_ptr() if bi is not None else None,
                                        y.data_ptr(), n, int(l.bits), int(l.group_size))
        self._calls.append(call)
        return outs

    def __len__(self) -> int:
        return len(self._calls)

    def finalize(self, debug_timeline: bool = False) -> "StreamChain":
        import ctypes

        lib = _lib.get()
        n = len(self._calls)
        arr = (_lib.StreamCall * max(n, 1))(*self._calls)
        info = _lib.StreamInfo()
        _lib.check(lib.gbxq_stream_plan(arr, n, self.m, _lib.BF16, None, 0, ctypes.byref(info)), "gbxq_stream_plan")
        host = torch.empty(int(info.blob_bytes), dtype=torch.uint8)
        _lib.check(lib.gbxq_stream_plan(arr, n, self.m, _lib.BF16, host.data_ptr(), host.numel(), ctypes.byref(info)),
                   "gbxq_stream_plan")
        if debug_timeline:  # development aid: 8 globaltimer stamps per call from CTA 0 (tools/stream_timeline.py)
            self.timeline = torch.zeros((n, 8), dtype=torch.int64, device=self.device)
            lib.gbxq_debug_stream_timeline.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
            lib.gbxq_debug_stream_timeline.restype = None
            lib.gbxq_debug_stream_timeline(host.data_ptr(), n, self.timeline.data_ptr())
        self._blob = host.to(self.device)
        self._counters = torch.zeros(int(info.counter_bytes) // 4, dtype=torch.int32, device=self.device)
        self._info = info
        return self

    @property
    def info(self) -> dict:
        i = self._info
        return {f: getattr(i, f) for f, _ in _lib.StreamInfo._fields_}

    def run(self) -> None:
        import ctypes

        if self._info is None:
            self.finalize()
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream().cuda_stream
            rc = _lib.get().gbxq_qmm_stream(ctypes.byref(self._info), self._blob.data_ptr(), self._counters.data_ptr(), st)
        _lib.check(rc, "gbxq_qmm_stream")

    def timed_out(self) -> bool:
        """True if a launch ever gave up waiting for a CTA (synchronises; for tests and health checks)."""
        return bool(self._counters[-1].item())


# ------------------------------------------------------------------------------------------ decode-step glue
def _stream():
    return torch.cuda.current_stream().cuda_stream


def _bf16c(*ts):
    for t in ts:
        if t is not None and (t.dtype != torch.bfloat16 or not t.is_contiguous() or not t.is_cuda):
            raise ValueError("decode glue ops take contiguous CUDA bf16 tensors")


def _check_keep(keep: Optional[int], max_len: int, where: str) -> Optional[int]:
    """The sink count of a rotating cache of window max_len: None (a flat cache) or an int in [0, max_len)."""
    if keep is None:
        return None
    if isinstance(keep, bool) or not isinstance(keep, int) or not 0 <= keep < max_len:
        raise ValueError(f"{where}: keep must be an int in [0, {max_len}) (the cache's window), got {keep!r}")
    return keep


def _pos_stride(position: torch.Tensor, b: int, q: torch.Tensor, where: str) -> int:
    """The pos_stride of the decode-step entry points for `position`: 0 for int64 [1] (one position shared by all rows),
    1 for int64 [B] (row b at position[b]).  The kernels read it, so it must be contiguous on the device of q."""
    if position.dim() != 1 or position.numel() not in (1, b):
        raise ValueError(f"{where}: position must be int64 [1] (shared) or [B] = [{b}] (one per row), "
                         f"got {tuple(position.shape)}")
    if position.dtype != torch.int64 or position.device != q.device or not position.is_contiguous():
        raise ValueError(f"{where}: position must be a contiguous int64 tensor on the device of q, "
                         f"got {position.dtype} on {position.device}")
    return 0 if position.numel() == 1 else 1


def _block(q: torch.Tensor, where: str, keep: Optional[int] = None):
    """(B, T, Hq, D) of q: [B, Hq, D] is one token per row (T = 1, the single-token entry point); [B, T, Hq, D] is a block
    of T consecutive tokens per row, at positions p_b .. p_b + T - 1 (the `_multi` entry points, flat caches only)."""
    if q.dim() == 3:
        return q.shape[0], 1, q.shape[1], q.shape[2]
    if q.dim() != 4:
        raise ValueError(f"{where}: q must be [B, Hq, D] or [B, T, Hq, D], got {tuple(q.shape)}")
    if keep is not None:
        raise ValueError(f"{where}: a block of T tokens per row needs a flat cache (keep=None)")
    return tuple(q.shape)


def rope_cache(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, position: torch.Tensor, inv_freq: torch.Tensor,
               k_cache: torch.Tensor, v_cache: torch.Tensor, keep: Optional[int] = None) -> torch.Tensor:
    """gbxq_rope_cache: q [B,Hq,D] rotated IN PLACE (returned), k rotated and v copied into the caches [B,Hkv,max_len,D] at
    `position` (int64 device tensor [1]).  Replaces RoPE + cache.update of a decode step (gbx_lm/models/qllama.py:83-88).
    keep = an int: the caches are a rotating window of max_len rows with `keep` sinks, and k / v go to row
    ring_slot(position) (cache.ring_slot).  position int64 [B]: row b at position[b].
    q [B,T,Hq,D] (k / v [B,T,Hkv,D]), 1 <= T <= 8: gbxq_rope_cache_multi, token t of row b at position[b] + t, bitwise T
    single-token calls; flat caches only."""
    _bf16c(q, k, v, k_cache, v_cache)
    b, t, hq, d = _block(q, "rope_cache", keep)
    hkv, max_len = k_cache.shape[1], k_cache.shape[2]
    kv_shape = (b, hkv, d) if q.dim() == 3 else (b, t, hkv, d)
    if tuple(k.shape) != kv_shape or tuple(v.shape) != kv_shape:
        raise ValueError(f"rope_cache: k / v must be {kv_shape}")
    if inv_freq.dtype != torch.float32 or inv_freq.numel() != d // 2:
        raise ValueError("rope_cache: inv_freq float32 [D/2]")
    keep = _check_keep(keep, max_len, "rope_cache")
    stride = _pos_stride(position, b, q, "rope_cache")
    lib = _lib.get()
    with torch.cuda.device(q.device):
        if q.dim() == 4:
            rc = lib.gbxq_rope_cache_multi(q.data_ptr(), k.data_ptr(), v.data_ptr(), position.data_ptr(), stride,
                                           inv_freq.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), b, t, hq, hkv, d,
                                           max_len, _stream())
        else:
            rc = lib.gbxq_rope_cache(q.data_ptr(), k.data_ptr(), v.data_ptr(), position.data_ptr(), stride,
                                     inv_freq.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), b, hq, hkv, d,
                                     max_len, -1 if keep is None else keep, _stream())
    _lib.check(rc, "gbxq_rope_cache")
    return q


def decode_attention(q: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor, position: torch.Tensor, scale: float,
                     attend_len: Optional[int] = None) -> torch.Tensor:
    """gbxq_decode_attention: one query row per head, q [B,Hq,D], against the static caches, keys 0..position visible
    (and < attend_len), GQA.  Returns [B,Hq,D].  Replaces mask + scaled_dot_product_attention (qllama.py:90-93).
    position int64 [B]: row b sees keys 0..position[b].  q [B,T,Hq,D], 1 <= T <= 8: gbxq_decode_attention_multi, query t
    of row b sees keys 0..position[b] + t (bitwise the single query there); returns [B,T,Hq,D]."""
    _bf16c(q, k_cache, v_cache)
    b, t, hq, d = _block(q, "decode_attention")
    hkv, max_len = k_cache.shape[1], k_cache.shape[2]
    stride = _pos_stride(position, b, q, "decode_attention")
    out = torch.empty_like(q)
    lib, attend_len = _lib.get(), int(attend_len or max_len)
    with torch.cuda.device(q.device):
        if q.dim() == 4:
            rc = lib.gbxq_decode_attention_multi(q.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), position.data_ptr(),
                                                 stride, out.data_ptr(), b, t, hq, hkv, d, max_len, attend_len,
                                                 float(scale), _stream())
        else:
            rc = lib.gbxq_decode_attention(q.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), position.data_ptr(),
                                           stride, out.data_ptr(), b, hq, hkv, d, max_len, attend_len, float(scale),
                                           _stream())
    _lib.check(rc, "gbxq_decode_attention")
    return out


def _check_qcache(q: torch.Tensor, k_cache3, v_cache3, group_size: int, bits: int):
    """Shapes of the quantized-cache glue: q [B,Hq,D] (or a block [B,T,Hq,D]) bf16, triples (codes uint32
    [B,Hkv,max_len,D*bits/32], scales / biases bf16 [B,Hkv,max_len,D/group_size]), all contiguous on one CUDA device.
    Returns (B, T, Hq, Hkv, D, max_len)."""
    if bits not in (2, 3, 4, 6, 8):
        raise ValueError(f"quantized cache: bits must be one of 2, 3, 4, 6, 8; got {bits}")
    if group_size not in (32, 64, 128):
        raise ValueError(f"quantized cache: group_size must be 32, 64 or 128; got {group_size}")
    if len(k_cache3) != 3 or len(v_cache3) != 3:
        raise ValueError("quantized cache: keys and values are (codes, scales, biases) triples")
    if q.dim() not in (3, 4) or q.dtype != torch.bfloat16:
        raise ValueError("quantized cache: q must be bf16 [B, Hq, D] or [B, T, Hq, D]")
    b, t, hq, d = _block(q, "quantized cache")
    kq = k_cache3[0]
    if kq.dim() != 4:
        raise ValueError("quantized cache: codes must be [B, Hkv, max_len, D*bits/32]")
    hkv, max_len = kq.shape[1], kq.shape[2]
    want = ((b, hkv, max_len, d * bits // 32), (b, hkv, max_len, d // group_size), (b, hkv, max_len, d // group_size))
    for side in (k_cache3, v_cache3):
        if side[0].dtype not in (torch.uint32, torch.int32) or side[1].dtype != torch.bfloat16 or side[2].dtype != torch.bfloat16:
            raise ValueError("quantized cache: codes uint32, scales / biases bf16")
        if tuple(tuple(t.shape) for t in side) != want:
            raise ValueError(f"quantized cache: triple shapes {[tuple(t.shape) for t in side]} do not match q {tuple(q.shape)} "
                             f"at bits={bits}, group_size={group_size} (want {list(want)})")
    if d % 32 or d % group_size or hkv < 1 or hq % hkv:
        raise ValueError(f"quantized cache: D={d}, group_size={group_size}, Hq={hq}, Hkv={hkv} are inconsistent")
    ts = [q, *k_cache3, *v_cache3]
    if not all(t.is_cuda and t.is_contiguous() for t in ts) or len({t.device for t in ts}) != 1:
        raise ValueError("quantized cache ops take contiguous tensors on one CUDA device (there is no CPU path)")
    return b, t, hq, hkv, d, max_len


def rope_cache_quantized(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, position: torch.Tensor, inv_freq: torch.Tensor,
                         k_cache3, v_cache3, group_size: int, bits: int, keep: Optional[int] = None) -> torch.Tensor:
    """gbxq_rope_cache_quantized: q [B,Hq,D] rotated IN PLACE (returned); k rotated and v copied, each quantized into row
    `position` (int64 device tensor [1]) of its (codes, scales, biases) triple -- bit-identical to `rope_cache` into a bf16
    row followed by `quantize_into` of that row.  The quantized counterpart of `rope_cache` (RoPE +
    QuantizedKVCache.update_and_fetch, gbx_lm/models/cache.py:172-185).  keep = an int: row ring_slot(position) of a
    rotating cache, as `rope_cache`.  position int64 [B]: row b at position[b].  q [B,T,Hq,D] (k / v [B,T,Hkv,D]):
    gbxq_rope_cache_quantized_multi, as `rope_cache` with a block; flat caches only."""
    group_size, bits = int(group_size), int(bits)
    _block(q, "rope_cache_quantized", keep)  # a block needs a flat cache
    b, t, hq, hkv, d, max_len = _check_qcache(q, k_cache3, v_cache3, group_size, bits)
    _bf16c(k, v)
    kv_shape = (b, hkv, d) if q.dim() == 3 else (b, t, hkv, d)
    if tuple(k.shape) != kv_shape or tuple(v.shape) != kv_shape:
        raise ValueError(f"rope_cache_quantized: k / v must be {kv_shape}")
    if inv_freq.dtype != torch.float32 or inv_freq.numel() != d // 2 or inv_freq.device != q.device:
        raise ValueError("rope_cache_quantized: inv_freq float32 [D/2] on the device of q")
    keep = _check_keep(keep, max_len, "rope_cache_quantized")
    stride = _pos_stride(position, b, q, "rope_cache_quantized")
    lib = _lib.get()
    ptrs = (q.data_ptr(), k.data_ptr(), v.data_ptr(), position.data_ptr(), stride, inv_freq.data_ptr(),
            *[x.data_ptr() for x in k_cache3], *[x.data_ptr() for x in v_cache3])
    with torch.cuda.device(q.device):
        if q.dim() == 4:
            rc = lib.gbxq_rope_cache_quantized_multi(*ptrs, b, t, hq, hkv, d, max_len, bits, group_size, _stream())
        else:
            rc = lib.gbxq_rope_cache_quantized(*ptrs, b, hq, hkv, d, max_len, -1 if keep is None else keep, bits,
                                               group_size, _stream())
    _lib.check(rc, "gbxq_rope_cache_quantized")
    return q


# partials of gbxq_decode_attention_quantized: one buffer per device (keyed by device, not stream, so that a graph
# captured on a side stream uses the buffer its warm-up sized; the decode loop issues these calls from one stream at a
# time), grown on demand.  Buffers that were outgrown stay alive, because a captured CUDA graph may still point at them.
_QATTN_WS: dict = {}


def _qattn_workspace(device: torch.device, need: int) -> torch.Tensor:
    bufs = _QATTN_WS.setdefault(device.index, [])
    if not bufs or bufs[-1].numel() < need:
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("decode_attention_quantized: call it once eagerly with the same attend_len before capture")
        bufs.append(torch.zeros((max(need, 1 << 20),), dtype=torch.uint8, device=device))
    return bufs[-1]


def decode_attention_quantized(q: torch.Tensor, k_cache3, v_cache3, position: torch.Tensor, scale: float, group_size: int,
                               bits: int, attend_len: Optional[int] = None) -> torch.Tensor:
    """gbxq_decode_attention_quantized: one query row per head, q [B,Hq,D], against the quantized triples, keys
    0..position visible (and < attend_len, default the whole cache), GQA.  Returns [B,Hq,D] bf16.  The result does not
    depend on attend_len beyond the clamp (bitwise).  Replaces quantized_scaled_dot_product_attention at decode
    (gbx_lm/models/base.py:65-98).  position int64 [B]: row b sees keys 0..position[b].  q [B,T,Hq,D], 1 <= T <= 8:
    gbxq_decode_attention_quantized_multi, query t of row b at position[b] + t, bitwise the single query there, with each
    chunk's codes read once for the T queries; returns [B,T,Hq,D]."""
    group_size, bits = int(group_size), int(bits)
    b, t, hq, hkv, d, max_len = _check_qcache(q, k_cache3, v_cache3, group_size, bits)
    attend_len = int(max_len if attend_len is None else attend_len)
    if not 1 <= attend_len <= max_len:
        raise ValueError(f"decode_attention_quantized: attend_len {attend_len} outside [1, {max_len}]")
    stride = _pos_stride(position, b, q, "decode_attention_quantized")
    lib = _lib.get()
    need = int(lib.gbxq_decode_attention_quantized_workspace_bytes(b * t, hq, hkv, d, attend_len))
    out = torch.empty_like(q)
    with torch.cuda.device(q.device):
        ws = _qattn_workspace(q.device, need)
        ptrs = (q.data_ptr(), *[x.data_ptr() for x in k_cache3], *[x.data_ptr() for x in v_cache3], position.data_ptr(),
                stride, out.data_ptr())
        if q.dim() == 4:
            rc = lib.gbxq_decode_attention_quantized_multi(*ptrs, b, t, hq, hkv, d, max_len, attend_len, float(scale),
                                                           bits, group_size, ws.data_ptr(), ws.numel(), _stream())
        else:
            rc = lib.gbxq_decode_attention_quantized(*ptrs, b, hq, hkv, d, max_len, attend_len, float(scale), bits,
                                                     group_size, ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "gbxq_decode_attention_quantized")
    return out


def add_rmsnorm(x: torch.Tensor, r: Optional[torch.Tensor], w: torch.Tensor, eps: float, want_h: bool = True):
    """gbxq_add_rmsnorm: h = x + r (r None: h = x), y = RMSNorm(h) * w over the last dimension.  Returns (h, y); h is None
    when want_h is False.  Replaces the residual add + nn.RMSNorm pair (qllama.py:137-141)."""
    _bf16c(x, r, w)
    hdim = x.shape[-1]
    rows = x.numel() // hdim
    y = torch.empty_like(x)
    h = torch.empty_like(x) if (want_h and r is not None) else None
    with torch.cuda.device(x.device):
        rc = _lib.get().gbxq_add_rmsnorm(x.data_ptr(), r.data_ptr() if r is not None else None, w.data_ptr(), float(eps),
                                         h.data_ptr() if h is not None else None, y.data_ptr(), rows, hdim, _stream())
    _lib.check(rc, "gbxq_add_rmsnorm")
    return (h if r is not None else (x if want_h else None)), y


def silu_mul(gate: torch.Tensor, up: torch.Tensor) -> torch.Tensor:
    """gbxq_silu_mul: silu(gate) * up (qllama.py:115), both roundings of the unfused expression kept."""
    _bf16c(gate, up)
    out = torch.empty_like(gate)
    with torch.cuda.device(gate.device):
        rc = _lib.get().gbxq_silu_mul(gate.data_ptr(), up.data_ptr(), out.data_ptr(), gate.numel(), _stream())
    _lib.check(rc, "gbxq_silu_mul")
    return out


# rows served by gbxq_head_gemv: measured (profiles/r02k_headbench.txt) 1.00-1.04 of the HBM peak at one row, as fast as the
# dense matmul; from 4 rows on the kernel is bound by its shared-memory reads of x (0.65 / 0.38 at 4 / 8 rows)
_HEAD_MAX_ROWS = 2


def head_linear(x: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
    """logits = x . weight^T with the UNQUANTIZED bf16 vocabulary matrix (`lm_head` / `embed_tokens.as_linear`,
    gbx_lm/models/qllama.py:183-184,194-198).  Decode-sized inputs (<= 8 rows) stream through gbxq_head_gemv; anything
    else (more rows, prefill, other dtypes) is the framework's dense matmul."""
    k = x.shape[-1]
    rows = x.numel() // k
    if (x.is_cuda and x.dtype == torch.bfloat16 and weight.dtype == torch.bfloat16 and weight.is_contiguous()
            and 1 <= rows <= _HEAD_MAX_ROWS and k % 256 == 0 and k * max(rows, 1) * 2 <= 100 * 1024):
        x2 = x.reshape(rows, k)
        if not x2.is_contiguous():
            x2 = x2.contiguous()
        v = weight.shape[0]
        y = torch.empty((rows, v), dtype=torch.bfloat16, device=x.device)
        with torch.cuda.device(x.device):
            rc = _lib.get().gbxq_head_gemv(x2.data_ptr(), weight.data_ptr(), y.data_ptr(), rows, v, k, 0, _stream())
        if rc != -9:
            _lib.check(rc, "gbxq_head_gemv")
            return y.reshape(*x.shape[:-1], v)
    return torch.nn.functional.linear(x, weight)


def dequantize(w: torch.Tensor, scales: torch.Tensor, biases: torch.Tensor, group_size: int = 64, bits: int = 4) -> torch.Tensor:
    """Drop-in for `mx.dequantize` (bit-exact: T(T(scale*q)+bias), T = scales.dtype)."""
    return _dequantize_op(w, scales, biases, int(group_size), int(bits))


def _check_quantize_args(w: torch.Tensor, group_size: int, bits: int) -> int:
    if bits not in (2, 3, 4, 6, 8):
        raise ValueError(f"[quantize] The requested number of bits {bits} is not supported. The supported bits are 2, 3, 4, 6 and 8.")
    if group_size not in (32, 64, 128):
        raise ValueError(f"[quantize] The requested group size {group_size} is not supported. The supported group sizes are 32, 64 and 128.")
    if w.dim() < 2:
        raise ValueError(f"[quantize] The matrix to be quantized must have at least 2 dimension but it has only {w.dim()}.")
    if w.shape[-1] % group_size:
        raise ValueError(f"[quantize] The last dimension of the matrix needs to be divisible by the quantization group size "
                         f"{group_size}. However the provided matrix has shape {tuple(w.shape)}")
    if w.dtype not in _DT:
        raise ValueError(f"[quantize] Only real floating types can be quantized (bf16, f16, f32), got {w.dtype}")
    _require_cuda(w)
    return _DT[w.dtype]


def quantize(w: torch.Tensor, group_size: int = 64, bits: int = 4):
    """Drop-in for `mx.quantize` (gbxq_quantize): returns `(w_q, scales, biases)` with `w_q` uint32 `[..., K*bits/32]` and
    `scales` / `biases` `[..., K/group_size]` in `w.dtype`, quantized along the last axis -- the call of
    KVCache.to_quantized (gbx_lm/models/cache.py:251-263) and of QuantizedKVCache.update_and_fetch (cache.py:176-177).
    Codes, scales and biases are bit-exact against the restatement of MLX's recipe (oracle/MLX_SPEC.md R6)."""
    group_size, bits = int(group_size), int(bits)
    dt = _check_quantize_args(w, group_size, bits)
    k = w.shape[-1]
    w = w.contiguous()
    lead = tuple(w.shape[:-1])
    rows = w.numel() // k
    wq = torch.empty((*lead, k * bits // 32), dtype=torch.uint32, device=w.device)
    scales = torch.empty((*lead, k // group_size), dtype=w.dtype, device=w.device)
    biases = torch.empty_like(scales)
    with torch.cuda.device(w.device):
        rc = _lib.get().gbxq_quantize(w.data_ptr(), wq.data_ptr(), scales.data_ptr(), biases.data_ptr(), rows, k, bits,
                                      group_size, dt, _stream())
    _lib.check(rc, "gbxq_quantize")
    return wq, scales, biases


def quantize_into(w: torch.Tensor, out, offset: int, group_size: int = 64, bits: int = 4) -> None:
    """`out[i][..., offset : offset + L, :] = mx.quantize(w, group_size, bits)[i]` for i = 0, 1, 2 in ONE launch
    (gbxq_quantize_rows): w `[..., L, K]`, out = (codes, scales, biases) contiguous buffers `[..., capacity, *]` with the
    same leading shape -- the cache write of QuantizedKVCache.update_and_fetch (gbx_lm/models/cache.py:176-180)."""
    group_size, bits = int(group_size), int(bits)
    dt = _check_quantize_args(w, group_size, bits)
    oq, os_, ob = out
    _require_cuda(w, oq, os_, ob)
    _as_u32_ptr_tensor(oq)
    if w.dim() < 2 or oq.dim() != w.dim():
        raise ValueError("[quantize_into] w must be [..., L, K] and the outputs [..., capacity, *] of the same rank")
    k, steps, cap = w.shape[-1], w.shape[-2], oq.shape[-2]
    lead = tuple(w.shape[:-2])
    if (tuple(oq.shape) != (*lead, cap, k * bits // 32) or tuple(os_.shape) != (*lead, cap, k // group_size)
            or ob.shape != os_.shape or os_.dtype != w.dtype or ob.dtype != w.dtype):
        raise ValueError(f"[quantize_into] outputs do not match w {tuple(w.shape)}: codes {tuple(oq.shape)}, scales "
                         f"{tuple(os_.shape)} {os_.dtype}, biases {tuple(ob.shape)} {ob.dtype}")
    if not (oq.is_contiguous() and os_.is_contiguous() and ob.is_contiguous()):
        raise ValueError("[quantize_into] the output buffers must be contiguous")
    if offset < 0 or offset + steps > cap:
        raise ValueError(f"[quantize_into] rows [{offset}, {offset + steps}) do not fit a capacity of {cap}")
    if steps == 0 or w.numel() == 0:
        return
    w = w.contiguous()
    with torch.cuda.device(w.device):
        rc = _lib.get().gbxq_quantize_rows(w.data_ptr(), oq.data_ptr(), os_.data_ptr(), ob.data_ptr(), w.numel() // k, k,
                                           bits, group_size, dt, steps, cap, int(offset), _stream())
    _lib.check(rc, "gbxq_quantize_rows")


def select_kernel(m: int, n: int, k: int, bits: int, group_size: int, dtype: torch.dtype = torch.bfloat16) -> str:
    rc = _lib.get().gbxq_select_kernel(m, n, k, bits, group_size, _DT[dtype])
    _lib.check(min(rc, 0), "gbxq_select_kernel")
    return {1: "generic", 2: "gemv", 3: "gemm", 4: "skinny", 5: "mmv", 6: "mmv8", 7: "gemm_ts"}[rc]


def set_pdl_mode(mode: int) -> None:
    """GBXQ_OPT_PDL (include/gbxq.h): 0 plain launches, 1 PDL with conservative waits, 2 (default) PDL with the
    frozen weights streamed ahead of the wait."""
    _lib.check(_lib.get().gbxq_set_option(_lib.OPT_PDL, int(mode)), "gbxq_set_option")


def launch_count() -> int:
    return int(_lib.get().gbxq_launch_count())
