"""CPU tests of the drop-in boundary: libgbxq.so loads without a GPU, exports every symbol that
include/gbxq.h declares, rejects bad arguments with the documented status codes before touching
CUDA, and the Python ops refuse CPU tensors (no fallback)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_functions():
    hdr = open(os.path.join(ROOT, "include", "gbxq.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(gbxq_[a-z_0-9]+)\s*\(", hdr)))


def test_header_symbols_exported_at_abi_version_2():
    from gbx_lm_b200 import _lib

    lib = _lib.get()
    names = _declared_functions()
    assert len(names) >= 10
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/gbxq.h but not exported"
    assert sorted(_lib.EXPORTS) == names
    assert lib.gbxq_abi_version() == 2


def test_no_torch_types_in_abi():
    hdr = open(os.path.join(ROOT, "include", "gbxq.h")).read()
    assert "torch" not in hdr and "at::" not in hdr and "#include <cuda" not in hdr


def test_argument_validation_without_gpu():
    from gbx_lm_b200 import _lib

    lib = _lib.get()
    p = ctypes.c_void_p(256)  # never dereferenced: validation fails first
    q = lambda **kw: lib.gbxq_qmm(p, p, p, p, None, p, kw.get("M", 1), kw.get("N", 8), kw.get("K", 64),
                                  kw.get("bits", 4), kw.get("gs", 64), kw.get("dt", 0), None, 0, None)
    assert q(bits=5) == -1 and q(bits=1) == -1 and q(bits=16) == -1
    assert q(gs=16) == -2 and q(gs=256) == -2
    assert q(K=48) == -3 and q(K=96, gs=64) == -3 and q(M=-1) == -3 and q(K=0) == -3
    assert q(dt=3) == -4
    assert q(M=0) == 0 and q(N=0) == 0  # empty problems are no-ops
    assert lib.gbxq_qmm(None, p, p, p, None, p, 1, 8, 64, 4, 64, 0, None, 0, None) == -6
    assert lib.gbxq_dequantize(p, p, p, ctypes.c_void_p(8), 8, 64, 4, 64, 0, None) == -5
    assert lib.gbxq_dequantize(p, p, p, p, 8, 64, 7, 64, 0, None) == -1
    assert lib.gbxq_workspace_bytes(1, 8, 64, 4, 64, 0) == 0
    assert b"bits" in lib.gbxq_status_string(-1)
    assert lib.gbxq_allreduce_oneshot(p, p, 64, 0, p, p, 64, 0, 2, 1, None) == -3  # capacity < 2*count
    assert lib.gbxq_allreduce_oneshot(p, p, 64, 0, p, p, 256, 2, 2, 1, None) == -3  # rank out of range


def test_stream_plan_is_host_only_and_validates():
    """gbxq_stream_plan never touches the device: sizes, ring geometry and refusals can be checked without a GPU."""
    from gbx_lm_b200 import _lib

    lib = _lib.get()
    p = 4096  # fake, 16-byte aligned device addresses; the planner never dereferences them

    def call(K, segs, dep=_lib.DEP_PREV):
        c = _lib.StreamCall()
        c.x, c.K, c.nseg, c.dep = p, K, len(segs), dep
        for i, (bits, N, gs) in enumerate(segs):
            c.segs[i] = _lib.Segment(p, p, p, None, p, N, bits, gs)
        return c

    def plan(calls, M=1, dt=0):
        arr = (_lib.StreamCall * len(calls))(*calls)
        info = _lib.StreamInfo()
        rc = lib.gbxq_stream_plan(arr, len(calls), M, dt, None, 0, ctypes.byref(info))
        return rc, info, arr

    block = [call(4096, [(4, 4096, 64), (2, 1024, 64), (4, 1024, 64)]), call(4096, [(4, 4096, 64)]),
             call(4096, [(4, 14336, 64), (4, 14336, 64)]), call(14336, [(4, 4096, 64)])]
    rc, info, arr = plan(block * 4)
    assert rc == 0 and info.ncalls == 16 and info.grid % 2 == 0 and info.group_size == 64 and info.mt == 1
    assert 2 <= info.stages <= 8 and info.smem_bytes <= 224 * 1024 and info.stages * info.slot_bytes < info.smem_bytes
    assert info.counter_bytes == (16 + 2) * 4 and info.blob_bytes > 0
    buf = ctypes.create_string_buffer(int(info.blob_bytes))
    assert lib.gbxq_stream_plan(arr, 16, 1, 0, buf, info.blob_bytes - 1, ctypes.byref(info)) == -8  # blob too small
    assert lib.gbxq_stream_plan(arr, 16, 1, 0, buf, info.blob_bytes, ctypes.byref(info)) == 0
    assert any(buf.raw)
    assert plan([call(4096, [(3, 64, 64)])])[0] == -9          # 3-bit: not served by the chain kernel
    assert plan([call(4096, [(4, 64, 64)])], M=5)[0] == -9      # prefill-sized M
    assert plan([call(4096, [(4, 64, 64)])], dt=1)[0] == -9     # fp16
    assert plan([call(4096, [(4, 64, 64)]), call(4096, [(4, 64, 128)])])[0] == -9  # mixed group sizes
    assert plan([call(4096, [(5, 64, 64)])])[0] == -1
    assert plan([call(4096, [(4, 64, 64)], dep=3)])[0] == -3    # dependency on a later call
    assert lib.gbxq_qmm_stream(None, None, None, None) == -6


def test_ops_refuse_cpu_tensors():
    import gbx_lm_b200 as g

    x = torch.zeros(1, 64, dtype=torch.bfloat16)
    w = torch.zeros(8, 8, dtype=torch.uint32)
    s = torch.ones(8, 1, dtype=torch.bfloat16)
    with pytest.raises((RuntimeError, NotImplementedError)):
        g.quantized_matmul(x, w, s, s, True, 64, 4)
    with pytest.raises((RuntimeError, NotImplementedError)):
        g.dequantize(w, s, s, 64, 4)


def test_python_shape_errors_are_value_errors():
    from gbx_lm_b200 import ops

    w = torch.zeros(8, 8, dtype=torch.uint32)
    s = torch.ones(8, 1, dtype=torch.bfloat16)
    with pytest.raises(ValueError):
        ops._check_shapes(w, s, s, 64, 5, None)
    with pytest.raises(ValueError):
        ops._check_shapes(w, s, s, 48, 4, None)
    with pytest.raises(ValueError):
        ops._check_shapes(w, torch.ones(8, 2, dtype=torch.bfloat16), torch.ones(8, 2, dtype=torch.bfloat16), 64, 4, None)
    with pytest.raises(ValueError):
        ops._check_shapes(w, s, s, 64, 4, 128)
    assert ops._check_shapes(w, s, s, 64, 4, 64) == (8, 64)


def test_quantized_linear_attribute_contract():
    """Constructor signature, attribute names, shapes and dtypes of quantized_linear_gba.py:36-117."""
    from gbx_lm_b200 import QuantizedLinear

    for bits in (2, 3, 4, 6, 8):
        for gs in (32, 64, 128):
            m = QuantizedLinear(256, 48, bias=(bits == 4), group_size=gs, bits=bits)
            assert m.qweight.shape == (48, 256 // 32 * bits) and m.qweight.dtype == torch.uint32
            assert m.scales.shape == (48, 256 // gs) == m.zeros.shape
            assert m.channel_scale.shape == (1, 1, 256) and m.channel_scale.dtype == torch.float16
            assert (m.bits, m.group_size, m.input_dims, m.output_dims) == (bits, gs, 256, 48)
            assert m.weight is m.qweight and m.biases is m.zeros
            assert (m.bias is not None) == (bits == 4)
            keys = set(m.state_dict().keys())
            assert {"qweight", "scales", "zeros", "channel_scale"} <= keys


def test_stream_plan_blob_invariants():
    """The descriptor blob gbxq_stream_plan writes (layout of StreamCallDev / Mmv8Params in gbxq_stream.cu and
    gbxq_mmv8_body.cuh, restated here): every row of every projection belongs to exactly one CTA, stages are whole MMA
    sets, a stage's weights, scales and biases fit the ring slot, and the ring fits the launch's shared memory."""
    import struct

    from gbx_lm_b200 import _lib

    lib = _lib.get()
    base = 1 << 20

    def call(K, segs, dep=_lib.DEP_PREV):
        c = _lib.StreamCall()
        c.x, c.K, c.nseg, c.dep = base, K, len(segs), dep
        for i, (bits, N, gs) in enumerate(segs):
            c.segs[i] = _lib.Segment(base + 4096 * (i + 1), base, base, None, base, N, bits, gs)
        return c

    chains = {
        1: [call(4096, [(4, 4096, 64), (2, 1024, 64), (8, 1024, 64)]), call(4096, [(4, 4096, 64)]),
            call(4096, [(4, 14336, 64), (2, 14336, 64)]), call(14336, [(4, 4096, 64)], dep=1),
            call(2048, [(4, 300, 64), (4, 1, 64)], dep=_lib.DEP_NONE), call(8192, [(2, 8192, 64)])],
        2: [call(4096, [(4, 4096, 128), (4, 1024, 128)]), call(8192, [(8, 4096, 128)])],
        4: [call(4096, [(4, 6144, 64)]), call(2048, [(2, 2048, 64), (4, 512, 64)])],
    }
    P, CALL = 144, 640  # sizeof(Mmv8Params), sizeof(StreamCallDev)
    for M, calls in chains.items():
        arr = (_lib.StreamCall * len(calls))(*calls)
        info = _lib.StreamInfo()
        assert lib.gbxq_stream_plan(arr, len(calls), M, 0, None, 0, ctypes.byref(info)) == 0
        assert info.blob_bytes == CALL * len(calls) and info.mt == {1: 1, 2: 2, 4: 4}[M]
        buf = ctypes.create_string_buffer(int(info.blob_bytes))
        assert lib.gbxq_stream_plan(arr, len(calls), M, 0, buf, info.blob_bytes, ctypes.byref(info)) == 0
        raw = buf.raw
        for ci, c in enumerate(calls):
            off = ci * CALL
            cta0 = struct.unpack_from("5i", raw, off + 4 * P)
            bits = struct.unpack_from("4i", raw, off + 4 * P + 20)
            nseg, variant, dep = struct.unpack_from("3i", raw, off + 4 * P + 36)
            assert nseg == c.nseg and 0 <= variant < 6
            assert dep == (ci - 1 if c.dep == _lib.DEP_PREV else c.dep) and dep < ci
            assert cta0[0] == 0 and all(cta0[i] <= cta0[i + 1] for i in range(4)) and cta0[4] <= info.grid
            assert cta0[nseg] == cta0[4]
            for s in range(nseg):
                po = off + s * P
                xq, wq, sq, bq, biasq, yq, N, K = struct.unpack_from("6Q2q", raw, po)
                Mv, G, row_bytes, nch, cw, rg, tr, stages, slot_bytes, sb_off, early = struct.unpack_from("2i2I4i2Ii", raw, po + 64)
                rows_base, rows_rem, spr0, spr1 = struct.unpack_from("4i", raw, po + 128)
                sg = c.segs[s]
                grid_s = cta0[s + 1] - cta0[s]
                assert (N, K, bits[s], Mv) == (sg.N, c.K, sg.bits, M) and wq == sg.qweight and xq == c.x
                assert G == K // sg.group_size and row_bytes == K * sg.bits // 8 and nch * 4 == G
                assert grid_s >= 1 and rows_base * grid_s + rows_rem == N and 0 <= rows_rem < grid_s  # every row once
                assert 1 <= cw * rg <= 16 and tr % 4 == 0 and spr0 % 4 == 0 and spr1 % 4 == 0 and 0 < spr0 <= tr and spr1 <= tr
                assert stages == info.stages and slot_bytes == info.slot_bytes and early == 1
                assert tr * row_bytes <= sb_off and sb_off + 2 * tr * G * 2 <= slot_bytes
        assert 4096 + info.stages * info.slot_bytes < info.smem_bytes <= 224 * 1024


def test_every_entry_point_is_documented():
    """INTEGRATION.md names each exported function next to the reference call it replaces."""
    from gbx_lm_b200 import _lib

    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    missing = [n for n in _lib.EXPORTS if n not in text and n.replace("_string", "[_string]") not in text]
    assert not missing, missing
