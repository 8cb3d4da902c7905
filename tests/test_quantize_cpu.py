"""CPU tests around the device-side quantiser (gbxq_quantize, SURVEY.md 8f rank 4): the restatement of mx.quantize
(oracle/MLX_SPEC.md R6) checked three ways, the argument validation of the C ABI (no GPU needed: it fails before any
CUDA call) and the host logic of the two KV caches (growth in blocks of 256, trim, state, to_quantized) with the
device operation stubbed by the oracle."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import indep_check as I
from oracle import mlx_affine as A


@pytest.mark.parametrize("dtype", ["bf16", "f16", "f32"])
@pytest.mark.parametrize("bits", A.SUPPORTED_BITS)
def test_quantize_numpy_vs_independent_scalar_checker(bits, dtype):
    rng = np.random.default_rng(bits)
    for gs in (32, 64, 128):
        w = rng.standard_normal((4, 2 * gs)).astype(np.float32) * np.float32(rng.choice([1e-3, 1.0, 50.0]))
        w[0, :gs] = 0.0          # all-zero group: scale = -1e-7, bias = 0, codes 0
        w[1, :gs] = 0.37         # constant group
        w[2, :gs] = -np.abs(w[2, :gs])  # all negative: the minimum is the anchored edge
        w = A._round_to(w, dtype)
        qw, s, b = A.quantize(w, gs, bits, dtype)
        codes = A.unpack_codes(qw, bits)
        for n in range(w.shape[0]):
            for g in range(2):
                c, sc, bi = I.quantize_group([float(v) for v in w[n, g * gs:(g + 1) * gs]], bits)
                assert list(codes[n, g * gs:(g + 1) * gs]) == c
                assert A._round_to(np.float32(sc), dtype) == s[n, g] and A._round_to(np.float32(bi), dtype) == b[n, g]
    assert (codes[0, :gs] == 0).all() and s[0, 0] == A._round_to(np.float32(-1e-7), dtype) and b[0, 0] == 0


@pytest.mark.parametrize("dtype", ["bf16", "f16", "f32"])
def test_quantize_numpy_vs_c_oracle(dtype):
    """Second independent implementation: the C restatement walks the matrix group by group as MLX's CPU quantiser does
    (oracle/gbxq_oracle.c::gbxq_oracle_quantize); codes and statistics equal the numpy one on every width x group size,
    including zero / constant / one-sided groups and magnitudes from 1e-6 to 1e4."""
    from oracle import c_oracle as C

    rng = np.random.default_rng(3)
    for bits in A.SUPPORTED_BITS:
        for gs in (32, 64, 128):
            w = rng.standard_normal((37, 3 * gs)).astype(np.float32) * rng.choice([1e-6, 1e-2, 1.0, 1e4], size=(37, 1)).astype(np.float32)
            w[0, :gs] = 0.0
            w[1, :gs] = -0.37
            w[2, :gs] = np.abs(w[2, :gs])
            w = A._round_to(w, dtype)
            qn, sn, bn = A.quantize(w, gs, bits, dtype)
            raw = w if dtype == "f32" else (A.f32_to_bf16_bits(w) if dtype == "bf16" else w.astype(np.float16).view(np.uint16))
            qc, sc, bc = C.quantize(raw, gs, bits, dtype)
            widen = (lambda a: a) if dtype == "f32" else (A.bf16_bits_to_f32 if dtype == "bf16" else (lambda a: a.view(np.float16).astype(np.float32)))
            assert np.array_equal(qc, qn), (bits, gs)
            assert np.array_equal(widen(sc), sn) and np.array_equal(widen(bc), bn), (bits, gs)


def test_quantize_hand_derived_known_answers():
    """Two groups whose answer follows from R6 by hand.  w = k mod 16 at 4 bits: max 15, min 0, |min| <= |max| so the
    scale is negative, -(15 / 15) = -1; the edge is the maximum, q0 = rint(15 / -1) = -15, scale = 15 / -15 = -1,
    bias = 15, code = rint((w - 15) / -1) = 15 - w.  Its mirror image w = -(k mod 16): |min| > |max|, scale = +1,
    edge = -15, bias = -15, code = w + 15 -- the same codes."""
    k = np.arange(64)
    for sign, scale, bias in ((1.0, -1.0, 15.0), (-1.0, 1.0, -15.0)):
        w = (sign * (k % 16)).astype(np.float32)[None]
        q, s, b = A.quantize(w, 64, 4, "bf16")
        assert s[0, 0] == scale and b[0, 0] == bias
        assert (A.unpack_codes(q, 4)[0] == 15 - (k % 16)).all()
        assert q[0, 0] == 0x89ABCDEF and q[0, 1] == 0x01234567   # codes 15..8 then 7..0, first code in the low nibble
        assert I.quantize_group([float(v) for v in w[0]], 4) == (list(15 - (k % 16)), scale, bias)


import json  # noqa: E402
import os  # noqa: E402

QG = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "quantize_golden.json")))


@pytest.mark.parametrize("case", QG["cases"], ids=lambda c: f"b{c['bits']}-g{c['group_size']}")
def test_quantize_golden_fixture(case):
    """tests/golden/quantize_golden.json was written by the C restatement; the numpy oracle reproduces it."""
    rows, K, bits, gs = case["rows"], case["K"], case["bits"], case["group_size"]
    w = A.bf16_bits_to_f32(np.array(case["w_bf16"], dtype=np.uint16).reshape(rows, K))
    q, s, b = A.quantize(w, gs, bits, "bf16")
    assert np.array_equal(q.reshape(-1), np.array(case["codes"], dtype=np.uint32))
    assert np.array_equal(A.f32_to_bf16_bits(s).reshape(-1), np.array(case["scales_bf16"], dtype=np.uint16))
    assert np.array_equal(A.f32_to_bf16_bits(b).reshape(-1), np.array(case["biases_bf16"], dtype=np.uint16))


@pytest.mark.parametrize("bits", A.SUPPORTED_BITS)
def test_quantize_properties(bits):
    """What holds whatever the exact recipe (R6, last sentence): the anchored edge is exact, the error is at most one
    step, codes span the range, and batch dimensions are just more rows."""
    rng = np.random.default_rng(7)
    gs = 64
    w = rng.standard_normal((2, 3, 5, 2 * gs)).astype(np.float32)
    qw, s, b = A.quantize(w, gs, bits, "f32")
    assert qw.shape == (2, 3, 5, 2 * gs * bits // 32) and s.shape == b.shape == (2, 3, 5, 2)
    flat = A.quantize(w.reshape(-1, 2 * gs), gs, bits, "f32")
    assert all(np.array_equal(a.reshape(c.shape), c) for a, c in zip((qw, s, b), flat))
    d = A.dequantize(flat[0], flat[1], flat[2], gs, bits, "f32").reshape(-1, 2, gs)
    g = w.reshape(-1, 2, gs)
    step = np.abs(flat[1])[..., None]
    assert (np.abs(d - g) <= 1.01 * step + 1e-6).all()
    edge = np.where(np.abs(g.min(-1)) > np.abs(g.max(-1)), g.min(-1), g.max(-1))
    hit = np.take_along_axis(d, np.abs(g).argmax(-1)[..., None], -1)[..., 0]
    assert np.array_equal(hit, edge)  # code 0 dequantises to the bias = the edge, bit for bit in fp32
    codes = A.unpack_codes(flat[0], bits).reshape(-1, 2, gs)
    assert codes.min() == 0 and codes.max() == (1 << bits) - 1


def test_packing_quantize_affine_agrees_with_oracle():
    from gbx_lm_b200 import packing

    rng = np.random.default_rng(1)
    for tdt, dtype in ((torch.bfloat16, "bf16"), (torch.float16, "f16"), (torch.float32, "f32")):
        for bits in A.SUPPORTED_BITS:
            for gs in (32, 64, 128):
                w = torch.from_numpy(rng.standard_normal((8, 2 * gs)).astype(np.float32)).to(tdt)
                qw, s, b = packing.quantize_affine(w, gs, bits)
                oq, os_, ob = A.quantize(w.float().numpy(), gs, bits, dtype)
                assert np.array_equal(qw.view(torch.int32).numpy().view(np.uint32), oq)
                assert np.array_equal(s.float().numpy(), os_) and np.array_equal(b.float().numpy(), ob)


def test_quantize_abi_validation_without_gpu():
    from gbx_lm_b200 import _lib

    lib = _lib.get()
    p = ctypes.c_void_p(256)  # never dereferenced: validation fails first
    q = lambda **kw: lib.gbxq_quantize(kw.get("w", p), p, p, p, kw.get("rows", 4), kw.get("K", 128), kw.get("bits", 4),
                                       kw.get("gs", 64), kw.get("dt", 0), None)
    assert q(bits=5) == -1 and q(bits=0) == -1
    assert q(gs=16) == -2
    assert q(K=96) == -3 and q(K=0) == -3 and q(rows=-1) == -3
    assert q(dt=7) == -4
    assert q(rows=0) == 0                       # empty input: no-op
    assert q(w=None) == -6
    assert q(w=ctypes.c_void_p(264)) == -5      # w must be 16-byte aligned
    r = lambda inner, stride, off, rows=4: lib.gbxq_quantize_rows(p, p, p, p, rows, 128, 4, 64, 0, inner, stride, off, None)
    assert r(0, 8, 0) == -3 and r(3, 8, 0) == -3   # inner_rows >= 1 and a divisor of rows
    assert r(2, 8, 7) == -3 and r(2, 1, 0) == -3   # the new rows must fit the capacity
    assert r(2, 8, -1) == -3
    assert r(2, 8, 6, rows=0) == 0


def test_ops_quantize_refuses_cpu_and_bad_arguments():
    from gbx_lm_b200 import ops

    w = torch.zeros((4, 128), dtype=torch.bfloat16)
    with pytest.raises(RuntimeError):
        ops.quantize(w)                              # no CPU path
    with pytest.raises(ValueError):
        ops.quantize(w, bits=5)
    with pytest.raises(ValueError):
        ops.quantize(w, group_size=48)
    with pytest.raises(ValueError):
        ops.quantize(w[:, :96], group_size=64)       # last dim not divisible
    with pytest.raises(ValueError):
        ops.quantize(w[0])                           # needs >= 2 dims
    with pytest.raises(ValueError):
        ops.quantize(w.to(torch.int32))


# ---------------------------------------------------------------------------------------------------------------
# host logic of the caches (gbx_lm/models/cache.py:133-266) with the device op stubbed by the oracle
# ---------------------------------------------------------------------------------------------------------------
def _oracle_quantize(x, group_size, bits):
    dt = {torch.bfloat16: "bf16", torch.float16: "f16", torch.float32: "f32"}[x.dtype]
    q, s, b = A.quantize(x.float().numpy(), group_size, bits, dt)
    return (torch.from_numpy(q.view(np.int32)).view(torch.uint32), torch.from_numpy(s).to(x.dtype), torch.from_numpy(b).to(x.dtype))


def _oracle_quantize_into(x, out, offset, group_size, bits):
    for o, v in zip(out, _oracle_quantize(x, group_size, bits)):
        o.view(torch.int32 if o.dtype == torch.uint32 else o.dtype)[..., offset:offset + x.shape[-2], :] = \
            v.view(torch.int32 if v.dtype == torch.uint32 else v.dtype)


@pytest.fixture()
def cache_on_oracle_ops(monkeypatch):
    from gbx_lm_b200 import cache, ops

    monkeypatch.setattr(ops, "quantize_into", _oracle_quantize_into)
    monkeypatch.setattr(ops, "quantize", _oracle_quantize)
    return cache


def _i32(t):
    return t.view(torch.int32) if t.dtype == torch.uint32 else t


def test_quantized_kv_cache_growth_trim_and_state_with_oracle_ops(cache_on_oracle_ops):
    cache = cache_on_oracle_ops
    B, H, D, gs, bits = 1, 2, 64, 32, 4
    gen = torch.Generator().manual_seed(0)
    c = cache.QuantizedKVCache(group_size=gs, bits=bits)
    ks, vs = [], []

    def feed(n):
        k = torch.randn((B, H, n, D), generator=gen).to(torch.bfloat16)
        v = torch.randn((B, H, n, D), generator=gen).to(torch.bfloat16)
        ks.append(k), vs.append(v)
        return c.update_and_fetch(k, v)

    qk, qv = feed(250)                                   # prompt: one block of 256 positions
    assert c.offset == 250 and c.keys[0].shape == (B, H, 256, D * bits // 32) and c.keys[1].shape == (B, H, 256, D // gs)
    assert qk[0].shape[-2] == 250 and qv[2].shape[-2] == 250
    for _ in range(6):
        feed(1)                                          # decode steps inside the block
    assert c.keys[0].shape[-2] == 256 and c.offset == 256
    qk, qv = feed(1)                                     # crosses the block border: grows by one block
    assert c.keys[0].shape[-2] == 512 and c.offset == 257 and qk[0].shape[-2] == 257
    want = _oracle_quantize(torch.cat(ks, 2), gs, bits)  # quantisation is per position: chunking does not matter
    for got, w in zip(qk, want):
        assert torch.equal(_i32(got), _i32(w))
    want_v = _oracle_quantize(torch.cat(vs, 2), gs, bits)
    assert all(torch.equal(_i32(g), _i32(w)) for g, w in zip(qv, want_v))
    assert (_i32(c.keys[0])[..., 257:, :] == 0).all()    # the tail of the buffers is untouched

    assert c.is_trimmable() and c.trim(7) == 7 and c.offset == 250 and c.trim(1000) == 250 and c.offset == 0
    c.offset = 250
    qk, _ = feed(5)
    assert c.keys[0].shape[-2] == 512 and c.offset == 255  # capacity suffices, nothing is reallocated
    assert c.meta_state == ("256", "255", str(gs), str(bits))
    k_state, v_state = c.state
    assert k_state[0].shape[-2] == 255
    c2 = cache.QuantizedKVCache()
    c2.state = (k_state, v_state)
    c2.meta_state = c.meta_state
    assert (c2.offset, c2.group_size, c2.bits, c2.step) == (255, gs, bits, 256)
    qk2, _ = c2.update_and_fetch(ks[0][:, :, :3], vs[0][:, :, :3])  # state from views: 255 + 3 > 255 -> grows from prev
    assert c2.offset == 258 and c2.keys[0].shape[-2] == 255 + 256 and c2.keys[0].is_contiguous()
    assert torch.equal(_i32(qk2[0])[..., :255, :], _i32(k_state[0]))


def test_quantized_kv_cache_straddling_widths_allocate_the_stream_length_with_oracle_ops(cache_on_oracle_ops):
    cache = cache_on_oracle_ops
    for bits in (3, 6):
        c = cache.QuantizedKVCache(group_size=64, bits=bits)
        k = torch.randn((1, 1, 2, 128)).to(torch.bfloat16)
        qk, _ = c.update_and_fetch(k, k)
        assert qk[0].shape == (1, 1, 2, 128 * bits // 32)
        want = _oracle_quantize(k, 64, bits)
        assert torch.equal(_i32(qk[0]), _i32(want[0]))


def test_kv_cache_to_quantized_and_maybe_quantize_with_oracle_ops(cache_on_oracle_ops):
    cache = cache_on_oracle_ops
    gen = torch.Generator().manual_seed(1)
    caches = [cache.KVCache() for _ in range(2)]
    k = torch.randn((1, 2, 10, 64), generator=gen).to(torch.bfloat16)
    v = torch.randn((1, 2, 10, 64), generator=gen).to(torch.bfloat16)
    for c in caches:
        kk, vv = c.update_and_fetch(k, v)
        assert kk.shape == (1, 2, 10, 64) and c.keys.shape[2] == 256 and torch.equal(kk, k)
    cache.maybe_quantize_kv_cache(caches, quantized_kv_start=10, kv_group_size=64, kv_bits=8)
    assert isinstance(caches[0], cache.KVCache)          # offset 10 is not > 10
    cache.maybe_quantize_kv_cache(caches, quantized_kv_start=0, kv_group_size=64, kv_bits=None)
    assert isinstance(caches[0], cache.KVCache)          # kv_bits None: never
    cache.maybe_quantize_kv_cache(caches, quantized_kv_start=5, kv_group_size=64, kv_bits=8)
    assert all(isinstance(c, cache.QuantizedKVCache) for c in caches)
    q = caches[0]
    assert q.offset == 10 and q.bits == 8 and q.group_size == 64 and q.keys[0].shape == (1, 2, 256, 16)
    want = _oracle_quantize(k, 64, 8)
    assert torch.equal(_i32(q.keys[0])[..., :10, :], _i32(want[0]))
    qk, qv = q.update_and_fetch(k[:, :, :1], v[:, :, :1])  # decode continues in the quantized cache
    assert q.offset == 11 and qk[0].shape[-2] == 11
    d = cache.KVCache()
    d.update_and_fetch(k, v)
    assert d.trim(4) == 4 and d.offset == 6 and d.state[0].shape[2] == 6
    d.update_and_fetch(k[:, :, :300], v[:, :, :300])     # 6 + 10 fits
    assert d.offset == 16
    big = torch.zeros((1, 2, 300, 64), dtype=torch.bfloat16)
    d.update_and_fetch(big, big)                          # 16 + 300 > 256: cut at prev (16 % 256 != 0), add two blocks
    assert d.offset == 316 and d.keys.shape[2] == 16 + 512


def test_cache_and_attention_flow_with_oracle_backed_ops(monkeypatch):
    """The body of the GPU test of the quantized cache + attention (tests/test_gpu_quantize.py) with the three device
    operations replaced by the oracle on the CPU: everything around the kernels -- cache growth across the block border,
    views handed to the attention wrapper, GQA reshapes, softmax, `to_quantized` -- is the code the GPU run executes."""
    from gbx_lm_b200 import ops
    import tests.test_gpu_quantize as T

    def deq(w, s, b, gs, bits):
        d = A.dequantize(w.contiguous().view(torch.int32).numpy().view(np.uint32).reshape(-1, w.shape[-1]),
                         s.float().numpy().reshape(-1, s.shape[-1]), b.float().numpy().reshape(-1, b.shape[-1]), gs, bits, "f32")
        return torch.from_numpy(d).reshape(*w.shape[:-1], -1)

    def qmm(x, w, s, b, transpose=True, group_size=64, bits=4, **kw):
        W = deq(w, s, b, group_size, bits)
        return (x.float() @ (W.transpose(-1, -2) if transpose else W)).to(x.dtype)

    def quantize_into(x, out, offset, group_size, bits):
        assert all(t.is_contiguous() for t in out)       # what gbxq_quantize_rows requires of the cache buffers
        _oracle_quantize_into(x.contiguous(), out, offset, group_size, bits)

    monkeypatch.setattr(ops, "quantize", _oracle_quantize)
    monkeypatch.setattr(ops, "quantize_into", quantize_into)
    monkeypatch.setattr(ops, "quantized_matmul", qmm)
    T.test_quantized_kv_cache_and_attention_on_device(torch.device("cpu"))
