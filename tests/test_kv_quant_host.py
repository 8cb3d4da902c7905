"""CPU tests of the quantized-KV decode path: the C-level argument validation of gbxq_rope_cache_quantized /
gbxq_decode_attention_quantized and the workspace query (no GPU needed: validation fails before any CUDA call), the
argument checks of the Python ops, the static caches of cache.py and their conversion rule, with the device quantiser
stubbed by the oracle."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import mlx_affine as A


def _rope_q(lib, stride=0, **kw):
    p = ctypes.c_void_p(256)  # never dereferenced: validation fails first
    a = dict(B=1, Hq=8, Hkv=2, D=128, max_len=64, bits=4, gs=64)
    a.update(kw)
    return lib.gbxq_rope_cache_quantized(p, p, p, p, stride, p, p, p, p, p, p, p, a["B"], a["Hq"], a["Hkv"], a["D"],
                                         a["max_len"], -1, a["bits"], a["gs"], None)


def _attn_q(lib, stride=0, ws=None, ws_bytes=1 << 30, **kw):
    p = ctypes.c_void_p(256)
    a = dict(B=1, Hq=8, Hkv=2, D=128, max_len=64, attend_len=64, bits=4, gs=64)
    a.update(kw)
    return lib.gbxq_decode_attention_quantized(p, p, p, p, p, p, p, p, stride, p, a["B"], a["Hq"], a["Hkv"], a["D"],
                                               a["max_len"], a["attend_len"], 0.1, a["bits"], a["gs"],
                                               ws if ws is not None else p, ws_bytes, None)


def test_quantized_decode_abi_validation_at_both_strides_without_gpu():
    from gbx_lm_b200 import _lib

    lib = _lib.get()
    for s in (0, 1):  # at B = 1 the shared and the per-row position are the same call
        for f in (_rope_q, _attn_q):
            assert f(lib, s, bits=5) == -1 and f(lib, s, bits=1) == -1 and f(lib, s, bits=16) == -1
            assert f(lib, s, gs=16) == -2 and f(lib, s, gs=256) == -2
            assert f(lib, s, D=64, gs=128) == -9                # group larger than the head
            assert f(lib, s, D=96, gs=32) == -9 and f(lib, s, D=256) == -9
            assert f(lib, s, Hq=6, Hkv=4) == -3                 # Hq % Hkv
            assert f(lib, s, Hq=32, Hkv=2) == -9                # GQA ratio above 8
            assert f(lib, s, B=0) == -3 and f(lib, s, Hkv=0) == -3 and f(lib, s, max_len=0) == -3
        assert _attn_q(lib, s, attend_len=0) == -3 and _attn_q(lib, s, attend_len=65) == -3
        assert _attn_q(lib, s, ws_bytes=16) == -8               # workspace too small
        assert _attn_q(lib, s, ws=ctypes.c_void_p(264)) == -5   # workspace not 16-byte aligned
        assert lib.gbxq_decode_attention_quantized(None, None, None, None, None, None, None, None, s, None, 1, 8, 2, 128,
                                                   64, 64, 0.1, 4, 64, None, 0, None) == -6


def test_quantized_decode_workspace_query():
    from gbx_lm_b200 import _lib

    w = _lib.get().gbxq_decode_attention_quantized_workspace_bytes
    # partials of 256-key chunks: (max, sum, o[D]) fp32 per (batch, query head, chunk)
    assert w(1, 32, 8, 128, 1) == 32 * 1 * 130 * 4
    assert w(1, 32, 8, 128, 256) == w(1, 32, 8, 128, 1)
    assert w(1, 32, 8, 128, 257) == 32 * 2 * 130 * 4
    assert w(2, 8, 2, 64, 70000) == 2 * 8 * 274 * 66 * 4
    assert w(1, 6, 4, 128, 64) == 0 and w(1, 8, 2, 96, 64) == 0 and w(1, 8, 2, 128, 0) == 0


def _triple(b, h, n, d, bits, gs, device="cpu", codes_dtype=torch.uint32):
    return (torch.zeros((b, h, n, d * bits // 32), dtype=torch.int32, device=device).view(codes_dtype),
            torch.zeros((b, h, n, d // gs), dtype=torch.bfloat16, device=device),
            torch.zeros((b, h, n, d // gs), dtype=torch.bfloat16, device=device))


def test_quantized_ops_refuse_cpu_tensors_and_bad_triples():
    from gbx_lm_b200 import ops

    q = torch.zeros((1, 8, 128), dtype=torch.bfloat16)
    kv = torch.zeros((1, 2, 128), dtype=torch.bfloat16)
    pos = torch.zeros((1,), dtype=torch.int64)
    inv = torch.zeros((64,), dtype=torch.float32)
    k3, v3 = _triple(1, 2, 32, 128, 4, 64), _triple(1, 2, 32, 128, 4, 64)
    with pytest.raises(ValueError):
        ops.rope_cache_quantized(q, kv, kv, pos, inv, k3, v3, 64, 4)       # CPU tensors: no CPU path
    with pytest.raises(ValueError):
        ops.decode_attention_quantized(q, k3, v3, pos, 0.1, 64, 4)
    # the shape checks themselves, on any device
    chk = ops._check_qcache
    with pytest.raises(ValueError):
        chk(q, k3, v3, 64, 5)
    with pytest.raises(ValueError):
        chk(q, k3, v3, 48, 4)
    with pytest.raises(ValueError):
        chk(q, _triple(1, 2, 32, 128, 8, 64), v3, 64, 4)                  # codes of another width
    with pytest.raises(ValueError):
        chk(q, k3, _triple(1, 2, 32, 128, 4, 32), 64, 4)                  # statistics of another group size
    with pytest.raises(ValueError):
        chk(q, k3[:2], v3, 64, 4)                                         # not a triple


def test_static_quantized_kv_cache_shapes():
    from gbx_lm_b200.cache import StaticQuantizedKVCache

    for bits in (2, 3, 4, 6, 8):
        for d, gss in ((64, (32, 64)), (128, (32, 64, 128))):
            for gs in gss:
                c = StaticQuantizedKVCache(2, 3, 40, d, "cpu", group_size=gs, bits=bits)
                for side in (c.keys, c.values):
                    assert side[0].shape == (2, 3, 40, d * bits // 32) and side[0].dtype == torch.uint32
                    assert side[1].shape == side[2].shape == (2, 3, 40, d // gs) and side[1].dtype == torch.bfloat16
                assert (c.offset, c.group_size, c.bits, c.max_len) == (0, gs, bits, 40)
    assert StaticQuantizedKVCache(1, 1, 8, 128, "cpu", 64, 3).keys[0].shape[-1] == 12   # 3-bit: 128 * 3 / 32 words
    assert StaticQuantizedKVCache(1, 1, 8, 64, "cpu", 32, 6).keys[0].shape[-1] == 12    # 6-bit: 64 * 6 / 32 words
    with pytest.raises(ValueError):
        StaticQuantizedKVCache(1, 1, 8, 64, "cpu", group_size=128, bits=4)


def _oracle_quantize(x, group_size, bits):
    q, s, b = A.quantize(x.float().numpy(), group_size, bits, "bf16")
    return (torch.from_numpy(q.view(np.int32)).view(torch.uint32), torch.from_numpy(s).to(x.dtype),
            torch.from_numpy(b).to(x.dtype))


def _i32(t):
    return t.view(torch.int32) if t.dtype == torch.uint32 else t


def test_static_kv_cache_to_quantized_and_conversion_rule(monkeypatch):
    from gbx_lm_b200 import cache, ops

    monkeypatch.setattr(ops, "quantize", _oracle_quantize)
    gen = torch.Generator().manual_seed(3)

    def filled(n):
        cs = [cache.StaticKVCache(1, 2, 32, 64, "cpu") for _ in range(3)]
        for c in cs:
            c.keys[:, :, :n] = torch.randn((1, 2, n, 64), generator=gen).to(torch.bfloat16)
            c.values[:, :, :n] = torch.randn((1, 2, n, 64), generator=gen).to(torch.bfloat16)
            c.offset = n
        return cs

    cs = filled(10)
    q = cs[0].to_quantized(group_size=32, bits=4)
    assert isinstance(q, cache.StaticQuantizedKVCache) and (q.offset, q.max_len, q.group_size, q.bits) == (10, 32, 32, 4)
    for got, want in zip(q.keys + q.values, _oracle_quantize(cs[0].keys, 32, 4) + _oracle_quantize(cs[0].values, 32, 4)):
        assert got.shape == want.shape and torch.equal(_i32(got), _i32(want))
    assert (_i32(q.keys[0])[:, :, 10:] == 0).all() and (q.keys[2][:, :, 10:] == 0).all()  # unused rows: zero groups

    # the reference's rule: convert exactly when offset > quantized_kv_start, never with kv_bits=None
    for start, kv_bits, converts in ((10, 8, False), (9, 8, True), (0, 8, True), (0, None, False), (100, 4, False)):
        cs = filled(10)
        cache.maybe_quantize_kv_cache(cs, quantized_kv_start=start, kv_group_size=64, kv_bits=kv_bits)
        kinds = {type(c) for c in cs}
        assert kinds == ({cache.StaticQuantizedKVCache} if converts else {cache.StaticKVCache}), (start, kv_bits)
        if converts:
            assert all(c.bits == kv_bits and c.group_size == 64 and c.offset == 10 for c in cs)
    # a list that is already quantized is left alone
    cs = filled(10)
    cache.maybe_quantize_kv_cache(cs, 0, 64, 8)
    first = cs[0]
    cache.maybe_quantize_kv_cache(cs, 0, 64, 4)
    assert cs[0] is first and cs[0].bits == 8

    # the cache.py caches keep their behaviour
    d = [cache.KVCache() for _ in range(2)]
    k = torch.randn((1, 2, 10, 64), generator=gen).to(torch.bfloat16)
    for c in d:
        c.update_and_fetch(k, k)
    cache.maybe_quantize_kv_cache(d, quantized_kv_start=10, kv_group_size=64, kv_bits=8)
    assert all(isinstance(c, cache.KVCache) for c in d)
    cache.maybe_quantize_kv_cache(d, quantized_kv_start=9, kv_group_size=64, kv_bits=8)
    assert all(isinstance(c, cache.QuantizedKVCache) for c in d)
