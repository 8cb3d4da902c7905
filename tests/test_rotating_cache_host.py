"""CPU tests of the rotating KV cache (`max_kv_size`): the ring-slot rule and the held-position map against a restatement
of the reference's in-place update, the window visibility rule against a brute-force set, the chunk write set, argument
validation (Python and C ABI), the conversion to the quantized rotating cache with the device quantiser replaced by the
oracle, and the choice of caches in `generate_step`."""
import ctypes
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import mlx_affine as A

SHAPES = [(W, keep) for W in (5, 8, 64) for keep in (0, 1, 4)]


def _reference_rows(W: int, keep: int, n: int):
    """The rows of a RotatingKVCache after n single-token updates, by the reference's bookkeeping
    (RotatingKVCache._update_in_place: write at `_idx`, which wraps to `keep` once it reaches `max_size`), and the row
    each token went to.  rows[s] is the absolute position row s holds (-1: never written)."""
    rows, slots, idx = [-1] * W, [], 0
    for p in range(n):
        if idx == W:
            idx = keep
        rows[idx] = p
        slots.append(idx)
        idx += 1
    return rows, slots


@pytest.mark.parametrize("W,keep", SHAPES)
def test_ring_slot_and_held_positions_match_reference_bookkeeping(W, keep):
    from gbx_lm_b200.cache import StaticRotatingKVCache, ring_slot

    c = StaticRotatingKVCache(1, 1, W, 8, "cpu", keep=keep)
    _, slots = _reference_rows(W, keep, 3 * W)
    assert [ring_slot(p, W, keep) for p in range(3 * W)] == slots
    assert [c.ring_slot(p) for p in range(3 * W)] == slots
    assert ring_slot(torch.arange(3 * W), W, keep).tolist() == slots
    for n in range(3 * W + 1):
        rows, _ = _reference_rows(W, keep, n)
        c.offset = n
        assert c.held_positions().tolist() == rows[:min(n, W)], n
        assert c.attend_len == min(n, W)


@pytest.mark.parametrize("W,keep", SHAPES)
def test_visibility_is_sinks_plus_last_window(W, keep):
    """A query at p sees the sinks and the last W - keep positions: min(p + 1, W) keys, exactly what the ring holds
    once p is written."""
    from gbx_lm_b200.cache import StaticRotatingKVCache

    c = StaticRotatingKVCache(1, 1, W, 8, "cpu", keep=keep)
    keys = torch.arange(4 * W)
    for p in range(3 * W):
        want = set(range(min(keep, p + 1))) | set(range(max(0, p - (W - keep) + 1), p + 1))
        got = set(keys[c.visible(keys, torch.tensor([p]))[0]].tolist())
        assert got == want and len(got) == min(p + 1, W), p
        c.offset = p + 1
        assert set(c.held_positions().tolist()) == want


def _filled(W, keep, off):
    """A float32 rotating cache after `off` tokens, every row's first element = the position it holds."""
    from gbx_lm_b200.cache import StaticRotatingKVCache

    c = StaticRotatingKVCache(1, 2, W, 4, "cpu", keep=keep, dtype=torch.float32)
    rows, _ = _reference_rows(W, keep, off)
    c.keys[..., 0] = torch.tensor(rows, dtype=torch.float32)
    c.values[..., 0] = -torch.tensor(rows, dtype=torch.float32)
    c.offset = off
    return c


@pytest.mark.parametrize("W,keep", SHAPES)
def test_chunk_write_set_matches_token_by_token(W, keep):
    """For chunks of L positions at off: the rows `window_with` hands the attention are the positions `held_positions`
    names, `store_runs` writes no row twice, and after `store` the ring holds what L single-token writes leave."""
    for off in sorted({0, 1, keep, W - 1, W, W + 3, 2 * W + 1}):
        for L in sorted({1, 2, W - keep - 1, W - keep, W, 2 * W + 3} - {0}):
            c = _filled(W, keep, off)
            chunk = torch.arange(off, off + L, dtype=torch.float32)
            k = torch.zeros((1, 2, L, 4))
            k[..., 0] = chunk
            keys, values, key_pos = c.window_with(k, -k, off)
            assert torch.equal(keys[0, 0, :, 0], key_pos.float()) and torch.equal(values, -keys)
            runs = c.store_runs(off, L)
            written = [r for _, n, row in runs for r in range(row, row + n)]
            assert len(written) == len(set(written)) and all(0 <= r < W for r in written), (off, L, runs)
            c.offset = off + L
            c.store(keys, values, off, L)
            rows, _ = _reference_rows(W, keep, off + L)
            assert c.keys[0, 0, :, 0].tolist() == [float(r) for r in rows], (off, L)
            assert torch.equal(c.values, -c.keys)


def test_rotating_cache_validation():
    from gbx_lm_b200 import ops
    from gbx_lm_b200.cache import StaticRotatingKVCache, StaticRotatingQuantizedKVCache

    for cls in (StaticRotatingKVCache, StaticRotatingQuantizedKVCache):
        for W, keep in ((8, 8), (8, 9), (8, -1), (0, 0), (-3, 0), (8, 1.5), (8, None)):
            with pytest.raises(ValueError):
                cls(1, 1, W, 64, "cpu", keep=keep)
        assert cls(1, 1, 8, 64, "cpu", keep=7).keep == 7
    for keep in (8, -1, 2.0, True):
        with pytest.raises(ValueError):
            ops._check_keep(keep, 8, "rope_cache")
    assert ops._check_keep(None, 8, "rope_cache") is None and ops._check_keep(0, 8, "rope_cache") == 0


def test_position_stride_rule():
    """The position of the four decode-step ops: a contiguous int64 [1] (pos_stride 0, shared by the rows) or [B]
    (pos_stride 1) on the device of q; anything else is a ValueError."""
    from gbx_lm_b200 import ops

    q = torch.zeros((3, 8, 64), dtype=torch.bfloat16)
    i64 = lambda *shape: torch.zeros(shape, dtype=torch.int64)  # noqa: E731
    assert ops._pos_stride(i64(1), 3, q, "rope_cache") == 0
    assert ops._pos_stride(i64(3), 3, q, "rope_cache") == 1
    assert ops._pos_stride(i64(1), 1, q[:1], "rope_cache") == 0
    for bad in (i64(2), i64(4), i64(3, 1), i64(), torch.zeros(1, dtype=torch.int32), torch.zeros(3, dtype=torch.int32),
                torch.zeros(3, dtype=torch.float32), i64(6)[::2]):
        with pytest.raises(ValueError, match="rope_cache: position"):
            ops._pos_stride(bad, 3, q, "rope_cache")


def test_keep_abi_validation_without_gpu():
    """The cache writes refuse keep >= max_len with GBXQ_ESHAPE before touching CUDA."""
    from gbx_lm_b200 import _lib

    lib = _lib.get()
    p = ctypes.c_void_p(256)  # never dereferenced: validation fails first
    for stride in (0, 1):  # at B = 1 the shared and the per-row position are the same call
        ring = lambda keep, max_len=64: lib.gbxq_rope_cache(p, p, p, p, stride, p, p, p, 1, 8, 2, 128, max_len, keep,
                                                            None)
        qring = lambda keep, max_len=64, bits=4: lib.gbxq_rope_cache_quantized(
            p, p, p, p, stride, p, p, p, p, p, p, p, 1, 8, 2, 128, max_len, keep, bits, 64, None)
        for f in (ring, qring):
            assert f(64) == -3 and f(100) == -3 and f(0, max_len=0) == -3
        assert qring(4, bits=5) == -1
        assert lib.gbxq_rope_cache(None, p, p, p, stride, p, p, p, 1, 8, 2, 128, 64, 4, None) == -6


def _oracle_quantize(x, group_size, bits):
    q, s, b = A.quantize(x.float().numpy(), group_size, bits, "bf16")
    return (torch.from_numpy(q.view(np.int32)).view(torch.uint32), torch.from_numpy(s).to(x.dtype),
            torch.from_numpy(b).to(x.dtype))


def _i32(t):
    return t.view(torch.int32) if t.dtype == torch.uint32 else t


def test_rotating_to_quantized_and_conversion_rule(monkeypatch):
    from gbx_lm_b200 import cache, ops

    monkeypatch.setattr(ops, "quantize", _oracle_quantize)
    gen = torch.Generator().manual_seed(3)

    def filled(offset):
        cs = [cache.StaticRotatingKVCache(1, 2, 16, 64, "cpu", keep=4) for _ in range(3)]
        for c in cs:
            c.keys.copy_(torch.randn(c.keys.shape, generator=gen).to(torch.bfloat16))
            c.values.copy_(torch.randn(c.values.shape, generator=gen).to(torch.bfloat16))
            c.offset = offset
        return cs

    cs = filled(40)  # wrapped: offset past the window
    q = cs[0].to_quantized(group_size=32, bits=4)
    assert type(q) is cache.StaticRotatingQuantizedKVCache and isinstance(q, cache.StaticQuantizedKVCache)
    assert (q.offset, q.max_len, q.window, q.keep, q.group_size, q.bits, q.attend_len) == (40, 16, 16, 4, 32, 4, 16)
    for got, want in zip(q.keys + q.values, _oracle_quantize(cs[0].keys, 32, 4) + _oracle_quantize(cs[0].values, 32, 4)):
        assert got.shape == want.shape and torch.equal(_i32(got), _i32(want))
    assert torch.equal(q.held_positions(), cs[0].held_positions())

    for start, converts in ((40, False), (39, True), (0, True)):
        cs = filled(40)
        cache.maybe_quantize_kv_cache(cs, quantized_kv_start=start, kv_group_size=64, kv_bits=8)
        want = cache.StaticRotatingQuantizedKVCache if converts else cache.StaticRotatingKVCache
        assert {type(c) for c in cs} == {want}
        assert all(c.keep == 4 and c.offset == 40 and c.max_len == 16 for c in cs)
        if converts:  # a list already quantized is left alone
            first = cs[0]
            cache.maybe_quantize_kv_cache(cs, 0, 64, 4)
            assert cs[0] is first and first.bits == 8


VOCAB = 64


class _StubModel(torch.nn.Module):
    """What the driver needs of `qllama.Model`: the attributes `make_prompt_cache` reads and a forward that advances the
    cache offsets; it records the cache classes it was called with.  Logits pick (last token * 5 + 3) % VOCAB."""

    def __init__(self):
        super().__init__()
        self.args = SimpleNamespace(head_dim=64, hidden_size=128, num_attention_heads=2, num_key_value_heads=2,
                                    num_hidden_layers=2)
        self.tp = SimpleNamespace(world=1)
        self.model = SimpleNamespace(embed_tokens=SimpleNamespace(weight=torch.zeros(1)))
        self.dummy = torch.nn.Parameter(torch.zeros(1), requires_grad=False)
        self.seen = []

    def forward(self, inputs, cache, positions=None, attend_len=None):
        B, L = inputs.shape
        off = cache[0].offset
        self.seen.append((type(cache[0]).__name__, cache[0].max_len, cache[0].keep))
        for c in cache:
            c.offset = off + L
        logits = torch.zeros((B, L, VOCAB))
        logits[0, torch.arange(L), (inputs[0] * 5 + 3) % VOCAB] = 1.0
        return logits


@pytest.mark.parametrize("max_kv_size,kv_bits", [(None, None), (16, None), (16, 4), (None, 8), (200, None)])
def test_generate_step_builds_rotating_caches_only_with_max_kv_size(monkeypatch, max_kv_size, kv_bits):
    from gbx_lm_b200 import ops, utils
    from gbx_lm_b200.cache import DEFAULT_KV_KEEP

    monkeypatch.setattr(ops, "quantize", _oracle_quantize)
    prompt = torch.randint(0, VOCAB, (12,), generator=torch.Generator().manual_seed(7))
    model = _StubModel()
    toks = [t for t, _ in utils.generate_step(prompt, model, max_tokens=30, use_cuda_graph=False, prefill_step_size=5,
                                              max_kv_size=max_kv_size, kv_bits=kv_bits, quantized_kv_start=20)]
    want = [(int(prompt[-1]) * 5 + 3) % VOCAB]
    while len(want) < 30:
        want.append((want[-1] * 5 + 3) % VOCAB)
    assert toks == want
    if max_kv_size is None:
        assert {(n, k) for n, _, k in model.seen} <= {("StaticKVCache", None), ("StaticQuantizedKVCache", None)}
        assert {m for _, m, _ in model.seen} == {12 + 30 + 1}
    else:
        assert {(m, k) for _, m, k in model.seen} == {(max_kv_size, DEFAULT_KV_KEEP)}
        assert {n for n, _, _ in model.seen} <= {"StaticRotatingKVCache", "StaticRotatingQuantizedKVCache"}
    assert ("Quantized" in model.seen[-1][0]) == (kv_bits is not None)
