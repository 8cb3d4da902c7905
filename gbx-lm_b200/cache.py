"""Every KV cache of the package, in two families.

The growable caches mirror the reference's `KVCache` (gbx_lm/models/cache.py:216-266) and `QuantizedKVCache`
(cache.py:133-213): attributes `keys`, `values`, `offset`, `step`, (`group_size`, `bits`), methods `update_and_fetch`,
`state`, `meta_state`, `trim`, `is_trimmable`, `to_quantized`, and the same growth rule, so that a caller written
against the reference (`maybe_quantize_kv_cache`, gbx_lm/utils.py:204-214; the attention layers) runs unchanged.
Built differently underneath: both are one block-grown store (`_BlockStore`), tuples of position-major CUDA buffers
`[B, H, capacity, width]` that share `offset`; the dense cache holds one buffer per side, the quantized one three
(codes, scales, biases).  What the reference does with `mx.quantize` followed by three slice assignments per side
(cache.py:176-180) is ONE `gbxq_quantize_rows` launch per side that writes codes and statistics at the offset
(`ops.quantize_into`); `to_quantized` (cache.py:251-263) is `gbxq_quantize` over the buffers.  The consumer is
`switch_layers.quantized_scaled_dot_product_attention` (gbx_lm/models/base.py:65-98).

The static caches, `StaticKVCache` and `StaticQuantizedKVCache`, are what `qllama.Model` reads and writes: allocated
once for `max_len` positions, so that the decode step is CUDA-graph capturable, in the same layouts.
`StaticRotatingKVCache` and `StaticRotatingQuantizedKVCache` are their rotating forms (the reference's RotatingKVCache,
`max_kv_size`): a window of `max_len` rows with `keep` sinks, written as a ring (`ring_slot`, `_Ring`).  The conversion
rule `maybe_quantize_kv_cache` decides for both families.  CUDA only, like everything in this package."""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence, Tuple

import torch

from . import ops

QTensor = Tuple[torch.Tensor, torch.Tensor, torch.Tensor]
Bufs = Tuple[torch.Tensor, ...]


def _zeros(shape, dtype: torch.dtype, device) -> torch.Tensor:
    # uint32 has few torch kernels: codes are allocated / concatenated as int32 and viewed
    if dtype == torch.uint32:
        return torch.zeros(shape, dtype=torch.int32, device=device).view(torch.uint32)
    return torch.zeros(shape, dtype=dtype, device=device)


def _cat_positions(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    if a.dtype == torch.uint32:
        return torch.cat([a.view(torch.int32), b.view(torch.int32)], dim=-2).view(torch.uint32)
    return torch.cat([a, b], dim=-2)


def _zero_triple(lead, n: int, head_dim: int, group_size: int, bits: int, dtype: torch.dtype, device) -> QTensor:
    """n zeroed positions of a quantized side: codes uint32 [*lead, n, D*bits/32], scales / biases [*lead, n, D/group_size].
    D * bits / 32 words per position: the reference's D // (32 // bits) (cache.py:150,156) is the same for 2/4/8-bit and
    mis-sized for the straddling 3-/6-bit packings (32 // 3 = 10)."""
    return (_zeros((*lead, n, head_dim * bits // 32), torch.uint32, device),
            _zeros((*lead, n, head_dim // group_size), dtype, device),
            _zeros((*lead, n, head_dim // group_size), dtype, device))


class _BlockStore:
    """`offset` valid positions in buffers that grow by whole blocks of `step` positions.

    Growth rule (the reference's, cache.py:145-171 / 224-239, kept because `state` exposes the capacity): when the new
    positions do not fit, ceil(new / step) blocks are appended -- after cutting the buffers back to `offset` if that is
    not a block border."""

    def __init__(self):
        self.offset = 0
        self.step = 256

    @staticmethod
    def _capacity(bufs: Optional[Bufs]) -> int:
        return 0 if bufs is None else bufs[0].shape[-2]

    def _make_room(self, sides: Sequence[Optional[Bufs]], new: int, fresh: Callable[[int], Sequence[Bufs]]):
        """The sides (tuples of buffers) with room for `new` more positions; `fresh(n)` allocates n zeroed positions
        of every buffer of every side."""
        if sides[0] is not None and self.offset + new <= self._capacity(sides[0]):
            return list(sides)
        blocks = -(-new // self.step) * self.step
        grown = []
        for old, add in zip(sides, fresh(blocks)):
            if old is None:
                grown.append(tuple(add))
                continue
            cut = self.offset if self.offset % self.step else self._capacity(old)
            grown.append(tuple(_cat_positions(o[..., :cut, :], a) for o, a in zip(old, add)))
        return grown

    def _valid(self, bufs: Bufs) -> Bufs:
        return tuple(t[..., : self.offset, :] for t in bufs)

    def is_trimmable(self) -> bool:
        return True

    def trim(self, n: int) -> int:
        n = min(self.offset, n)
        self.offset -= n
        return n


class QuantizedKVCache(_BlockStore):
    """cache.py:133-213.  `keys` / `values` are (codes uint32 [B, H, capacity, D*bits/32], scales, biases [B, H,
    capacity, D/group_size]) triples; `update_and_fetch` returns views of the first `offset` positions."""

    def __init__(self, group_size: int = 64, bits: int = 8):
        super().__init__()
        self.keys: Optional[QTensor] = None
        self.values: Optional[QTensor] = None
        self.group_size = group_size
        self.bits = bits

    def _fresh(self, lead, dims, like: torch.Tensor):
        return lambda n: [_zero_triple(lead, n, d, self.group_size, self.bits, like.dtype, like.device) for d in dims]

    def update_and_fetch(self, keys: torch.Tensor, values: torch.Tensor) -> Tuple[QTensor, QTensor]:
        new = keys.shape[-2]
        k_side, v_side = self._make_room((self.keys, self.values), new,
                                         self._fresh(keys.shape[:-2], (keys.shape[-1], values.shape[-1]), keys))
        # the kernel writes into the buffers in place: they must be dense (a `state` set from views is not)
        self.keys = tuple(t if t.is_contiguous() else t.contiguous() for t in k_side)
        self.values = tuple(t if t.is_contiguous() else t.contiguous() for t in v_side)
        at = self.offset
        self.offset = at + new
        ops.quantize_into(keys, self.keys, at, self.group_size, self.bits)
        ops.quantize_into(values, self.values, at, self.group_size, self.bits)
        return self._valid(self.keys), self._valid(self.values)

    @property
    def state(self):
        if self.offset == self._capacity(self.keys):
            return self.keys, self.values
        return self._valid(self.keys), self._valid(self.values)

    @state.setter
    def state(self, v):
        self.keys, self.values = v

    @property
    def meta_state(self):
        return tuple(str(v) for v in (self.step, self.offset, self.group_size, self.bits))

    @meta_state.setter
    def meta_state(self, v):
        self.step, self.offset, self.group_size, self.bits = (int(s) for s in v)


class KVCache(_BlockStore):
    """cache.py:216-266: the dense cache a prompt is processed into before `to_quantized`."""

    def __init__(self):
        super().__init__()
        self.keys: Optional[torch.Tensor] = None
        self.values: Optional[torch.Tensor] = None

    def update_and_fetch(self, keys: torch.Tensor, values: torch.Tensor):
        new = keys.shape[-2]

        def fresh(n: int):
            return [(_zeros((*t.shape[:-2], n, t.shape[-1]), t.dtype, t.device),) for t in (keys, values)]

        sides = self._make_room([None if t is None else (t,) for t in (self.keys, self.values)], new, fresh)
        self.keys, self.values = sides[0][0], sides[1][0]
        at = self.offset
        self.offset = at + new
        self.keys[..., at: self.offset, :] = keys
        self.values[..., at: self.offset, :] = values
        return self._valid((self.keys, self.values))

    @property
    def state(self):
        if self.offset == self.keys.shape[-2]:
            return self.keys, self.values
        return self._valid((self.keys, self.values))

    @state.setter
    def state(self, v):
        self.keys, self.values = v
        self.offset = self.keys.shape[-2]

    def to_quantized(self, group_size: int = 64, bits: int = 4) -> QuantizedKVCache:
        """The whole buffers are quantized (unused positions are zero groups), `offset` carries over."""
        q = QuantizedKVCache(group_size=group_size, bits=bits)
        q.offset = self.offset
        if self.keys is not None:
            q.keys = ops.quantize(self.keys, group_size, bits)
            q.values = ops.quantize(self.values, group_size, bits)
        return q


# The most keys gbxq_decode_attention attends: its kernel holds one float of shared memory per visible key
# (gbxq_glue.cu, launch_decode_attention).  A longer bf16 cache takes the unfused decode path.
DECODE_ATTENTION_MAX_KEYS = 49152


class StaticKVCache:
    """Static pre-allocated KV cache [B, n_kv, max_len, D] (the reference grows in steps of 256,
    models/cache.py:215-277; a static buffer keeps the decode step CUDA-graph capturable).  `offset` is the host-side
    count of valid positions (eager mode)."""

    keep: Optional[int] = None  # sink rows of a rotating cache; None: a flat cache, position p in row p

    def __init__(self, batch: int, n_kv: int, max_len: int, head_dim: int, device, dtype=torch.bfloat16):
        self.keys = torch.zeros((batch, n_kv, max_len, head_dim), device=device, dtype=dtype)
        self.values = torch.zeros((batch, n_kv, max_len, head_dim), device=device, dtype=dtype)
        self.max_len = max_len
        self.offset = 0

    @property
    def device(self) -> torch.device:
        return self.keys.device

    @property
    def attend_len(self) -> int:
        """Rows a model call attends once `offset` counts its positions."""
        return self.offset

    def fused_decode_fits(self, head_dim: int, n_heads: int, n_kv_heads: int) -> bool:
        """Shapes gbxq_rope_cache + gbxq_decode_attention serve (include/gbxq.h)."""
        return head_dim in (64, 128) and self.max_len <= DECODE_ATTENTION_MAX_KEYS

    def update(self, k: torch.Tensor, v: torch.Tensor, positions: torch.Tensor):
        """k / v [B, n_kv, L, D] at positions int64 [L] shared by the rows, or at per-row positions [B, L]."""
        if positions.dim() == 2:
            rows = torch.arange(k.shape[0], device=k.device)[:, None]
            self.keys[rows, :, positions] = k.transpose(1, 2)  # the indexed view is [B, L, n_kv, D]
            self.values[rows, :, positions] = v.transpose(1, 2)
            return
        self.keys.index_copy_(2, positions, k)
        self.values.index_copy_(2, positions, v)

    # the reference's interface: `trim(n)` moves `offset` back by n positions.  The rows past it are dead -- every later
    # call writes a position before any query can see it
    is_trimmable = _BlockStore.is_trimmable
    trim = _BlockStore.trim

    def to_quantized(self, group_size: int = 64, bits: int = 4) -> "StaticQuantizedKVCache":
        """The static quantized cache holding these positions (as `KVCache.to_quantized`): the whole buffers are
        quantized, unused zero rows become zero groups, `offset` carries over."""
        q = StaticQuantizedKVCache.__new__(StaticQuantizedKVCache)
        q.keys = tuple(ops.quantize(self.keys, group_size, bits))
        q.values = tuple(ops.quantize(self.values, group_size, bits))
        q.max_len, q.offset, q.group_size, q.bits = self.max_len, self.offset, group_size, bits
        return q


class StaticQuantizedKVCache:
    """Static pre-allocated group-quantized KV cache: the counterpart of `StaticKVCache` in the layout of
    `QuantizedKVCache` -- `keys` / `values` are (codes uint32 [B, n_kv, max_len, D*bits/32], scales, biases
    [B, n_kv, max_len, D/group_size]) triples, with `offset`, `group_size` and `bits`.  The decode step writes and
    reads it with gbxq_rope_cache_quantized / gbxq_decode_attention_quantized."""

    keep: Optional[int] = None  # as StaticKVCache.keep

    def __init__(self, batch: int, n_kv: int, max_len: int, head_dim: int, device, group_size: int = 64, bits: int = 8,
                 dtype=torch.bfloat16):
        if bits not in (2, 3, 4, 6, 8) or group_size not in (32, 64, 128) or head_dim % group_size or head_dim % 32:
            raise ValueError(f"StaticQuantizedKVCache: bits {bits} / group_size {group_size} do not fit head_dim {head_dim}")
        self.keys, self.values = (_zero_triple((batch, n_kv), max_len, head_dim, group_size, bits, dtype, device)
                                  for _ in range(2))
        self.max_len = max_len
        self.offset = 0
        self.group_size, self.bits = group_size, bits

    @property
    def device(self) -> torch.device:
        return self.keys[0].device

    @property
    def attend_len(self) -> int:
        """Rows a model call attends once `offset` counts its positions."""
        return self.offset

    def fused_decode_fits(self, head_dim: int, n_heads: int, n_kv_heads: int) -> bool:
        """Shapes gbxq_rope_cache_quantized + gbxq_decode_attention_quantized serve (include/gbxq.h)."""
        return (head_dim in (64, 128) and self.group_size <= head_dim
                and n_heads % n_kv_heads == 0 and n_heads // n_kv_heads <= 8)

    def update(self, k: torch.Tensor, v: torch.Tensor, at: int):
        """k / v [B, n_kv, L, D] quantized into positions [at, at + L) (ops.quantize_into, one launch per side)."""
        ops.quantize_into(k, self.keys, at, self.group_size, self.bits)
        ops.quantize_into(v, self.values, at, self.group_size, self.bits)

    def update_row(self, b: int, k: torch.Tensor, v: torch.Tensor, at: int):
        """`update` of batch row b alone: k / v [1, n_kv, L, D] into that row's positions [at, at + L)."""
        ops.quantize_into(k, tuple(t[b:b + 1] for t in self.keys), at, self.group_size, self.bits)
        ops.quantize_into(v, tuple(t[b:b + 1] for t in self.values), at, self.group_size, self.bits)

    def prefix(self, n: int):
        return tuple(t[:, :, :n] for t in self.keys), tuple(t[:, :, :n] for t in self.values)

    is_trimmable = _BlockStore.is_trimmable  # as StaticKVCache
    trim = _BlockStore.trim


# The sink count of the reference's rotating caches: generate_step builds them through make_prompt_cache, which passes
# keep=4 (gbx_lm/models/cache.py:280-420, RotatingKVCache; SURVEY.md section 2 row 5).
DEFAULT_KV_KEEP = 4


def ring_slot(p, window: int, keep: int):
    """Row of a rotating cache (`window` rows, the first `keep` of them sinks) that holds absolute position p (an int or
    an int64 tensor of positions):

        ring_slot(p) = p                                       if p < window
                     = keep + (p - keep) mod (window - keep)   otherwise

    -- where the reference's in-place update puts a token (RotatingKVCache._update_in_place: the write index wraps to
    `keep` at `max_size`).  The device computes the same rule (kv_cache_row, gbxq_common.cuh)."""
    if isinstance(p, torch.Tensor):
        return torch.where(p < window, p, keep + (p - keep) % (window - keep))
    return p if p < window else keep + (p - keep) % (window - keep)


class _Ring:
    """What the two rotating caches add to their flat bases.  The buffers hold `window` = `max_len` rows for good;
    `offset` counts every position processed (absolute, as the reference's `offset`).  Position p lives in row
    ring_slot(p), and a query at position p sees key position j iff

        j <= p  and  (j < keep  or  j > p - (window - keep))

    -- the sinks and the last window - keep positions: min(p + 1, window) keys, the set a reference decode step sees.

    A decode step writes its row on the device (the `keep` argument of gbxq_rope_cache) and attends the first
    `attend_len` rows, which are exactly the ring's contents in some order.  A call of L positions at off .. off + L - 1 that takes the ring past its
    window (`wraps`) attends `window_with` (the valid rows plus its own keys) under `visible`, then `store`s the
    positions that survive it."""

    def _set_ring(self, window: int, keep: int):
        if isinstance(window, bool) or not isinstance(window, int) or window < 1:
            raise ValueError(f"rotating KV cache: window must be an int >= 1, got {window!r}")
        if isinstance(keep, bool) or not isinstance(keep, int) or not 0 <= keep < window:
            raise ValueError(f"rotating KV cache: keep must be an int in [0, window = {window}), got {keep!r}")
        self.keep = keep

    @property
    def window(self) -> int:
        return self.max_len

    @property
    def attend_len(self) -> int:
        return min(self.offset, self.max_len)

    def ring_slot(self, p):
        return ring_slot(p, self.max_len, self.keep)

    def held_positions(self, offset: Optional[int] = None) -> torch.Tensor:
        """int64 [min(offset, window)] on the cache's device: the absolute position in each valid row after `offset`
        positions (default: the cache's).  Row s >= keep of a wrapped ring holds last - ((last - s) mod (window - keep)),
        last = offset - 1."""
        offset = self.offset if offset is None else offset
        s = torch.arange(min(offset, self.max_len), device=self.device)
        if offset <= self.max_len:
            return s
        last = offset - 1
        return torch.where(s < self.keep, s, last - (last - s) % (self.max_len - self.keep))

    def visible(self, key_positions: torch.Tensor, positions: torch.Tensor) -> torch.Tensor:
        """bool [L, T]: whether the query at positions[i] sees the key at key_positions[j]."""
        j, p = key_positions[None, :], positions[:, None]
        return (j <= p) & ((j < self.keep) | (j > p - (self.max_len - self.keep)))

    def is_trimmable(self) -> bool:
        """False: a ring that has wrapped has overwritten the rows a rewind would expose (the reference refuses it too)."""
        return False

    def trim(self, n: int) -> int:
        raise ValueError("a rotating KV cache cannot be rewound")

    def wraps(self) -> bool:
        """Whether the model call that has just advanced `offset` past its positions reaches beyond the window."""
        return self.offset > self.max_len

    def store_runs(self, off: int, L: int) -> List[Tuple[int, int, int]]:
        """(first chunk index, count, first row) of each contiguous run of the chunk at off .. off + L - 1 that survives
        it: the positions p < keep and p >= off + L - (window - keep), each to ring_slot(p).  At most three runs (the
        sinks, then the ring part, split where it wraps); no row is written twice."""
        end, runs = off + L, []
        if off < self.keep:
            runs.append((0, min(end, self.keep) - off, off))
        p = max(off, self.keep, end - (self.max_len - self.keep))
        while p < end:
            row = self.ring_slot(p)
            n = min(end - p, self.max_len - row)
            runs.append((p - off, n, row))
            p += n
        return runs


class StaticRotatingKVCache(_Ring, StaticKVCache):
    """`StaticKVCache` as a rotating window of `window` positions with `keep` sinks (the reference's RotatingKVCache,
    gbx_lm/models/cache.py:280-420, as a static buffer; the rule is `_Ring`'s)."""

    def __init__(self, batch: int, n_kv: int, window: int, head_dim: int, device, keep: int = DEFAULT_KV_KEEP,
                 dtype=torch.bfloat16):
        self._set_ring(window, keep)
        super().__init__(batch, n_kv, window, head_dim, device, dtype)

    def window_with(self, k: torch.Tensor, v: torch.Tensor, off: int):
        """(keys, values, key positions): the valid rows before the chunk k / v [B, n_kv, L, D] at `off`, then the chunk."""
        n = min(off, self.max_len)
        pos = torch.arange(off, off + k.shape[-2], device=self.device)
        return (torch.cat([self.keys[:, :, :n], k], 2), torch.cat([self.values[:, :, :n], v], 2),
                torch.cat([self.held_positions(off), pos]))

    def store(self, keys: torch.Tensor, values: torch.Tensor, off: int, L: int):
        """The surviving positions of the chunk (the last L rows of `keys` / `values`) into their rows."""
        base = keys.shape[-2] - L
        for i, n, row in self.store_runs(off, L):
            self.keys[:, :, row:row + n] = keys[:, :, base + i:base + i + n]
            self.values[:, :, row:row + n] = values[:, :, base + i:base + i + n]

    def to_quantized(self, group_size: int = 64, bits: int = 4) -> "StaticRotatingQuantizedKVCache":
        """As `StaticKVCache.to_quantized`; rows, `keep` and `offset` carry over."""
        q = StaticRotatingQuantizedKVCache.__new__(StaticRotatingQuantizedKVCache)
        q.keys = tuple(ops.quantize(self.keys, group_size, bits))
        q.values = tuple(ops.quantize(self.values, group_size, bits))
        q.max_len, q.offset, q.group_size, q.bits, q.keep = self.max_len, self.offset, group_size, bits, self.keep
        return q


class StaticRotatingQuantizedKVCache(_Ring, StaticQuantizedKVCache):
    """`StaticQuantizedKVCache` as a rotating window (the rule is `_Ring`'s).  The reference raises NotImplementedError
    for a quantized rotating cache; here `kv_bits` and `max_kv_size` compose (DESIGN.md section 7)."""

    def __init__(self, batch: int, n_kv: int, window: int, head_dim: int, device, keep: int = DEFAULT_KV_KEEP,
                 group_size: int = 64, bits: int = 8, dtype=torch.bfloat16):
        self._set_ring(window, keep)
        super().__init__(batch, n_kv, window, head_dim, device, group_size, bits, dtype)

    def window_with(self, k: torch.Tensor, v: torch.Tensor, off: int):
        """As `StaticRotatingKVCache.window_with` on triples: the chunk is quantized first (ops.quantize)."""
        n = min(off, self.max_len)
        pos = torch.arange(off, off + k.shape[-2], device=self.device)
        kq, vq = ops.quantize(k, self.group_size, self.bits), ops.quantize(v, self.group_size, self.bits)
        return (tuple(_cat_positions(t[:, :, :n], c) for t, c in zip(self.keys, kq)),
                tuple(_cat_positions(t[:, :, :n], c) for t, c in zip(self.values, vq)),
                torch.cat([self.held_positions(off), pos]))

    def store(self, keys, values, off: int, L: int):
        """The surviving rows of the already quantized chunk (the last L rows of each triple) copied into their rows."""
        base = keys[0].shape[-2] - L
        for i, n, row in self.store_runs(off, L):
            for dst, src in zip(self.keys + self.values, tuple(keys) + tuple(values)):
                _rows(dst)[:, :, row:row + n] = _rows(src)[:, :, base + i:base + i + n]


def _rows(t: torch.Tensor) -> torch.Tensor:
    # uint32 codes have no copy kernel of their own: copied as int32
    return t.view(torch.int32) if t.dtype == torch.uint32 else t


def maybe_quantize_kv_cache(prompt_cache: list, quantized_kv_start: int, kv_group_size: int, kv_bits: Optional[int]) -> None:
    """gbx_lm/utils.py:204-214: once the prompt is longer than `quantized_kv_start`, every dense cache of the list is
    replaced by its quantized form (the list is edited in place; a list that already starts quantized is left alone).
    The same rule decides for the growable and for the static caches."""
    if (kv_bits is None or isinstance(prompt_cache[0], (QuantizedKVCache, StaticQuantizedKVCache))
            or prompt_cache[0].offset <= quantized_kv_start):
        return
    prompt_cache[:] = [c.to_quantized(group_size=kv_group_size, bits=kv_bits) if isinstance(c, (KVCache, StaticKVCache))
                       else c for c in prompt_cache]


def can_trim_prompt_cache(cache: list) -> bool:
    """gbx_lm/models/cache.py: whether every cache of the list can be rewound."""
    return all(c.is_trimmable() for c in cache)


def trim_prompt_cache(cache: list, num_tokens: int) -> int:
    """gbx_lm/models/cache.py: moves every cache of the list back by num_tokens positions; returns how many positions
    were trimmed (0 when the list cannot be rewound)."""
    if not cache or not can_trim_prompt_cache(cache):
        return 0
    return [c.trim(num_tokens) for c in cache][0]
