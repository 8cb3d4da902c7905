"""Llama / Mistral decoder built from `QuantizedLinear` -- the CALLERS of the hot path
(reference: gbx_lm/models/qllama.py:39-209).  Same module tree and parameter names as the
reference so a gba2mlx checkpoint loads by key:

    model.embed_tokens.weight, model.layers.N.{input,post_attention}_layernorm.weight,
    model.layers.N.self_attn.{q,k,v,o}_proj.{qweight,scales,zeros[,bias]},
    model.layers.N.mlp.{gate,up,down}_proj.{qweight,scales,zeros}, model.norm.weight, lm_head.weight

Attention / RoPE / RMSNorm are glue (SURVEY.md section 2.1 row 5) written with PyTorch ops; at DECODE (one new token,
cache present) the glue of a block runs as four libgbxq launches instead (SURVEY.md 8f rank 2: rope + cache write,
one-query attention, residual add + RMSNorm, silu * up).  The seven projections per block go through libgbxq.  Tensor parallelism
(SURVEY.md 8e, new work): q/k/v/gate/up column-parallel, o/down row-parallel + sum all-reduce.
"""
from __future__ import annotations

import inspect
import math
import os
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Union

import torch
import torch.nn.functional as F
from torch import nn

from . import ops
from .cache import StaticKVCache, StaticQuantizedKVCache, StaticRotatingKVCache
from .quantized_linear import QuantizedLinear
from .switch_layers import quantized_scaled_dot_product_attention
from .tp import TPContext


@dataclass
class BaseModelArgs:
    @classmethod
    def from_dict(cls, params):  # gbx_lm/models/base.py:15-24
        return cls(**{k: v for k, v in params.items() if k in inspect.signature(cls).parameters})


@dataclass
class ModelArgs(BaseModelArgs):  # gbx_lm/models/qllama.py:15-36
    model_type: str
    hidden_size: int
    num_hidden_layers: int
    intermediate_size: int
    num_attention_heads: int
    rms_norm_eps: float
    vocab_size: int
    head_dim: Optional[int] = None
    max_position_embeddings: Optional[int] = None
    num_key_value_heads: Optional[int] = None
    attention_bias: bool = False
    mlp_bias: bool = False
    rope_theta: float = 10000
    rope_traditional: bool = False
    rope_scaling: Optional[Dict[str, Union[float, str]]] = None
    tie_word_embeddings: bool = True

    def __post_init__(self):
        if self.num_key_value_heads is None:
            self.num_key_value_heads = self.num_attention_heads


# ------------------------------------------------------------------------------------------ glue
def rope_inv_freq(dims: int, base: float, scaling: Optional[dict]) -> torch.Tensor:
    """Inverse frequencies as the reference's initialize_rope produces them
    (gbx_lm/models/rope_utils.py:197-257: default / linear / llama3)."""
    rope_type = "default"
    if scaling is not None:
        rope_type = scaling.get("type") or scaling.get("rope_type", "default")
    freqs = base ** (torch.arange(0, dims, 2, dtype=torch.float32) / dims)  # "wavelength-like", inv = 1/freqs
    if rope_type == "default":
        return 1.0 / freqs
    if rope_type == "linear":
        return (1.0 / freqs) / float(scaling["factor"])
    if rope_type == "llama3":  # rope_utils.py:70-108
        factor = scaling["factor"]
        low = scaling.get("low_freq_factor", 1.0)
        high = scaling.get("high_freq_factor", 4.0)
        old = scaling.get("original_max_position_embeddings", 8192)
        low_wl, high_wl = old / low, old / high
        wavelens = 2 * math.pi * freqs
        f = torch.where(wavelens > low_wl, freqs * factor, freqs)
        medium = (wavelens > high_wl) & (wavelens < low_wl)
        smooth = (old / wavelens - low) / (high - low)
        smooth_f = f / ((1 - smooth) / factor + smooth)
        return 1.0 / torch.where(medium, smooth_f, f)
    raise ValueError(f"Unsupported RoPE type {rope_type} (yarn/longrope are outside the configs)")


# Decode-step glue through libgbxq (rope_cache / decode_attention / add_rmsnorm / silu_mul) instead of ~45 framework
# launches per block; GBXQ_FUSED_DECODE=0 keeps the plain torch glue (the tests compare the two).
FUSED_DECODE = os.environ.get("GBXQ_FUSED_DECODE", "1") != "0"


# The most tokens per row of one fused step: the `_multi` entry points of the decode-step kernels (include/gbxq.h)
MAX_BLOCK_TOKENS = 8


def fused_decode_ok(x: torch.Tensor, L: int, cache, block: bool = False) -> bool:
    """Whether a model call of L tokens per row may take the fused decode step: L == 1, or with `block` (explicit
    consecutive positions, Model.forward) 2 <= L <= MAX_BLOCK_TOKENS on a flat cache -- a verify block."""
    if not (FUSED_DECODE and cache is not None and x.is_cuda and x.dtype == torch.bfloat16):
        return False
    return L == 1 or (block and 2 <= L <= MAX_BLOCK_TOKENS and cache.keep is None)


class RoPE(nn.Module):
    """Non-traditional (half-split) rotary embedding, like mx.fast.rope(traditional=False)."""

    def __init__(self, dims: int, base: float, traditional: bool, scaling: Optional[dict]):
        super().__init__()
        if traditional:
            raise NotImplementedError("rope_traditional=True is not used by the configs")
        self.dims = dims
        self.register_buffer("inv_freq", rope_inv_freq(dims, base, scaling), persistent=False)

    def forward(self, x: torch.Tensor, positions: torch.Tensor) -> torch.Tensor:
        # x [B, H, L, D]; positions int64 [L] (shared by the rows) or [B, L] (per row)
        ang = positions.to(torch.float32)[..., None] * self.inv_freq  # [L, D/2] or [B, L, D/2]
        ang = ang[None, None] if ang.dim() == 2 else ang[:, None]
        cos, sin = ang.cos(), ang.sin()
        h = self.dims // 2
        x1, x2 = x[..., :h].float(), x[..., h : 2 * h].float()
        out = torch.cat([x1 * cos - x2 * sin, x1 * sin + x2 * cos], dim=-1)
        return out.to(x.dtype)


def make_prompt_cache(model, batch: int = 1, max_len: int = 4096, keep: Optional[int] = None) -> List[StaticKVCache]:
    """One static bf16 cache per layer: flat caches of max_len positions, or with `keep` an int, rotating caches of
    window max_len with `keep` sinks (the reference's RotatingKVCache)."""
    a = model.args
    hd = a.head_dim or a.hidden_size // a.num_attention_heads
    dev = model.model.embed_tokens.weight.device
    n_kv = a.num_key_value_heads // model.tp.world
    if keep is not None:
        return [StaticRotatingKVCache(batch, n_kv, max_len, hd, dev, keep) for _ in range(a.num_hidden_layers)]
    return [StaticKVCache(batch, n_kv, max_len, hd, dev) for _ in range(a.num_hidden_layers)]


class Attention(nn.Module):  # gbx_lm/models/qllama.py:39-96
    def __init__(self, args: ModelArgs, tp: TPContext, qkv_bias: Optional[bool] = None):
        super().__init__()
        dim = args.hidden_size
        self.tp = tp
        assert args.num_attention_heads % tp.world == 0 and args.num_key_value_heads % tp.world == 0, \
            "tensor parallel degree must divide the head counts (kv heads bound tp <= 8)"
        self.n_heads = args.num_attention_heads // tp.world
        self.n_kv_heads = args.num_key_value_heads // tp.world
        self.head_dim = head_dim = args.head_dim or args.hidden_size // args.num_attention_heads
        self.scale = head_dim ** -0.5
        attention_bias = getattr(args, "attention_bias", False) if qkv_bias is None else qkv_bias
        o_bias = getattr(args, "attention_bias", False) if qkv_bias is None else False
        self.q_proj = QuantizedLinear(dim, self.n_heads * head_dim, bias=attention_bias)
        self.k_proj = QuantizedLinear(dim, self.n_kv_heads * head_dim, bias=attention_bias)
        self.v_proj = QuantizedLinear(dim, self.n_kv_heads * head_dim, bias=attention_bias)
        self.o_proj = QuantizedLinear(self.n_heads * head_dim, dim, bias=o_bias)
        self.rope = RoPE(head_dim, args.rope_theta, args.rope_traditional, args.rope_scaling)

    def takes_fused_decode(self, cache: Union[StaticKVCache, StaticQuantizedKVCache]) -> bool:
        """Whether a decode step on `cache` runs the fused kernel pair of the cache's type: GBXQ_FUSED_DECODE on and
        shapes the pair serves."""
        return FUSED_DECODE and cache.fused_decode_fits(self.head_dim, self.n_heads, self.n_kv_heads)

    def forward(self, x, positions, cache: Optional[Union[StaticKVCache, StaticQuantizedKVCache]],
                attend_len: Optional[int], block: bool = False):
        B, L, _ = x.shape
        # one grouped launch for the three projections of x (ref qllama.py:76 calls them back to back)
        q, k, v = ops.quantized_matmul_grouped(x, (self.q_proj, self.k_proj, self.v_proj))
        quantized = isinstance(cache, StaticQuantizedKVCache)
        per_row = positions.dim() == 2  # [B, L]: rows that sit at different positions
        if fused_decode_ok(x, L, cache, block) and self.takes_fused_decode(cache):
            # the first position of each row (or of all rows): a block's tokens sit at start .. start + L - 1
            start = positions[:, 0].contiguous() if per_row else positions[:1]
            # decode step: RoPE + cache write in one launch, attention in another (SURVEY.md 8f rank 2); over the
            # quantized cache the attention is split-K on the codes (+ its combine launch).  L > 1: a verify block, the
            # same launches over [B, L, heads, D]
            lead = (B,) if L == 1 else (B, L)
            qh = q.view(*lead, self.n_heads, self.head_dim)
            kh, vh = k.view(*lead, self.n_kv_heads, self.head_dim), v.view(*lead, self.n_kv_heads, self.head_dim)
            # (a rotating cache: the row is the position's ring slot, and the attention reads the whole window)
            if quantized:
                gs, bits = cache.group_size, cache.bits
                ops.rope_cache_quantized(qh, kh, vh, start, self.rope.inv_freq, cache.keys, cache.values, gs, bits,
                                         keep=cache.keep)
                out = ops.decode_attention_quantized(qh, cache.keys, cache.values, start, self.scale, gs, bits,
                                                     attend_len)
            else:
                ops.rope_cache(qh, kh, vh, start, self.rope.inv_freq, cache.keys, cache.values, keep=cache.keep)
                out = ops.decode_attention(qh, cache.keys, cache.values, start, self.scale, attend_len)
            return self.tp.row_parallel(self.o_proj, out.view(B, L, -1))
        if per_row and cache is not None and cache.keep is not None:
            raise ValueError("per-row positions on a rotating cache need the fused decode path (the unfused ring glue "
                             "works on one shared offset)")
        q = self.rope(q.view(B, L, self.n_heads, -1).transpose(1, 2), positions)
        k = self.rope(k.view(B, L, self.n_kv_heads, -1).transpose(1, 2), positions)
        v = v.view(B, L, self.n_kv_heads, -1).transpose(1, 2)
        # a rotating cache that this call takes past its window: the positions attend the ring's rows and the call's own
        # keys under the window rule, and only then are the positions that survive the call stored (prefill glue, host
        # offsets: not graph-capturable).  Until then a rotating cache is written and read as the flat cache is.
        ring = cache is not None and cache.keep is not None and cache.wraps()
        if cache is None:
            T, keys, values = L, k, v
        elif ring:
            keys, values, key_positions = cache.window_with(k, v, cache.offset - L)
            T = key_positions.numel()
        elif quantized:
            # the rows are written at the HOST offset (Model.forward has already advanced it past these L positions), so
            # this path is not graph-capturable
            T = cache.offset
            if per_row:  # each row at its own (consecutive) positions, read back to the host
                for b, p in enumerate(positions[:, 0].tolist()):
                    cache.update_row(b, k[b:b + 1], v[b:b + 1], p)
            else:
                cache.update(k, v, T - L)
            keys, values = cache.prefix(T)
        else:
            cache.update(k, v, positions)
            T = attend_len if attend_len is not None else cache.max_len
            keys, values = cache.keys[:, :, :T], cache.values[:, :, :T]
        if ring:
            visible = cache.visible(key_positions, positions)
        else:  # causal over absolute positions: key j visible to query at position p iff j <= p
            visible = torch.arange(T, device=x.device) <= positions[..., None]  # [L, T], per row [B, L, T]
        if quantized:
            # the reference's attention on the codes (gbx_lm/models/base.py:65-98), with its additive mask
            mask = torch.zeros(visible.shape, dtype=q.dtype, device=x.device).masked_fill_(~visible, float("-inf"))
            if per_row:  # against the scores [B, Hq, L, T], or [B, Hkv, Hq / Hkv, L, T] under GQA
                mask = mask.view(B, *[1] * (1 if self.n_heads == self.n_kv_heads else 2), L, T)
            out = quantized_scaled_dot_product_attention(q, keys, values, self.scale, mask, cache.group_size, cache.bits)
        else:
            mask = visible[:, None] if per_row else visible[None, None]
            out = F.scaled_dot_product_attention(q, keys, values, attn_mask=mask, scale=self.scale,
                                                 enable_gqa=self.n_heads != self.n_kv_heads)
        if ring:
            cache.store(keys, values, cache.offset - L, L)
        out = out.transpose(1, 2).reshape(B, L, -1)
        return self.tp.row_parallel(self.o_proj, out)


class MLP(nn.Module):  # gbx_lm/models/qllama.py:99-115
    def __init__(self, args: ModelArgs, tp: TPContext):
        super().__init__()
        dim, hidden_dim = args.hidden_size, args.intermediate_size
        assert hidden_dim % tp.world == 0
        self.tp = tp
        mlp_bias = getattr(args, "mlp_bias", False)
        self.gate_proj = QuantizedLinear(dim, hidden_dim // tp.world, bias=mlp_bias)
        self.down_proj = QuantizedLinear(hidden_dim // tp.world, dim, bias=mlp_bias)
        self.up_proj = QuantizedLinear(dim, hidden_dim // tp.world, bias=mlp_bias)

    def forward(self, x):
        gate, up = ops.quantized_matmul_grouped(x, (self.gate_proj, self.up_proj))  # ref qllama.py:115
        if gate.is_cuda and gate.dtype == torch.bfloat16 and gate.numel() % 8 == 0 and FUSED_DECODE:
            act = ops.silu_mul(gate, up)
        else:
            act = F.silu(gate) * up
        return self.tp.row_parallel(self.down_proj, act)


class TransformerBlock(nn.Module):  # gbx_lm/models/qllama.py:118-141
    def __init__(self, args: ModelArgs, tp: TPContext, qkv_bias: Optional[bool] = None):
        super().__init__()
        self.self_attn = Attention(args, tp, qkv_bias)
        self.mlp = MLP(args, tp)
        self.input_layernorm = nn.RMSNorm(args.hidden_size, eps=args.rms_norm_eps)
        self.post_attention_layernorm = nn.RMSNorm(args.hidden_size, eps=args.rms_norm_eps)

    def forward(self, x, positions, cache, attend_len):
        h = x + self.self_attn(self.input_layernorm(x), positions, cache, attend_len)
        return h + self.mlp(self.post_attention_layernorm(h))


class LlamaModel(nn.Module):  # gbx_lm/models/qllama.py:144-174
    def __init__(self, args: ModelArgs, tp: TPContext, qkv_bias: Optional[bool] = None):
        super().__init__()
        assert args.vocab_size > 0
        self.embed_tokens = nn.Embedding(args.vocab_size, args.hidden_size)
        self.layers = nn.ModuleList([TransformerBlock(args, tp, qkv_bias) for _ in range(args.num_hidden_layers)])
        self.norm = nn.RMSNorm(args.hidden_size, eps=args.rms_norm_eps)

    def forward(self, inputs, positions, cache, attend_len, block: bool = False):
        h = self.embed_tokens(inputs)
        if cache is None:
            cache = [None] * len(self.layers)
        if fused_decode_ok(h, inputs.shape[1], cache[0], block) and h.shape[-1] % 8 == 0:
            # decode step: every residual add travels with the RMSNorm that follows it (one launch each); the add of a
            # block's MLP output happens in the next block's (or the final) norm launch
            resid, pend = h.contiguous(), None
            for layer, c in zip(self.layers, cache):
                resid, n = ops.add_rmsnorm(resid, pend, layer.input_layernorm.weight, layer.input_layernorm.eps)
                a = layer.self_attn(n, positions, c, attend_len, block)
                resid, n = ops.add_rmsnorm(resid, a, layer.post_attention_layernorm.weight, layer.post_attention_layernorm.eps)
                pend = layer.mlp(n)
            return ops.add_rmsnorm(resid, pend, self.norm.weight, self.norm.eps, want_h=False)[1]
        for layer, c in zip(self.layers, cache):
            h = layer(h, positions, c, attend_len)
        return self.norm(h)


class Model(nn.Module):  # gbx_lm/models/qllama.py:177-209
    QKV_BIAS: Optional[bool] = None  # None -> follow args.attention_bias (Llama); Qwen2 overrides

    def __init__(self, args: ModelArgs, tp: Optional[TPContext] = None):
        super().__init__()
        self.args = args
        self.model_type = args.model_type
        self.tp = tp or TPContext()
        self.model = LlamaModel(args, self.tp, self.QKV_BIAS)
        if not args.tie_word_embeddings:
            self.lm_head = nn.Linear(args.hidden_size, args.vocab_size, bias=False)

    def forward(self, inputs: torch.Tensor, cache: Optional[List[Union[StaticKVCache, StaticQuantizedKVCache]]] = None,
                positions: Optional[torch.Tensor] = None, attend_len: Optional[int] = None, hidden_states: bool = False,
                head_columns: Optional[torch.Tensor] = None):
        """inputs int64 [B, L].  positions int64 [L] (absolute, shared by the rows); default = cache offset .. offset+L.
        A decode step (L = 1) may instead give each row its own position, int64 [B, 1]; the caller keeps the caches'
        offsets then.  Explicit positions with 2 <= L <= 8 must be consecutive in each row (int64 [L] shared, or [B, L]
        per row): a verify block of speculative decoding, which takes the fused decode step on flat caches (its tokens
        written at their positions, query t seeing keys 0 .. p_b + t); the caller keeps the offsets.  attend_len: number of cache positions attended (None = whole static cache, for graph replay).
        head_columns int64 [B]: only column head_columns[b] of row b goes through the vocabulary projection (logits
        [B, 1, V], hidden states [B, 1, H]) -- what a batched prefill needs, without the [B, L, V] logits of every
        position; None: every position."""
        L = inputs.shape[1]
        block = positions is not None and L > 1
        if positions is None:
            off = cache[0].offset if cache is not None else 0
            positions = torch.arange(off, off + L, device=inputs.device)
            if cache is not None:
                for c in cache:
                    c.offset = off + L
                attend_len = cache[0].attend_len  # off + L; at most the window on a rotating cache
        out = self.model(inputs, positions, cache, attend_len, block)
        if head_columns is not None:
            out = out[torch.arange(out.shape[0], device=out.device), head_columns][:, None]
        # vocabulary projection (qllama.py:194-198): decode-sized inputs go through the streaming bf16 GEMV
        # (gbxq_head_gemv), prefill through the dense matmul
        head = self.model.embed_tokens.weight if self.args.tie_word_embeddings else self.lm_head.weight
        logits = ops.head_linear(out, head) if FUSED_DECODE else F.linear(out, head)
        return (logits, out) if hidden_states else logits

    def sanitize(self, weights: Dict[str, Any]) -> Dict[str, Any]:  # qllama.py:201-205
        return {k: v for k, v in weights.items() if "self_attn.rotary_emb.inv_freq" not in k}

    @property
    def layers(self):
        return self.model.layers
