"""Layer-mix weight loader, checkpoint writer and decode loop -- host-side mirror of the parts of
`gbx_lm/utils.py` that sit on either side of the quantized-matmul path:

    load_model / load        gbx_lm/utils.py:752-920   (strategy -> reinit_module -> load_weights)
    make_shards/save_weights gbx_lm/utils.py:967-988, 1055-1104
    save_config              gbx_lm/utils.py:1107-1127
    generate_step            gbx_lm/utils.py:217-338   (batch-1 prefill in 2048-token chunks + greedy decode)
    speculative_generate_step gbx_lm/utils.py:341-522  (a draft model proposes, the target verifies k + 1 tokens a step)
    batch_generate           (new) greedy decode of B prompts of different lengths in one batch

The on-disk layout is exactly what gba2mlx emits (gbx_lm/gba2mlx.py:47-65): `model*.safetensors` with
`<module>.{qweight,scales,zeros[,bias]}`, metadata {"format": "mlx"}, `config.json` carrying
`"quantization": {"group_size", "bits"}` and an optional `quant_strategy.json`.
Tensor-parallel loading (new work) slices each projection for this rank before it reaches the GPU.
"""
from __future__ import annotations

import glob
import json
import logging
import time
from pathlib import Path
from typing import Any, Callable, Dict, Generator, List, Optional, Tuple, Type, Union

import torch
from torch import nn

from . import qllama, qqwen2
from .cache import (DEFAULT_KV_KEEP, StaticKVCache, StaticQuantizedKVCache, maybe_quantize_kv_cache,
                    trim_prompt_cache)
from .quantized_linear import QuantizedLinear
from .tp import TPContext, proj_kind, shard_tensor

MODEL_MAPPING = {  # subset of gbx_lm/utils.py:52-61 that BASELINE.json's configs use
    "llama": qllama,
    "mistral": qllama,  # same remapping as the reference (utils.py:141-159)
    "qwen2": qqwen2,
}
MAX_FILE_SIZE_GB = 5


def _get_classes(config: dict):
    model_type = config["model_type"]
    if model_type not in MODEL_MAPPING:
        msg = f"Model type {model_type} not supported."
        logging.error(msg)
        raise ValueError(msg)
    arch = MODEL_MAPPING[model_type]
    return arch.Model, arch.ModelArgs


def get_parameter_usage_info(weights: Dict[str, Any]) -> Tuple[bool, bool]:
    """(double-quantised statistics present, q_perm present) -- gbx_lm/utils.py:696-719; one implementation, shared
    with the converter."""
    from .gba_convert import parameter_usage

    return parameter_usage(weights)


def _load_safetensors(path: str) -> Dict[str, torch.Tensor]:
    from safetensors.torch import load_file

    return load_file(path, device="cpu")


def load_weights(model: nn.Module, weights: Dict[str, torch.Tensor], strict: bool = False, device=None) -> List[str]:
    """`model.load_weights(list(weights.items()), strict=False)` (utils.py:862): assign by dotted key.
    Unlike MLX (which does not check shapes with strict=False -- SURVEY 3.1) a shape mismatch raises."""
    targets = dict(model.named_buffers())
    targets.update(dict(model.named_parameters()))
    missing = []
    for key, t in weights.items():
        if key not in targets:
            if strict:
                raise KeyError(f"unexpected weight {key}")
            missing.append(key)
            continue
        mod_name, _, leaf = key.rpartition(".")
        mod = model.get_submodule(mod_name) if mod_name else model
        cur = targets[key]
        if cur is not None and tuple(cur.shape) != tuple(t.shape):
            raise ValueError(f"{key}: checkpoint shape {tuple(t.shape)} != module shape {tuple(cur.shape)}")
        t = t.to(device) if device is not None else t
        if leaf in mod._parameters:
            mod._parameters[leaf] = nn.Parameter(t, requires_grad=False)
        else:
            mod._buffers[leaf] = t
    return missing


def load_model(
    model_path: Union[str, Path],
    lazy: bool = False,
    model_config: dict = {},
    bits: int = 4,
    group_size: int = 64,
    is_conversion: bool = False,
    get_model_classes: Callable[[dict], Tuple[Type[nn.Module], Type]] = _get_classes,
    device: Union[str, torch.device] = "cuda",
    tp: Optional[TPContext] = None,
) -> Tuple[nn.Module, dict]:
    """Mirror of gbx_lm/utils.py:752-879 (same steps, same order, same error behaviour)."""
    model_path = Path(model_path)
    tp = tp or TPContext()
    # ======== load strategy.json file ========= #  (utils.py:787-792)
    strategy = None
    try:
        with open(model_path / "quant_strategy.json", "r") as f:
            strategy = json.load(f)["measurement"]
    except FileNotFoundError:
        logging.info(f"[WARNING] Strategy config file not found in {model_path}")
    # ===== load quantization config file ====== #  (utils.py:795-803)
    try:
        with open(model_path / "config.json", "r") as f:
            config = json.load(f)
            quantization = config.get("quantization", None)
            if quantization is None:
                quantization = {"group_size": group_size, "bits": bits}
    except FileNotFoundError:
        logging.info(f"[WARNING] Quantization config file not found in {model_path}")
        raise
    config.update(model_config)

    weight_files = glob.glob(str(model_path / "model*.safetensors"))
    if not weight_files:
        logging.error(f"No safetensors found in {model_path}")
        raise FileNotFoundError(f"No safetensors found in {model_path}")
    weights: Dict[str, torch.Tensor] = {}
    for wf in weight_files:
        weights.update(_load_safetensors(wf))

    use_double_quantization, use_q_perm = get_parameter_usage_info(weights)
    if not use_q_perm:
        assert quantization["group_size"] in [32, 64, 128], \
            f"The group size value ({group_size}) must be 32, 64 or 128."
    if is_conversion or use_double_quantization:
        # an original GBA checkpoint (K-major qweight / statistics, subtractive zeros, optionally double-quantised
        # statistics): brought to the layout of the path on the host, before any module sees it -- the reference's
        # transposes (utils.py:828-838), `prepare_scales_zeros` and `post_processing_and_release` (:864-873)
        from .gba_convert import convert_gba_weights, expand_statistics
        from .quantized_linear import strategy_params

        def gs_of(mod_name: str) -> int:
            return strategy_params(mod_name, strategy, quantization["bits"], quantization["group_size"])[1]

        weights = convert_gba_weights(weights, gs_of) if is_conversion else expand_statistics(weights, gs_of)
        for k in [k for k in weights if k.endswith(".q_perm")]:
            weights[k] = weights[k].reshape(1, 1, -1)  # quantized_linear_gba.py:157-158
        use_double_quantization = False  # plain scales / zeros from here on
    # scales / zeros -> bf16 (utils.py:841-843)
    for k, v in weights.items():
        if "scale" in k or "zeros" in k:
            weights[k] = v.to(torch.bfloat16)

    model_class, model_args_class = get_model_classes(config=config)
    model_args = model_args_class.from_dict(config)
    model = model_class(model_args, tp) if tp.world > 1 else model_class(model_args)
    if hasattr(model, "sanitize"):
        weights = model.sanitize(weights)

    # per-layer (bits, group_size) from the strategy (utils.py:854-860 -> quantized_linear_gba.py:210-283)
    QuantizedLinear.reinit_module(
        model, **quantization, strategy=strategy, use_double_quantization=use_double_quantization, use_q_perm=use_q_perm
    )
    if tp.world > 1:
        mods = dict(model.named_modules())
        sharded = {}
        for k, v in weights.items():
            mod_name = k.rpartition(".")[0]
            m = mods.get(mod_name)
            if isinstance(m, QuantizedLinear) and proj_kind(mod_name) is not None:
                sharded[k] = shard_tensor(k, v, m.bits, m.group_size, tp.rank, tp.world)
            else:
                sharded[k] = v
        weights = sharded
    # embeddings / norms / head follow the activation dtype of the path
    for k, v in list(weights.items()):
        if v.is_floating_point() and v.dtype != torch.bfloat16 and "channel_scale" not in k:
            weights[k] = v.to(torch.bfloat16)

    dev = torch.device(device)
    load_weights(model, weights, strict=False, device=dev)
    # anything the checkpoint did not provide (RoPE tables, absent optional buffers) moves too
    model.to(dev)
    for m in model.modules():
        if isinstance(m, (nn.RMSNorm, nn.Embedding, nn.Linear)):
            m.to(torch.bfloat16)
    if not lazy and dev.type == "cuda":
        torch.cuda.synchronize(dev)
    model.eval()
    for prm in model.parameters():
        prm.requires_grad_(False)
    return model, config


def load(path: Union[str, Path], model_config: dict = {}, lazy: bool = False, device="cuda", tp: Optional[TPContext] = None):
    """gbx_lm.load without the tokenizer / hub download (no network; token ids in, token ids out)."""
    model, config = load_model(Path(path), lazy, model_config=model_config, device=device, tp=tp)
    return model, config


# ------------------------------------------------------------------------------------------ writer
def _nbytes(t: torch.Tensor) -> int:
    return t.numel() * t.element_size()


def make_shards(weights: dict, max_file_size_gb: int = MAX_FILE_SIZE_GB) -> list:
    """The on-disk split of gbx_lm/utils.py:967-988: tensors in insertion order, a tensor that would take the current
    file over the cap opens the next one.  (The reference also emits an EMPTY first shard when the very first tensor is
    over the cap; no empty file is written here.)"""
    cap = max_file_size_gb << 30
    shards, used = [{}], 0
    for name, t in weights.items():
        if shards[-1] and used + _nbytes(t) > cap:
            shards.append({})
            used = 0
        shards[-1][name] = t
        used += _nbytes(t)
    return shards


def save_weights(save_path: Union[str, Path], weights: Dict[str, torch.Tensor], *, donate_weights: bool = False,
                 max_file_size_gb: int = MAX_FILE_SIZE_GB) -> None:
    """The layout `load_model` (and gbx_lm/utils.py:1055-1104) expects: `model.safetensors`, or
    `model-0000i-of-0000n.safetensors` when the split has n > 1 files, each with metadata {"format": "mlx"}, plus
    `model.safetensors.index.json` = {"metadata": {"total_size"}, "weight_map": name -> file, sorted by name}."""
    from safetensors.torch import save_file

    out = Path(save_path)
    out.mkdir(parents=True, exist_ok=True)
    shards = make_shards(weights, max_file_size_gb)
    n = len(shards)
    index = {"metadata": {"total_size": sum(_nbytes(t) for t in weights.values())}, "weight_map": {}}
    if donate_weights:
        weights.clear()  # the shards hold the only references from here on
    for i in range(1, n + 1):
        shard = shards.pop(0)  # dropped after the write, so that a donated checkpoint is freed file by file
        fname = f"model-{i:05d}-of-{n:05d}.safetensors" if n > 1 else "model.safetensors"
        save_file({k: v.contiguous().cpu() for k, v in shard.items()}, str(out / fname), metadata={"format": "mlx"})
        index["weight_map"].update(dict.fromkeys(shard, fname))
    index["weight_map"] = dict(sorted(index["weight_map"].items()))
    (out / "model.safetensors.index.json").write_text(json.dumps(index, indent=4))


def save_config(config: dict, config_path: Union[str, Path]) -> None:
    """gbx_lm/utils.py:1107-1127: keys sorted, `_name_or_path` dropped (from the written copy only)."""
    Path(config_path).write_text(json.dumps({k: config[k] for k in sorted(config) if k != "_name_or_path"}, indent=4))


def write_synthetic_checkpoint(path: Union[str, Path], dims, strategy: Optional[dict], seed: int = 0,
                               default_bits: int = 4, default_gs: int = 64, embed_scale: float = 1.0) -> dict:
    """Random-init checkpoint of `dims` (workloads.ModelDims) in the gba2mlx layout, with the synthetic
    recipe of SURVEY.md 8d.  `strategy` is a quant_strategy.json dict or None (uniform bits/gs from
    config["quantization"], the `strategy is None` branch of reinit_module)."""
    from . import packing
    from .workloads import PROJS, layer_plan

    path = Path(path)
    path.mkdir(parents=True, exist_ok=True)
    gen = torch.Generator().manual_seed(seed)
    weights: Dict[str, torch.Tensor] = {}
    h = dims.hidden
    weights["model.embed_tokens.weight"] = (torch.randn((dims.vocab, h), generator=gen) * embed_scale).to(torch.bfloat16)
    weights["model.norm.weight"] = (1.0 + 0.05 * torch.randn((h,), generator=gen)).to(torch.bfloat16)
    if not dims.tie:
        weights["lm_head.weight"] = (torch.randn((dims.vocab, h), generator=gen) / h ** 0.5).to(torch.bfloat16)
    for (i, p, n, k, b, g) in layer_plan(dims, strategy, default_bits, default_gs):
        sub = "self_attn" if p in ("q_proj", "k_proj", "v_proj", "o_proj") else "mlp"
        L = packing.synth_layer(n, k, b, g, seed=seed * 100003 + i * 7 + PROJS.index(p),
                                with_bias=dims.qkv_bias and p in ("q_proj", "k_proj", "v_proj"))
        base = f"model.layers.{i}.{sub}.{p}"
        weights[base + ".qweight"] = L["qweight"]
        weights[base + ".scales"] = L["scales"]
        weights[base + ".zeros"] = L["zeros"]
        if "bias" in L:
            weights[base + ".bias"] = L["bias"]
    for i in range(dims.layers):
        for nm in ("input_layernorm", "post_attention_layernorm"):
            weights[f"model.layers.{i}.{nm}.weight"] = (1.0 + 0.05 * torch.randn((h,), generator=gen)).to(torch.bfloat16)
    config = {
        "model_type": dims.model_type, "hidden_size": h, "num_hidden_layers": dims.layers,
        "intermediate_size": dims.inter, "num_attention_heads": dims.heads, "num_key_value_heads": dims.kv_heads,
        "rms_norm_eps": dims.rms_eps, "vocab_size": dims.vocab, "rope_theta": dims.rope_theta,
        "rope_scaling": dims.rope_scaling, "tie_word_embeddings": dims.tie, "max_position_embeddings": dims.max_pos,
        "head_dim": dims.head_dim, "quantization": {"group_size": default_gs, "bits": default_bits},
    }
    if dims.model_type == "qwen2":
        config.pop("head_dim")
    save_weights(path, weights)
    save_config(config, path / "config.json")
    if strategy is not None:
        with open(path / "quant_strategy.json", "w") as f:
            json.dump(strategy, f)
    return config


# ------------------------------------------------------------------------------------------ decode loop
def fast_argmax(x: torch.Tensor) -> torch.Tensor:
    """argmax over the last (vocabulary) dimension, first occurrence on ties like torch.argmax, as two row-parallel
    reductions: a [B, V] single-row argmax is one slow block on the GPU (~0.5 ms at V = 128256, profiles/README.md), a
    [B*a, V/a] max followed by an argmax over the a segment maxima is not."""
    v = x.shape[-1]
    a = next((c for c in (256, 192, 128, 96, 64, 48, 32) if v % c == 0 and v // c >= 64), 0)
    if not a:
        return torch.argmax(x, dim=-1)
    seg = x.reshape(*x.shape[:-1], a, v // a)
    m, i = seg.max(dim=-1)              # first maximal index inside every segment
    j = m.argmax(dim=-1, keepdim=True)  # first segment holding the global maximum
    return (j * (v // a) + i.gather(-1, j)).squeeze(-1)



class DecodeGraph:
    """One decode step (token ids [B,1] -> logits) captured in a CUDA graph: the whole step --
    7*L QuantizedLinear launches plus the glue -- replays as one submission (SURVEY.md 7.2 item 1).
    per_row: the B rows sit at their own positions, `pos` int64 [B] (prompts of different lengths), instead of one
    shared position `pos` [1]."""

    def __init__(self, model, cache, batch: int = 1, per_row: bool = False):
        # the unfused quantized and rotating paths write at the HOST offset, which a replay cannot advance
        if any((isinstance(c, StaticQuantizedKVCache) or c.keep is not None) and not layer.self_attn.takes_fused_decode(c)
               for layer, c in zip(model.layers, cache)):
            raise ValueError("DecodeGraph: a quantized or rotating KV cache is graph-capturable only on the fused decode "
                             "path")
        self.model, self.cache = model, cache
        dev = cache[0].device
        self.tok = torch.zeros((batch, 1), dtype=torch.long, device=dev)
        self.pos = torch.zeros((batch if per_row else 1,), dtype=torch.long, device=dev)
        self.per_row = per_row
        self.logits = None
        self.graph = None

    def _set(self, tokens: torch.Tensor, position) -> None:
        self.tok.copy_(tokens.reshape(self.tok.shape))
        if self.per_row:
            self.pos.copy_(position)
        else:
            self.pos.fill_(position)

    def _positions(self) -> torch.Tensor:
        return self.pos[:, None] if self.per_row else self.pos

    def capture(self, tokens: torch.Tensor, position, device_loop: int = 0):
        """Warm-up + capture at (tokens, position) = the step that will be replayed first, so the KV
        entries written during warm-up/capture are exactly the ones that step writes anyway.
        device_loop = n > 0: the greedy sampler is part of the graph -- argmax of the logits (= argmax of the
        log-probabilities, utils.py:285,305-306), fed back as the next step's token, position advanced and the token
        appended to `self.out` [n] on the device -- so that n steps replay back to back without a host round trip.
        position: an int, or with per_row an int64 [B] device tensor."""
        self._set(tokens, position)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s), torch.no_grad():
            for _ in range(2):
                self.model(self.tok, self.cache, positions=self._positions(), attend_len=None)
        torch.cuda.current_stream().wait_stream(s)
        if device_loop:
            self.out = torch.zeros((device_loop, self.tok.shape[0]), dtype=torch.long, device=self.tok.device)
            self.idx = torch.zeros((1,), dtype=torch.long, device=self.tok.device)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph), torch.no_grad():
            self.logits = self.model(self.tok, self.cache, positions=self._positions(), attend_len=None)
            if device_loop:
                nxt = fast_argmax(self.logits[:, -1, :])  # [B]; bf16 -> fp32 is order preserving, so no cast
                self.out.index_copy_(0, self.idx, nxt[None])
                self.tok.copy_(nxt[:, None])
                self.pos.add_(1)
                self.idx.add_(1)
        return self

    def step(self, tokens: torch.Tensor, position) -> torch.Tensor:
        """One replay at `position` (as in `capture`); the caches' offset becomes the largest position + 1."""
        self._set(tokens, position)
        self.graph.replay()
        last = int(position.max()) if self.per_row else position
        for c in self.cache:
            c.offset = last + 1
        return self.logits[:, -1, :]


def _kv_quantizer(cache: list, kv_bits: Optional[int], kv_group_size: int, quantized_kv_start: int) -> Callable[[], bool]:
    """The reference's check after every model call (gbx_lm/utils.py:204-214, 268-270): maybe_quantize_kv_cache on the
    list; returns True when this call converted it."""
    def step() -> bool:
        before = cache[0]
        maybe_quantize_kv_cache(cache, quantized_kv_start, kv_group_size, kv_bits)
        return cache[0] is not before

    return step


def _decode_graph(model, cache, tok, position, device_loop: int = 0) -> Optional[DecodeGraph]:
    """A captured decode step for the rows of `tok` [B] at `position` (an int, or an int64 [B] device tensor of per-row
    positions), or None where the cache cannot be captured (a quantized or rotating cache off the fused path)."""
    try:
        dg = DecodeGraph(model, cache, batch=tok.numel(), per_row=isinstance(position, torch.Tensor))
    except ValueError:
        return None
    return dg.capture(tok, position, device_loop=device_loop)


def _prompt_cache(model, run_len: int, max_kv_size: Optional[int], batch: int = 1) -> list:
    """Flat caches for a run of `run_len` positions, or rotating caches of window max_kv_size."""
    if max_kv_size is None:
        return qllama.make_prompt_cache(model, batch, run_len)
    return qllama.make_prompt_cache(model, batch, max_kv_size, keep=DEFAULT_KV_KEEP)


def _prefill_chunks(model, tokens: torch.Tensor, cache: list, prefill_step_size: int, kv: dict,
                    last: Optional[List[int]] = None) -> torch.Tensor:
    """tokens [B, L] through the model in `prefill_step_size` chunks at the shared positions 0 .. L-1, with the conversion
    rule of `generate_step` applied after every model call.  Returns the logits [B, V] of the final column, or with
    `last` (one column per row) those of column last[b] of row b: each chunk sends only those columns through the
    vocabulary projection (Model.forward head_columns)."""
    quantize_cache = _kv_quantizer(cache, **kv)
    L = tokens.shape[1]
    out = None
    with torch.no_grad():
        for c0 in range(0, L, prefill_step_size):
            chunk = tokens[:, c0:c0 + prefill_step_size]
            n = chunk.shape[1]
            if last is None:
                logits = model(chunk, cache)
                if c0 + n == L:
                    out = logits[:, -1, :]
            else:
                here = [c0 <= j < c0 + n for j in last]
                cols = torch.tensor([min(max(j - c0, 0), n - 1) for j in last], device=tokens.device)
                logits = model(chunk, cache, head_columns=cols)[:, 0]
                if any(here):
                    keep = torch.tensor(here, device=tokens.device)[:, None]
                    out = logits if out is None else torch.where(keep, logits, out)
            quantize_cache()
    return out


def prefill(model, prompt: torch.Tensor, cache: list, prefill_step_size: int = 2048, kv_bits: Optional[int] = None,
            kv_group_size: int = 64, quantized_kv_start: int = 0) -> torch.Tensor:
    """The prompt (token ids [n], on the model's device) through the model in `prefill_step_size` chunks, with the
    conversion rule of `generate_step` applied after every model call; returns the logits of the last position [1, V]."""
    kv = dict(kv_bits=kv_bits, kv_group_size=kv_group_size, quantized_kv_start=quantized_kv_start)
    return _prefill_chunks(model, prompt.reshape(1, -1), cache, prefill_step_size, kv)


def _conversion_segments(cache: list, steps: int, pos0: int, kv_bits: Optional[int], quantized_kv_start: int) -> List[int]:
    """Replay counts of the captured decode: replay i takes the caches' offset to pos0 + i + 1, and the reference
    converts after the call that takes the offset past quantized_kv_start, i.e. after replay
    max(0, quantized_kv_start - pos0): the replays up to there are one segment, the rest a second one on a graph of the
    quantized step."""
    head = steps
    if kv_bits is not None and isinstance(cache[0], StaticKVCache):
        head = min(max(quantized_kv_start - pos0, 0) + 1, steps)
    return [head] + ([steps - head] if head < steps else [])


def _device_decode(model, cache: list, tok: torch.Tensor, position, pos0: int, steps: int, kv: dict, where: str):
    """`steps` greedy decode steps as replays of captured steps with the sampler inside (DecodeGraph device_loop), split
    at the kv_bits conversion (_conversion_segments).  tok [B]: the first tokens; position: the first replay's position
    (an int, or int64 [B] per row); pos0: the caches' offset before it.  Returns (first tokens as a list, the time after
    the first capture, [n, B] token tensors of the segments); the caches' offset is left at pos0 + steps."""
    per_row = isinstance(position, torch.Tensor)
    outs, offset = [], pos0
    for i, n in enumerate(_conversion_segments(cache, steps, pos0, kv["kv_bits"], kv["quantized_kv_start"])):
        if i:  # at the conversion: convert the caches, continue from the last token on a graph of the quantized step
            for c in cache:
                c.offset = offset
            maybe_quantize_kv_cache(cache, kv["quantized_kv_start"], kv["kv_group_size"], kv["kv_bits"])
            tok = dg.tok[:, 0].clone()
            position = dg.pos.clone() if per_row else position
        # captured even for zero replays (max_tokens 1): the cache is checked for capturability all the same
        dg = _decode_graph(model, cache, tok, position, device_loop=max(n, 1))
        if dg is None:
            raise ValueError(f"{where}: the quantized cache cannot be captured (unfused decode path)")
        if i == 0:  # the capture of the first graph counts as prompt time
            first = tok.tolist()
            t_first = time.perf_counter()
        for _ in range(n):
            dg.graph.replay()
        outs.append(dg.out[:n])
        offset += n
        if not per_row:
            position += n
    for c in cache:
        c.offset = offset
    return first, t_first, outs


def generate_step(
    prompt: torch.Tensor,
    model: nn.Module,
    *,
    max_tokens: int = 256,
    sampler: Optional[Callable[[torch.Tensor], torch.Tensor]] = None,
    prompt_cache: Optional[Any] = None,
    prefill_step_size: int = 2048,
    max_kv_size: Optional[int] = None,
    use_cuda_graph: bool = True,
    kv_bits: Optional[int] = None,
    kv_group_size: int = 64,
    quantized_kv_start: int = 0,
) -> Generator[Tuple[int, torch.Tensor], None, None]:
    """Mirror of gbx_lm/utils.py:217-338 for the greedy path: batch-1 prompt of token ids,
    prefill in `prefill_step_size` chunks, then one token per step; yields (token, logprobs).
    The default sampler is the argmax of the log-probabilities (utils.py:285,305-306).
    kv_bits / kv_group_size / quantized_kv_start: the reference's quantized KV cache -- after every model call, prefill
    chunks included, the caches are converted to `kv_bits`-bit group-quantized ones once their offset exceeds
    `quantized_kv_start` (maybe_quantize_kv_cache); kv_bits=None keeps the bf16 cache.  A decode graph captured before the
    conversion is captured again once, after it.
    max_kv_size = W: rotating caches of W positions with DEFAULT_KV_KEEP sinks (the reference's RotatingKVCache), so the
    memory and the attention of every step stay bounded however long the run; they compose with kv_bits."""
    y = prompt.reshape(-1).to(next(model.parameters()).device)
    sampler = sampler or (lambda lp: torch.argmax(lp, dim=-1))
    cache = prompt_cache if prompt_cache is not None else _prompt_cache(model, y.numel() + max_tokens + 1, max_kv_size)
    kv = dict(kv_bits=kv_bits, kv_group_size=kv_group_size, quantized_kv_start=quantized_kv_start)
    quantize_cache = _kv_quantizer(cache, **kv)

    with torch.no_grad():
        lp = _logprobs(prefill(model, y, cache, prefill_step_size, **kv))
        tok = sampler(lp)
        use_graph = use_cuda_graph and tok.is_cuda
        dg = _decode_graph(model, cache, tok, cache[0].offset) if use_graph else None
        n = 0
        while True:
            if n == max_tokens:
                break
            yield int(tok.item()), lp.squeeze(0)
            n += 1
            pos = cache[0].offset
            if dg is not None:
                logits = dg.step(tok, pos)
            else:
                logits = model(tok.reshape(1, 1), cache)[:, -1, :]
            converted = quantize_cache()
            lp = _logprobs(logits)
            tok = sampler(lp)
            if converted and use_graph:  # the captured step wrote the bf16 buffers: capture the quantized step
                dg = _decode_graph(model, cache, tok, cache[0].offset)


def _logprobs(logits: torch.Tensor) -> torch.Tensor:
    logits = logits.float()
    return logits - torch.logsumexp(logits, dim=-1, keepdim=True)


# ------------------------------------------------------------------------------------------ speculative decoding
def _check_speculative(model, draft_model, num_draft_tokens: int, max_kv_size: Optional[int] = None) -> None:
    if max_kv_size is not None:
        raise ValueError("speculative decoding: max_kv_size (a rotating cache) cannot be rewound; use a flat cache")
    if isinstance(num_draft_tokens, bool) or not isinstance(num_draft_tokens, int) or not 1 <= num_draft_tokens <= 7:
        raise ValueError(f"speculative decoding: num_draft_tokens must be an int in 1..7, got {num_draft_tokens!r}")
    if model.args.vocab_size != draft_model.args.vocab_size:
        raise ValueError(f"speculative decoding: the draft's vocabulary ({draft_model.args.vocab_size}) differs from the "
                         f"target's ({model.args.vocab_size})")
    if model.tp.world > 1 or draft_model.tp.world > 1:
        raise ValueError("speculative decoding: tensor-parallel models are not supported")


def _spec_cache(model, draft_model, run_len: int) -> list:
    """The target's flat caches, then the draft's (the reference's prompt_cache layout)."""
    return qllama.make_prompt_cache(model, 1, run_len) + qllama.make_prompt_cache(draft_model, 1, run_len)


def _draft_and_verify(model, draft_model, tc: list, dc: list, prev: torch.Tensor, y: torch.Tensor, P: torch.Tensor,
                      k: int, pick: Callable[[torch.Tensor], torch.Tensor], host_P: Optional[int] = None):
    """Steps 1 and 2 of a round (DESIGN.md section 10).  prev / y [1]: the tokens at P - 1 and P (int64 [1] on the
    device).  The draft takes one T = 2 step on [prev, y] at P - 1, P, then k - 1 single-token steps, each token picked
    from the last logits (`pick`: logits [V] -> token [1]); the target verifies [y, d_1 .. d_k] at P .. P + k in one
    step of k + 1 tokens.  Returns (d [k], the verify logits [k + 1, V]).  host_P: P as an int, to keep the caches'
    offsets (the unfused glue writes a quantized cache at them); None inside a captured graph, which needs the fused
    path."""
    ar = torch.arange(k + 1, device=P.device)

    def call(m, cache, toks, pos, end):
        if host_P is not None:
            for c in cache:
                c.offset = host_P + end
        return m(toks[None], cache, positions=pos)[0]

    d = [pick(call(draft_model, dc, torch.cat([prev, y]), P - 1 + ar[:2], 1)[-1])]
    for i in range(1, k):
        d.append(pick(call(draft_model, dc, d[-1], P + i, i + 1)[-1]))
    d = torch.cat(d)
    return d, call(model, tc, torch.cat([y, d]), P + ar, k + 1)


def speculative_generate_step(prompt: torch.Tensor, model: nn.Module, draft_model: nn.Module, *, num_draft_tokens: int = 2,
                              max_tokens: int = 256, sampler: Optional[Callable[[torch.Tensor], torch.Tensor]] = None,
                              prompt_cache: Optional[list] = None, prefill_step_size: int = 2048,
                              kv_bits: Optional[int] = None, kv_group_size: int = 64, quantized_kv_start: int = 0
                              ) -> Generator[Tuple[int, torch.Tensor, bool], None, None]:
    """Mirror of gbx_lm/utils.py:341-522: `draft_model` proposes num_draft_tokens = k tokens a round and `model` checks
    them in one step of k + 1 tokens; yields (token, logprobs, from_draft).  prompt_cache: the target's caches, then the
    draft's (default: flat caches of prompt + max_tokens + k + 2 positions).  `sampler` picks every token from its
    log-probabilities (default argmax).  kv_bits / kv_group_size / quantized_kv_start as in generate_step: both lists
    are converted after the verify step that takes the target's offset past quantized_kv_start.

    The round schedule (DESIGN.md section 10) keeps the block at k + 1 tokens in every round, the last one included, and
    drops the tokens past max_tokens, so that at a fixed k the tokens do not depend on the draft."""
    k = num_draft_tokens
    _check_speculative(model, draft_model, k)
    dev = next(model.parameters()).device
    y0 = prompt.reshape(-1).to(dev)
    sampler = sampler or (lambda lp: torch.argmax(lp, dim=-1))
    cache = prompt_cache if prompt_cache is not None else _spec_cache(model, draft_model, y0.numel() + max_tokens + k + 2)
    nt = len(model.layers)
    kv = dict(kv_bits=kv_bits, kv_group_size=kv_group_size, quantized_kv_start=quantized_kv_start)
    if max_tokens <= 0:
        return
    with torch.no_grad():
        tc, dc = cache[:nt], cache[nt:]
        lp = _logprobs(prefill(model, y0, tc, prefill_step_size, **kv))[0]
        prefill(draft_model, y0, dc, prefill_step_size, **kv)
        cache[:] = tc + dc
        y = sampler(lp).reshape(1)
        prev, P = y0[-1:], y0.numel()  # the target holds positions < P, y sits at P, the draft holds < P - 1 at least
        yield int(y), lp, False
        ntoks = 1
        while ntoks < max_tokens:
            tc, dc = cache[:nt], cache[nt:]
            d, logits = _draft_and_verify(model, draft_model, tc, dc, prev, y, torch.tensor([P], device=dev), k,
                                          lambda lg: sampler(_logprobs(lg)).reshape(1), host_P=P)
            maybe_quantize_kv_cache(cache, quantized_kv_start, kv_group_size, kv_bits)  # by the target's offset
            lps = _logprobs(logits)
            a = sampler(lps).reshape(-1)
            a_l, d_l = a.tolist(), d.tolist()
            n = 0
            while n < k and a_l[n] == d_l[n]:
                n += 1
            for i in range(n + 1):
                yield a_l[i], lps[i], i < n
                ntoks += 1
                if ntoks == max_tokens:
                    break
            # rewind: the target keeps positions < P + n + 1, the draft < P + n (its next T = 2 step rewrites P + n)
            block = torch.cat([y, d])
            prev, y, P = block[n:n + 1], a[n:n + 1], P + n + 1
            trim_prompt_cache(cache[:nt], k - n)
            trim_prompt_cache(cache[nt:], k - n)


def _check_fused(model, draft_model, cache: list) -> None:
    """The device driver captures its rounds: every cache of the list (the target's, then the draft's) must be on the
    fused decode path, whose positions live on the device."""
    nt = len(model.layers)
    for m, cs in ((model, cache[:nt]), (draft_model, cache[nt:])):
        if not all(qllama.FUSED_DECODE and layer.self_attn.takes_fused_decode(c) for layer, c in zip(m.layers, cs)):
            raise ValueError("speculative decoding on the device: a cache is off the fused decode path (raise "
                             "GBXQ_FUSED_DECODE or use a quantized cache for contexts above 49152 keys)")


class _SpecGraph:
    """One round of speculative decoding captured in a CUDA graph: the draft's steps with their argmax fed back, the
    verify step, the accept rule, the write of a_0 .. a_k into `out` at `idx`, and the advance of P / prev / y -- all
    on device tensors, so rounds replay back to back without the host."""

    def __init__(self, model, draft_model, cache: list, k: int, prev, y, P: int, out: torch.Tensor, idx: torch.Tensor,
                 accepted: torch.Tensor):
        nt = len(model.layers)
        self.k, self.tc, self.dc = k, cache[:nt], cache[nt:]
        _check_fused(model, draft_model, cache)
        dev = out.device
        self.prev, self.y = prev.clone(), y.clone()
        self.P = torch.tensor([P], dtype=torch.long, device=dev)
        self.out, self.idx, self.accepted = out, idx, accepted
        self.model, self.draft_model = model, draft_model
        state = (self.prev, self.y, self.P, self.out, self.idx, self.accepted)
        snap = [t.clone() for t in state]
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s), torch.no_grad():
            for _ in range(2):  # warm-up (workspaces, libraries); it writes the rows the first replay writes anyway
                self._round()
                for t, v in zip(state, snap):
                    t.copy_(v)
        torch.cuda.current_stream().wait_stream(s)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph), torch.no_grad():
            self._round()

    def _round(self):
        k = self.k
        d, logits = _draft_and_verify(self.model, self.draft_model, self.tc, self.dc, self.prev, self.y, self.P, k,
                                      lambda lg: fast_argmax(lg).reshape(1))
        a = fast_argmax(logits)  # [k + 1]
        n = (a[:k] == d).long().cumprod(0).sum().reshape(1)  # leading matches
        self.out.index_copy_(0, self.idx + torch.arange(k + 1, device=a.device), a)
        self.prev.copy_(torch.cat([self.y, d]).index_select(0, n))
        self.y.copy_(a.index_select(0, n))
        self.P.add_(n + 1)
        self.idx.add_(n + 1)
        self.accepted.add_(n)


def _speculative_device(model, draft_model, y0: torch.Tensor, max_tokens: int, k: int, prefill_step_size: int,
                        kv: dict) -> Tuple[List[int], float, dict]:
    """generate_tokens_device with a draft: rounds of _SpecGraph, r = ceil(remaining / (k + 1)) replays between host
    synchronisations (each round emits 1 .. k + 1 tokens, so at most k past max_tokens, dropped).  Before the kv_bits
    conversion the host synchronises every round, converts both lists after the round whose verify takes the target's
    offset past quantized_kv_start, and captures the round again."""
    dev = y0.device
    cache = _spec_cache(model, draft_model, y0.numel() + max_tokens + k + 2)
    # refused before the prefill when the rounds start on these bf16 caches; when the prefill converts them (kv_bits,
    # a prompt longer than quantized_kv_start), the converted caches are checked right after it
    if kv["kv_bits"] is None or y0.numel() <= kv["quantized_kv_start"]:
        _check_fused(model, draft_model, cache)
    nt = len(model.layers)
    tc, dc = cache[:nt], cache[nt:]
    tok = fast_argmax(prefill(model, y0, tc, prefill_step_size, **kv)[0]).reshape(1)
    prefill(draft_model, y0, dc, prefill_step_size, **kv)
    cache[:] = tc + dc
    _check_fused(model, draft_model, cache)
    out = torch.zeros((max_tokens + k + 1,), dtype=torch.long, device=dev)
    out[:1] = tok
    idx = torch.ones((1,), dtype=torch.long, device=dev)
    accepted = torch.zeros((1,), dtype=torch.long, device=dev)
    P, rounds = y0.numel(), 0
    pending = kv["kv_bits"] is not None and isinstance(cache[0], StaticKVCache)  # a conversion still to come
    sg = _SpecGraph(model, draft_model, cache, k, y0[-1:], tok, P, out, idx, accepted) if max_tokens > 1 else None
    t_first = time.perf_counter()
    emitted = 1
    while emitted < max_tokens:
        r = 1 if pending else -(-(max_tokens - emitted) // (k + 1))
        for _ in range(r):
            sg.graph.replay()
        rounds += r
        if pending:
            P_start = int(sg.P) - (int(sg.idx) - emitted)
            for i, c in enumerate(cache):  # the offsets after this round's verify (target) and last draft step
                c.offset = P_start + k + (1 if i < nt else 0)
            maybe_quantize_kv_cache(cache, kv["quantized_kv_start"], kv["kv_group_size"], kv["kv_bits"])
            if not isinstance(cache[0], StaticKVCache):
                pending = False
                sg = _SpecGraph(model, draft_model, cache, k, sg.prev, sg.y, int(sg.P), out, idx, accepted)
        emitted = int(idx)
    if sg is not None:
        P = int(sg.P)
    for i, c in enumerate(cache):
        c.offset = P if i < nt else P - 1
    stats = {"draft_tokens": rounds * k, "accepted_tokens": int(accepted),
             "acceptance_rate": int(accepted) / max(rounds * k, 1)}
    return out[:max_tokens].tolist(), t_first, stats


def generate_tokens_device(model, prompt: torch.Tensor, max_tokens: int = 128, prefill_step_size: int = 2048,
                           kv_bits: Optional[int] = None, kv_group_size: int = 64, quantized_kv_start: int = 0,
                           max_kv_size: Optional[int] = None, draft_model: Optional[nn.Module] = None,
                           num_draft_tokens: int = 2) -> Tuple[List[int], dict]:
    """Greedy generation with the sampler inside the captured decode step (DecodeGraph device_loop): the same tokens as
    `generate_tokens` (argmax of the log-probabilities = argmax of the logits), but the host only enqueues replays and
    reads the tokens once at the end -- the per-token host round trip of utils.py:299-337 (~0.3-0.6 ms on a B200 box)
    is gone.  Same timing definitions as generate_tokens.  kv_bits / kv_group_size / quantized_kv_start as in
    generate_step: when the conversion falls inside the decode, the graph replays up to that step, the caches are
    converted, and a graph of the quantized step replays the rest.  max_kv_size as in generate_step: the captured step
    writes the ring slot of its device-side position, so the replays wrap without the host.
    draft_model: speculative decoding with num_draft_tokens = k drafts a round (speculative_generate_step's schedule and
    tokens), each round one captured graph (_SpecGraph); the stats add draft_tokens, accepted_tokens and
    acceptance_rate."""
    y = prompt.reshape(-1).to(next(model.parameters()).device)
    n_prompt = y.numel()
    if draft_model is not None:
        _check_speculative(model, draft_model, num_draft_tokens, max_kv_size)
        kv = dict(kv_bits=kv_bits, kv_group_size=kv_group_size, quantized_kv_start=quantized_kv_start)
        t0 = time.perf_counter()
        with torch.no_grad():
            toks, t_first, spec = _speculative_device(model, draft_model, y, max_tokens, num_draft_tokens,
                                                      prefill_step_size, kv)
        t1 = time.perf_counter()
        return toks, {"prompt_tokens": int(n_prompt), "prompt_tps": n_prompt / max(t_first - t0, 1e-9),
                      "generation_tokens": len(toks), "generation_tps": max(len(toks) - 1, 1) / max(t1 - t_first, 1e-9),
                      **spec}
    cache = _prompt_cache(model, n_prompt + max_tokens + 1, max_kv_size)
    kv = dict(kv_bits=kv_bits, kv_group_size=kv_group_size, quantized_kv_start=quantized_kv_start)
    t0 = time.perf_counter()
    tok = torch.argmax(prefill(model, y, cache, prefill_step_size, **kv).float(), dim=-1)
    pos0 = cache[0].offset
    first, t_first, outs = _device_decode(model, cache, tok, pos0, pos0, max(max_tokens - 1, 0), kv,
                                          "generate_tokens_device")
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    toks = first + [int(t) for o in outs for t in o[:, 0].tolist()]
    stats = {
        "prompt_tokens": int(n_prompt), "prompt_tps": n_prompt / max(t_first - t0, 1e-9),
        "generation_tokens": len(toks), "generation_tps": max(len(toks) - 1, 1) / max(t1 - t_first, 1e-9),
    }
    return toks, stats


def _pad_prompts(prompts, pad_id: int, max_kv_size: Optional[int]) -> Tuple[torch.Tensor, List[int]]:
    """The prompts (1-D token-id tensors) right-padded with pad_id into one [B, Lmax] matrix, and their lengths."""
    if len(prompts) == 0:
        raise ValueError("batch_generate: no prompts")
    if any(p.dim() != 1 for p in prompts):
        raise ValueError("batch_generate: each prompt must be a 1-D tensor of token ids")
    lens = [int(p.numel()) for p in prompts]
    if min(lens) == 0:
        raise ValueError(f"batch_generate: prompt {lens.index(0)} is empty")
    if max_kv_size is not None and max(lens) > max_kv_size:
        # the prefill ring logic (window_with / store_runs) runs on one shared offset: pads would push real tokens out
        raise ValueError(f"batch_generate: the longest prompt ({max(lens)} tokens) exceeds max_kv_size = {max_kv_size}")
    tokens = torch.full((len(prompts), max(lens)), int(pad_id), dtype=torch.long)
    for b, p in enumerate(prompts):
        tokens[b, :lens[b]] = p.to(torch.long)
    return tokens, lens


def batch_generate(model, prompts: List[torch.Tensor], max_tokens: int = 128, *, prefill_step_size: int = 2048,
                   kv_bits: Optional[int] = None, kv_group_size: int = 64, quantized_kv_start: int = 0,
                   max_kv_size: Optional[int] = None, pad_id: int = 0,
                   use_cuda_graph: bool = True) -> Tuple[List[List[int]], dict]:
    """Greedy generation of `max_tokens` tokens for each of B prompts of any lengths (1-D token-id tensors), in one batch.

    The prompts are padded on the right to the longest, Lmax, and prefilled together at the shared positions
    0 .. Lmax-1: under the causal mask no real token sees a pad, and row b's first token is the argmax at its column
    len_b - 1.  Each decode step then runs the B rows at their own positions (row b's s-th step at len_b + s): the
    step writes that row's cache row and attends that row's keys 0 .. len_b + s, so the pad keys of row b are
    overwritten before any of its queries can see them, and no row's tokens depend on the pads or on the other rows.
    kv_bits / kv_group_size / quantized_kv_start / max_kv_size as in generate_step (the conversion rule reads the
    caches' offset, Lmax + steps so far); the longest prompt must fit max_kv_size.  use_cuda_graph: the captured step
    with the sampler inside (as generate_tokens_device); False: eager steps, the same tokens.

    Returns (the tokens of each row, stats) with the reference's timing definitions summed over the rows:
    prompt_tps = prompt tokens / time to the first tokens, generation_tps = generated tokens / decode time."""
    dev = next(model.parameters()).device
    tokens, lens = _pad_prompts(prompts, pad_id, max_kv_size)
    B, Lmax = tokens.shape
    tokens = tokens.to(dev)
    kv = dict(kv_bits=kv_bits, kv_group_size=kv_group_size, quantized_kv_start=quantized_kv_start)
    cache = _prompt_cache(model, Lmax + max_tokens + 1, max_kv_size, batch=B)
    steps = max(max_tokens - 1, 0)
    t0 = time.perf_counter()
    tok = fast_argmax(_prefill_chunks(model, tokens, cache, prefill_step_size, kv, last=[n - 1 for n in lens]))
    position = torch.tensor(lens, dtype=torch.long, device=dev)  # of each row's first decode step
    if use_cuda_graph:
        first, t_first, outs = _device_decode(model, cache, tok, position, Lmax, steps, kv, "batch_generate")
        rows = [first] + [r for o in outs for r in o.tolist()]
    else:
        quantize_cache = _kv_quantizer(cache, **kv)
        rows = [tok.tolist()]
        t_first = time.perf_counter()
        with torch.no_grad():
            for s in range(steps):
                for c in cache:
                    c.offset = Lmax + s + 1
                logits = model(tok[:, None], cache, positions=position[:, None], attend_len=cache[0].attend_len)
                quantize_cache()
                tok = fast_argmax(logits[:, -1, :])
                position = position + 1
                rows.append(tok.tolist())
    if tok.is_cuda:
        torch.cuda.synchronize(dev)
    t1 = time.perf_counter()
    out = [list(r) for r in zip(*rows)]  # rows: the B tokens of each step
    stats = {
        "prompt_tokens": int(sum(lens)), "prompt_tps": sum(lens) / max(t_first - t0, 1e-9),
        "generation_tokens": B * len(out[0]), "generation_tps": B * max(len(out[0]) - 1, 1) / max(t1 - t_first, 1e-9),
    }
    return out, stats


def generate_tokens(model, prompt: torch.Tensor, max_tokens: int = 128, **kw) -> Tuple[List[int], dict]:
    """Greedy generation + the reference's timing definitions (utils.py:590-607):
    prompt_tps = prompt_len / time_to_first_token, generation_tps = n / (t_now - t_first).  Keyword arguments
    (use_cuda_graph, prefill_step_size, kv_bits, kv_group_size, quantized_kv_start, ...) go to generate_step; with
    draft_model (and num_draft_tokens) to speculative_generate_step."""
    toks = []
    t0 = time.perf_counter()
    t_first = None
    draft_model = kw.pop("draft_model", None)
    if draft_model is not None:
        _check_speculative(model, draft_model, kw.get("num_draft_tokens", 2), kw.pop("max_kv_size", None))
        kw.pop("use_cuda_graph", None)
        steps = ((t, lp) for t, lp, _ in speculative_generate_step(prompt, model, draft_model, max_tokens=max_tokens, **kw))
    else:
        steps = generate_step(prompt, model, max_tokens=max_tokens, **kw)
    for tok, _ in steps:
        if t_first is None:
            t_first = time.perf_counter()
        toks.append(tok)
    t1 = time.perf_counter()
    stats = {
        "prompt_tokens": int(prompt.numel()), "prompt_tps": prompt.numel() / max(t_first - t0, 1e-9),
        "generation_tokens": len(toks), "generation_tps": max(len(toks) - 1, 1) / max(t1 - t_first, 1e-9),
    }
    return toks, stats
