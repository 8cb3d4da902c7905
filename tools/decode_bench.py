#!/usr/bin/env python
"""End-to-end decode through the CALLERS of the hot path (SURVEY.md 8a A4-A7, BASELINE.json configs[0]): synthetic
layer-mix checkpoint in the gba2mlx layout -> load_model (quant_strategy.json, safetensors) -> greedy generate of N
tokens at batch 1 (CUDA-graph decode step: 7 L QuantizedLinear forwards through libgbxq + torch glue + bf16 head),
timed with the reference's own definitions (gbx_lm/utils.py:590-607).  Prints one JSON line.

    python tools/decode_bench.py [--model llama-3.2-1b] [--strategy bpw-4.0] [--tokens 128] [--prompt 32]
                                 [--kv-bits none,8,4] [--kv-group-size 64] [--quantized-kv-start N]
                                 [--max-kv-size none,W] [--graph-positions P1,P2,...] [--batch B1,B2,... [--ragged]]

--kv-bits takes a comma-separated list (none = the bf16 cache); one JSON line per entry, from one model load.  With a
width the caches are converted to the group-quantized cache after the model call that takes them past
--quantized-kv-start (the reference's generate_step rule); a start one below the prompt length prefills on bf16 and
converts once before the decode.

--max-kv-size takes a comma-separated list too (none = the flat cache, W = rotating caches of W positions with 4 sinks,
`generate_step(max_kv_size=W)`); every (kv-bits, max-kv-size) pair is one JSON line.  --graph-positions times the
captured step at each listed position as well (default: the prompt length); on a rotating cache every position past
the window attends the same W keys.

--batch takes a comma-separated list of batch sizes B: each (B, kv-bits, max-kv-size) is one JSON line of
`utils.batch_generate` on B prompts of --prompt tokens each, or with --ragged of lengths spread evenly over
[prompt/2, prompt]: the aggregate generation rate of the rows (device sampler inside the captured step), the captured
step's device time at the rows' first decode positions, and the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gbx_lm_b200 import ops, utils  # noqa: E402
from gbx_lm_b200.cache import DEFAULT_KV_KEEP  # noqa: E402
from gbx_lm_b200 import workloads as W  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="llama-3.2-1b")
    ap.add_argument("--strategy", default="bpw-4.0", choices=["bpw-4.0", "bpw-2.2", "uniform"])
    ap.add_argument("--tokens", type=int, default=128)
    ap.add_argument("--prompt", type=int, default=32)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--kv-bits", default="none")
    ap.add_argument("--kv-group-size", type=int, default=64)
    ap.add_argument("--quantized-kv-start", type=int, default=0)
    ap.add_argument("--max-kv-size", default="none")
    ap.add_argument("--graph-positions", default="")
    ap.add_argument("--batch", default="")
    ap.add_argument("--ragged", action="store_true")
    args = ap.parse_args()
    dims = W.MODELS[args.model]
    strat = None if args.strategy == "uniform" else W.STRATEGIES[args.strategy](dims.layers)
    d = Path(tempfile.mkdtemp(prefix="gbxq_ckpt_"))
    try:
        t0 = time.perf_counter()
        utils.write_synthetic_checkpoint(d, dims, strat, seed=0, default_bits=4, default_gs=64, embed_scale=1.0)
        t_write = time.perf_counter() - t0
        t0 = time.perf_counter()
        model, cfg = utils.load_model(d, device="cuda")
        torch.cuda.synchronize()
        t_load = time.perf_counter() - t0
    finally:
        shutil.rmtree(d, ignore_errors=True)
    prompt = torch.randint(0, dims.vocab, (args.prompt,), generator=torch.Generator().manual_seed(1))
    none_or_int = lambda s: None if s.strip().lower() == "none" else int(s)
    for size in args.max_kv_size.split(","):
        for kv in args.kv_bits.split(","):
            if args.batch:
                for B in args.batch.split(","):
                    run_batch(args, dims, model, int(B), none_or_int(kv), none_or_int(size))
            else:
                run(args, dims, strat, model, prompt, none_or_int(kv), none_or_int(size), t_write, t_load)


def gpu_name_and_power_limit():
    """(name, power limit in W) of GPU 0, read now: a rate is a number of the card and the limit it ran at."""
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        limit = float(r.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        limit = None
    return torch.cuda.get_device_name(0), limit


def batch_lengths(prompt: int, B: int, ragged: bool):
    """B prompt lengths: all `prompt`, or spread evenly over [prompt // 2, prompt] (the last row the longest)."""
    if not ragged or B == 1:
        return [prompt] * B
    lo = prompt // 2
    return [lo + round(b * (prompt - lo) / (B - 1)) for b in range(B)]


def run_batch(args, dims, model, B, kv_bits, max_kv_size):
    lens = batch_lengths(args.prompt, B, args.ragged)
    gen = torch.Generator().manual_seed(1)
    prompts = [torch.randint(0, dims.vocab, (n,), generator=gen) for n in lens]
    kw = dict(kv_bits=kv_bits, kv_group_size=args.kv_group_size, quantized_kv_start=args.quantized_kv_start,
              max_kv_size=max_kv_size)
    toks0, best = utils.batch_generate(model, prompts, args.tokens, **kw)  # warm-up (allocator, library state)
    for _ in range(args.repeat):
        toks, stats = utils.batch_generate(model, prompts, args.tokens, **kw)
        assert toks == toks0, "batched greedy decode is not reproducible run to run"
        if stats["generation_tps"] > best["generation_tps"]:
            best = stats
    # device time of the captured per-row step at the rows' first decode positions, on the cache the decode runs on
    from gbx_lm_b200.cache import StaticQuantizedKVCache

    Lmax = max(lens)
    cache = utils._prompt_cache(model, Lmax + args.tokens + 1, max_kv_size, batch=B)
    kv = {k: v for k, v in kw.items() if k != "max_kv_size"}
    pad = torch.zeros((B, Lmax), dtype=torch.long)
    for b, p in enumerate(prompts):
        pad[b, :lens[b]] = p
    tok = utils.fast_argmax(utils._prefill_chunks(model, pad.cuda(), cache, 2048, kv, last=[n - 1 for n in lens]))
    quantized = isinstance(cache[0], StaticQuantizedKVCache)
    dg = utils.DecodeGraph(model, cache, batch=B, per_row=True).capture(tok, torch.tensor(lens, device="cuda"))
    for _ in range(5):
        dg.graph.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(50):
        dg.graph.replay()
    e1.record()
    torch.cuda.synchronize()
    graph_ms = e0.elapsed_time(e1) / 50
    del dg, cache
    name, limit = gpu_name_and_power_limit()
    print(json.dumps({
        "tool": "decode_bench", "mode": "batch_generate", "model": args.model, "strategy": args.strategy, "batch": B,
        "ragged": bool(args.ragged and B > 1), "prompt_lengths": lens, "prompt_tokens": sum(lens),
        "kv_bits": kv_bits, "kv_group_size": args.kv_group_size if kv_bits else None,
        "quantized_kv_start": args.quantized_kv_start if kv_bits else None, "decode_cache": "quantized" if quantized else "bf16",
        "max_kv_size": max_kv_size, "tokens_per_row": args.tokens, "generation_tokens": best["generation_tokens"],
        "generation_tps": round(best["generation_tps"], 1), "generation_tps_per_row": round(best["generation_tps"] / B, 1),
        "prompt_tps": round(best["prompt_tps"], 1), "graph_ms_per_step": round(graph_ms, 4),
        "graph_tps_per_step": round(B * 1e3 / graph_ms, 1), "repeat": args.repeat,
        "data": "synthetic (random-init, seed 0)", "gpu": name, "power_limit_w": limit,
        "note": "generation_tps: aggregate over the rows, batch_generate with the greedy sampler inside the captured step "
                "(best of --repeat runs after one warm-up run); graph_ms_per_step: device time of the captured per-row "
                "step at the rows' first decode positions, mean of 50 replays",
    }), flush=True)


def run(args, dims, strat, model, prompt, kv_bits, max_kv_size, t_write, t_load):
    from gbx_lm_b200.cache import StaticQuantizedKVCache

    kw = dict(kv_bits=kv_bits, kv_group_size=args.kv_group_size, quantized_kv_start=args.quantized_kv_start,
              max_kv_size=max_kv_size)
    best, toks0 = None, None
    for r in range(args.repeat):
        n0 = ops.launch_count()
        toks, stats = utils.generate_tokens(model, prompt, max_tokens=args.tokens, use_cuda_graph=True, **kw)
        stats["gbxq_launches"] = ops.launch_count() - n0
        if toks0 is None:
            toks0 = toks
        assert toks == toks0, "greedy decode is not reproducible run to run"
        if best is None or stats["generation_tps"] > best["generation_tps"]:
            best = stats
    d_toks, d_stats = utils.generate_tokens_device(model, prompt, max_tokens=args.tokens, **kw)
    d_toks, d_stats = utils.generate_tokens_device(model, prompt, max_tokens=args.tokens, **kw)
    assert d_toks == toks0, "device-side greedy sampler diverged from the host-side one"
    # device time of the captured decode step alone (no sampling, no host sync between steps), on the cache the decode
    # runs on: converted after the prompt when kv_bits is set and the prompt is past quantized_kv_start
    # (and the prefill alone, device-synchronised, on that cache)
    cache = utils._prompt_cache(model, args.prompt + args.tokens + 1, max_kv_size)
    kv = {k: v for k, v in kw.items() if k != "max_kv_size"}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    utils.prefill(model, prompt.cuda(), cache, **kv)
    torch.cuda.synchronize()
    prefill_ms = (time.perf_counter() - t0) * 1e3
    quantized = isinstance(cache[0], StaticQuantizedKVCache)
    graph_ms = {}
    for pos in [args.prompt] + [int(p) for p in args.graph_positions.split(",") if p]:
        # the step's cost depends on the position (the keys it attends), not on the cache's contents
        dg = utils.DecodeGraph(model, cache).capture(torch.tensor([1], device="cuda"), pos)
        for _ in range(5):
            dg.graph.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(50):
            dg.graph.replay()
        e1.record()
        torch.cuda.synchronize()
        graph_ms[pos] = round(e0.elapsed_time(e1) / 50, 4)
        del dg
    del cache
    plan = W.layer_plan(dims, strat, 4, 64)
    body = sum(W.qmm_bytes(1, n, k, b, g) for (_, _, n, k, b, g) in plan)
    head = dims.vocab * dims.hidden * 2
    hd = dims.head_dim or dims.hidden // dims.heads
    row = hd * kv_bits // 8 + 2 * 2 * (hd // args.kv_group_size) if quantized else hd * 2
    kv_per_token = dims.layers * dims.kv_heads * 2 * row
    ctx = args.prompt + args.tokens // 2  # mean visible keys over the decode
    if max_kv_size is not None:
        ctx = min(ctx, max_kv_size)
    print(json.dumps({
        "tool": "decode_bench", "model": args.model, "strategy": args.strategy, "batch": 1, "prompt_tokens": args.prompt,
        "kv_bits": kv_bits, "kv_group_size": args.kv_group_size if kv_bits else None,
        "quantized_kv_start": args.quantized_kv_start if kv_bits else None, "decode_cache": "quantized" if quantized else "bf16",
        "max_kv_size": max_kv_size, "kv_keep": DEFAULT_KV_KEEP if max_kv_size else None,
        "kv_bytes_per_token": kv_per_token, "kv_bytes_per_step_at_mean_context": kv_per_token * ctx,
        "generation_tokens": best["generation_tokens"], "generation_tps": round(best["generation_tps"], 1),
        "prompt_tps": round(best["prompt_tps"], 1), "ms_per_token": round(1e3 / best["generation_tps"], 4),
        "generation_tps_device_sampler": round(d_stats["generation_tps"], 1), "graph_ms_per_step": graph_ms[args.prompt],
        "graph_ms_at_position": graph_ms, "prefill_ms": round(prefill_ms, 2), "gbxq_launches_per_generate": best["gbxq_launches"],
        "device_tokens_equal_host_tokens": True,
        "qmm_bytes_per_token": body, "head_bytes_per_token": head,
        "hbm_gbs_body_plus_head": round((body + head) * best["generation_tps"] / 1e9, 1),
        "checkpoint_write_s": round(t_write, 1), "load_s": round(t_load, 1), "data": "synthetic (random-init, seed 0)",
        "gpu": torch.cuda.get_device_name(0),
        "note": "whole decode step: quantized forwards + decode glue through libgbxq (GBXQ_FUSED_DECODE=0: torch glue), bf16 head via cuBLAS; generation_tps syncs with the host every token, generation_tps_device_sampler does not; graph_ms_per_step is the captured step at position prompt_tokens; prefill_ms is utils.prefill of the prompt alone",
    }), flush=True)


if __name__ == "__main__":
    main()
