#!/usr/bin/env python
"""Speculative decoding on synthetic checkpoints: what a draft-and-verify round costs against the plain decode step.

    python tools/spec_bench.py [--target llama-3-8b] [--draft llama-3.2-1b] [--prompts 512,8000] [--ks 1,2,3,4,7]
                               [--kv-bits none,4] [--tokens 128]

For each cache (bf16, or converted to --kv-bits at prefill) and prompt length, one JSON line per k with:
- t1_step_ms: the captured T = 1 decode step of the target (utils.DecodeGraph), verify_step_ms: the captured step of
  T = k + 1 tokens (Model.forward with explicit positions), both at the prompt's position;
- draft_t2_ms / draft_t1_ms: the draft's T = 2 and T = 1 steps, for the --draft model and for the target as its own
  draft (its t1 is t1_step_ms);
- round_ms: one captured round with the --draft model (utils._SpecGraph), timed over replays;
- e2e tok/s of generate_tokens_device: plain, with draft = target (acceptance about 1, the upper bound), with the --draft
  model on random weights (acceptance about 0, the cost of speculating for nothing);
- projected_tps: (1 - a^(k+1)) / (1 - a) tokens per measured round at a in {0.5, 0.7, 0.9} -- a PROJECTION: synthetic
  weights say nothing about the acceptance a real draft reaches.
Every line carries the GPU's name and power limit, read in the same run.  Times are CUDA events over graph replays."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gbx_lm_b200 import qllama, utils  # noqa: E402
from gbx_lm_b200 import workloads as W  # noqa: E402
from gbx_lm_b200.cache import maybe_quantize_kv_cache  # noqa: E402


def gpu_info() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers are still device times; say what could not be read
        return f"unknown ({e})"


def load(name: str, seed: int, root: Path):
    dims = W.MODELS[name]
    d = root / name
    utils.write_synthetic_checkpoint(d, dims, W.STRATEGIES["bpw-4.0"](dims.layers), seed=seed, default_bits=4,
                                     default_gs=64, embed_scale=dims.hidden ** -0.5)
    model, _ = utils.load_model(d, device="cuda")
    shutil.rmtree(d)
    return model


def time_graph(graph: torch.cuda.CUDAGraph, n: int = 50) -> float:
    for _ in range(3):
        graph.replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        graph.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def capture(fn) -> torch.cuda.CUDAGraph:
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s), torch.no_grad():
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g), torch.no_grad():
        fn()
    return g


def prefilled(model, prompt, run_len: int, kv_bits):
    cache = qllama.make_prompt_cache(model, 1, run_len)
    utils.prefill(model, prompt, cache, kv_bits=kv_bits, kv_group_size=64, quantized_kv_start=0)
    return cache


def block_step_ms(model, prompt, kv_bits, T: int) -> float:
    """The captured step of T tokens at the prompt's position (T = 1: the decode step of DecodeGraph)."""
    P = prompt.numel()
    cache = prefilled(model, prompt, P + 16, kv_bits)
    if T == 1:
        dg = utils.DecodeGraph(model, cache).capture(prompt[-1:], P)
        return time_graph(dg.graph)
    toks = prompt[-T:][None].clone()
    pos = torch.arange(P, P + T, device=prompt.device)
    return time_graph(capture(lambda: model(toks, cache, positions=pos)))


def round_ms(model, draft, prompt, kv_bits, k: int, n: int = 30) -> float:
    P = prompt.numel()
    cache = prefilled(model, prompt, P + n * (k + 1) + 64, kv_bits) + prefilled(draft, prompt, P + n * (k + 1) + 64,
                                                                              kv_bits)
    out = torch.zeros((n * (k + 1) + 64,), dtype=torch.long, device=prompt.device)
    idx, acc = torch.zeros((1,), dtype=torch.long, device=out.device), torch.zeros((1,), dtype=torch.long, device=out.device)
    sg = utils._SpecGraph(model, draft, cache, k, prompt[-1:], prompt[-1:], P, out, idx, acc)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        sg.graph.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--target", default="llama-3-8b")
    ap.add_argument("--draft", default="llama-3.2-1b")
    ap.add_argument("--prompts", default="512,8000")
    ap.add_argument("--ks", default="1,2,3,4,7")
    ap.add_argument("--kv-bits", default="none,4")
    ap.add_argument("--tokens", type=int, default=128)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("spec_bench needs a GPU")
    gpu = gpu_info()
    root = Path(tempfile.mkdtemp(prefix="gbxq_spec_"))
    try:
        target, draft = load(args.target, 1, root), load(args.draft, 2, root)
        for kvs in args.kv_bits.split(","):
            kv_bits = None if kvs == "none" else int(kvs)
            for plen in (int(x) for x in args.prompts.split(",")):
                prompt = torch.randint(0, target.args.vocab_size, (plen,), generator=torch.Generator().manual_seed(plen))
                prompt = prompt.cuda()
                kw = dict(kv_bits=kv_bits, kv_group_size=64, quantized_kv_start=0)
                t1 = block_step_ms(target, prompt, kv_bits, 1)
                d1, d2 = block_step_ms(draft, prompt, kv_bits, 1), block_step_ms(draft, prompt, kv_bits, 2)
                t2 = block_step_ms(target, prompt, kv_bits, 2)
                with torch.no_grad():
                    _, plain = utils.generate_tokens_device(target, prompt, args.tokens, **kw)
                for k in (int(x) for x in args.ks.split(",")):
                    with torch.no_grad():
                        verify = block_step_ms(target, prompt, kv_bits, k + 1)
                        rnd = round_ms(target, draft, prompt, kv_bits, k)
                        _, self_st = utils.generate_tokens_device(target, prompt, args.tokens, draft_model=target,
                                                                  num_draft_tokens=k, **kw)
                        _, rand_st = utils.generate_tokens_device(target, prompt, args.tokens, draft_model=draft,
                                                                  num_draft_tokens=k, **kw)
                    proj = {str(a): round((1 - a ** (k + 1)) / (1 - a) / (rnd * 1e-3), 1) for a in (0.5, 0.7, 0.9)}
                    print(json.dumps({
                        "gpu": gpu, "target": args.target, "draft": args.draft, "kv_bits": kv_bits, "prompt": plen,
                        "k": k, "t1_step_ms": round(t1, 4), "verify_step_ms": round(verify, 4),
                        "draft_t1_ms": round(d1, 4), "draft_t2_ms": round(d2, 4), "target_as_draft_t2_ms": round(t2, 4),
                        "round_ms": round(rnd, 4), "plain_tps": round(plain["generation_tps"], 1),
                        "self_draft_tps": round(self_st["generation_tps"], 1),
                        "self_draft_acceptance": round(self_st["acceptance_rate"], 3),
                        "random_draft_tps": round(rand_st["generation_tps"], 1),
                        "random_draft_acceptance": round(rand_st["acceptance_rate"], 3),
                        "projected_tps_at_acceptance": proj}), flush=True)
    finally:
        shutil.rmtree(root, ignore_errors=True)


if __name__ == "__main__":
    main()
