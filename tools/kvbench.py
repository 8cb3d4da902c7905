#!/usr/bin/env python
"""Decode attention over the KV cache, one query token (B = 1), at the attention shapes of Llama-3-8B (Hq 32), Llama-3.2-3B
(Hq 24) with Hkv 8 / D 128, and Llama-3.2-1B (Hq 32, Hkv 8, D 64), for 1K .. 128K visible keys:

    bf16        gbxq_decode_attention (one CTA per query head; refuses more than 49 152 keys)
    q8 / q4     gbxq_decode_attention_quantized on an 8- / 4-bit group-64 cache (split-K over 256-key chunks + combine)
    qsdpa4      switch_layers.quantized_scaled_dot_product_attention on the 4-bit cache (two gbxq_gather_qmm launches and
                a torch softmax: the reference's own formulation, the prefill path)

Timing: CUDA events around replays of a CUDA graph that holds one call per layer cache (no host launch cost inside).
One layer's cache at 32K keys fits the 126 MB L2, so the timed loop rotates over `--layers` (default 32) distinct layer
caches, as a decode step does.  Bytes are the algorithm's: the visible keys' codes +
scales + biases (bf16: the rows) for K and V, plus q and out.  Share of peak = bytes / time / HBM peak
(MEASURED_PEAKS.json hbm_gbs as bench.py reads it, else the data-sheet 7.7 TB/s, labelled).  Prints one line per case and
a JSON summary.

    python tools/kvbench.py [--contexts 1024,4096,16384,32768,131072] [--layers 32] [--iters 20] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gbx_lm_b200 import ops, switch_layers  # noqa: E402
from gbx_lm_b200.cache import DECODE_ATTENTION_MAX_KEYS  # noqa: E402

SHAPES = [("llama-3-8b", 32, 8, 128), ("llama-3.2-3b", 24, 8, 128), ("llama-3.2-1b", 32, 8, 64)]


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except (KeyError, ValueError):
            pass
    return 7700.0, "data sheet (HGX B200, 7.7 TB/s per GPU; not measured here)"


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                            capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        pl = f"unavailable ({e})"
    return name, pl


def kv_bytes(kind, n, hkv, d):
    if kind == "bf16":
        return 2 * n * hkv * d * 2
    bits = 8 if kind == "q8" else 4
    return 2 * n * hkv * (d * bits // 8 + 2 * 2 * (d // 64))


def time_calls(fn, layers, iters):
    """µs per call: one rotation over the layer caches captured in a CUDA graph (no host launch cost in the window),
    replayed `iters` times between two events."""
    for i in range(layers):  # warm-up every layer cache once (also sizes the attention workspace before capture)
        fn(i)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(layers):
            fn(i)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (iters * layers)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--contexts", default="1024,4096,16384,32768,131072")
    ap.add_argument("--layers", type=int, default=32)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("kvbench needs a CUDA device")
    dev = torch.device("cuda:0")
    peak, peak_src = hbm_peak()
    name, power = gpu_info()
    print(f"# {name}; power.limit, clocks.max.sm = {power}; HBM peak {peak:.0f} GB/s ({peak_src})")
    print(f"# timed loop rotates over {args.layers} distinct layer caches (one 32K-key layer fits in L2), one CUDA graph of "
          f"{args.layers} calls replayed {args.iters} times")
    rows = []
    g = torch.Generator(device=dev).manual_seed(0)
    for model, hq, hkv, d in SHAPES:
        for n in [int(c) for c in args.contexts.split(",")]:
            q = torch.randn((1, hq, d), generator=g, device=dev).to(torch.bfloat16)
            pos = torch.tensor([n - 1], device=dev)
            scale = d ** -0.5
            for kind in ("bf16", "q8", "q4", "qsdpa4"):
                if kind == "bf16" and n > DECODE_ATTENTION_MAX_KEYS:
                    rows.append({"model": model, "keys": n, "cache": kind, "us": None, "note": "above the kernel's 49 152-key cap"})
                    print(f"{model:13s} keys {n:7d} {kind:7s}  -- above the bf16 kernel's 49 152-key cap")
                    continue
                caches = []
                for _ in range(args.layers):
                    if kind == "bf16":
                        kc = torch.randn((1, hkv, n, d), generator=g, device=dev).to(torch.bfloat16)
                        vc = torch.randn((1, hkv, n, d), generator=g, device=dev).to(torch.bfloat16)
                        caches.append((kc, vc))
                    else:
                        bits = 8 if kind == "q8" else 4
                        kv = torch.randn((2, 1, hkv, n, d), generator=g, device=dev).to(torch.bfloat16)
                        caches.append((ops.quantize(kv[0], 64, bits), ops.quantize(kv[1], 64, bits)))
                        del kv
                if kind == "bf16":
                    fn = lambda i: ops.decode_attention(q, caches[i][0], caches[i][1], pos, scale, n)  # noqa: E731
                elif kind in ("q8", "q4"):
                    bits = 8 if kind == "q8" else 4
                    fn = lambda i: ops.decode_attention_quantized(q, caches[i][0], caches[i][1], pos, scale, 64, bits, n)  # noqa: E731
                else:
                    fn = lambda i: switch_layers.quantized_scaled_dot_product_attention(  # noqa: E731
                        q[:, :, None], caches[i][0], caches[i][1], scale, None, 64, 4)
                us = time_calls(fn, args.layers, args.iters)
                nbytes = kv_bytes("bf16" if kind == "bf16" else ("q8" if kind == "q8" else "q4"), n, hkv, d) + 2 * hq * d * 2
                frac = nbytes / (us * 1e-6) / (peak * 1e9)
                rows.append({"model": model, "hq": hq, "hkv": hkv, "d": d, "keys": n, "cache": kind, "us": round(us, 2),
                             "bytes": nbytes, "gbs": round(nbytes / us / 1e3, 1), "frac_hbm_peak": round(frac, 3)})
                print(f"{model:13s} keys {n:7d} {kind:7s} {us:9.2f} us  {nbytes / 1e6:8.2f} MB  {nbytes / us / 1e3:7.0f} GB/s  "
                      f"{frac:.3f} of peak", flush=True)
                del caches, fn
                torch.cuda.empty_cache()
    summary = {"tool": "kvbench", "gpu": name, "power_limit_and_max_sm_clock": power, "hbm_peak_gbs": peak,
               "hbm_peak_source": peak_src, "layers_rotated": args.layers, "rounds": args.iters, "rows": rows}
    print(json.dumps(summary))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
