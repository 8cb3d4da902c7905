#!/usr/bin/env python
"""Digests of the single-token decode-step ops on seeded inputs, to compare two builds of libgbxq bit for bit:

    GBXQ_LIB=/path/to/other/libgbxq.so python tools/decode_step_ab.py > a.json
    python tools/decode_step_ab.py > b.json && cmp a.json b.json

The inputs are those of the kernel tests: every (bf16 | bits, D, group size, Hq/Hkv) of tests/test_gpu_rotating_cache.py
KERNEL_CASES, shared and per-row positions around the 256-key chunk borders, flat and rotating (keep) caches.  One line
of JSON: case -> sha256 of the rotated q, the cache buffers after the write, and the attention output."""
import hashlib
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gbx_lm_b200 import ops, qllama  # noqa: E402
from tests.test_gpu_rotating_cache import KERNEL_CASES, _i32, _side  # noqa: E402


def digest(ts) -> str:
    h = hashlib.sha256()
    for t in ts:
        t = t.view(torch.int16) if t.dtype == torch.bfloat16 else _i32(t)  # the bits (numpy has no bf16)
        h.update(t.contiguous().cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def main():
    dev = torch.device("cuda")
    out = {}
    B, max_len = 2, 700
    for kind, bits, D, gs, Hq, Hkv in KERNEL_CASES:
        g = torch.Generator(device=dev).manual_seed(bits * 1000 + D + gs + Hq)
        inv = qllama.RoPE(D, 500000.0, False, None).to(dev).inv_freq
        ks, vs = (_side(kind, B, Hkv, max_len, D, bits, gs, dev, g) for _ in range(2))
        if kind == "q":  # valid triples (scales from the quantizer), as a filled cache holds them
            kb = (torch.randn((B, Hkv, max_len, D), generator=g, device=dev) * 2).to(torch.bfloat16)
            ks, vs = tuple(ops.quantize(kb, gs, bits)), tuple(ops.quantize(kb.flip(2).contiguous(), gs, bits))
        for pos, keep in (([0], None), ([255], None), ([256, 600], None), ([511, 257], None), ([699], 4), ([900], 4)):
            q = torch.randn((B, Hq, D), generator=g, device=dev).to(torch.bfloat16)
            k = (torch.randn((B, Hkv, D), generator=g, device=dev) * 3).to(torch.bfloat16)
            v = torch.randn((B, Hkv, D), generator=g, device=dev).to(torch.bfloat16)
            p = torch.tensor(pos, device=dev)
            if kind == "bf16":
                ops.rope_cache(q, k, v, p, inv, ks[0], vs[0], keep=keep)
                o = ops.decode_attention(q, ks[0], vs[0], p, D ** -0.5)
            else:
                ops.rope_cache_quantized(q, k, v, p, inv, ks, vs, gs, bits, keep=keep)
                o = ops.decode_attention_quantized(q, ks, vs, p, D ** -0.5, gs, bits)
            out[f"{kind}-b{bits}-D{D}-g{gs}-{Hq}/{Hkv}-p{pos}-keep{keep}"] = digest([q, *ks, *vs, o])
    torch.cuda.synchronize()
    print(json.dumps(out, sort_keys=True))


if __name__ == "__main__":
    main()
