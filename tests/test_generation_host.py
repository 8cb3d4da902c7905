"""CPU tests of the generation driver: `utils.generate_step` (eager, no CUDA graph) on a stub model that only advances
the cache offsets, with the device quantiser replaced by the oracle.  They pin the schedule -- the prefill chunks, the
conversion to the quantized cache after every model call once the offset passes `quantized_kv_start`, and the tokens."""
import numpy as np
import pytest
import torch
from types import SimpleNamespace

from oracle import mlx_affine as A

VOCAB = 64


def _oracle_quantize(x, group_size, bits):
    q, s, b = A.quantize(x.float().numpy(), group_size, bits, "bf16")
    return (torch.from_numpy(q.view(np.int32)).view(torch.uint32), torch.from_numpy(s).to(x.dtype),
            torch.from_numpy(b).to(x.dtype))


def _next(tok: int) -> int:
    return (tok * 5 + 3) % VOCAB


class _StubModel(torch.nn.Module):
    """What the driver needs of `qllama.Model`: the attributes `make_prompt_cache` reads, and a forward that advances
    every cache's offset by the input length as `Model.forward` does.  Its logits pick `_next(last input token)`."""

    def __init__(self):
        super().__init__()
        self.args = SimpleNamespace(head_dim=64, hidden_size=128, num_attention_heads=2, num_key_value_heads=2,
                                    num_hidden_layers=2)
        self.tp = SimpleNamespace(world=1)
        self.model = SimpleNamespace(embed_tokens=SimpleNamespace(weight=torch.zeros(1)))
        self.dummy = torch.nn.Parameter(torch.zeros(1), requires_grad=False)
        self.calls = []

    def forward(self, inputs, cache, positions=None, attend_len=None):
        assert positions is None and attend_len is None
        B, L = inputs.shape
        off = cache[0].offset
        self.calls.append((L, off, hasattr(cache[0], "bits")))
        for c in cache:
            c.offset = off + L
        logits = torch.zeros((B, L, VOCAB))
        logits[0, torch.arange(L), (inputs[0] * 5 + 3) % VOCAB] = 1.0
        return logits


def _decode(first: int, n: int, quantized_from: int):
    return [(1, o, o >= quantized_from) for o in range(first, first + n)]


NEVER = 1 << 30
# (kv_bits, prefill_step_size, quantized_kv_start, max_tokens, model calls as (length, offset on entry, quantized))
# With a 12-token prompt.  Every yielded token is followed by one decode call, the last one included.
CASES = {
    "bf16": (None, 2048, 0, 8, [(12, 0, False)] + _decode(12, 8, NEVER)),
    "mid_prefill": (4, 5, 6, 8, [(5, 0, False), (5, 5, False), (2, 10, True)] + _decode(12, 8, 12)),
    "after_prompt": (8, 2048, 11, 8, [(12, 0, False)] + _decode(12, 8, 12)),
    "mid_decode": (4, 2048, 20, 16, [(12, 0, False)] + _decode(12, 16, 21)),
    "beyond_end": (8, 2048, 100, 16, [(12, 0, False)] + _decode(12, 16, NEVER)),
    "one_token": (4, 2048, 12, 1, [(12, 0, False), (1, 12, False)]),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_generate_step_prefill_and_conversion_schedule(monkeypatch, case):
    from gbx_lm_b200 import ops, qllama, utils

    kv_bits, step, start, max_tokens, want_calls = CASES[case]
    monkeypatch.setattr(ops, "quantize", _oracle_quantize)
    model = _StubModel()
    prompt = torch.randint(0, VOCAB, (12,), generator=torch.Generator().manual_seed(7))
    cache = qllama.make_prompt_cache(model, 1, 64)
    toks = [t for t, _ in utils.generate_step(prompt, model, max_tokens=max_tokens, prompt_cache=cache,
                                              prefill_step_size=step, use_cuda_graph=False, kv_bits=kv_bits,
                                              kv_group_size=64, quantized_kv_start=start)]
    assert model.calls == want_calls
    want_toks = [_next(int(prompt[-1]))]
    while len(want_toks) < max_tokens:
        want_toks.append(_next(want_toks[-1]))
    assert toks == want_toks
    # the conversion rule is applied after the last call too
    end = 12 + max_tokens
    converted = kv_bits is not None and end > start
    assert all(hasattr(c, "bits") == converted and c.offset == end for c in cache)
    if converted:
        assert all(c.bits == kv_bits and c.group_size == 64 for c in cache)
