"""CPU tests of speculative decoding: the four `_multi` entry points of libgbxq refuse bad arguments with the documented
status codes before touching CUDA, the static caches rewind (`trim`), and `utils.speculative_generate_step` follows its
round schedule on stub target and draft models -- the tokens are the target's whatever the draft proposes, with the
`from_draft` flags, the `max_tokens` truncation, the caches' offsets after every round and the kv_bits conversion after
the verify step that crosses `quantized_kv_start`."""
import ctypes
import random
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import mlx_affine as A

ESHAPE, ENULL, EINVAL_BITS, EINVAL_GROUP, EWORKSPACE, EUNSUPPORTED = -3, -6, -1, -2, -8, -9


def _multi_entries(lib):
    """The four `_multi` entry points at pos_stride 0; every other argument is valid unless a keyword overrides it."""
    p = ctypes.c_void_p(256)  # never dereferenced: validation fails first

    def rope(T=3, B=2, Hq=8, Hkv=2, D=128, max_len=64, stride=0, null=False):
        return lib.gbxq_rope_cache_multi(None if null else p, p, p, p, stride, p, p, p, B, T, Hq, Hkv, D, max_len, None)

    def qrope(T=3, B=2, Hq=8, Hkv=2, D=128, max_len=64, bits=4, gs=64, stride=0, null=False):
        return lib.gbxq_rope_cache_quantized_multi(p, p, p, None if null else p, stride, p, p, p, p, p, p, p, B, T, Hq,
                                                   Hkv, D, max_len, bits, gs, None)

    def attn(T=3, B=2, Hq=8, Hkv=2, D=128, max_len=64, attend_len=64, stride=0, null=False):
        return lib.gbxq_decode_attention_multi(p, p, p, None if null else p, stride, p, B, T, Hq, Hkv, D, max_len,
                                               attend_len, 0.1, None)

    def qattn(T=3, B=2, Hq=8, Hkv=2, D=128, max_len=64, attend_len=64, bits=4, gs=64, ws=1 << 30, stride=0, null=False):
        return lib.gbxq_decode_attention_quantized_multi(p, p, p, p, p, p, p, None if null else p, stride, p, B, T, Hq,
                                                         Hkv, D, max_len, attend_len, 0.1, bits, gs, p, ws, None)

    return rope, qrope, attn, qattn


def test_multi_abi_validation_without_gpu():
    from gbx_lm_b200 import _lib

    lib = _lib.get()
    rope, qrope, attn, qattn = _multi_entries(lib)
    for f in (rope, qrope, attn, qattn):
        assert f(null=True) == ENULL
        assert f(T=0) == ESHAPE and f(T=9) == ESHAPE and f(T=-1) == ESHAPE
        assert f(B=0) == ESHAPE
        assert f(stride=2) == ESHAPE and f(stride=-1) == ESHAPE
        assert f(B=8192, T=8) == ESHAPE  # B * T rows above the 65535 of a grid's y dimension
    assert rope(D=63) == ESHAPE and rope(max_len=0) == ESHAPE
    assert qrope(bits=5) == EINVAL_BITS and qrope(gs=16) == EINVAL_GROUP
    assert qrope(D=96) == EUNSUPPORTED and qrope(Hq=16, Hkv=1) == EUNSUPPORTED
    assert attn(attend_len=65) == ESHAPE and attn(attend_len=0) == ESHAPE and attn(Hq=6, Hkv=4) == ESHAPE
    assert attn(attend_len=49153, max_len=49153) == EUNSUPPORTED  # the bf16 kernel's cap holds for blocks too
    assert qattn(attend_len=65) == ESHAPE and qattn(Hq=6, Hkv=4) == ESHAPE
    assert qattn(D=96) == EUNSUPPORTED and qattn(bits=7) == EINVAL_BITS
    # the partials of B * T query rows: the existing size query at B * T
    need = lib.gbxq_decode_attention_quantized_workspace_bytes(2 * 3, 8, 2, 128, 64)
    assert need == 3 * lib.gbxq_decode_attention_quantized_workspace_bytes(2, 8, 2, 128, 64)
    assert qattn(ws=need - 1) == EWORKSPACE


def test_static_caches_trim():
    from gbx_lm_b200 import cache as C

    flat = [C.StaticKVCache(1, 2, 32, 64, "cpu"), C.StaticQuantizedKVCache(1, 2, 32, 64, "cpu", 64, 4)]
    ring = [C.StaticRotatingKVCache(1, 2, 32, 64, "cpu", 4), C.StaticRotatingQuantizedKVCache(1, 2, 32, 64, "cpu", 4, 64, 4)]
    for c in flat:
        c.offset = 10
        assert c.is_trimmable()
        assert c.trim(3) == 3 and c.offset == 7
        assert c.trim(100) == 7 and c.offset == 0
    for c in ring:
        c.offset = 10
        assert not c.is_trimmable()
        with pytest.raises(ValueError):
            c.trim(1)
    for c in flat:
        c.offset = 10
    assert C.can_trim_prompt_cache(flat) and C.trim_prompt_cache(flat, 4) == 4
    assert [c.offset for c in flat] == [6, 6]
    assert not C.can_trim_prompt_cache(flat + ring) and C.trim_prompt_cache(flat + ring, 4) == 0
    assert [c.offset for c in flat] == [6, 6]


VOCAB = 64


def _next(tok: int) -> int:
    return (tok * 5 + 3) % VOCAB


def _oracle_quantize(x, group_size, bits):
    q, s, b = A.quantize(x.float().numpy(), group_size, bits, "bf16")
    return (torch.from_numpy(q.view(np.int32)).view(torch.uint32), torch.from_numpy(s).to(x.dtype),
            torch.from_numpy(b).to(x.dtype))


RULES = {
    "right": lambda tok, pos: _next(tok),
    "wrong": lambda tok, pos: (_next(tok) + 1) % VOCAB,
    "random": lambda tok, pos: _next(tok) if random.Random(tok * 1009 + pos).random() < 0.6 else (tok * 11 + 1) % VOCAB,
}


class _StubModel(torch.nn.Module):
    """What the driver needs of `qllama.Model`: the attributes `make_prompt_cache` reads and the forward's interface.
    Column t of the logits picks rule(inputs[0, t], its position).  A prefill call (no positions) advances the offsets as
    `Model.forward` does; a call with explicit positions checks that they are consecutive and that the driver has set
    the offsets past them.  Every call is recorded as (tokens, first position, quantized cache)."""

    def __init__(self, rule, vocab=VOCAB, fused=True, world=1):
        super().__init__()
        self.args = SimpleNamespace(head_dim=64, hidden_size=128, num_attention_heads=2, num_key_value_heads=2,
                                    num_hidden_layers=2, vocab_size=vocab)
        self.tp = SimpleNamespace(world=world)
        self.model = SimpleNamespace(embed_tokens=SimpleNamespace(weight=torch.zeros(1)))
        self.layers = [SimpleNamespace(self_attn=SimpleNamespace(takes_fused_decode=lambda c: fused))] * 2
        self.dummy = torch.nn.Parameter(torch.zeros(1), requires_grad=False)
        self.rule = rule
        self.calls = []

    def forward(self, inputs, cache, positions=None, attend_len=None):
        B, L = inputs.shape
        if positions is None:
            off = cache[0].offset
            for c in cache:
                c.offset = off + L
            pos = list(range(off, off + L))
        else:
            pos = positions.tolist()
            assert pos == list(range(pos[0], pos[0] + L))
            assert all(c.offset == pos[-1] + 1 for c in cache)
        self.calls.append((L, pos[0], hasattr(cache[0], "bits")))
        logits = torch.zeros((B, L, VOCAB))
        for t in range(L):
            logits[0, t, self.rule(int(inputs[0, t]), pos[t])] = 1.0
        return logits


def _chain(last: int, n: int):
    out = []
    while len(out) < n:
        last = _next(last)
        out.append(last)
    return out


def _run(draft_rule, k, max_tokens, n_prompt=12, **kw):
    from gbx_lm_b200 import utils

    target, draft = _StubModel(RULES["right"]), _StubModel(RULES[draft_rule])
    prompt = torch.randint(0, VOCAB, (n_prompt,), generator=torch.Generator().manual_seed(3))
    cache = utils._spec_cache(target, draft, n_prompt + max_tokens + k + 2)
    seen = []
    for tok, lp, from_draft in utils.speculative_generate_step(prompt, target, draft, num_draft_tokens=k,
                                                               max_tokens=max_tokens, prompt_cache=cache, **kw):
        assert lp.shape == (VOCAB,) and int(lp.argmax()) == tok
        seen.append((tok, from_draft, [c.offset for c in cache]))
    return prompt, target, draft, cache, seen


@pytest.mark.parametrize("k", [1, 2, 4, 7])
@pytest.mark.parametrize("draft_rule", sorted(RULES))
@pytest.mark.parametrize("max_tokens", [1, 2, 9, 24])
def test_speculative_tokens_are_the_targets(draft_rule, k, max_tokens):
    n_prompt = 12
    prompt, target, draft, cache, seen = _run(draft_rule, k, max_tokens, n_prompt)
    assert [t for t, _, _ in seen] == _chain(int(prompt[-1]), max_tokens)
    flags = [f for _, f, _ in seen]
    assert flags[0] is False  # the prefill's token
    # the rounds: n accepted drafts (from_draft) then the target's own token, all cut at max_tokens
    rounds, i = [], 1
    while i < len(flags):
        n = 0
        while i + n < len(flags) and flags[i + n]:
            n += 1
        assert n <= k
        rounds.append((i, n))
        i += n + 1
    if draft_rule == "right":
        assert all(n == k for _, n in rounds[:-1])
    if draft_rule == "wrong":
        assert not any(flags)
    # every round: the draft's T = 2 step at P - 1 then k - 1 single steps, the target's k + 1 verify at P; the offsets
    # at the round's tokens are those after the verify (target P + k + 1, draft P + k)
    nt = len(target.layers)
    assert seen[0][2] == [n_prompt] * len(cache)
    assert target.calls[0] == (n_prompt, 0, False) and draft.calls[0] == (n_prompt, 0, False)
    assert len(target.calls) == 1 + len(rounds)
    for r, (i, n) in enumerate(rounds):
        P = n_prompt + i - 1
        assert target.calls[1 + r] == (k + 1, P, False)
        assert draft.calls[1 + r * k: 1 + (r + 1) * k] == [(2, P - 1, False)] + [(1, P + j, False) for j in range(1, k)]
        assert seen[i][2] == [P + k + 1] * nt + [P + k] * nt
    # after the last round's rewind: the target holds < P + n + 1 (dropped tokens included), the draft one less
    end = [c.offset for c in cache]
    if rounds:
        P = n_prompt + rounds[-1][0] - 1
        assert end[:nt] == [end[0]] * nt and end[nt:] == [end[0] - 1] * nt
        assert P + 1 <= end[0] <= P + k + 1 and end[0] >= n_prompt + max_tokens - 1
    else:  # max_tokens 1: the prefill's token alone
        assert end == [n_prompt] * len(cache)


def test_speculative_kv_bits_converts_after_the_crossing_verify(monkeypatch):
    from gbx_lm_b200 import ops

    monkeypatch.setattr(ops, "quantize", _oracle_quantize)
    k, start = 2, 20
    prompt, target, draft, cache, seen = _run("random", k, 24, kv_bits=4, kv_group_size=64, quantized_kv_start=start)
    assert [t for t, _, _ in seen] == _chain(int(prompt[-1]), 24)
    verifies = target.calls[1:]
    crossing = next(i for i, (L, P, _) in enumerate(verifies) if P + L > start)
    assert all(not q for _, _, q in verifies[:crossing + 1]) and all(q for _, _, q in verifies[crossing + 1:])
    # the draft's steps of the crossing round ran on bf16, the later ones on the converted caches
    drafts = draft.calls[1:]
    assert all(not q for _, _, q in drafts[:(crossing + 1) * k]) and all(q for _, _, q in drafts[(crossing + 1) * k:])
    assert all(c.bits == 4 and c.group_size == 64 for c in cache)


def test_speculative_kv_bits_at_prefill(monkeypatch):
    from gbx_lm_b200 import ops

    monkeypatch.setattr(ops, "quantize", _oracle_quantize)
    prompt, target, draft, cache, seen = _run("right", 3, 10, kv_bits=8, kv_group_size=64, quantized_kv_start=0)
    assert [t for t, _, _ in seen] == _chain(int(prompt[-1]), 10)
    assert all(q for _, _, q in target.calls[1:] + draft.calls[1:])


def test_speculative_refusals():
    from gbx_lm_b200 import utils

    target, prompt = _StubModel(RULES["right"]), torch.arange(5)
    for k in (0, 8, 2.0, True):
        with pytest.raises(ValueError, match="num_draft_tokens"):
            next(utils.speculative_generate_step(prompt, target, _StubModel(RULES["right"]), num_draft_tokens=k))
    with pytest.raises(ValueError, match="vocabulary"):
        next(utils.speculative_generate_step(prompt, target, _StubModel(RULES["right"], vocab=VOCAB + 1)))
    with pytest.raises(ValueError, match="tensor-parallel"):
        next(utils.speculative_generate_step(prompt, target, _StubModel(RULES["right"], world=2)))
    with pytest.raises(ValueError, match="max_kv_size"):
        utils.generate_tokens(target, prompt, 8, draft_model=_StubModel(RULES["right"]), max_kv_size=16)
    with pytest.raises(ValueError, match="max_kv_size"):
        utils.generate_tokens_device(target, prompt, 8, draft_model=_StubModel(RULES["right"]), max_kv_size=16)
    with pytest.raises(ValueError, match="fused decode path"):
        utils.generate_tokens_device(target, prompt, 8, draft_model=_StubModel(RULES["right"], fused=False))
    with pytest.raises(ValueError, match="fused decode path"):
        utils.generate_tokens_device(_StubModel(RULES["right"], fused=False), prompt, 8, draft_model=target)


def test_generate_tokens_routes_a_draft_to_the_speculative_generator():
    from gbx_lm_b200 import utils

    target, draft = _StubModel(RULES["right"]), _StubModel(RULES["wrong"])
    prompt = torch.arange(7)
    toks, stats = utils.generate_tokens(target, prompt, 11, draft_model=draft, num_draft_tokens=3)
    assert toks == _chain(6, 11) and stats["generation_tokens"] == 11
    assert draft.calls and draft.calls[1] == (2, 6, False)
