"""CPU tests of batched generation with per-row prompt lengths: the four decode-step entry points of libgbxq refuse bad
arguments with the documented status codes before touching CUDA, at both position strides, and `utils.batch_generate`
checks its arguments, pads the prompts on the right, reads each row's first token at its own last column and steps each
row at its own position (a stub model stands in for qllama.Model)."""
import ctypes
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import mlx_affine as A

ESHAPE, ENULL, EINVAL_BITS, EINVAL_GROUP, EWORKSPACE, EUNSUPPORTED = -3, -6, -1, -2, -8, -9


def _decode_entries(lib, stride):
    """gbxq_rope_cache, gbxq_rope_cache_quantized, gbxq_decode_attention and gbxq_decode_attention_quantized at one
    pos_stride; every other argument is valid unless a keyword overrides it."""
    p = ctypes.c_void_p(256)  # never dereferenced: validation fails first

    def rope(keep=-1, max_len=64, B=2, Hq=8, Hkv=2, D=128, null=False):
        return lib.gbxq_rope_cache(None if null else p, p, p, p, stride, p, p, p, B, Hq, Hkv, D, max_len, keep, None)

    def qrope(keep=-1, max_len=64, B=2, Hq=8, Hkv=2, D=128, bits=4, gs=64, null=False):
        return lib.gbxq_rope_cache_quantized(p, p, p, None if null else p, stride, p, p, p, p, p, p, p, B, Hq, Hkv, D,
                                             max_len, keep, bits, gs, None)

    def attn(attend_len=64, max_len=64, B=2, Hq=8, Hkv=2, D=128, null=False):
        return lib.gbxq_decode_attention(p, p, p, None if null else p, stride, p, B, Hq, Hkv, D, max_len, attend_len, 0.1,
                                         None)

    def qattn(attend_len=64, max_len=64, B=2, Hq=8, Hkv=2, D=128, bits=4, gs=64, ws=1 << 30, null=False):
        return lib.gbxq_decode_attention_quantized(p, p, p, p, p, p, p, None if null else p, stride, p, B, Hq, Hkv, D,
                                                   max_len, attend_len, 0.1, bits, gs, p, ws, None)

    return rope, qrope, attn, qattn


def test_decode_step_abi_validation_without_gpu():
    from gbx_lm_b200 import _lib

    lib = _lib.get()
    for stride in (0, 1):  # one position for every row, one per row
        rope, qrope, attn, qattn = _decode_entries(lib, stride)
        for f in (rope, qrope):
            assert f(keep=64) == ESHAPE and f(keep=100) == ESHAPE and f(keep=0, max_len=0) == ESHAPE  # keep >= max_len
            assert f(null=True) == ENULL and f(keep=4, null=True) == ENULL  # flat and ring
            assert f(B=0) == ESHAPE
        assert rope(D=63) == ESHAPE
        assert qrope(bits=5) == EINVAL_BITS and qrope(gs=16) == EINVAL_GROUP
        assert qrope(D=96) == EUNSUPPORTED and qrope(Hq=16, Hkv=1) == EUNSUPPORTED and qrope(D=64, gs=128) == EUNSUPPORTED
        assert qrope(Hq=6, Hkv=4) == ESHAPE
        assert attn(null=True) == ENULL
        assert attn(attend_len=65) == ESHAPE and attn(attend_len=0) == ESHAPE and attn(Hq=6, Hkv=4) == ESHAPE
        assert attn(B=0) == ESHAPE
        assert attn(attend_len=49153, max_len=49153) == EUNSUPPORTED  # one float of shared memory per visible key
        assert qattn(null=True) == ENULL
        assert qattn(attend_len=65) == ESHAPE and qattn(Hq=6, Hkv=4) == ESHAPE
        assert qattn(D=96) == EUNSUPPORTED and qattn(Hq=16, Hkv=1) == EUNSUPPORTED
        assert qattn(bits=7) == EINVAL_BITS
        need = lib.gbxq_decode_attention_quantized_workspace_bytes(2, 8, 2, 128, 64)
        assert need > 0 and qattn(ws=need - 1) == EWORKSPACE
    for stride in (-1, 2):  # neither
        assert [f() for f in _decode_entries(lib, stride)] == [ESHAPE] * 4


VOCAB = 64


def _next(t: int) -> int:
    return (t * 5 + 3) % VOCAB


class _StubModel(torch.nn.Module):
    """What batch_generate needs of `qllama.Model`: the attributes `make_prompt_cache` reads and the forward's
    interface.  Row b's logits at column j pick _next(inputs[b, j]); it records every call."""

    def __init__(self):
        super().__init__()
        self.args = SimpleNamespace(head_dim=64, hidden_size=128, num_attention_heads=2, num_key_value_heads=2,
                                    num_hidden_layers=2)
        self.tp = SimpleNamespace(world=1)
        self.model = SimpleNamespace(embed_tokens=SimpleNamespace(weight=torch.zeros(1)))
        self.dummy = torch.nn.Parameter(torch.zeros(1), requires_grad=False)
        self.calls = []

    def forward(self, inputs, cache, positions=None, attend_len=None, head_columns=None):
        B, L = inputs.shape
        self.calls.append(dict(inputs=inputs.clone(), offset=cache[0].offset, kind=type(cache[0]).__name__,
                               max_len=cache[0].max_len, batch=cache[0].keys[0].shape[0] if isinstance(cache[0].keys, tuple)
                               else cache[0].keys.shape[0],
                               positions=None if positions is None else positions.clone(), attend_len=attend_len,
                               head_columns=None if head_columns is None else head_columns.clone()))
        if positions is None:  # as Model.forward: the shared positions of the offset, which advances
            for c in cache:
                c.offset += L
        cols = torch.arange(L).expand(B, L) if head_columns is None else head_columns[:, None]
        picked = torch.gather(inputs, 1, cols)
        logits = torch.zeros((B, cols.shape[1], VOCAB))
        logits.scatter_(2, _next(picked)[..., None], 1.0)
        return logits


def _oracle_quantize(x, group_size, bits):
    q, s, b = A.quantize(x.float().numpy(), group_size, bits, "bf16")
    return (torch.from_numpy(q.view(np.int32)).view(torch.uint32), torch.from_numpy(s).to(x.dtype),
            torch.from_numpy(b).to(x.dtype))


def _prompts(lens, seed=7):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, VOCAB, (n,), generator=g) for n in lens]


def test_batch_generate_rejects_bad_arguments():
    from gbx_lm_b200 import utils

    model = _StubModel()
    kw = dict(use_cuda_graph=False)
    with pytest.raises(ValueError, match="no prompts"):
        utils.batch_generate(model, [], **kw)
    with pytest.raises(ValueError, match="empty"):
        utils.batch_generate(model, _prompts([3]) + [torch.zeros(0, dtype=torch.long)], **kw)
    with pytest.raises(ValueError, match="1-D"):
        utils.batch_generate(model, [torch.zeros((1, 4), dtype=torch.long)], **kw)
    with pytest.raises(ValueError, match="max_kv_size"):
        utils.batch_generate(model, _prompts([3, 17]), max_kv_size=16, **kw)
    assert model.calls == []  # refused before any model call


def test_pad_prompts_right_pads_with_pad_id():
    from gbx_lm_b200 import utils

    prompts = _prompts([3, 7, 1])
    tokens, lens = utils._pad_prompts(prompts, 63, None)
    assert lens == [3, 7, 1] and tokens.shape == (3, 7) and tokens.dtype == torch.long
    for b, p in enumerate(prompts):
        assert torch.equal(tokens[b, :lens[b]], p) and (tokens[b, lens[b]:] == 63).all()
    assert utils._pad_prompts(prompts, 0, 7)[1] == lens  # the longest prompt may fill the window


@pytest.mark.parametrize("max_kv_size,kv_bits", [(None, None), (None, 8), (16, None), (16, 4)])
@pytest.mark.parametrize("step", (2048, 5, 1))
def test_batch_generate_bookkeeping(monkeypatch, step, max_kv_size, kv_bits):
    from gbx_lm_b200 import ops, utils

    monkeypatch.setattr(ops, "quantize", _oracle_quantize)
    lens, max_tokens, pad = [3, 12, 7, 1], 9, 61
    prompts = _prompts(lens)
    model = _StubModel()
    toks, stats = utils.batch_generate(model, prompts, max_tokens, prefill_step_size=step, pad_id=pad,
                                       max_kv_size=max_kv_size, kv_bits=kv_bits, quantized_kv_start=14,
                                       use_cuda_graph=False)
    for b, p in enumerate(prompts):  # each row continues its own last prompt token, never a pad
        want = [_next(int(p[-1]))]
        while len(want) < max_tokens:
            want.append(_next(want[-1]))
        assert toks[b] == want, b
    assert stats["prompt_tokens"] == sum(lens) and stats["generation_tokens"] == len(lens) * max_tokens
    assert stats["prompt_tps"] > 0 and stats["generation_tps"] > 0
    Lmax = max(lens)
    prefill = [c for c in model.calls if c["positions"] is None]
    decode = [c for c in model.calls if c["positions"] is not None]
    assert len(prefill) == -(-Lmax // step) and len(decode) == max_tokens - 1
    padded = torch.cat([c["inputs"] for c in prefill], 1)
    for b, p in enumerate(prompts):
        assert torch.equal(padded[b, :lens[b]], p) and (padded[b, lens[b]:] == pad).all()
    for c0, c in zip(range(0, Lmax, step), prefill):  # every chunk sends one column per row through the head
        n = c["inputs"].shape[1]
        assert c["offset"] == c0 and c["head_columns"].shape == (len(lens),)
        assert all(0 <= int(j) < n for j in c["head_columns"])
        for b, n_b in enumerate(lens):
            if c0 <= n_b - 1 < c0 + n:
                assert int(c["head_columns"][b]) == n_b - 1 - c0
    for s, c in enumerate(decode):  # row b's s-th step at position len_b + s; the offset is the longest row's count
        assert c["positions"].shape == (len(lens), 1)
        assert c["positions"][:, 0].tolist() == [n + s for n in lens]
        assert c["offset"] == Lmax + s + 1
        assert c["attend_len"] == (Lmax + s + 1 if max_kv_size is None else min(Lmax + s + 1, max_kv_size))
    assert {c["batch"] for c in model.calls} == {len(lens)}
    assert {c["max_len"] for c in model.calls} == {Lmax + max_tokens + 1 if max_kv_size is None else max_kv_size}
    kinds = [c["kind"] for c in model.calls]
    if kv_bits is None:
        assert not any("Quantized" in k for k in kinds)
    else:  # converted after the first call that takes the offset past quantized_kv_start = 14
        after = [c["offset"] + (c["inputs"].shape[1] if c["positions"] is None else 0) for c in model.calls]
        first_q = next(i for i, c in enumerate(model.calls) if "Quantized" in c["kind"])
        assert after[first_q - 1] > 14 and all(a <= 14 for a in after[:first_q - 1])
        assert all("Quantized" in k for k in kinds[first_q:])
    assert ("Rotating" in kinds[0]) == (max_kv_size is not None)
