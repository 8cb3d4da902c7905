"""GPU tests of batched generation with per-row prompt lengths: the cache-write and attention ops with per-row
positions (pos_stride 1) against one shared position (pos_stride 0; bitwise, with equal positions) and against B = 1
calls row by row (bitwise, with distinct positions; nothing else written), `batch_generate` against the shared-position
path, each row's independence of the pads and of the other rows at batches that reach every matmul kernel family, the
fp32 reference (flat, 8-bit and wrapping rotating caches), graph / eager / in-decode conversion, fused against unfused
per-row decode, and the launches of a ragged decode step."""
import copy

import pytest
import torch
from safetensors.torch import load_file

from gbx_lm_b200 import ops, qllama, utils, workloads as W
from gbx_lm_b200.cache import DEFAULT_KV_KEEP, ring_slot
from tests import ref_model
from tests.test_gpu_rotating_cache import KERNEL_CASES, _i32, _ref_forward, _side

pytestmark = pytest.mark.gpu

RW, RKEEP = 40, 4  # the cache of the kernel tests: max_len rows, RKEEP sinks when it is a ring
FLAT_POS = (0, RKEEP - 1, RW - 1, RW, 17, 5)  # RW: past the flat cache (no write, attention clamps)
RING_POS = (0, RKEEP - 1, RW - 1, RW, 3 * RW + 7, 10 ** 6)


def _write(kind, q, k, v, p, inv, ks, vs, bits, gs, keep):
    if kind == "bf16":
        return ops.rope_cache(q, k, v, p, inv, ks[0], vs[0], keep=keep)
    return ops.rope_cache_quantized(q, k, v, p, inv, ks, vs, gs, bits, keep=keep)


def _attend(kind, q, ks, vs, p, bits, gs, attend_len):
    if kind == "bf16":
        return ops.decode_attention(q, ks[0], vs[0], p, 0.125, attend_len)
    return ops.decode_attention_quantized(q, ks, vs, p, 0.125, gs, bits, attend_len)


def _inputs(g, dev, B, Hq, Hkv, D):
    q = torch.randn((B, Hq, D), generator=g, device=dev).to(torch.bfloat16)
    k = (torch.randn((B, Hkv, D), generator=g, device=dev) * 3).to(torch.bfloat16)
    v = torch.randn((B, Hkv, D), generator=g, device=dev).to(torch.bfloat16)
    return q, k, v


@pytest.mark.parametrize("keep", (None, RKEEP), ids=("flat", "ring"))
@pytest.mark.parametrize("kind,bits,D,gs,Hq,Hkv", KERNEL_CASES)
def test_rows_with_equal_positions_are_the_shared_entries(cuda_device, kind, bits, D, gs, Hq, Hkv, keep):
    g = torch.Generator(device=cuda_device).manual_seed(bits * 1000 + D + gs + Hq + (keep or 0))
    inv = qllama.RoPE(D, 500000.0, False, None).to(cuda_device).inv_freq
    B = 3
    for pos in ((7, RW - 1) if keep is None else (7, RW + 5)):
        ks, vs = (_side(kind, B, Hkv, RW, D, bits, gs, cuda_device, g) for _ in range(2))
        ks2, vs2 = tuple(t.clone() for t in ks), tuple(t.clone() for t in vs)
        q, k, v = _inputs(g, cuda_device, B, Hq, Hkv, D)
        shared = torch.tensor([pos], device=cuda_device)
        rows = torch.full((B,), pos, device=cuda_device)
        assert torch.equal(_write(kind, q.clone(), k, v, shared, inv, ks, vs, bits, gs, keep),
                           _write(kind, q.clone(), k, v, rows, inv, ks2, vs2, bits, gs, keep))
        for a, b in zip(ks + vs, ks2 + vs2):
            assert torch.equal(_i32(a), _i32(b))
        for attend_len in (min(pos + 1, RW), RW):
            assert torch.equal(_attend(kind, q, ks, vs, shared, bits, gs, attend_len),
                               _attend(kind, q, ks, vs, rows, bits, gs, attend_len)), (pos, attend_len)


@pytest.mark.parametrize("keep", (None, RKEEP), ids=("flat", "ring"))
@pytest.mark.parametrize("kind,bits,D,gs,Hq,Hkv", KERNEL_CASES)
def test_rows_are_independent_b1_calls(cuda_device, kind, bits, D, gs, Hq, Hkv, keep):
    """Distinct positions per row: row b of q, of every cache buffer and of the attention is bitwise the B = 1 call on
    row b's slices at its position; no other cache row changes."""
    g = torch.Generator(device=cuda_device).manual_seed(bits * 7 + D + gs * 3 + Hq + (keep or 0))
    inv = qllama.RoPE(D, 500000.0, False, None).to(cuda_device).inv_freq
    positions = FLAT_POS if keep is None else RING_POS
    B = len(positions)
    ks, vs = (_side(kind, B, Hkv, RW, D, bits, gs, cuda_device, g) for _ in range(2))
    before = [t.clone() for t in ks + vs]
    q, k, v = _inputs(g, cuda_device, B, Hq, Hkv, D)
    pos = torch.tensor(positions, device=cuda_device)
    got_q = _write(kind, q.clone(), k, v, pos, inv, ks, vs, bits, gs, keep)
    eager = min(max(positions) + 1, RW)  # and 18: some rows' positions are past it, the kernel clamps them
    got_o = {a: _attend(kind, got_q, ks, vs, pos, bits, gs, a) for a in (eager, 18, RW)}
    for b, p in enumerate(positions):
        one = [t[b:b + 1].clone() for t in before]
        k1, v1 = tuple(one[:len(ks)]), tuple(one[len(ks):])
        p1 = torch.tensor([p], device=cuda_device)
        want_q = _write(kind, q[b:b + 1].clone(), k[b:b + 1], v[b:b + 1], p1, inv, k1, v1, bits, gs, keep)
        assert torch.equal(got_q[b:b + 1], want_q), (b, p)
        for got, want in zip(ks + vs, k1 + v1):
            assert torch.equal(_i32(got)[b:b + 1], _i32(want)), (b, p)
        for a, o in got_o.items():
            assert torch.equal(o[b:b + 1], _attend(kind, want_q, k1, v1, p1, bits, gs, a)), (b, p, a)
        # nothing outside the row's own slot (if any) was written
        slot = p if keep is None else ring_slot(p, RW, keep)
        others = torch.ones(RW, dtype=torch.bool, device=cuda_device)
        if slot < RW:
            others[slot] = False
        for got, old in zip(ks + vs, before):
            assert torch.equal(_i32(got)[b, :, others], _i32(old)[b, :, others]), (b, p)


# ------------------------------------------------------------------------------------------ the model and generation
_MODELS = {}


@pytest.fixture(scope="module")
def model_of(tmp_path_factory, cuda_device):
    def get(name):
        if name not in _MODELS:
            dims = W.MODELS[name]
            strat = W.STRATEGIES["bpw-4.0"](dims.layers) if name == "tiny-llama" else None
            d = tmp_path_factory.mktemp(name)
            cfg = utils.write_synthetic_checkpoint(d, dims, strat, seed=11, default_bits=4, default_gs=64,
                                                   embed_scale=1.0)
            model, _ = utils.load_model(d, device=cuda_device)
            _MODELS[name] = (dims, cfg, model, d, strat)
        return _MODELS[name]

    yield get
    _MODELS.clear()


def _prompts(dims, lens, seed=3):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, dims.vocab, (n,), generator=g) for n in lens]


def _ragged_logits(model, prompts, steps, pad_id=0, kv_bits=None, start=0, prefill_step_size=2048, tokens=None):
    """batch_generate's eager computation with the per-step logits kept: [B, steps + 1, V] fp32 and the tokens [B, steps
    + 1].  tokens [B, steps + 1]: teacher-forced instead of greedy."""
    dev = next(model.parameters()).device
    pad, lens = utils._pad_prompts(prompts, pad_id, None)
    B, Lmax = pad.shape
    kv = dict(kv_bits=kv_bits, kv_group_size=64, quantized_kv_start=start)
    cache = utils._prompt_cache(model, Lmax + steps + 2, None, batch=B)
    convert = utils._kv_quantizer(cache, **kv)
    out = [utils._prefill_chunks(model, pad.to(dev), cache, prefill_step_size, kv, last=[n - 1 for n in lens])]
    toks = [utils.fast_argmax(out[0]) if tokens is None else tokens[:, 0].to(dev)]
    pos = torch.tensor(lens, device=dev)
    with torch.no_grad():
        for s in range(steps):
            for c in cache:
                c.offset = Lmax + s + 1
            out.append(model(toks[-1][:, None], cache, positions=pos[:, None], attend_len=cache[0].attend_len)[:, -1])
            convert()
            toks.append(utils.fast_argmax(out[-1]) if tokens is None else tokens[:, s + 1].to(dev))
            pos = pos + 1
    return torch.stack(out, 1).float(), torch.stack(toks, 1)


@pytest.mark.parametrize("kv_bits", (None, 4))
@pytest.mark.parametrize("B", (2, 5, 12))
def test_equal_lengths_are_the_shared_position_path(cuda_device, model_of, B, kv_bits):
    """B prompts of one length: batch_generate's tokens are bitwise those of the shared-position DecodeGraph path, and
    the per-row captured step gives bitwise its per-step logits."""
    dims, _, model, _, _ = model_of("tiny-llama")
    L, n = 9, 20
    prompts = _prompts(dims, [L] * B)
    kv = dict(kv_bits=kv_bits, kv_group_size=64, quantized_kv_start=L + 6)
    toks, _ = utils.batch_generate(model, prompts, n, **kv)
    tokens = torch.stack(prompts).to(cuda_device)
    cache = utils._prompt_cache(model, L + n + 1, None, batch=B)
    tok = utils.fast_argmax(utils._prefill_chunks(model, tokens, cache, 2048, kv, last=[L - 1] * B))
    first, _, outs = utils._device_decode(model, cache, tok, L, L, n - 1, kv, "test")
    want = [list(r) for r in zip(*([first] + [r for o in outs for r in o.tolist()]))]
    assert toks == want
    # per-step logits of the captured steps, from one prefilled cache: shared position against one position per row
    cache = utils._prompt_cache(model, L + n + 1, None, batch=B)
    tok = utils.fast_argmax(utils._prefill_chunks(model, tokens, cache, 2048, kv, last=[L - 1] * B))
    if kv_bits:
        cache[:] = [c.to_quantized(64, kv_bits) for c in cache]
    cache2 = copy.deepcopy(cache)
    shared = utils.DecodeGraph(model, cache, batch=B).capture(tok, L)
    rows = utils.DecodeGraph(model, cache2, batch=B, per_row=True).capture(tok, torch.full((B,), L, device=cuda_device))
    for s in range(n):
        a = shared.step(tok, L + s)
        b = rows.step(tok, torch.full((B,), L + s, device=cuda_device))
        assert torch.equal(a, b), s
        tok = utils.fast_argmax(a)


@pytest.mark.parametrize("kv_bits", (None, 8))
@pytest.mark.parametrize("B", (2, 5, 12))
def test_rows_do_not_depend_on_pads_or_neighbours(cuda_device, model_of, B, kv_bits):
    """Row b's tokens and per-step logits are bitwise unchanged when the other rows' prompts (same lengths) or the pad
    token change.  B = 2 / 5 / 12 run the decode matmuls on mmv8 / skinny / gemm_ts and the head on head_gemv (<= 8
    rows) and on the dense matmul."""
    dims, _, model, _, _ = model_of("tiny-llama")
    lens = [3 + (7 * b) % 17 for b in range(B)]
    base = _prompts(dims, lens, seed=5)
    other = _prompts(dims, lens, seed=6)
    n = 16
    kw = dict(kv_bits=kv_bits, start=max(lens) + 4)
    ref_l, ref_t = _ragged_logits(model, base, n, pad_id=0, **kw)
    toks, _ = utils.batch_generate(model, base, n + 1, kv_bits=kv_bits, kv_group_size=64, quantized_kv_start=kw["start"])
    assert toks == ref_t.tolist()  # batch_generate is this computation
    for b in (0, B - 1):
        mixed = [base[i] if i == b else other[i] for i in range(B)]
        for pad_id in (0, dims.vocab - 1):
            got_l, got_t = _ragged_logits(model, mixed, n, pad_id=pad_id, **kw)
            assert torch.equal(got_t[b], ref_t[b]), (b, pad_id)
            assert torch.equal(got_l[b], ref_l[b]), (b, pad_id)
        g_toks, _ = utils.batch_generate(model, mixed, n + 1, kv_bits=kv_bits, kv_group_size=64,
                                         quantized_kv_start=kw["start"], pad_id=dims.vocab - 1)
        assert g_toks[b] == toks[b]


def _dense(name, dims, d, strat):
    ckpt = load_file(str(d / "model.safetensors"))
    plan = {}
    for (i, p, n, k, b, g) in W.layer_plan(dims, strat, 4, 64):
        sub = "self_attn" if p in ("q_proj", "k_proj", "v_proj", "o_proj") else "mlp"
        plan[f"model.layers.{i}.{sub}.{p}"] = (b, g)
    return ref_model.dense_weights(ckpt, lambda m: plan[m])


REF_CASES = {  # (prompt lengths, max_tokens, kv_bits, max_kv_size)
    "bf16": ([5, 12, 9, 1], 24, None, None),
    "kv8": ([5, 12, 9, 1], 24, 8, None),
    "ring": ([5, 12, 18], 30, None, 20),  # the rows wrap at decode steps 15, 8 and 2
}


@pytest.mark.parametrize("case", sorted(REF_CASES))
@pytest.mark.parametrize("name", ("tiny-llama", "tiny-qwen2"))
def test_rows_match_reference_on_clear_steps(cuda_device, model_of, name, case):
    """Each row's greedy tokens against the fp32 reference on its own prompt and tokens, teacher-forced, under the
    causal mask or the window mask of a rotating cache."""
    lens, n, kv_bits, window = REF_CASES[case]
    dims, cfg, model, d, strat = model_of(name)
    dense = _dense(name, dims, d, strat)
    prompts = _prompts(dims, lens, seed=8)
    toks, _ = utils.batch_generate(model, prompts, n, kv_bits=kv_bits, max_kv_size=window, pad_id=dims.vocab - 1)
    clear_total = 0
    for p, t in zip(prompts, toks):
        seq = torch.cat([p, torch.tensor(t)])[None]
        i, j = torch.arange(seq.shape[1])[:, None], torch.arange(seq.shape[1])[None, :]
        visible = j <= i
        if window is not None:
            visible = visible & ((j < DEFAULT_KV_KEEP) | (j > i - (window - DEFAULT_KV_KEEP)))
        with torch.no_grad():
            ref = _ref_forward(dense, cfg, seq, visible)[0, len(p) - 1:-1]
        top2 = ref.topk(2, -1).values
        clear = (top2[:, 0] - top2[:, 1]) > 0.05 * ref.abs().max()
        clear_total += int(clear.sum())
        assert (ref.argmax(-1)[clear] == torch.tensor(t)[clear]).all()
    assert clear_total >= 10, f"only {clear_total} decisive steps"


GRAPH_CASES = {  # (prompt lengths, max_tokens, kv_bits, quantized_kv_start, max_kv_size, prefill_step_size)
    "bf16": ([5, 12, 9], 24, None, 0, None, 2048),
    "kv4-in-decode": ([5, 12, 9], 24, 4, 20, None, 2048),
    "kv8-in-prefill": ([5, 12, 9], 24, 8, 6, None, 4),
    "ring": ([5, 12, 18], 30, None, 0, 20, 2048),
    "ring-kv4-in-decode": ([5, 12, 18], 30, 4, 25, 20, 7),
    "max1": ([5, 12, 9], 1, 4, 0, None, 2048),
}


@pytest.mark.parametrize("case", sorted(GRAPH_CASES))
@pytest.mark.parametrize("name", ("tiny-llama", "tiny-qwen2"))
def test_graph_and_eager_give_the_same_tokens(cuda_device, model_of, name, case):
    lens, n, kv_bits, start, window, step = GRAPH_CASES[case]
    dims, _, model, _, _ = model_of(name)
    prompts = _prompts(dims, lens, seed=4)
    kw = dict(kv_bits=kv_bits, kv_group_size=64, quantized_kv_start=start, max_kv_size=window, prefill_step_size=step)
    g_toks, stats = utils.batch_generate(model, prompts, n, **kw)
    e_toks, _ = utils.batch_generate(model, prompts, n, use_cuda_graph=False, **kw)
    assert g_toks == e_toks and [len(t) for t in g_toks] == [n] * len(lens)
    assert stats["prompt_tokens"] == sum(lens) and stats["generation_tokens"] == n * len(lens)


@pytest.mark.parametrize("kv_bits", (None, 4, 8))
@pytest.mark.parametrize("name", ("tiny-llama", "tiny-qwen2"))
def test_fused_and_unfused_per_row_decode_agree(cuda_device, model_of, monkeypatch, name, kv_bits):
    dims, _, model, _, _ = model_of(name)
    prompts = _prompts(dims, [4, 11, 7, 1], seed=12)
    forced = torch.randint(0, dims.vocab, (4, 25), generator=torch.Generator().manual_seed(2))
    runs = []
    for fused in (True, False):
        monkeypatch.setattr(qllama, "FUSED_DECODE", fused)
        runs.append(_ragged_logits(model, prompts, 24, kv_bits=kv_bits, start=0, tokens=forced)[0])
    a, b = runs
    assert (a - b).abs().max() <= 3e-2 * b.abs().max()
    top2 = b.topk(2, -1).values
    clear = (top2[..., 0] - top2[..., 1]) > 0.05 * b.abs().max()
    assert clear.sum() >= 10 and (a.argmax(-1)[clear] == b.argmax(-1)[clear]).all()


def test_per_row_positions_on_a_ring_need_the_fused_path(cuda_device, model_of, monkeypatch):
    dims, _, model, _, _ = model_of("tiny-llama")
    monkeypatch.setattr(qllama, "FUSED_DECODE", False)
    cache = qllama.make_prompt_cache(model, 2, 16, keep=DEFAULT_KV_KEEP)
    with torch.no_grad():
        model(torch.zeros((2, 5), dtype=torch.long, device=cuda_device), cache)
        with pytest.raises(ValueError, match="rotating"):
            model(torch.zeros((2, 1), dtype=torch.long, device=cuda_device), cache,
                  positions=torch.tensor([[3], [5]], device=cuda_device), attend_len=6)
    with pytest.raises(ValueError, match="max_kv_size"):
        utils.batch_generate(model, _prompts(dims, [3, 17]), 4, max_kv_size=16)


@pytest.mark.parametrize("kv_bits", (None, 4))
@pytest.mark.parametrize("keep", (None, DEFAULT_KV_KEEP))
def test_ragged_decode_step_launches(cuda_device, model_of, kv_bits, keep):
    """A decode step with one position per row enqueues exactly the libgbxq launches of a shared-position step."""
    dims, _, model, _, _ = model_of("tiny-llama")
    B = 4
    tok = torch.arange(B, device=cuda_device)[:, None]
    counts = {}
    for name, positions in (("shared", torch.tensor([20], device=cuda_device)),
                            ("rows", torch.tensor([[3], [20], [11], [7]], device=cuda_device))):
        cache = qllama.make_prompt_cache(model, B, 64 if keep is None else 24, keep=keep)
        with torch.no_grad():
            model(torch.zeros((B, 20), dtype=torch.long, device=cuda_device), cache)
            if kv_bits:
                cache[:] = [c.to_quantized(64, kv_bits) for c in cache]
            for c in cache:
                c.offset = 21
            torch.cuda.synchronize()
            n0 = ops.launch_count()
            model(tok, cache, positions=positions, attend_len=cache[0].attend_len)
            counts[name] = ops.launch_count() - n0
    assert counts["rows"] == counts["shared"], counts
