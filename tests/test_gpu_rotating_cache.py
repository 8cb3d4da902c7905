"""GPU tests of the rotating KV cache (`max_kv_size`): the ring cache writes against the flat ones (bit-exact, nothing
else written), runs that never wrap against the flat cache (bitwise), wrapping runs on the graph / eager / device-sampler
paths, fused against unfused decode on a wrapped ring, prefill chunking invariance, the fp32 reference under the window
mask, and the launches of a decode step."""
import pytest
import torch

from gbx_lm_b200 import ops, qllama, utils, workloads as W
from gbx_lm_b200.cache import DEFAULT_KV_KEEP, StaticRotatingKVCache, StaticRotatingQuantizedKVCache, ring_slot
from tests import ref_model

pytestmark = pytest.mark.gpu

WIDTHS = (2, 3, 4, 6, 8)
DGS = [(64, 32), (64, 64), (128, 32), (128, 64), (128, 128)]
GQA = [(2, 2), (8, 2), (16, 2)]  # (Hq, Hkv): ratios 1, 4, 8
KERNEL_CASES = ([("bf16", 0, D, 0, hq, hkv) for D in (64, 128) for hq, hkv in GQA]
                + [("q", bits, D, gs, hq, hkv) for bits in WIDTHS for D, gs in DGS for hq, hkv in GQA])
RW, RKEEP = 40, 4  # the ring of the kernel tests
POSITIONS = (0, RKEEP - 1, RKEEP, RW - 1, RW, RW + 1, 3 * RW + 7, 10 ** 6)


def _i32(t):
    return t.view(torch.int32) if t.dtype == torch.uint32 else t


def _side(kind, B, Hkv, n, D, bits, gs, dev, g=None):
    """One cache side: (bf16 [B, Hkv, n, D],) or a (codes, scales, biases) triple; random with a generator, else zero."""
    if kind == "bf16":
        shapes = [((B, Hkv, n, D), torch.bfloat16)]
    else:
        shapes = [((B, Hkv, n, D * bits // 32), torch.int32), ((B, Hkv, n, D // gs), torch.bfloat16),
                  ((B, Hkv, n, D // gs), torch.bfloat16)]
    out = []
    for shape, dt in shapes:
        if g is None:
            t = torch.zeros(shape, dtype=dt, device=dev)
        elif dt == torch.int32:
            t = torch.randint(-2 ** 31, 2 ** 31 - 1, shape, generator=g, device=dev, dtype=torch.int32)
        else:
            t = torch.randn(shape, generator=g, device=dev).to(dt)
        out.append(t.view(torch.uint32) if dt == torch.int32 else t)
    return tuple(out)


def _write(kind, q, k, v, p, inv, ks, vs, bits, gs, keep=None):
    if kind == "bf16":
        return ops.rope_cache(q, k, v, p, inv, ks[0], vs[0], keep=keep)
    return ops.rope_cache_quantized(q, k, v, p, inv, ks, vs, gs, bits, keep=keep)


@pytest.mark.parametrize("kind,bits,D,gs,Hq,Hkv", KERNEL_CASES)
def test_ring_cache_write_is_the_flat_write_at_the_ring_slot(cuda_device, kind, bits, D, gs, Hq, Hkv):
    g = torch.Generator(device=cuda_device).manual_seed(bits * 1000 + D + gs + Hq)
    inv = qllama.RoPE(D, 500000.0, False, None).to(cuda_device).inv_freq
    for pos in POSITIONS:
        B = 1 if pos >= 10 ** 6 else 2  # the flat buffer of 10^6 rows: about 0.5 GB per bf16 side at B = 1
        ring_k, ring_v = (_side(kind, B, Hkv, RW, D, bits, gs, cuda_device, g) for _ in range(2))
        before = [t.clone() for t in ring_k + ring_v]
        flat_k, flat_v = (_side(kind, B, Hkv, pos + 1, D, bits, gs, cuda_device) for _ in range(2))
        q = torch.randn((B, Hq, D), generator=g, device=cuda_device).to(torch.bfloat16)
        k = (torch.randn((B, Hkv, D), generator=g, device=cuda_device) * 3).to(torch.bfloat16)
        v = torch.randn((B, Hkv, D), generator=g, device=cuda_device).to(torch.bfloat16)
        p = torch.tensor([pos], device=cuda_device)
        want_q = _write(kind, q.clone(), k, v, p, inv, flat_k, flat_v, bits, gs)
        got_q = _write(kind, q.clone(), k, v, p, inv, ring_k, ring_v, bits, gs, keep=RKEEP)
        assert torch.equal(got_q, want_q), pos
        slot = ring_slot(pos, RW, RKEEP)
        others = torch.ones(RW, dtype=torch.bool, device=cuda_device)
        others[slot] = False
        for got, flat, old in zip(ring_k + ring_v, flat_k + flat_v, before):
            assert torch.equal(_i32(got)[:, :, slot], _i32(flat)[:, :, pos]), pos
            assert torch.equal(_i32(got)[:, :, others], _i32(old)[:, :, others]), pos  # no other row changes
        if pos < RW:  # below the window the ring entry point is the flat one
            old_k, old_v = tuple(before[:len(ring_k)]), tuple(before[len(ring_k):])
            assert torch.equal(_write(kind, q.clone(), k, v, p, inv, old_k, old_v, bits, gs), got_q)
            for a, b in zip(old_k + old_v, ring_k + ring_v):
                assert torch.equal(_i32(a), _i32(b)), pos
        del flat_k, flat_v


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
            _MODELS[name] = (dims, cfg, model, d)
        return _MODELS[name]

    yield get
    _MODELS.clear()


def _prompt(dims, n, seed=3):
    return torch.randint(0, dims.vocab, (n,), generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("kv_bits", (None, 4, 8))
@pytest.mark.parametrize("name", ("tiny-llama", "tiny-qwen2"))
def test_unwrapped_ring_is_the_flat_cache_bitwise(cuda_device, model_of, name, kv_bits):
    """A window at least as long as the run: per-step logits and the tokens and log-probabilities of the graph, eager
    and device-sampler paths are bitwise those of the flat cache."""
    dims, _, model, _ = model_of(name)
    prompt = _prompt(dims, 12)
    toks = prompt.to(cuda_device)[None]

    def logits(keep):
        cache = qllama.make_prompt_cache(model, 1, 64, keep=keep)
        outs = []
        with torch.no_grad():
            outs.append(model(toks[:, :7], cache))
            outs.append(model(toks[:, 7:], cache))
            if kv_bits:
                cache[:] = [c.to_quantized(64, kv_bits) for c in cache]
            for i in range(20):
                outs.append(model(torch.tensor([[i * 7 % dims.vocab]], device=cuda_device), cache))
        assert (cache[0].keep is None) == (keep is None)
        return outs

    for a, b in zip(logits(None), logits(DEFAULT_KV_KEEP)):
        assert torch.equal(a, b)
    kw = dict(kv_bits=kv_bits, kv_group_size=64, quantized_kv_start=15)
    for graph in (True, False):
        flat = list(utils.generate_step(prompt, model, max_tokens=24, use_cuda_graph=graph, **kw))
        ring = list(utils.generate_step(prompt, model, max_tokens=24, use_cuda_graph=graph, max_kv_size=37, **kw))
        assert [t for t, _ in flat] == [t for t, _ in ring]
        assert all(torch.equal(a, b) for (_, a), (_, b) in zip(flat, ring))
    d_flat, _ = utils.generate_tokens_device(model, prompt, max_tokens=24, **kw)
    d_ring, _ = utils.generate_tokens_device(model, prompt, max_tokens=24, max_kv_size=37, **kw)
    assert d_flat == d_ring == [t for t, _ in flat]


WRAP_CASES = {  # (prompt, window, max_tokens, prefill_step_size, kv_bits, quantized_kv_start)
    "decode": (12, 24, 40, 2048, None, 0),
    "prefill": (40, 24, 24, 2048, None, 0),
    "prefill-chunked": (40, 24, 24, 16, None, 0),
    "max1": (40, 24, 1, 2048, None, 0),
    "kv4-before": (12, 24, 40, 2048, 4, 5),
    "kv8-after": (12, 24, 40, 2048, 8, 30),
    "kv4-prefill": (40, 24, 24, 16, 4, 20),
    "kv8-max1": (40, 24, 1, 2048, 8, 0),
}


@pytest.mark.parametrize("case", sorted(WRAP_CASES))
@pytest.mark.parametrize("name", ("tiny-llama", "tiny-qwen2"))
def test_wrapping_runs_graph_eager_device(cuda_device, model_of, name, case):
    """Runs that wrap during prefill or during decode, with the quantized conversion before or after the wrap: the
    three decode paths give the same tokens, and the buffers stay `window` positions long."""
    n_prompt, window, max_tokens, step, kv_bits, start = WRAP_CASES[case]
    dims, _, model, _ = model_of(name)
    prompt = _prompt(dims, n_prompt)
    kw = dict(kv_bits=kv_bits, kv_group_size=64, quantized_kv_start=start, prefill_step_size=step)
    cache = qllama.make_prompt_cache(model, 1, window, keep=DEFAULT_KV_KEEP)
    g_toks, _ = utils.generate_tokens(model, prompt, max_tokens=max_tokens, use_cuda_graph=True, prompt_cache=cache,
                                      **kw)
    e_toks, _ = utils.generate_tokens(model, prompt, max_tokens=max_tokens, use_cuda_graph=False, max_kv_size=window,
                                      **kw)
    d_toks, _ = utils.generate_tokens_device(model, prompt, max_tokens=max_tokens, max_kv_size=window, **kw)
    assert len(g_toks) == max_tokens and g_toks == e_toks == d_toks
    want = StaticRotatingQuantizedKVCache if kv_bits is not None else StaticRotatingKVCache
    assert all(type(c) is want for c in cache)
    assert cache[0].offset == n_prompt + max_tokens and cache[0].keep == DEFAULT_KV_KEEP
    for c in cache:
        for t in ((c.keys,) if kv_bits is None else c.keys) + ((c.values,) if kv_bits is None else c.values):
            assert t.shape[2] == window


@pytest.mark.parametrize("kv_bits", (None, 4, 8))
@pytest.mark.parametrize("name", ("tiny-llama", "tiny-qwen2"))
def test_fused_decode_on_wrapped_ring_matches_unfused(cuda_device, model_of, monkeypatch, name, kv_bits):
    dims, _, model, _ = model_of(name)
    toks = torch.randint(0, dims.vocab, (1, 56), generator=torch.Generator().manual_seed(4)).to(cuda_device)

    def run(fused):
        monkeypatch.setattr(qllama, "FUSED_DECODE", fused)
        cache = qllama.make_prompt_cache(model, 1, 24, keep=DEFAULT_KV_KEEP)
        outs = []
        with torch.no_grad():
            outs.append(model(toks[:, :8], cache)[:, -1:].float())
            if kv_bits:
                cache[:] = [c.to_quantized(64, kv_bits) for c in cache]
            for i in range(8, 56):
                outs.append(model(toks[:, i:i + 1], cache).float())
        assert cache[0].offset == 56 and cache[0].attend_len == 24
        return torch.cat(outs, 1)

    a, b = run(True), run(False)
    assert (a - b).abs().max() <= 3e-2 * b.abs().max()
    top2 = b.topk(2, -1).values
    clear = (top2[..., 0] - top2[..., 1]) > 0.05 * b.abs().max()
    assert clear.sum() >= 10 and (a.argmax(-1)[clear] == b.argmax(-1)[clear]).all()


@pytest.mark.parametrize("kv_bits", (None, 8))
def test_prefill_chunking_invariance_on_a_wrapping_prompt(cuda_device, model_of, kv_bits):
    """Every query sees the keys its decode step would see, so the chunk size changes only the order of summation."""
    dims, _, model, _ = model_of("tiny-llama")
    window = 24
    prompt = _prompt(dims, 70, seed=9).to(cuda_device)
    outs = []
    for step in (1, 5, window - DEFAULT_KV_KEEP - 1, 2048):
        if kv_bits is None:
            cache = qllama.make_prompt_cache(model, 1, window, keep=DEFAULT_KV_KEEP)
        else:  # quantized from the first position, so that every chunk size attends the same quantized keys
            cache = [StaticRotatingQuantizedKVCache(1, dims.kv_heads, window, dims.head_dim, cuda_device, DEFAULT_KV_KEEP,
                                                    64, kv_bits) for _ in range(dims.layers)]
        outs.append(utils.prefill(model, prompt, cache, step).float())
        assert cache[0].offset == 70
    for o in outs[1:]:
        assert (o - outs[0]).abs().max() <= 3e-2 * outs[0].abs().max()


def _ref_forward(Wd, cfg, tokens, visible):
    """`tests/ref_model.forward` (fp32, no cache) with the attention mask given: visible bool [L, L], query i sees key j.
    The same steps, built from its helpers."""
    H, nh, nkv = cfg["hidden_size"], cfg["num_attention_heads"], cfg["num_key_value_heads"]
    hd = cfg.get("head_dim") or H // nh
    eps = cfg["rms_norm_eps"]
    inv = ref_model._inv_freq(hd, cfg["rope_theta"], cfg.get("rope_scaling"))
    B, L = tokens.shape
    pos = torch.arange(L)
    h = Wd["model.embed_tokens.weight"][tokens]
    lin = lambda x, name: torch.nn.functional.linear(x, Wd[name + ".weight"], Wd.get(name + ".bias"))
    for i in range(cfg["num_hidden_layers"]):
        p = f"model.layers.{i}."
        x = ref_model._rms(h, Wd[p + "input_layernorm.weight"], eps)
        q = lin(x, p + "self_attn.q_proj").view(B, L, nh, hd).transpose(1, 2)
        k = lin(x, p + "self_attn.k_proj").view(B, L, nkv, hd).transpose(1, 2)
        v = lin(x, p + "self_attn.v_proj").view(B, L, nkv, hd).transpose(1, 2)
        q, k = ref_model._rope(q, pos, inv), ref_model._rope(k, pos, inv)
        k = k.repeat_interleave(nh // nkv, 1)
        v = v.repeat_interleave(nh // nkv, 1)
        att = ((q @ k.transpose(-1, -2)) * hd ** -0.5).masked_fill(~visible, float("-inf")).softmax(-1)
        o = (att @ v).transpose(1, 2).reshape(B, L, -1)
        h = h + lin(o, p + "self_attn.o_proj")
        x = ref_model._rms(h, Wd[p + "post_attention_layernorm.weight"], eps)
        h = h + lin(torch.nn.functional.silu(lin(x, p + "mlp.gate_proj")) * lin(x, p + "mlp.up_proj"), p + "mlp.down_proj")
    h = ref_model._rms(h, Wd["model.norm.weight"], eps)
    head = Wd["model.embed_tokens.weight"] if cfg.get("tie_word_embeddings", True) else Wd["lm_head.weight"]
    return h @ head.t()


def test_ring_tokens_match_reference_on_clear_steps(cuda_device, model_of):
    """Greedy tokens on a wrapping ring against the fp32 reference under the window mask, teacher-forced."""
    from safetensors.torch import load_file

    dims, cfg, model, d = model_of("tiny-llama")
    ckpt = load_file(str(d / "model.safetensors"))
    plan = {}
    for (i, p, n, k, b, g) in W.layer_plan(dims, W.STRATEGIES["bpw-4.0"](dims.layers), 4, 64):
        sub = "self_attn" if p in ("q_proj", "k_proj", "v_proj", "o_proj") else "mlp"
        plan[f"model.layers.{i}.{sub}.{p}"] = (b, g)
    dense = ref_model.dense_weights(ckpt, lambda m: plan[m])
    window, keep = 20, DEFAULT_KV_KEEP
    prompt = _prompt(dims, 12)
    toks, _ = utils.generate_tokens(model, prompt, max_tokens=48, max_kv_size=window)
    seq = torch.cat([prompt, torch.tensor(toks)])[None]
    i, j = torch.arange(seq.shape[1])[:, None], torch.arange(seq.shape[1])[None, :]
    visible = (j <= i) & ((j < keep) | (j > i - (window - keep)))
    with torch.no_grad():
        # under the causal mask the restatement is the reference itself, bitwise
        assert torch.equal(_ref_forward(dense, cfg, seq, j <= i), ref_model.forward(dense, cfg, seq))
        ref = _ref_forward(dense, cfg, seq, visible)[0, len(prompt) - 1:-1]
    top2 = ref.topk(2, -1).values
    clear = (top2[:, 0] - top2[:, 1]) > 0.05 * ref.abs().max()
    assert clear.sum() >= 10, f"only {int(clear.sum())} decisive steps"
    assert (ref.argmax(-1)[clear] == torch.tensor(toks)[clear]).all()


@pytest.mark.parametrize("kv_bits", (None, 4))
def test_ring_decode_step_launches(cuda_device, model_of, kv_bits):
    """A decode step on a wrapped ring enqueues exactly the libgbxq launches of a step on the flat cache."""
    dims, _, model, _ = model_of("tiny-llama")
    tok = torch.tensor([[3]], device=cuda_device)
    counts = {}
    for keep, size in ((None, 64), (DEFAULT_KV_KEEP, 16)):
        cache = qllama.make_prompt_cache(model, 1, size, keep=keep)
        with torch.no_grad():
            model(torch.arange(20, device=cuda_device)[None], cache)
            if kv_bits:
                cache[:] = [c.to_quantized(64, kv_bits) for c in cache]
            torch.cuda.synchronize()
            n0 = ops.launch_count()
            model(tok, cache)
            counts[keep] = ops.launch_count() - n0
        assert cache[0].keep == keep
    assert counts[DEFAULT_KV_KEEP] == counts[None], counts
