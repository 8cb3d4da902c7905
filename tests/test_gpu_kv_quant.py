"""GPU tests of the quantized-KV decode path: gbxq_rope_cache_quantized against gbxq_rope_cache + gbxq_quantize_rows
(bit-exact), gbxq_decode_attention_quantized against an fp64 evaluation on the oracle-dequantised cache and against
quantized_scaled_dot_product_attention, its determinism across attend_len / max_len, and the model + generation with
kv_bits (fused vs unfused decode, graph vs eager vs device sampler, the fp32 reference on clear-margin steps, launches
per step)."""
import numpy as np
import pytest
import torch

from gbx_lm_b200 import ops, qllama, switch_layers, utils, workloads as W
from gbx_lm_b200.cache import DECODE_ATTENTION_MAX_KEYS, StaticQuantizedKVCache
from oracle import mlx_affine as A
from tests import ref_model

pytestmark = pytest.mark.gpu

WIDTHS = (2, 3, 4, 6, 8)
DGS = [(64, 32), (64, 64), (128, 32), (128, 64), (128, 128)]
GQA = [(2, 2), (8, 2), (16, 2)]  # (Hq, Hkv): ratios 1, 4, 8


def _triple(b, h, n, d, bits, gs, device):
    return (torch.zeros((b, h, n, d * bits // 32), dtype=torch.int32, device=device).view(torch.uint32),
            torch.zeros((b, h, n, d // gs), dtype=torch.bfloat16, device=device),
            torch.zeros((b, h, n, d // gs), dtype=torch.bfloat16, device=device))


def _i32(t):
    return t.view(torch.int32) if t.dtype == torch.uint32 else t


@pytest.mark.parametrize("Hq,Hkv", GQA)
@pytest.mark.parametrize("D,gs", DGS)
@pytest.mark.parametrize("bits", WIDTHS)
def test_rope_cache_quantized_is_rope_cache_then_quantize(cuda_device, bits, D, gs, Hq, Hkv):
    B, max_len = 2, 300
    g = torch.Generator(device=cuda_device).manual_seed(bits * 1000 + D + gs + Hq)
    rope = qllama.RoPE(D, 500000.0, False, None).to(cuda_device)
    k3, v3 = _triple(B, Hkv, max_len, D, bits, gs, cuda_device), _triple(B, Hkv, max_len, D, bits, gs, cuda_device)
    want_k3, want_v3 = _triple(B, Hkv, max_len, D, bits, gs, cuda_device), _triple(B, Hkv, max_len, D, bits, gs, cuda_device)
    kc = torch.zeros((B, Hkv, max_len, D), dtype=torch.bfloat16, device=cuda_device)
    vc = torch.zeros_like(kc)
    for pos in (0, 256, max_len - 1):  # first row, a key-chunk border, last row
        q = torch.randn((B, Hq, D), generator=g, device=cuda_device).to(torch.bfloat16)
        k = (torch.randn((B, Hkv, D), generator=g, device=cuda_device) * 3).to(torch.bfloat16)
        v = torch.randn((B, Hkv, D), generator=g, device=cuda_device).to(torch.bfloat16)
        p = torch.tensor([pos], device=cuda_device)
        want_q = ops.rope_cache(q.clone(), k, v, p, rope.inv_freq, kc, vc)
        ops.quantize_into(kc[:, :, pos:pos + 1], want_k3, pos, gs, bits)
        ops.quantize_into(vc[:, :, pos:pos + 1], want_v3, pos, gs, bits)
        got_q = ops.rope_cache_quantized(q.clone(), k, v, p, rope.inv_freq, k3, v3, gs, bits)
        assert torch.equal(got_q, want_q)
        for got, want in zip(k3 + v3, want_k3 + want_v3):
            assert torch.equal(_i32(got), _i32(want)), pos
    written = torch.zeros(max_len, dtype=torch.bool)
    written[[0, 256, max_len - 1]] = True
    for t in k3 + v3:  # every other position untouched
        assert not _i32(t)[:, :, ~written.to(cuda_device)].any()


def _oracle_deq(t3, gs, bits):
    q, s, b = (x.cpu() for x in t3)
    d = A.dequantize(q.contiguous().view(torch.int32).numpy().view(np.uint32).reshape(-1, q.shape[-1]),
                     s.float().numpy().reshape(-1, s.shape[-1]), b.float().numpy().reshape(-1, b.shape[-1]), gs, bits, "f32")
    return torch.from_numpy(d).reshape(*q.shape[:-1], -1).double()


def _ref_attention(q, kd, vd, pos, scale):
    """fp64 softmax(scale q.K^T) V over keys 0..pos, GQA; kd / vd [B, Hkv, T, D] float64 (any device)."""
    B, Hq, D = q.shape
    rep = Hq // kd.shape[1]
    k = kd[:, :, : pos + 1].repeat_interleave(rep, 1)
    v = vd[:, :, : pos + 1].repeat_interleave(rep, 1)
    s = torch.einsum("bhd,bhtd->bht", q.double(), k) * scale
    return torch.einsum("bht,bhtd->bhd", torch.softmax(s, -1), v)


def _fill(B, Hkv, n, D, bits, gs, device, seed):
    g = torch.Generator(device=device).manual_seed(seed)
    k = (torch.randn((B, Hkv, n, D), generator=g, device=device) * 2).to(torch.bfloat16)
    v = torch.randn((B, Hkv, n, D), generator=g, device=device).to(torch.bfloat16)
    return ops.quantize(k, gs, bits), ops.quantize(v, gs, bits)


def _close(got, want):
    err = (got.double().cpu() - want.cpu()).abs().max().item()
    assert err <= 1e-2 * want.abs().max().item() + 1e-3, err


@pytest.mark.parametrize("Hq,Hkv", GQA)
@pytest.mark.parametrize("D,gs", DGS)
@pytest.mark.parametrize("bits", WIDTHS)
def test_decode_attention_quantized_matches_fp64(cuda_device, bits, D, gs, Hq, Hkv):
    B, max_len = 2, 600
    k3, v3 = _fill(B, Hkv, max_len, D, bits, gs, cuda_device, bits * 7 + D + gs + Hq)
    kd, vd = _oracle_deq(k3, gs, bits).to(cuda_device), _oracle_deq(v3, gs, bits).to(cuda_device)
    g = torch.Generator(device=cuda_device).manual_seed(5)
    q = torch.randn((B, Hq, D), generator=g, device=cuda_device).to(torch.bfloat16)
    scale = D ** -0.5
    for pos in (0, 1, 255, 256, 257, 511, 512, max_len - 1):  # chunk borders +- 1
        p = torch.tensor([pos], device=cuda_device)
        want = _ref_attention(q, kd, vd, pos, scale)
        got = ops.decode_attention_quantized(q, k3, v3, p, scale, gs, bits)
        _close(got, want)
        # eager form (attend_len = pos + 1): bitwise the same as the whole-cache form
        assert torch.equal(ops.decode_attention_quantized(q, k3, v3, p, scale, gs, bits, attend_len=pos + 1), got)
    # attend_len clamps the visible prefix
    got = ops.decode_attention_quantized(q, k3, v3, torch.tensor([max_len - 1], device=cuda_device), scale, gs, bits,
                                         attend_len=300)
    _close(got, _ref_attention(q, kd, vd, 299, scale))


@pytest.mark.parametrize("bits", (4, 8))
def test_decode_attention_quantized_long_context(cuda_device, bits):
    """70 000 keys: above the 49 152-key limit of the bf16 kernel; ~18 MB of 4-bit cache with Hkv 2."""
    B, Hq, Hkv, D, gs, n = 1, 8, 2, 128, 64, 70000
    k3, v3 = _fill(B, Hkv, n, D, bits, gs, cuda_device, 11)
    g = torch.Generator(device=cuda_device).manual_seed(6)
    q = torch.randn((B, Hq, D), generator=g, device=cuda_device).to(torch.bfloat16)
    kd, vd = _oracle_deq(k3, gs, bits).to(cuda_device), _oracle_deq(v3, gs, bits).to(cuda_device)
    for pos in (n - 1, DECODE_ATTENTION_MAX_KEYS, 1000):
        p = torch.tensor([pos], device=cuda_device)
        got = ops.decode_attention_quantized(q, k3, v3, p, D ** -0.5, gs, bits)
        _close(got, _ref_attention(q, kd, vd, pos, D ** -0.5))


@pytest.mark.parametrize("bits", (2, 3, 4, 6, 8))
def test_decode_attention_quantized_is_deterministic_and_independent_of_max_len(cuda_device, bits):
    B, Hq, Hkv, D, gs, n = 2, 32, 8, 128, 64, 900
    k3, v3 = _fill(B, Hkv, n, D, bits, gs, cuda_device, 21)
    big_k3, big_v3 = _triple(B, Hkv, 2000, D, bits, gs, cuda_device), _triple(B, Hkv, 2000, D, bits, gs, cuda_device)
    for dst, src in zip(big_k3 + big_v3, k3 + v3):
        _i32(dst)[:, :, :n] = _i32(src)
    g = torch.Generator(device=cuda_device).manual_seed(8)
    q = torch.randn((B, Hq, D), generator=g, device=cuda_device).to(torch.bfloat16)
    for pos in (0, 300, n - 1):
        p = torch.tensor([pos], device=cuda_device)
        a = ops.decode_attention_quantized(q, k3, v3, p, 0.1, gs, bits)
        assert torch.equal(a, ops.decode_attention_quantized(q, k3, v3, p, 0.1, gs, bits))  # run to run
        for attend_len in (pos + 1, n, 1500, 2000):
            b = ops.decode_attention_quantized(q, big_k3, big_v3, p, 0.1, gs, bits, attend_len=attend_len)
            assert torch.equal(a, b), (pos, attend_len)
    # within bf16 noise of the two-launch path (quantized_scaled_dot_product_attention) on the same triples
    pos = n - 1
    want = switch_layers.quantized_scaled_dot_product_attention(q[:, :, None], k3, v3, 0.1, None, gs, bits)[:, :, 0]
    got = ops.decode_attention_quantized(q, k3, v3, torch.tensor([pos], device=cuda_device), 0.1, gs, bits)
    assert (got.float() - want.float()).abs().max() <= 2e-2 * want.float().abs().max() + 2e-3


# ------------------------------------------------------------------------------------------ the model and generation
def _model(tmp_path, name, cuda_device, seed=5):
    dims = W.MODELS[name]
    strat = W.STRATEGIES["bpw-4.0"](dims.layers) if name == "tiny-llama" else None
    cfg = utils.write_synthetic_checkpoint(tmp_path, dims, strat, seed=seed, default_bits=4, default_gs=64, embed_scale=1.0)
    model, _ = utils.load_model(tmp_path, device=cuda_device)
    return dims, cfg, model


@pytest.mark.parametrize("kv_bits", (4, 8))
@pytest.mark.parametrize("name", ("tiny-llama", "tiny-qwen2"))
def test_fused_decode_on_static_quantized_cache_matches_unfused(cuda_device, tmp_path, monkeypatch, name, kv_bits):
    dims, _, model = _model(tmp_path, name, cuda_device)
    toks = torch.randint(0, dims.vocab, (1, 40), generator=torch.Generator().manual_seed(4)).to(cuda_device)

    def run(fused):
        monkeypatch.setattr(qllama, "FUSED_DECODE", fused)
        cache = qllama.make_prompt_cache(model, 1, 64)
        outs = []
        with torch.no_grad():
            outs.append(model(toks[:, :8], cache)[:, -1:].float())
            cache[:] = [c.to_quantized(64, kv_bits) for c in cache]
            for i in range(8, 40):
                outs.append(model(toks[:, i:i + 1], cache).float())
        assert isinstance(cache[0], StaticQuantizedKVCache) and cache[0].offset == 40
        return torch.cat(outs, 1)

    a, b = run(True), run(False)
    assert (a - b).abs().max() <= 3e-2 * b.abs().max()
    top2 = b.topk(2, -1).values
    clear = (top2[..., 0] - top2[..., 1]) > 0.05 * b.abs().max()
    assert clear.sum() >= 10 and (a.argmax(-1)[clear] == b.argmax(-1)[clear]).all()


@pytest.mark.parametrize("kv_bits,start,max_tokens",
                         [(4, 0, 40), (8, 0, 40), (4, 20, 40), (8, 20, 40), (4, 11, 40), (8, 100, 40), (4, 12, 1), (8, 0, 1)],
                         ids=["4-0", "8-0", "4-20", "8-20", "4-11", "8-100", "4-12-max1", "8-0-max1"])
@pytest.mark.parametrize("name", ("tiny-llama", "tiny-qwen2"))
def test_generate_with_quantized_cache_graph_eager_device(cuda_device, tmp_path, name, kv_bits, start, max_tokens):
    """With a 12-token prompt: start 0 converts after the first prefill call, start 11 right after the prompt, start 20
    mid-decode (the graph is captured again, the device loop replays up to the conversion and continues on a new graph),
    start 100 never; max_tokens 1 yields the prefill's token alone."""
    dims, _, model = _model(tmp_path, name, cuda_device, seed=11)
    prompt = torch.randint(0, dims.vocab, (12,), generator=torch.Generator().manual_seed(3))
    kw = dict(kv_bits=kv_bits, kv_group_size=64, quantized_kv_start=start)
    g_toks, _ = utils.generate_tokens(model, prompt, max_tokens=max_tokens, use_cuda_graph=True, **kw)
    e_toks, _ = utils.generate_tokens(model, prompt, max_tokens=max_tokens, use_cuda_graph=False, **kw)
    d_toks, stats = utils.generate_tokens_device(model, prompt, max_tokens=max_tokens, **kw)
    assert len(g_toks) == max_tokens and g_toks == e_toks and d_toks == g_toks and stats["generation_tps"] > 0
    c_toks, _ = utils.generate_tokens(model, prompt, max_tokens=16, prefill_step_size=5, **kw)  # conversion mid-prefill
    assert len(c_toks) == 16


def test_kv8_tokens_match_reference_on_clear_steps(cuda_device, tmp_path):
    from safetensors.torch import load_file

    dims, cfg, model = _model(tmp_path, "tiny-llama", cuda_device, seed=11)
    ckpt = load_file(str(tmp_path / "model.safetensors"))
    strat = W.STRATEGIES["bpw-4.0"](dims.layers)
    plan = {}
    for (i, p, n, k, b, g) in W.layer_plan(dims, strat, 4, 64):
        sub = "self_attn" if p in ("q_proj", "k_proj", "v_proj", "o_proj") else "mlp"
        plan[f"model.layers.{i}.{sub}.{p}"] = (b, g)
    dense = ref_model.dense_weights(ckpt, lambda m: plan[m])
    prompt = torch.randint(0, dims.vocab, (12,), generator=torch.Generator().manual_seed(3))
    q_toks, _ = utils.generate_tokens(model, prompt, max_tokens=48, kv_bits=8, kv_group_size=64, quantized_kv_start=0)
    # teacher-forced on the 8-bit run's tokens: the fp32 reference and the bf16-cache model (a full forward, no cache)
    seq = torch.cat([prompt, torch.tensor(q_toks)])[None]
    with torch.no_grad():
        ref = ref_model.forward(dense, cfg, seq)[0, len(prompt) - 1:-1]
        bf16 = model(seq.to(cuda_device)).float().cpu()[0, len(prompt) - 1:-1]
    top2 = ref.topk(2, -1).values
    clear = (top2[:, 0] - top2[:, 1]) > 0.05 * ref.abs().max()
    assert clear.sum() >= 24, f"only {int(clear.sum())} decisive steps"
    got = torch.tensor(q_toks)
    assert (ref.argmax(-1)[clear] == got[clear]).all()
    assert (bf16.argmax(-1)[clear] == got[clear]).all()


def test_quantized_decode_step_launches(cuda_device, tmp_path):
    """One decode step enqueues, per layer, one cache write and one attention launch as the bf16 step does, plus the
    combine launch of the split-K attention: layers more libgbxq launches than the bf16 step."""
    dims, _, model = _model(tmp_path, "tiny-llama", cuda_device)
    tok = torch.tensor([[3]], device=cuda_device)
    counts = {}
    for kv_bits in (None, 4):
        cache = qllama.make_prompt_cache(model, 1, 64)
        with torch.no_grad():
            model(torch.arange(8, device=cuda_device)[None], cache)
            if kv_bits:
                cache[:] = [c.to_quantized(64, kv_bits) for c in cache]
            torch.cuda.synchronize()
            n0 = ops.launch_count()
            model(tok, cache)
            counts[kv_bits] = ops.launch_count() - n0
    assert counts[4] == counts[None] + dims.layers, counts
