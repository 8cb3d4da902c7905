"""GPU tests of the decode-step glue kernels (gbxq_rope_cache / gbxq_decode_attention / gbxq_add_rmsnorm /
gbxq_silu_mul, include/gbxq.h) against the plain PyTorch expressions they replace in the callers
(gbx_lm/models/qllama.py:76-141 restated in gbx_lm_b200/qllama.py), and of the fused decode path of the model against
the unfused one."""
import pytest
import torch
import torch.nn.functional as F

from gbx_lm_b200 import ops, qllama, utils, workloads as W

pytestmark = pytest.mark.gpu


def _ulp_close(a, b, frac=0.999, tol=1.0 / 64):
    """bf16 results of the same fp32 expression: equal almost everywhere, never more than ~1 ulp apart."""
    a, b = a.float(), b.float()
    same = (a == b).float().mean().item()
    rel = ((a - b).abs() / b.abs().clamp_min(1e-3)).max().item()
    assert same >= frac and rel <= tol, (same, rel)


@pytest.mark.parametrize("D,Hq,Hkv", [(64, 8, 2), (128, 4, 4), (128, 32, 8)])
def test_rope_cache_matches_torch(cuda_device, D, Hq, Hkv):
    g = torch.Generator(device=cuda_device).manual_seed(D + Hq)
    B, max_len, pos = 2, 96, 37
    rope = qllama.RoPE(D, 500000.0, False, None).to(cuda_device)
    q = torch.randn((B, Hq, D), generator=g, device=cuda_device).to(torch.bfloat16)
    k = torch.randn((B, Hkv, D), generator=g, device=cuda_device).to(torch.bfloat16)
    v = torch.randn((B, Hkv, D), generator=g, device=cuda_device).to(torch.bfloat16)
    p = torch.tensor([pos], device=cuda_device)
    want_q = rope(q[:, :, None, :], p)[:, :, 0]
    want_k = rope(k[:, :, None, :], p)[:, :, 0]
    kc = torch.zeros((B, Hkv, max_len, D), device=cuda_device, dtype=torch.bfloat16)
    vc = torch.zeros_like(kc)
    got_q = ops.rope_cache(q.clone(), k, v, p, rope.inv_freq, kc, vc)
    _ulp_close(got_q, want_q)
    _ulp_close(kc[:, :, pos], want_k)
    assert torch.equal(vc[:, :, pos], v)
    kc[:, :, pos] = 0
    vc[:, :, pos] = 0
    assert not kc.any() and not vc.any()  # nothing else was touched


@pytest.mark.parametrize("D,Hq,Hkv,pos", [(64, 8, 2, 0), (64, 8, 2, 70), (128, 32, 8, 200), (128, 4, 4, 5)])
def test_decode_attention_matches_sdpa(cuda_device, D, Hq, Hkv, pos):
    g = torch.Generator(device=cuda_device).manual_seed(pos + D)
    B, max_len = 2, 256
    q = torch.randn((B, Hq, D), generator=g, device=cuda_device).to(torch.bfloat16)
    kc = torch.randn((B, Hkv, max_len, D), generator=g, device=cuda_device).to(torch.bfloat16)
    vc = torch.randn((B, Hkv, max_len, D), generator=g, device=cuda_device).to(torch.bfloat16)
    p = torch.tensor([pos], device=cuda_device)
    scale = D ** -0.5
    got = ops.decode_attention(q, kc, vc, p, scale).float()
    mask = torch.arange(max_len, device=cuda_device)[None, :] <= p[:, None]
    rep = Hq // Hkv
    want = F.scaled_dot_product_attention(q[:, :, None].float(), kc.float().repeat_interleave(rep, 1),
                                          vc.float().repeat_interleave(rep, 1), attn_mask=mask[None, None], scale=scale)[:, :, 0]
    assert (got - want).abs().max() <= 1e-2 * want.abs().max() + 1e-3
    # attend_len clamps the visible prefix
    got2 = ops.decode_attention(q, kc, vc, torch.tensor([max_len - 1], device=cuda_device), scale, attend_len=pos + 1).float()
    assert (got2 - want).abs().max() <= 1e-2 * want.abs().max() + 1e-3


@pytest.mark.parametrize("op", ("rope_cache", "decode_attention", "rope_cache_quantized", "decode_attention_quantized"))
def test_ops_refuse_positions_the_kernels_cannot_read(cuda_device, op):
    """The kernels read `position` as int64 in device memory: an int32 [1] or a host int64 [1] position is a ValueError
    before anything is launched."""
    B, Hq, Hkv, D, max_len, bits, gs = 2, 8, 2, 128, 64, 4, 64
    bf = dict(dtype=torch.bfloat16, device=cuda_device)
    q, k = torch.zeros((B, Hq, D), **bf), torch.zeros((B, Hkv, D), **bf)
    kc = torch.zeros((B, Hkv, max_len, D), **bf)
    inv = torch.ones(D // 2, dtype=torch.float32, device=cuda_device)
    c3 = (torch.zeros((B, Hkv, max_len, D * bits // 32), dtype=torch.int32, device=cuda_device).view(torch.uint32),
          torch.zeros((B, Hkv, max_len, D // gs), **bf), torch.zeros((B, Hkv, max_len, D // gs), **bf))
    call = {
        "rope_cache": lambda p: ops.rope_cache(q, k, k, p, inv, kc, kc),
        "decode_attention": lambda p: ops.decode_attention(q, kc, kc, p, 0.1),
        "rope_cache_quantized": lambda p: ops.rope_cache_quantized(q, k, k, p, inv, c3, c3, gs, bits),
        "decode_attention_quantized": lambda p: ops.decode_attention_quantized(q, c3, c3, p, 0.1, gs, bits),
    }[op]
    call(torch.zeros(1, dtype=torch.int64, device=cuda_device))  # the same call with a valid position launches
    for bad in (torch.zeros(1, dtype=torch.int32, device=cuda_device), torch.zeros(1, dtype=torch.int64)):
        n0 = ops.launch_count()
        with pytest.raises(ValueError, match=f"{op}: position"):
            call(bad)
        assert ops.launch_count() == n0, (op, bad.dtype, bad.device)
    torch.cuda.synchronize()


@pytest.mark.parametrize("H", (256, 4096, 8192))
def test_add_rmsnorm_and_silu_mul_match_torch(cuda_device, H):
    g = torch.Generator(device=cuda_device).manual_seed(H)
    x = torch.randn((3, 1, H), generator=g, device=cuda_device).to(torch.bfloat16)
    r = torch.randn((3, 1, H), generator=g, device=cuda_device).to(torch.bfloat16)
    w = (1 + 0.1 * torch.randn((H,), generator=g, device=cuda_device)).to(torch.bfloat16)
    h, y = ops.add_rmsnorm(x, r, w, 1e-5)
    want_h = x + r
    assert torch.equal(h, want_h)
    want_y = F.rms_norm(want_h.float(), (H,), w.float(), 1e-5)
    assert (y.float() - want_y).abs().max() <= 1e-2 * want_y.abs().max()
    h2, y2 = ops.add_rmsnorm(x, None, w, 1e-5)
    assert h2 is x
    assert (y2.float() - F.rms_norm(x.float(), (H,), w.float(), 1e-5)).abs().max() <= 1e-2 * want_y.abs().max()
    _, y3 = ops.add_rmsnorm(x, r, w, 1e-5, want_h=False)
    assert torch.equal(y3, y)
    _ulp_close(ops.silu_mul(x, r), F.silu(x) * r, frac=0.99)


def test_fused_decode_matches_unfused_model(cuda_device, tmp_path, monkeypatch):
    """The same checkpoint decoded with the glue kernels and with the plain torch glue: logits agree within bf16 noise
    at every step, and the greedy tokens agree wherever the unfused top-1 margin is clear."""
    dims = W.MODELS["tiny-llama"]
    utils.write_synthetic_checkpoint(tmp_path, dims, W.STRATEGIES["bpw-4.0"](dims.layers), seed=5, default_bits=4,
                                     default_gs=64, embed_scale=1.0)
    model, _ = utils.load_model(tmp_path, device=cuda_device)
    toks = torch.randint(0, dims.vocab, (1, 40), generator=torch.Generator().manual_seed(4)).to(cuda_device)

    def run(fused):
        monkeypatch.setattr(qllama, "FUSED_DECODE", fused)
        cache = qllama.make_prompt_cache(model, 1, 64)
        outs = []
        with torch.no_grad():
            outs.append(model(toks[:, :8], cache)[:, -1:].float())
            for i in range(8, 40):
                outs.append(model(toks[:, i:i + 1], cache).float())
        return torch.cat(outs, 1)

    a, b = run(True), run(False)
    assert (a - b).abs().max() <= 3e-2 * b.abs().max()
    top2 = b.topk(2, -1).values
    clear = (top2[..., 0] - top2[..., 1]) > 0.05 * b.abs().max()
    assert clear.sum() >= 10 and (a.argmax(-1)[clear] == b.argmax(-1)[clear]).all()


@pytest.mark.parametrize("shape", [(1, 128256, 2048), (1, 128256, 4096), (2, 512, 256), (1, 1000, 3072), (2, 152064, 5120), (1, 7, 8192)])
def test_head_gemv_matches_fp32_linear(cuda_device, shape):
    """gbxq_head_gemv (the unquantized vocabulary projection, qllama.py:183-184,194-198) against F.linear evaluated in
    fp32 on the same bf16 operands: one bf16 rounding of the exact sum (relative tolerance 2^-8 plus fp32 summation
    noise), and bitwise reproducible."""
    from gbx_lm_b200 import ops

    m, v, k = shape
    g = torch.Generator(device=cuda_device).manual_seed(m + v + k)
    w = (torch.randn((v, k), generator=g, device=cuda_device) / k ** 0.5).to(torch.bfloat16)
    x = torch.randn((m, k), generator=g, device=cuda_device).to(torch.bfloat16)
    n0 = ops.launch_count()
    y = ops.head_linear(x, w)
    assert ops.launch_count() == n0 + 1, "the head did not go through gbxq_head_gemv"
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ref = torch.nn.functional.linear(x.float(), w.float())
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    assert y.shape == (m, v) and y.dtype == torch.bfloat16
    err = (y.float() - ref).abs().max() / ref.abs().max()
    assert err <= 2.0 ** -8, err
    # where the fp32 reference is not within rounding of a bf16 tie the bf16 result is exactly the rounded reference
    assert (y == ref.to(torch.bfloat16)).float().mean() > 0.99
    assert torch.equal(y, ops.head_linear(x, w))
    # 3-D input, as the model passes it
    assert torch.equal(ops.head_linear(x[:, None, :], w)[:, 0], y)
    # the C entry point itself serves up to 8 rows (the Python dispatch stops at 2: shared-memory bound beyond)
    from gbx_lm_b200 import _lib

    x8 = torch.randn((8, k), generator=g, device=cuda_device).to(torch.bfloat16)
    y8 = torch.empty((8, v), dtype=torch.bfloat16, device=cuda_device)
    if 8 * k * 2 <= 100 * 1024:
        rc = _lib.get().gbxq_head_gemv(x8.data_ptr(), w.data_ptr(), y8.data_ptr(), 8, v, k, 0, torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        ref8 = torch.nn.functional.linear(x8.float(), w.float())
        assert (y8.float() - ref8).abs().max() <= 2.0 ** -8 * ref8.abs().max()
    # prefill-sized input falls back to the dense matmul (no gbxq launch)
    xl = torch.randn((9, k), generator=g, device=cuda_device).to(torch.bfloat16)
    n1 = ops.launch_count()
    yl = ops.head_linear(xl, w)
    assert ops.launch_count() == n1 and yl.shape == (9, v)
