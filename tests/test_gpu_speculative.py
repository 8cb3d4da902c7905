"""GPU tests of speculative decoding: the T-token cache writes are bitwise T single-token writes (and write nothing else),
the T-query attention is bitwise the single-query attention at each query's position whatever attend_len, block position
or row start, and close to fp64; the fused T-token model step against the unfused path, T single steps and its graph
replay; generation whose tokens do not depend on the draft, on the host or device driver, and agree with the fp32
reference."""
import dataclasses
import json

import pytest
import torch

from gbx_lm_b200 import ops, qllama, utils, workloads as W
from tests import ref_model
from tests.test_gpu_kv_quant import _close, _fill, _oracle_deq, _ref_attention
from tests.test_gpu_rotating_cache import KERNEL_CASES, _i32, _side

pytestmark = pytest.mark.gpu

TS = (1, 2, 3, 5, 8)


def _write(kind, q, k, v, p, inv, ks, vs, bits, gs):
    if kind == "bf16":
        return ops.rope_cache(q, k, v, p, inv, ks[0], vs[0])
    return ops.rope_cache_quantized(q, k, v, p, inv, ks, vs, gs, bits)


@pytest.mark.parametrize("kind,bits,D,gs,Hq,Hkv", KERNEL_CASES)
def test_block_cache_write_is_t_single_writes(cuda_device, kind, bits, D, gs, Hq, Hkv):
    g = torch.Generator(device=cuda_device).manual_seed(bits * 1000 + D + gs + Hq)
    inv = qllama.RoPE(D, 500000.0, False, None).to(cuda_device).inv_freq
    B, max_len = 2, 48
    for T in TS:
        # shared start, per-row starts, and blocks that end past max_len (those positions are not written)
        for starts in ([5], [0, 17], [max_len - 3, 40], [max_len - 1]):
            base_k, base_v = (_side(kind, B, Hkv, max_len, D, bits, gs, cuda_device, g) for _ in range(2))
            q = torch.randn((B, T, Hq, D), generator=g, device=cuda_device).to(torch.bfloat16)
            k = (torch.randn((B, T, Hkv, D), generator=g, device=cuda_device) * 3).to(torch.bfloat16)
            v = torch.randn((B, T, Hkv, D), generator=g, device=cuda_device).to(torch.bfloat16)
            p = torch.tensor(starts, device=cuda_device)
            mk, mv = tuple(t.clone() for t in base_k), tuple(t.clone() for t in base_v)
            mq = q.clone()
            _write(kind, mq, k, v, p, inv, mk, mv, bits, gs)
            sk, sv = tuple(t.clone() for t in base_k), tuple(t.clone() for t in base_v)
            sq = q.clone()
            for t in range(T):
                qt = sq[:, t].contiguous()
                _write(kind, qt, k[:, t].contiguous(), v[:, t].contiguous(), p + t, inv, sk, sv, bits, gs)
                sq[:, t] = qt
            assert torch.equal(mq, sq), (T, starts)
            for a, b in zip(mk + mv, sk + sv):
                assert torch.equal(_i32(a), _i32(b)), (T, starts)
            # nothing outside the block's rows, and nothing at or past max_len
            written = torch.zeros((B, max_len), dtype=torch.bool)
            for b in range(B):
                s = starts[0] if len(starts) == 1 else starts[b]
                written[b, s:min(s + T, max_len)] = True
            for a, b in zip(mk + mv, base_k + base_v):
                same = (_i32(a) == _i32(b)).all(-1).all(1).cpu()  # [B, max_len]
                assert same[~written].all(), (T, starts)


ATTN_CASES = [("bf16", 0, 128, 0, 32, 8), ("bf16", 0, 64, 0, 16, 2), ("q", 4, 128, 64, 32, 8), ("q", 8, 128, 128, 16, 2),
              ("q", 3, 64, 32, 8, 2), ("q", 2, 128, 64, 2, 2), ("q", 6, 64, 64, 16, 2)]
CONTEXTS = (1, 255, 256, 257, 4097)


def _attn(kind, q, ks, vs, p, scale, bits, gs, attend_len=None):
    if kind == "bf16":
        return ops.decode_attention(q, ks[0], vs[0], p, scale, attend_len)
    return ops.decode_attention_quantized(q, ks, vs, p, scale, gs, bits, attend_len)


@pytest.mark.parametrize("kind,bits,D,gs,Hq,Hkv", ATTN_CASES)
def test_block_attention_is_the_single_query_attention(cuda_device, kind, bits, D, gs, Hq, Hkv):
    B, max_len, scale = 2, 4200, D ** -0.5
    g = torch.Generator(device=cuda_device).manual_seed(bits * 31 + D + Hq)
    if kind == "bf16":
        kb = (torch.randn((B, Hkv, max_len, D), generator=g, device=cuda_device) * 2).to(torch.bfloat16)
        vb = torch.randn((B, Hkv, max_len, D), generator=g, device=cuda_device).to(torch.bfloat16)
        ks, vs = (kb,), (vb,)
        kd, vd = kb.double(), vb.double()
    else:
        ks, vs = _fill(B, Hkv, max_len, D, bits, gs, cuda_device, bits + D + Hq)
        kd, vd = _oracle_deq(ks, gs, bits).to(cuda_device), _oracle_deq(vs, gs, bits).to(cuda_device)
    for T in TS:
        q = torch.randn((B, T, Hq, D), generator=g, device=cuda_device).to(torch.bfloat16)
        for n in CONTEXTS:  # the keys the block's last query sees
            if n < T:
                continue
            starts = [n - T, max(n - T - 37, 0)]  # rows with different starts
            p = torch.tensor(starts, device=cuda_device)
            got = _attn(kind, q, ks, vs, p, scale, bits, gs)
            assert got.shape == q.shape
            # attend_len: the eager form (the last query's keys) and anything above give the same bits
            for attend_len in (n, min(n + 300, max_len), max_len - 1):
                assert torch.equal(_attn(kind, q, ks, vs, p, scale, bits, gs, attend_len), got), (T, n, attend_len)
            for b in range(B):
                for t in range(T):
                    pos = torch.tensor([starts[b] + t], device=cuda_device)
                    one = _attn(kind, q[b:b + 1, t].contiguous(), tuple(x[b:b + 1] for x in ks),
                                tuple(x[b:b + 1] for x in vs), pos, scale, bits, gs)
                    assert torch.equal(got[b, t], one[0]), (T, n, b, t)
            # a query at x as t = 0 of a block at x and as t = 3 of a block at x - 3
            if T >= 4 and n >= T + 3:
                x = starts[0]
                q2 = q.clone()
                q2[:, 3] = q[:, 0]
                other = _attn(kind, q2, ks, vs, torch.tensor([x - 3, starts[1]], device=cuda_device), scale, bits, gs)
                assert torch.equal(other[0, 3], got[0, 0]), (T, n)
            if T in (3, 8):
                for b in range(B):
                    for t in range(T):
                        want = _ref_attention(q[b:b + 1, t], kd[b:b + 1], vd[b:b + 1], starts[b] + t, scale)
                        _close(got[b:b + 1, t], want)


def test_block_attention_quantized_beyond_the_bf16_cap(cuda_device):
    """50 000 keys: above the 49 152 keys of the bf16 kernel."""
    B, Hq, Hkv, D, gs, bits, n, T = 1, 8, 2, 128, 64, 4, 50000, 5
    ks, vs = _fill(B, Hkv, n, D, bits, gs, cuda_device, 13)
    kd, vd = _oracle_deq(ks, gs, bits).to(cuda_device), _oracle_deq(vs, gs, bits).to(cuda_device)
    g = torch.Generator(device=cuda_device).manual_seed(9)
    q = torch.randn((B, T, Hq, D), generator=g, device=cuda_device).to(torch.bfloat16)
    p0 = n - T
    got = ops.decode_attention_quantized(q, ks, vs, torch.tensor([p0], device=cuda_device), D ** -0.5, gs, bits)
    for t in range(T):
        pos = torch.tensor([p0 + t], device=cuda_device)
        one = ops.decode_attention_quantized(q[:, t].contiguous(), ks, vs, pos, D ** -0.5, gs, bits)
        assert torch.equal(got[:, t], one)
        _close(got[:, t], _ref_attention(q[:, t], kd, vd, p0 + t, D ** -0.5))


# ------------------------------------------------------------------------------------------ the model and generation
def _model(tmp_path, name, cuda_device, seed=5, dims=None):
    dims = dims or W.MODELS[name]
    strat = W.STRATEGIES["bpw-4.0"](dims.layers) if name in ("tiny-llama", "llama-3.2-1b") else None
    cfg = utils.write_synthetic_checkpoint(tmp_path, dims, strat, seed=seed, default_bits=4, default_gs=64, embed_scale=1.0)
    model, _ = utils.load_model(tmp_path, device=cuda_device)
    return dims, cfg, model


def _varied_model(tmp_path, name, cuda_device, seed):
    """The architecture of `name` with an untied head and embeddings at 1/sqrt(hidden): on random weights its greedy
    chain keeps changing token (a tied head on large embeddings repeats one token)."""
    dims = dataclasses.replace(W.MODELS[name], tie=False)
    cfg = utils.write_synthetic_checkpoint(tmp_path, dims, W.STRATEGIES["bpw-4.0"](dims.layers), seed=seed,
                                           default_bits=4, default_gs=64, embed_scale=dims.hidden ** -0.5)
    model, _ = utils.load_model(tmp_path, device=cuda_device)
    return dims, cfg, model


def _drafts(tmp_path, dims, cuda_device):
    """(a draft right part of the time, an unrelated one): the target's checkpoint loaded again with its final norm
    weights perturbed (same layers, its argmax agrees with the target's on some steps only), and a random 2-layer model
    of the target's vocabulary with its own head."""
    partial, _ = utils.load_model(tmp_path / "target", device=cuda_device)
    w = partial.model.norm.weight
    g = torch.Generator(device=cuda_device).manual_seed(1)
    w.mul_(1 + 0.15 * torch.randn(w.shape, generator=g, device=cuda_device))
    ddims = W.ModelDims("draft", "llama", 256, 512, 2, 4, 2, 64, dims.vocab, False)
    _, _, unrelated = _model(tmp_path / "draft", "draft", cuda_device, seed=77, dims=ddims)
    return partial, unrelated


def _rounds(flags, k):
    """The accepted counts n of the rounds of a host run, from its from_draft flags."""
    out, i = [], 1
    while i < len(flags):
        n = 0
        while i + n < len(flags) and flags[i + n]:
            n += 1
        out.append(n)
        i += n + 1
    return out


def _prefilled(model, toks, kv_bits):
    cache = qllama.make_prompt_cache(model, 1, 64)
    with torch.no_grad():
        model(toks, cache)
    if kv_bits:
        cache[:] = [c.to_quantized(64, kv_bits) for c in cache]
    return cache


@pytest.mark.parametrize("kv_bits", (None, 4))
@pytest.mark.parametrize("T", (2, 3, 5, 8))
def test_fused_block_step_matches_unfused_sequential_and_graph(cuda_device, tmp_path, monkeypatch, T, kv_bits):
    dims, _, model = _model(tmp_path, "tiny-llama", cuda_device)
    toks = torch.randint(0, dims.vocab, (1, 20 + T), generator=torch.Generator().manual_seed(T)).to(cuda_device)
    P = 20
    pos = torch.arange(P, P + T, device=cuda_device)
    block = toks[:, P:]

    def block_step(fused, positions):
        monkeypatch.setattr(qllama, "FUSED_DECODE", fused)
        cache = _prefilled(model, toks[:, :P], kv_bits)
        for c in cache:
            c.offset = P + T
        with torch.no_grad():
            return model(block, cache, positions=positions, attend_len=P + T).float(), cache

    fused, cache = block_step(True, pos)
    unfused, _ = block_step(False, pos)
    per_row, _ = block_step(True, pos[None])  # [B, T] positions: the same launches at pos_stride 1
    assert torch.equal(per_row, fused)
    monkeypatch.setattr(qllama, "FUSED_DECODE", True)
    seq_cache = _prefilled(model, toks[:, :P], kv_bits)
    with torch.no_grad():
        seq = torch.cat([model(block[:, t:t + 1], seq_cache).float() for t in range(T)], 1)
    scale = unfused.abs().max()
    assert (fused - unfused).abs().max() <= 3e-2 * scale
    assert (fused - seq).abs().max() <= 3e-2 * scale
    # graph replay of the block step: bitwise the eager call
    gcache = _prefilled(model, toks[:, :P], kv_bits)
    static_pos = pos.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s), torch.no_grad():
        for _ in range(2):
            model(block, gcache, positions=static_pos)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph), torch.no_grad():
        out = model(block, gcache, positions=static_pos)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out.float(), fused)


def _reference_check(model, cfg, dims, strat_plan, prompt, toks, ckpt_dir, cuda_device, label):
    import os

    from safetensors.torch import load_file

    ckpt = {}
    for f in sorted(os.listdir(ckpt_dir)):
        if f.endswith(".safetensors"):
            ckpt.update(load_file(str(ckpt_dir / f)))
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        dense = ref_model.dense_weights_c(ckpt, lambda m: strat_plan[m], device=cuda_device)
        seq = torch.cat([prompt, torch.tensor(toks)])[None].to(cuda_device)
        with torch.no_grad():
            ref = ref_model.forward(dense, cfg, seq)[0, len(prompt) - 1:-1].float()
            ours = model(seq).float()[0, len(prompt) - 1:-1]
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    noise_t = (ours - ref).abs().max(-1).values.cpu()
    top2 = ref.topk(2, -1).values
    margin = (top2[:, 0] - top2[:, 1]).cpu()
    decisive = margin > 2.0 * noise_t
    match = ref.argmax(-1).cpu() == torch.tensor(toks)
    print(f"{label}: decisive {int(decisive.sum())}, matching {int(match.sum())} of {len(toks)}")
    assert float(noise_t.max()) <= 3e-2 * float(ref.abs().max())
    assert bool(match[decisive].all()), f"{label}: a decisive step disagrees with the fp32 reference"
    return int(match.sum())


def _plan(dims):
    strat = W.STRATEGIES["bpw-4.0"](dims.layers)
    plan = {}
    for (i, p, n, k, b, g) in W.layer_plan(dims, strat, 4, 64):
        sub = "self_attn" if p in ("q_proj", "k_proj", "v_proj", "o_proj") else "mlp"
        plan[f"model.layers.{i}.{sub}.{p}"] = (b, g)
    return plan


@pytest.mark.parametrize("name", ("tiny-llama", "llama-3.2-1b"))
def test_speculative_tokens_do_not_depend_on_the_draft(cuda_device, tmp_path, name):
    dims, cfg, model = _varied_model(tmp_path / "target", name, cuda_device, seed=20261018)
    partial, unrelated = _drafts(tmp_path, dims, cuda_device)
    prompt = torch.randint(0, dims.vocab, (16,), generator=torch.Generator().manual_seed(5))
    n = 128
    report = {}
    for kv_bits in (None, 4):
        kw = dict(kv_bits=kv_bits, kv_group_size=64, quantized_kv_start=0)
        for k in (1, 2, 4, 7):
            runs, rates = {}, {}
            for label, draft in (("self", model), ("partial", partial), ("unrelated", unrelated)):
                steps = list(utils.speculative_generate_step(prompt, model, draft, num_draft_tokens=k, max_tokens=n, **kw))
                runs["host_" + label] = [t for t, _, _ in steps]
                if label == "partial":
                    accepted = _rounds([f for _, _, f in steps], k)
                if label == "self":  # the target's top-2 margin where it rejected its own draft
                    i, tie_margins = 1, []
                    for a in _rounds([f for _, _, f in steps], k):
                        if a < k and i + a < len(steps):
                            top2 = steps[i + a][1].topk(2).values
                            tie_margins.append(float(top2[0] - top2[1]))
                        i += a + 1
                runs["device_" + label], st = utils.generate_tokens_device(model, prompt, n, draft_model=draft,
                                                                           num_draft_tokens=k, **kw)
                rates[label] = round(st["acceptance_rate"], 3)
            toks = runs["host_self"]
            assert len(toks) == n and all(r == toks for r in runs.values()), (kv_bits, k)
            # not one repeated token: the accept rule, prev, y and the advance of P all change what comes next
            assert len(set(toks)) >= 5, f"a degenerate chain: {sorted(set(toks))}"
            # the partial draft: rounds that accept none, some and (k > 1) not all of the drafts
            assert 0 in accepted and any(a > 0 for a in accepted), (kv_bits, k, accepted)
            if k > 1:
                assert any(0 < a < k for a in accepted), (kv_bits, k, accepted)
            # draft = target disagrees only where the verify (M = k + 1 rows) and the draft's steps (M = 1, 2) round a
            # near tie differently (logits of these models reach about 5); one such step ends a round and drops the
            # rest of its drafts, so at k = 7 on the 1B chain the rate falls to about 0.7
            assert all(m <= 0.25 for m in tie_margins), (kv_bits, k, tie_margins)
            assert rates["self"] >= (0.8 if k <= 4 else 0.6) and 0 < rates["partial"] < 1, (kv_bits, k, rates)
            report[f"kv{kv_bits}_k{k}"] = dict(rates, distinct=len(set(toks)),
                                                self_rejection_margin_max=round(max(tie_margins, default=0.0), 4),
                                                changes=sum(a != b for a, b in zip(toks, toks[1:])),
                                                partial_rounds_0_some_all=[sum(a == 0 for a in accepted),
                                                                           sum(0 < a < k for a in accepted),
                                                                           sum(a == k for a in accepted)])
            if kv_bits is None:
                matching = _reference_check(model, cfg, dims, _plan(dims), prompt, toks, tmp_path / "target",
                                            cuda_device, f"{name} k={k}")
                if name == "llama-3.2-1b":
                    assert matching >= 110
    print("acceptance:", json.dumps(report))


@pytest.mark.parametrize("start", (20, 23))
def test_speculative_conversion_inside_the_decode_host_equals_device(cuda_device, tmp_path, start):
    dims, _, model = _varied_model(tmp_path / "target", "tiny-llama", cuda_device, seed=11)
    partial, unrelated = _drafts(tmp_path, dims, cuda_device)
    prompt = torch.randint(0, dims.vocab, (12,), generator=torch.Generator().manual_seed(3))
    # The conversion follows the verify step that crosses quantized_kv_start, so which positions run on the bf16 cache
    # depends on where the rounds fall: the tokens may depend on the draft here, host and device must still agree.
    for d in (model, partial, unrelated):
        kw = dict(kv_bits=4, kv_group_size=64, quantized_kv_start=start, draft_model=d, num_draft_tokens=3)
        host, _ = utils.generate_tokens(model, prompt, 40, **kw)
        dev, _ = utils.generate_tokens_device(model, prompt, 40, **kw)
        assert len(host) == 40 and host == dev
        assert len(set(host)) >= 5, f"a degenerate chain: {sorted(set(host))}"
