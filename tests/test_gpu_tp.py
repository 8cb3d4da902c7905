"""2-GPU tests (one process per GPU, NCCL for plumbing) of the tensor-parallel path (SURVEY.md 8e):
  * gbxq_qmm_rowpar_allreduce: the row-parallel matmul with the all-reduce inside the kernel -- against the oracle's
    fp64 truth of the UNSHARDED layer, bitwise equal on both ranks, M = 1..4, repeated, different sizes back to back,
    and under CUDA-graph replay for more than two epoch wraps of the double-buffered staging;
  * gbxq_allreduce_oneshot: bitwise equal on both ranks and equal to the fp32 sum rounded once, different sizes back
    to back, CUDA-graph replay;
  * a TP-sharded tiny Llama (column-parallel q/k/v/gate/up, row-parallel o/down) against the unsharded model.
Skipped when fewer than two GPUs are visible."""
import os
import traceback

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _u32(t):
    return t.view(torch.int32).numpy().view(np.uint32)


def _u16(t):
    return t.view(torch.int16).numpy().view(np.uint16)


def _worker(rank, world, port, tmp, out):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
        import torch.distributed as dist

        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        from gbx_lm_b200 import QuantizedLinear, packing, tp as tpmod, utils, workloads as W
        from oracle import mlx_affine as A

        res = {}
        say = lambda *a: print(f"[tp rank {rank}]", *a, flush=True) if rank == 0 else None
        fused = tpmod.FusedRowParallel(None, dev, max_elems=4 * 4096)
        oneshot = tpmod.OneShotAllReduce(None, dev, capacity_elems=1 << 16)

        def same_on_all_ranks(t):
            g = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(g, t.contiguous())
            return all(torch.equal(g[0].view(torch.int16), gi.view(torch.int16)) for gi in g)

        # ---------------- fused row-parallel matmul + all-reduce
        worst = 0.0
        for (n, k, bits, gs) in ((512, 2048, 4, 64), (4096, 4096, 4, 64), (1024, 4096, 2, 64), (768, 4096, 8, 128)):
            L = packing.synth_layer(n, k, bits, gs, seed=n + k + bits)  # identical on both ranks
            lin = QuantizedLinear(k // world, n, bias=False, group_size=gs, bits=bits)
            for leaf in ("qweight", "scales", "zeros"):
                lin._set(leaf, tpmod.shard_tensor(f"model.layers.0.mlp.down_proj.{leaf}", L[leaf], bits, gs, rank, world).to(dev))
            lin._set("channel_scale", None)
            for m in (1, 2, 4, 3):
                x = A.synth_x(m, k, seed=m + n)
                xt = torch.from_numpy(x.view(np.int16)).view(torch.bfloat16)
                xs = xt[:, rank * (k // world):(rank + 1) * (k // world)].contiguous().to(dev)
                y = fused(lin, xs)
                assert y is not None, (n, k, bits, gs, m)
                truth = A.quantized_matmul(x, _u32(L["qweight"]), _u16(L["scales"]), _u16(L["zeros"]), gs, bits, "bf16", "f64")
                err = float(np.abs(y.float().cpu().numpy() - truth).max() / np.abs(truth).max())
                worst = max(worst, err)
                assert err <= 1e-2, (n, k, bits, gs, m, err)
                assert same_on_all_ranks(y), "fused all-reduce differs between ranks"
        res["fused_worst_rel_err"] = worst
        say("fused eager ok, worst rel err", worst)
        # graph replay: epochs advance on the device; 7 replays x 2 calls = 14 epochs (staging halves wrap 7 times)
        L = packing.synth_layer(1024, 2048, 4, 64, seed=5)
        lin = QuantizedLinear(2048 // world, 1024, bias=False, group_size=64, bits=4)
        for leaf in ("qweight", "scales", "zeros"):
            lin._set(leaf, tpmod.shard_tensor(f"model.layers.0.mlp.down_proj.{leaf}", L[leaf], 4, 64, rank, world).to(dev))
        lin._set("channel_scale", None)
        xg = torch.zeros((2, 2048 // world), dtype=torch.bfloat16, device=dev)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            fused(lin, xg)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            y1 = fused(lin, xg)
            y2 = fused(lin, xg[:1])  # a different size straight after
        for it in range(7):
            x = A.synth_x(2, 2048, seed=100 + it)
            xt = torch.from_numpy(x.view(np.int16)).view(torch.bfloat16)
            xg.copy_(xt[:, rank * (2048 // world):(rank + 1) * (2048 // world)])
            graph.replay()
            torch.cuda.synchronize()
            truth = A.quantized_matmul(x, _u32(L["qweight"]), _u16(L["scales"]), _u16(L["zeros"]), 64, 4, "bf16", "f64")
            for yy, tt in ((y1, truth), (y2, truth[:1])):
                err = float(np.abs(yy.float().cpu().numpy() - tt).max() / np.abs(tt).max())
                assert err <= 1e-2, ("replay", it, err)
                assert same_on_all_ranks(yy)
        assert not fused.timed_out()
        res["fused_graph_replays"] = 7
        say("fused graph replay ok")

        # ---------------- stand-alone one-shot all-reduce
        gen = torch.Generator(device=dev).manual_seed(17 + rank)
        for count in (4096, 8, 8192 * 4, 1024, 4096):
            t = torch.randn(count, generator=gen, device=dev).to(torch.bfloat16)
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            want = sum(p.float() for p in parts).to(torch.bfloat16)  # rank-order fp32 sum, one rounding
            got = oneshot(t.clone())
            assert torch.equal(got.view(torch.int16), want.view(torch.int16)), ("oneshot", count)
            assert same_on_all_ranks(got)
        buf = torch.zeros(4096, dtype=torch.bfloat16, device=dev)
        with torch.cuda.stream(s):
            oneshot(buf)
        torch.cuda.synchronize()
        g2 = torch.cuda.CUDAGraph()
        work = torch.zeros(4096, dtype=torch.bfloat16, device=dev)
        with torch.cuda.graph(g2):
            work.copy_(buf)
            oneshot(work)
            small = work[:512].clone()
            oneshot(small)
        for it in range(5):
            t = torch.randn(4096, generator=gen, device=dev).to(torch.bfloat16)
            buf.copy_(t)
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            want = sum(p.float() for p in parts).to(torch.bfloat16)
            g2.replay()
            torch.cuda.synchronize()
            assert torch.equal(work.view(torch.int16), want.view(torch.int16)), ("oneshot replay", it)
            want2 = (want[:512].float() * world).to(torch.bfloat16)
            assert torch.equal(small.view(torch.int16), want2.view(torch.int16)), ("oneshot replay small", it)
        res["oneshot_ok"] = True
        say("oneshot ok")

        # ---------------- TP-sharded tiny Llama against the unsharded model (same checkpoint, both loaded here)
        dims = W.MODELS["tiny-llama"]
        strat = W.STRATEGIES["bpw-4.0"](dims.layers)
        if rank == 0:
            utils.write_synthetic_checkpoint(tmp, dims, strat, seed=7, default_bits=4, default_gs=64, embed_scale=1.0)
        dist.barrier()
        full, _ = utils.load_model(tmp, device=dev)
        ctx = tpmod.TPContext(rank, world, None, oneshot, fused)
        shard, _ = utils.load_model(tmp, device=dev, tp=ctx)
        toks = torch.randint(0, dims.vocab, (2, 9), generator=torch.Generator().manual_seed(1)).to(dev)
        with torch.no_grad():
            ref = full(toks).float()
            got = shard(toks).float()
        err = float((got - ref).abs().max() / ref.abs().max())
        assert err < 3e-2, ("tp prefill", err)
        # greedy decode (M = 1: the fused row-parallel kernel inside the captured decode step)
        res["tp_prefill_rel_err"] = err
        say("tp prefill ok", err)
        try:
            tf, _ = utils.generate_tokens(full, toks[:1], max_tokens=12)
            ts, _ = utils.generate_tokens(shard, toks[:1], max_tokens=12)
            res["tp_decode_tokens_equal"] = tf == ts
            res["tp_decode_tokens"] = (tf, ts)
        except Exception as e:  # noqa: BLE001
            res["tp_decode_error"] = repr(e)
        assert same_on_all_ranks(got.to(torch.bfloat16))
        dist.barrier()
        torch.cuda.synchronize()
        if rank == 0:
            out.put(("ok", res))
    except Exception:  # noqa: BLE001
        out.put(("fail", f"rank {rank}: {traceback.format_exc()}"))
    finally:
        out.close()
        out.join_thread()  # flush the result to the pipe before leaving without interpreter teardown
        os._exit(0)  # NCCL teardown with captured graphs alive can hang (profiles/README.md r01j)


def test_tp2_fused_rowparallel_oneshot_and_model(tmp_path):
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, str(tmp_path), out), daemon=True) for r in range(2)]
    for p in procs:
        p.start()
    try:
        status, res = out.get(timeout=240)
    except Exception:  # noqa: BLE001
        status, res = "fail", "no result within 240 s (a rank hangs)"
    for p in procs:
        p.join(10)
        if p.is_alive():  # a rank stuck in a collective after its peer failed: never outlive the test
            p.kill()
    assert status == "ok", res
    print("tp2:", {k: v for k, v in res.items() if k != "tp_decode_tokens"})
    assert res["fused_worst_rel_err"] <= 1e-2
    assert res.get("tp_decode_error") is None, res.get("tp_decode_error")
    # greedy tokens of the sharded and the unsharded model: equal unless a step is a rounding tie
    tf, ts = res["tp_decode_tokens"]
    assert len(tf) == len(ts) and sum(a == b for a, b in zip(tf, ts)) >= len(tf) - 2, (tf, ts)
