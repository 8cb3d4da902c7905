#!/usr/bin/env python
"""bench.py -- headline benchmark of the gbx-lm quantized-matmul hot path on B200.

Metric (BASELINE.json): "4-bit qmatmul HBM GB/s (M=1) & decode tok/s, Llama-3-8B, 1-8 B200".

One STEP = one decode token through the quantized-matmul path of the workload: the 7*L
`QuantizedLinear` forwards (q,k,v,o,gate,up,down of every block) at M = batch rows, on synthetic
layer-mix weights (SURVEY.md 8d).  `value` = ALGORITHMIC bytes of a step (packed weights + scales +
biases + x + y, BASELINE.md section 3) / device time of a step, inputs resident in HBM, the step
replayed from a CUDA graph.  The body of Llama-3-8B (3.4 GB) is 27x the 126 MB L2, so every step
streams its weights from HBM (L2 defeated by input size).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl gbxq|reference]
                    [--model llama-3-8b] [--strategy bpw-4.0] [--batch 1] [--dump-outputs DIR]

Every timed loop runs exactly K steps.  --dump-outputs DIR writes what the last timed step computed, one
`DIR/layer<i>_<proj>.npy` (float32, [rows, N]) per QuantizedLinear forward; inputs are seeded, so two builds run with the
same arguments can be compared output for output.  When all rows would exceed 64 MB, a fixed seeded sample of the rows
(the same for every layer) is written.

N > 1 (launched by torch.distributed.run): tensor-parallel shards of the same model (strong scaling):
column-parallel q/k/v/gate/up, row-parallel o/down followed by a sum all-reduce (SURVEY.md 8e).
`--impl reference` times the CPU restatement of the reference path (oracle/, OpenMP over all host
cores; MLX itself is not installable here -- DESIGN.md) on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "qmatmul_hbm_gbs_m1"
UNIT = "GB/s"
DUMP_BUDGET_BYTES = 64 << 20


def dump_rows(m_rows: int, row_elems: int, budget_bytes: int = DUMP_BUDGET_BYTES):
    """Rows of the outputs --dump-outputs writes: None (all rows) when the whole step fits the budget as float32, else a
    sorted seeded sample of rows, the same for every layer."""
    import numpy as np

    keep = budget_bytes // (4 * row_elems)
    if keep < 1:
        raise SystemExit(f"--dump-outputs: one row of every output ({4 * row_elems} bytes) exceeds {budget_bytes} bytes")
    if keep >= m_rows:
        return None
    return np.sort(np.random.default_rng(0).choice(m_rows, keep, replace=False))


def load_tensor_peak():
    """Sustained dense bf16 peak (the GEMM is timed inside a long step), MEASURED_PEAKS.json else the profiling guide's fallback."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
        except Exception:
            pass
    return 1400.0, "fallback (B200_PROFILING.md)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle-reason sampler running during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def build_plan(args):
    from gbx_lm_b200 import workloads as W

    dims = W.MODELS[args.model]
    strat = None if args.strategy == "uniform" else W.STRATEGIES[args.strategy](dims.layers)
    plan = W.layer_plan(dims, strat, args.bits, args.group_size)
    return dims, plan


def shard_plan(plan, tp: int):
    """TP shard shapes: column-parallel splits N, row-parallel (o_proj, down_proj) splits K."""
    out = []
    for (i, p, n, k, b, g) in plan:
        if p in ("o_proj", "down_proj"):
            assert k % tp == 0 and (k // tp) % g == 0 and ((k // tp) * b) % 32 == 0
            out.append((i, p, n, k // tp, b, g))
        else:
            assert n % tp == 0
            out.append((i, p, n // tp, k, b, g))
    return out


# ------------------------------------------------------------------------------------------ GPU arm
def run_gbxq(args):
    import torch
    import torch.distributed as dist

    from gbx_lm_b200 import QuantizedLinear, ops
    from gbx_lm_b200 import workloads as W

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # row-parallel layers under TP (--allreduce): "fused" = the all-reduce inside the matmul kernel
    # (gbxq_qmm_rowpar_allreduce: P2P pushes of fp32 partials over NVLink, per-CTA flags, rank-order sum);
    # "oneshot" = matmul, then the stand-alone peer-memory all-reduce kernel; "nccl" = matmul, then ncclAllReduce.
    # Every choice is self-checked against NCCL before it is trusted; what actually ran is recorded in the line.
    from gbx_lm_b200 import workloads as _W
    from gbx_lm_b200.tp import TPContext

    dims_hidden = _W.MODELS[args.model].hidden
    tpctx, ar_kind = TPContext(), "none"
    if world > 1:
        ar_kind, oneshot, fused = "nccl", None, None
        if args.allreduce in ("oneshot", "fused"):
            try:
                from gbx_lm_b200.tp import OneShotAllReduce

                oneshot = OneShotAllReduce(None, dev, capacity_elems=max(1 << 16, 4 * args.batch * 8192))
                for i in range(3):  # both staging halves and a wrap
                    t = torch.randn(args.batch * dims_hidden, generator=torch.Generator(device=dev).manual_seed(7 * rank + i), device=dev).to(torch.bfloat16)
                    want = t.float()
                    dist.all_reduce(want)
                    got = oneshot(t.clone()).float()
                    if not torch.allclose(got, want, rtol=2e-2, atol=2e-2):
                        raise RuntimeError("one-shot all-reduce self-check failed")
                ar_kind = "gbxq_allreduce_oneshot (peer memory over NVLink, separate PDL launch)"
            except Exception as e:  # noqa: BLE001
                oneshot = None
                ar_kind = f"nccl (one-shot unavailable: {type(e).__name__}: {str(e)[:80]})"
        if args.allreduce == "fused":
            try:
                from gbx_lm_b200.tp import FusedRowParallel

                fused = FusedRowParallel(None, dev, max_elems=max(4 * 8192, args.batch * dims_hidden))
                # self-check: a K-sharded layer through the fused kernel against matmul + NCCL sum of the same shards
                gchk = torch.Generator(device=dev).manual_seed(99 + rank)
                lin = QuantizedLinear(1024, dims_hidden, bias=False, group_size=64, bits=4)
                lin._set("qweight", torch.randint(-(2 ** 31), 2 ** 31 - 1, (dims_hidden, 128), generator=gchk, device=dev, dtype=torch.int64).to(torch.int32).view(torch.uint32))
                lin._set("scales", ((torch.rand((dims_hidden, 16), generator=gchk, device=dev) + 0.5) * 0.004).to(torch.bfloat16))
                lin._set("zeros", (-lin.scales.float() * 7.5).to(torch.bfloat16))
                lin._set("channel_scale", None)
                for i in range(3):
                    xx = torch.randn((min(args.batch, 4), 1024), generator=gchk, device=dev).to(torch.bfloat16)
                    want = lin(xx).float()
                    dist.all_reduce(want)
                    got = fused(lin, xx)
                    if got is None:
                        raise RuntimeError("fused row-parallel kernel does not serve this batch")
                    if not torch.allclose(got.float(), want, rtol=3e-2, atol=3e-2):
                        raise RuntimeError("fused row-parallel self-check failed")
                    chk = got.float().clone()
                    dist.all_reduce(chk, op=dist.ReduceOp.MAX)
                    if not torch.equal(chk, got.float()):
                        raise RuntimeError("fused row-parallel result differs between ranks")
                ar_kind = "fused into the row-parallel matmul kernel (gbxq_qmm_rowpar_allreduce: P2P fp32 pushes over NVLink, per-CTA flags)"
            except Exception as e:  # noqa: BLE001
                fused = None
                ar_kind += f" [fused unavailable: {type(e).__name__}: {str(e)[:80]}]"
        tpctx = TPContext(rank, world, None, oneshot, fused)

    ops.set_pdl_mode(args.pdl)
    dims, full_plan = build_plan(args)
    prefill = args.phase == "prefill"
    M = args.prefill_tokens if prefill else args.batch
    # --parallelism: how N > 1 GPUs are used.  tp = tensor-parallel shards of ONE model instance (column-parallel
    # q/k/v/gate/up, row-parallel o/down + sum all-reduce; strong scaling) -- what the 32B / 70B configurations need;
    # dp = one full model replica per GPU, independent decode streams, no data-path collective (weak scaling) -- the
    # deployment of a model that fits one GPU.  auto = tp (the headline at N > 1); the other mode is measured as well
    # and reported under "also".
    mode = args.parallelism
    if mode == "auto":
        mode = "tp"  # north_star: N > 1 = tensor-parallel shards of ONE model with an all-reduce after o_proj / down_proj
    if world == 1:
        mode = "single"

    def measure(tp: int, m_rows=None, dump=False):
        Mr = M if m_rows is None else m_rows  # rows of x of this measurement
        plan = shard_plan(full_plan, tp) if tp > 1 else full_plan

        # ---- synthetic weights created directly in HBM (seeded); SURVEY.md 8d recipe
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        layers = []
        for (i, p, n, k, b, g) in plan:
            m = QuantizedLinear(k, n, bias=False, group_size=g, bits=b)
            nb = (1 << b) - 1
            qw = torch.randint(-(2 ** 31), 2 ** 31 - 1, (n, k * b // 32), generator=gen, device=dev, dtype=torch.int64).to(torch.int32).view(torch.uint32)
            s = ((torch.rand((n, k // g), generator=gen, device=dev) + 0.5) * (2.0 / (k ** 0.5) / nb)).to(torch.bfloat16)
            eps = torch.rand((n, k // g), generator=gen, device=dev) * 0.1 - 0.05
            z = (-s.float() * (nb / 2.0) * (1.0 + eps)).to(torch.bfloat16)
            m._set("qweight", qw)
            m._set("scales", s)
            m._set("zeros", z)
            m._set("channel_scale", None)
            layers.append((p, m))
        xbuf = {}
        for (_, _, n, k, _, _) in plan:
            if k not in xbuf:
                xbuf[k] = torch.randn((Mr, k), generator=gen, device=dev).to(torch.bfloat16)
        h_in = torch.randn((Mr, dims.hidden)).to(torch.bfloat16).pin_memory()
        h_out = torch.empty((Mr, dims.hidden), dtype=torch.bfloat16).pin_memory()
        x_hidden = xbuf[dims.hidden]

        outs = [None]

        # the callers' launch structure (gbx_lm/models/qllama.py:76,115): q|k|v and gate|up read the same activations
        # and go out as ONE grouped call each, o_proj and down_proj as single calls -> 4 library calls per block
        calls, i = [], 0
        while i < len(layers):
            names = [p for p, _ in layers[i:i + 3]]
            if args.grouped and names == ["q_proj", "k_proj", "v_proj"]:
                calls.append(("qkv", [m for _, m in layers[i:i + 3]])); i += 3
            elif args.grouped and names[:2] == ["gate_proj", "up_proj"]:
                calls.append(("gate_up", [m for _, m in layers[i:i + 2]])); i += 2
            else:
                calls.append((layers[i][0], [layers[i][1]])); i += 1

        # --stream 1: the calls of a step as a chain executed by ONE persistent launch (gbxq_qmm_stream), every call
        # ordered after the one before it (dep = previous: exactly the semantics of the launch-per-call step below).
        # Under TP the chain is cut at each all-reduce (after o_proj / down_proj).
        chains, stream_ys = [], []
        if args.stream:
            cur = ops.StreamChain(Mr)
            for p, ms in calls:
                ys = cur.add(xbuf[ms[0].input_dims], ms)
                stream_ys += ys
                if tp > 1 and p in ("o_proj", "down_proj"):
                    chains.append((cur.finalize(), ys[0]))
                    cur = ops.StreamChain(Mr)
            if len(cur):
                chains.append((cur.finalize(), None))

        # a step's result: the output of every forward, in plan order (all kept alive, so that --dump-outputs can read
        # every one of them after the last timed step)
        def step():
            if args.stream:
                for ch, ar in chains:
                    ch.run()
                    if ar is not None:
                        tpctx.all_reduce(ar)
                outs[0] = stream_ys
                return
            ys = []
            for p, ms in calls:
                if len(ms) == 1:
                    if tp > 1 and p in ("o_proj", "down_proj"):
                        ys.append(tpctx.row_parallel(ms[0], xbuf[ms[0].input_dims]))
                    else:
                        ys.append(ms[0](xbuf[ms[0].input_dims]))
                else:
                    ys += ops.quantized_matmul_grouped(xbuf[ms[0].input_dims], ms)
            outs[0] = ys

        # ---- warm-up eagerly (also sets kernel attributes), then capture one step into a CUDA graph
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            step()
            step()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        n0 = ops.launch_count()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            step()
        launches_per_step = ops.launch_count() - n0
        assert len(outs[0]) == len(plan)
        y_last = outs[0][-1]

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        for _ in range(max(args.warmup, 3)):
            graph.replay()
        barrier()

        # ---- timed region: EXACTLY K steps, CUDA events on the launching stream, max over ranks
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
            time.sleep(0.25)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            graph.replay()
        e1.record()
        barrier()
        ms_total = e0.elapsed_time(e1)
        clocks = sampler.stop() if rank == 0 else None
        if world > 1:
            t = torch.tensor([ms_total], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_total = float(t.item())
        ms_step = ms_total / args.steps
        if args.stream and any(ch.timed_out() for ch, _ in chains):
            raise SystemExit("gbxq_qmm_stream: a CTA gave up waiting (grid not co-resident); the measurement is void")

        # the outputs of the last timed step, copied to the host before the e2e steps below overwrite x_hidden
        dumped = None
        if dump:
            rows = dump_rows(Mr, sum(y.shape[-1] for y in outs[0]))
            sel = None if rows is None else torch.from_numpy(rows).to(dev)
            dumped = {f"layer{i:02d}_{p}": (y if sel is None else y.index_select(0, sel)).float().cpu().numpy()
                      for (i, p, *_), y in zip(plan, outs[0])}

        # ---- e2e: the same step through the public API with HOST buffers (pinned), copies inside the timed region
        def e2e_step():
            x_hidden.copy_(h_in, non_blocking=True)
            graph.replay()
            h_out.copy_(y_last if y_last.shape == h_out.shape else y_last[:, : dims.hidden], non_blocking=True)
            torch.cuda.current_stream().synchronize()

        for _ in range(3):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            e2e_step()
        f1.record()
        barrier()
        e2e_wall = (time.perf_counter() - t0) * 1e3 / args.steps
        e2e_ms = max(f0.elapsed_time(f1) / args.steps, e2e_wall)  # host-visible time per step (>= device time)
        if world > 1:
            t = torch.tensor([e2e_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_ms = float(t.item())

        return {"ms_step": ms_step, "e2e_ms": e2e_ms, "e2e_wall": e2e_wall, "launches_per_step": launches_per_step,
                "calls": len(calls), "plan": plan, "layers": layers, "clocks": clocks, "chains": chains,
                "h2d": int(h_in.numel() * 2), "d2h": int(h_out.numel() * 2), "outputs": dumped}

    r = measure(world if mode == "tp" else 1, dump=args.dump_outputs is not None and rank == 0)
    dumped = r["outputs"]
    ms_step, e2e_ms, e2e_wall, launches_per_step, plan, layers, clocks, chains = (
        r["ms_step"], r["e2e_ms"], r["e2e_wall"], r["launches_per_step"], r["plan"], r["layers"], r["clocks"], r["chains"])
    ncalls, r_h2d, r_d2h = r["calls"], r["h2d"], r["d2h"]
    replicas = world if mode == "dp" else 1
    also = None
    if world > 1 and not args.no_also:
        del r
        r2 = measure(1 if mode == "tp" else world)
        other = "dp" if mode == "tp" else "tp"
        rep2 = world if other == "dp" else 1
        b2 = sum(W.qmm_bytes(M, n, k, b, g) for (_, _, n, k, b, g) in full_plan) * rep2
        also = {"parallelism": f"{other}{world}", "scaling": "weak" if other == "dp" else "strong",
                "allreduce": ar_kind if other == "tp" else "none (independent replicas)",
                "value": round(b2 / (r2["ms_step"] * 1e-3) / 1e9, 2), "unit": UNIT, "ms_per_step": round(r2["ms_step"], 5),
                "decode_tok_s_qmm_only": round(1e3 / r2["ms_step"] * M * rep2, 2)}
        del r2

    # N = 1, default decode run: the other two regimes of the same model, measured the same way in the same process
    # (CUDA graph, CUDA events, inputs resident, --steps timed steps), so that one result line carries them: a decode
    # batch of 16 rows (HBM roofline) and a prefill chunk of 2048 tokens (tensor roofline, TFLOP/s against the sustained
    # bf16 peak).
    if world == 1 and not prefill and not args.stream and args.batch == 1 and not args.no_also:
        del r
        also = {}
        rb = measure(1, 16)
        bb = sum(W.qmm_bytes(16, n, k, b, g) for (_, _, n, k, b, g) in full_plan)
        also["decode_batch_16"] = {"value": round(bb / (rb["ms_step"] * 1e-3) / 1e9, 2), "unit": UNIT, "ms_per_step": round(rb["ms_step"], 5),
                                   "decode_tok_s_qmm_only": round(16e3 / rb["ms_step"], 1), "launches_per_step": rb["launches_per_step"],
                                   "frac_of_hbm_peak": round(bb / (rb["ms_step"] * 1e-3) / 1e9 / load_peaks()[0], 4)}
        del rb
        rp = measure(1, 2048)
        fl = sum(2.0 * 2048 * n * k for (_, _, n, k, _, _) in full_plan)
        tpk, tsrc = load_tensor_peak()
        also["prefill_2048"] = {"value": round(fl / (rp["ms_step"] * 1e-3) / 1e12, 2), "unit": "TFLOP/s", "ms_per_step": round(rp["ms_step"], 4),
                                "prefill_tok_s_qmm_only": round(2048e3 / rp["ms_step"], 1), "launches_per_step": rp["launches_per_step"],
                                "frac_of_tensor_peak": round(fl / (rp["ms_step"] * 1e-3) / 1e12 / tpk, 4), "peak": tpk, "peak_source": tsrc,
                                "kernel": "gbxq::gemm_ts_kernel (tcgen05.mma, weights as the TMEM operand)"}
        del rp

    bytes_step = sum(W.qmm_bytes(M, n, k, b, g) for (_, _, n, k, b, g) in full_plan) * replicas
    value = bytes_step / (ms_step * 1e-3) / 1e9
    peak, peak_src = load_peaks()
    # roofline of the dominant kernel (the streaming GEMV: every launch of the timed region is one):
    # per-launch algorithmic bytes / per-launch average duration == per-rank bytes / step time
    rank_bytes = sum(W.qmm_bytes(M, n, k, b, g) for (_, _, n, k, b, g) in plan)
    achieved = rank_bytes / (ms_step * 1e-3) / 1e9
    # DRAM traffic per launch comes from an ncu capture of the SAME command (tools/traffic_from_ncu.py writes
    # profiles/traffic.json with the workload it was taken on); it is reported only when this run is that workload
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            same = (tj.get("model", "llama-3-8b") == args.model and tj.get("strategy", "bpw-4.0") == args.strategy and
                    int(tj.get("batch", 1)) == args.batch and world == 1 and not prefill and not args.stream)
            if same:
                traffic = tj.get("dram_bytes_per_launch")
                traffic_src = tj.get("source")
        except Exception:
            traffic = None

    def finish():
        # NCCL teardown with a captured graph alive was seen to hang on the box (profiles/README.md, r01j): make sure
        # every rank is done, then leave without destroy_process_group
        if world > 1:
            sys.stdout.flush()
            dist.barrier()
            torch.cuda.synchronize()
            os._exit(0)

    if rank != 0:
        finish()
        return
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 5), "higher_is_better": True,
        "scaling": "strong" if mode == "tp" else "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {
            "workload": f"{args.model} layer-mix {args.strategy} decode batch {M}: {len(full_plan)} QuantizedLinear "
                        f"forwards/step (stored bpw {W.stored_bpw(full_plan):.3f})",
            "bytes_per_step": bytes_step, "l2": "inputs larger than L2 (weights per step >> 126 MB)",
            "parallelism": f"{mode}{world}" if world > 1 else "single", "launch": "cuda_graph",
            "allreduce": ar_kind if mode == "tp" else "none (independent replicas)" if world > 1 else "none",
            "calls_per_step": ncalls, "grouped_qkv_gate_up": bool(args.grouped),
            "chain_launch": ({"launches_per_step": len(chains), **chains[0][0].info} if args.stream else None),
        },
        "decode_tok_s_qmm_only": round(1e3 / ms_step * M * replicas, 2),
        "roofline": {"bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "kernel": ("gbxq::stream_kernel (persistent chain launch: the mmv8 body over every call of the step)"
                                if args.stream else "gbxq::mmv8_kernel / mmv8_grouped_kernel (all launches of the step)"),
                     "bytes_per_launch_avg": rank_bytes // max(launches_per_step, 1),
                     "avg_launch_us": round(ms_step * 1e3 / max(launches_per_step, 1), 3)},
        "e2e": {"value": round(bytes_step / (e2e_ms * 1e-3) / 1e9, 2), "unit": UNIT,
                "h2d_bytes_per_step": r_h2d * replicas, "d2h_bytes_per_step": r_d2h * replicas,
                "ms_per_step": round(e2e_ms, 5), "wall_ms_per_step": round(e2e_wall, 5)},
        "gpu_launches": int(launches_per_step * args.steps),
        "also": also,
        "clocks": clocks,
    }
    if prefill:
        # prefill leg: the same 7*L forwards at M = prefill chunk (gbx_lm/utils.py:312-319: 2048-token chunks), a dense
        # contraction on the tcgen05 kernel: TFLOP/s (2*M*N*K per forward; dequant ALU work not counted) against the
        # measured sustained bf16 peak
        flops = sum(2.0 * M * n * k for (_, _, n, k, _, _) in full_plan) * replicas
        rank_flops = sum(2.0 * M * n * k for (_, _, n, k, _, _) in plan)
        tpeak, tsrc = load_tensor_peak()
        tf = flops / (ms_step * 1e-3) / 1e12
        line.update({"metric": "qmatmul_prefill_tflops", "value": round(tf, 2), "unit": "TFLOP/s"})
        line["config"]["workload"] = (f"{args.model} layer-mix {args.strategy} prefill chunk of {M} tokens: {len(full_plan)} "
                                      f"QuantizedLinear forwards/step (stored bpw {W.stored_bpw(full_plan):.3f})")
        line["config"]["flops_per_step"] = flops
        line["config"]["l2"] = "weights + activations per step >> 126 MB L2"
        line.pop("decode_tok_s_qmm_only", None)
        line["prefill_tok_s_qmm_only"] = round(M * replicas / (ms_step * 1e-3), 1)
        ach = rank_flops / (ms_step * 1e-3) / 1e12
        line["roofline"] = {"bound": "tensor", "achieved": round(ach, 2), "peak": tpeak, "unit": "TFLOP/s", "frac": round(ach / tpeak, 4),
                            "traffic": None, "peak_source": tsrc, "kernel": "gbxq::gemm_ts_kernel (tcgen05.mma swap-AB, dequantised weights as the TMEM operand)",
                            "flops_per_launch_avg": rank_flops / max(launches_per_step, 1),
                            "avg_launch_us": round(ms_step * 1e3 / max(launches_per_step, 1), 3)}
        line["e2e"]["value"] = round(flops / (e2e_ms * 1e-3) / 1e12, 2)
        line["e2e"]["unit"] = "TFLOP/s"
    if world == 1 and not args.no_cpu_baseline and not prefill:
        line["cpu_baseline"] = cpu_sample(args, layers_for_cpu=[(p, m) for (p, m) in layers[:7]], M=M, budget_s=args.cpu_seconds)
    if dumped is not None:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line), flush=True)
    finish()


# ------------------------------------------------------------------------------------------ CPU arm
_CPU_BLOCK0: dict = {}


def cpu_sample(args, layers_for_cpu=None, M=1, budget_s=12.0):
    """Times the CPU restatement of the reference path (oracle/gbxq_oracle.c, OpenMP) on a bounded
    sample: the 7 projections of block 0 of the workload, repeated until ~budget_s seconds."""
    import numpy as np

    from gbx_lm_b200 import workloads as W
    from oracle import c_oracle as C
    from oracle import mlx_affine as A

    dims, plan = build_plan(args)
    block0 = [e for e in plan if e[0] == 0]
    data = []
    if layers_for_cpu is not None:
        import torch

        for (p, m) in layers_for_cpu:
            data.append((m.qweight.cpu().view(torch.int32).numpy().view(np.uint32),
                         m.scales.cpu().view(torch.int16).numpy().view(np.uint16),
                         m.zeros.cpu().view(torch.int16).numpy().view(np.uint16), m.bits, m.group_size))
    else:
        key = (args.model, args.strategy, args.bits, args.group_size)
        if key not in _CPU_BLOCK0:  # generated once per process: the reference arm samples the same block every step
            _CPU_BLOCK0[key] = []
            for (i, p, n, k, b, g) in block0:
                L = A.synth_layer(n, k, b, g, seed=i * 7 + len(_CPU_BLOCK0[key]))
                _CPU_BLOCK0[key].append((L["qweight"], L["scales"], L["zeros"], b, g))
        data = _CPU_BLOCK0[key]
    xs = {k: A.synth_x(M, k, seed=3) for k in {d[0].shape[1] * 32 // d[3] for d in data}}
    threads = max(C.max_threads(), int(os.environ.get("GBXQ_CPU_THREADS", "0")))  # explicit omp_set_num_threads in the C call
    nbytes = sum(W.qmm_bytes(M, d[0].shape[0], d[0].shape[1] * 32 // d[3], d[3], d[4]) for d in data)

    def one_pass():
        for (qw, s, z, b, g) in data:
            C.qmm_fast(xs[qw.shape[1] * 32 // b], qw, s, z, g, b, nthreads=threads)

    one_pass()  # warm
    passes, t0 = 0, time.perf_counter()
    while True:
        one_pass()
        passes += 1
        el = time.perf_counter() - t0
        if el >= budget_s or passes >= 5000:
            break
    per = el / passes
    return {"value": round(nbytes / per / 1e9, 3), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"block 0 of {args.model} {args.strategy} (7 projections, M={M}), {passes} passes in {el:.1f} s, "
                      f"C/OpenMP restatement of MLX's CPU quantized_matmul (oracle/gbxq_oracle.c)",
            "ms_per_sample": round(per * 1e3, 3)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torch.distributed.run exports OMP_NUM_THREADS=1 to every rank; only rank 0 works here, on all host cores
    os.environ["GBXQ_CPU_THREADS"] = str(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    from gbx_lm_b200 import workloads as W

    dims, plan = build_plan(args)
    per_step_budget = max(1.0, min(8.0, 120.0 / max(args.steps + args.warmup, 1)))
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_sample(args, None, args.batch, budget_s=per_step_budget)
        if i >= args.warmup:
            vals.append(r)
    v = round(statistics.median([r["value"] for r in vals]), 3)
    ms = statistics.median([r["ms_per_sample"] for r in vals])
    bytes_step = sum(W.qmm_bytes(args.batch, n, k, b, g) for (_, _, n, k, b, g) in plan)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(bytes_step / (v * 1e9) * 1e3, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.model} layer-mix {args.strategy} decode batch {args.batch} (CPU: block-0 sample per step)",
                   "bytes_per_step": bytes_step, "parallelism": "host threads"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": vals[-1]["cores"], "kind": "port", "sample": vals[-1]["sample"]},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "MLX (the reference's numerical backend) is not installable offline; this is the C/OpenMP restatement of its "
                "CPU quantized_matmul, ms_per_step extrapolated from the sampled block to the whole step",
        "ms_per_sample": ms,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="gbxq", choices=["gbxq", "reference"])
    ap.add_argument("--model", default="llama-3-8b")
    ap.add_argument("--strategy", default="bpw-4.0", choices=["bpw-4.0", "bpw-2.2", "uniform"])
    ap.add_argument("--bits", type=int, default=4)
    ap.add_argument("--group-size", type=int, default=64)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--phase", default="decode", choices=["decode", "prefill"], help="prefill: the forwards at M = --prefill-tokens, reported in TFLOP/s against the tensor roofline")
    ap.add_argument("--prefill-tokens", type=int, default=2048)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--grouped", type=int, default=1, help="1: q|k|v and gate|up as one gbxq_qmm_grouped call each (as the model does)")
    ap.add_argument("--stream", type=int, default=0, help="1: the step's calls as one persistent chain launch (gbxq_qmm_stream); 0: one launch per call")
    ap.add_argument("--parallelism", default="auto", choices=["auto", "tp", "dp"], help="N > 1: tensor-parallel shards or independent replicas")
    ap.add_argument("--no-also", action="store_true", help="N > 1: skip the measurement of the other parallelism mode")
    ap.add_argument("--allreduce", default="fused", choices=["fused", "oneshot", "nccl"], help="row-parallel layers under TP: all-reduce fused into the matmul kernel, stand-alone peer-memory kernel, or NCCL")
    ap.add_argument("--pdl", type=int, default=2, help="GBXQ_OPT_PDL (0 plain launches, 1 PDL, 2 PDL + early weight streaming)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs is not None and args.impl != "gbxq":
        ap.error("--dump-outputs applies to --impl gbxq")
    sys.dont_write_bytecode = True  # the benchmark may run from a read-only tree and writes nothing into it
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gbxq(args)


if __name__ == "__main__":
    main()
