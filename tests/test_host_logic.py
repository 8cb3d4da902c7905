"""CPU tests of host-side logic around the path: TP shard plans of the benchmark configurations, the two-stage
vocabulary argmax of the device-side sampler, and the DRAM-traffic figure bench.py reports (profiles/traffic.json) being
reproducible from the committed ncu launch list."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_shard_plans_of_the_configurations():
    """SURVEY.md 8e: column-parallel splits N, row-parallel splits K on group and word borders, for every model of
    BASELINE.json's configs at every TP degree the kv heads allow; bytes are conserved up to the replicated x / y."""
    from gbx_lm_b200 import workloads as W

    b = _bench()
    for model, strat in (("llama-3-8b", "bpw-4.0"), ("llama-3-70b", "bpw-4.0"), ("qwen2.5-32b", None), ("llama-3.2-3b", "bpw-4.0")):
        dims = W.MODELS[model]
        plan = W.layer_plan(dims, W.STRATEGIES[strat](dims.layers) if strat else None, 4, 128 if strat is None else 64)
        full_w = sum(n * k * bits // 8 + 4 * n * (k // g) for (_, _, n, k, bits, g) in plan)
        for tp in (2, 4, 8):
            sh = b.shard_plan(plan, tp)
            assert len(sh) == len(plan)
            for (i, p, n, k, bits, g), (_, _, n0, k0, _, _) in zip(sh, plan):
                if p in ("o_proj", "down_proj"):
                    assert n == n0 and k * tp == k0 and k % g == 0 and (k * bits) % 32 == 0
                else:
                    assert k == k0 and n * tp == n0
            assert sum(n * k * bits // 8 + 4 * n * (k // g) for (_, _, n, k, bits, g) in sh) * tp == full_w


def test_dump_rows_fit_the_budget_and_are_fixed():
    """bench.py --dump-outputs: every row while a step's outputs fit the budget as float32, else the same seeded rows."""
    b = _bench()
    n = 43008 * 32  # outputs of one token through the 224 forwards of a Llama-3-8B step
    assert b.dump_rows(1, n) is None
    rows = b.dump_rows(2048, n)
    assert len(rows) == b.DUMP_BUDGET_BYTES // (4 * n) and len(rows) * 4 * n <= b.DUMP_BUDGET_BYTES
    assert bool((np.diff(rows) > 0).all()) and 0 <= rows[0] and rows[-1] < 2048
    assert np.array_equal(rows, b.dump_rows(2048, n))
    with pytest.raises(SystemExit):
        b.dump_rows(1, b.DUMP_BUDGET_BYTES)


def test_fast_argmax_first_occurrence():
    from gbx_lm_b200 import utils

    g = torch.Generator().manual_seed(0)
    for v in (128256, 152064, 512, 1000, 32000, 2048):
        x = torch.randn((2, 3, v), generator=g).to(torch.bfloat16)
        x[0, 1, 7] = x[0, 1, v - 5] = x[0, 1].max() + 1
        x[1, 2, v - 1] = 100.0
        assert torch.equal(utils.fast_argmax(x), torch.argmax(x, dim=-1)), v


def test_traffic_json_reproducible_from_launch_list(tmp_path):
    csv = os.path.join(ROOT, "profiles", "r03b_launches.csv")
    want = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    out = tmp_path / "t.json"
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "traffic_from_ncu.py"), csv, "128", str(out)], check=True,
                   capture_output=True)
    got = json.load(open(out))
    assert got["launches"] == 128 and got["dram_bytes_per_launch"] == want["dram_bytes_per_launch"]
    assert sum(k["launches"] for k in got["kernels"].values()) == 128
    # no re-reads: DRAM traffic within 2 % of the algorithmic bytes of the step (bench.py config.bytes_per_step)
    assert 1.0 <= got["dram_read_bytes_step"] / 3461349376 < 1.02


def test_switch_glu_sort_and_unsort_are_inverse():
    """switch_layers.py:11-23 of the reference: (token, slot) pairs ordered by expert for the sorted gather_qmm path and
    put back afterwards; the oracle-side statement of what SwitchGLU relies on (host logic, no kernel)."""
    from gbx_lm_b200 import switch_layers as SL

    gen = torch.Generator().manual_seed(0)
    T, topk, H, E = 40, 2, 8, 5
    x = torch.randn((1, T, 1, 1, H), generator=gen)
    idx = torch.randint(0, E, (1, T, topk), generator=gen)
    xs, flat, inv = SL._gather_sort(x, idx)
    assert xs.shape == (T * topk, 1, H) and flat.shape == (T * topk,)
    assert bool((flat[1:] >= flat[:-1]).all())                       # ordered by expert
    # row j of the sorted activations is the token that owns pair order[j]
    order = torch.argsort(idx.flatten(), stable=True)
    assert torch.equal(xs, x.flatten(0, -3)[order // topk])
    # a per-pair payload survives the round trip: y[pair] = (token, expert)
    y = torch.stack([(order // topk).float(), flat.float()], -1)
    back = SL._scatter_unsort(y, inv, idx.shape)
    want = torch.stack([torch.arange(T).repeat_interleave(topk).float().reshape(1, T, topk), idx.float()], -1)
    assert torch.equal(back, want)
