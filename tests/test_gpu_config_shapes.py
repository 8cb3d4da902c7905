"""Decode-sized quantized matmuls at the shapes the model configs reach, against the fp64 oracle.

The decode kernels branch on shape far more than a few hand-picked cases can cover: `mmv8` is instantiated per (bits,
group size, token tile, chunk columns per warp, rows per stage, half-full last column), `make_plan` picks the
instantiation and the row split from K / group_size, the packed row width and N, and `select` picks the kernel by M,
width and alignment.  The cases here are derived from `workloads.MODELS` x `workloads.STRATEGIES` x the
tensor-parallel degrees, so every branch a config reaches is run:

* every (bits, group size, K) of the configs at N = 260 and M = 1..16, with auto dispatch and every kernel that
  accepts the call, each against the fp64 truth;
* layers of real size (generated on the device), where the per-CTA row loop, the row tail and the ring refills run;
* the q|k|v and gate|up groups of layers 0 and 1 through `quantized_matmul_grouped`.
"""
import math
import zlib
from collections import defaultdict

import numpy as np
import pytest
import torch

from gbx_lm_b200 import workloads as W
from oracle import mlx_affine as A
from tests.gpu_util import assert_close_to_truth, bf16_from_bits, bits_from_bf16, layer_to_cuda

TPS = (1, 2, 4, 8)
ROW_PARALLEL = ("o_proj", "down_proj")  # split K under tensor parallelism; the other projections split N
GROUPS = (("q_proj", "k_proj", "v_proj"), ("gate_proj", "up_proj"))  # the projections the callers issue as one call
KERNELS = ("mmv8", "mmv", "skinny", "gemv", "gemm_ts", "gemm")
# bar against the fp64 truth, as in test_gpu_parity: 2^-7 of max |y| for the kernels that apply the affine map exactly;
# the path's 1e-2 for the tensor-core GEMMs, which round each weight s*q+z once to bf16 (with a bias add rounded on
# top, b6g64K4096 at M = 2 lands 2 bf16 ulps = 7.97e-3 of max |y| from the truth, exactly what that rounding predicts)
TOL = {"gemm": 1e-2, "gemm_ts": 1e-2}
DECODE_M = (1, 2, 3, 4, 8, 16)  # every branch of select at decode sizes: mmv8 / mmv, skinny or mmv8, gemm_ts
BIAS_M = 2
N_SMALL = 260  # a multiple of 4 (the 4-row unit refuses others), but of no row tile and not of 148
SAMPLED_ROWS = 64


def config_shards():
    """(model, strategy, tp, layer, projection, N, K, bits, group size) of every projection shard of the configs:
    column-parallel projections keep K and split N, row-parallel ones split K where the shard is legal (DESIGN §6)."""
    for name, dims in W.MODELS.items():
        if name.startswith("tiny-"):
            continue
        for sname, strategy in W.STRATEGIES.items():
            for layer, proj, N, K, bits, gs in W.layer_plan(dims, strategy(dims.layers)):
                for tp in TPS:
                    if proj in ROW_PARALLEL:
                        k = K // tp
                        if K % tp or k % gs or k * bits % 32:
                            continue
                        yield name, sname, tp, layer, proj, N, k, bits, gs
                    else:
                        yield name, sname, tp, layer, proj, N // tp, K, bits, gs


def config_triples():
    return sorted({(bits, gs, K) for *_, K, bits, gs in config_shards()})


def real_layer_shapes():
    """(N, K, bits, gs): every shard with K >= 8192, and the largest shard of every other (bits, gs, K) -- together
    they put every decode geometry the configs reach under a layer as tall as the configs' own."""
    shapes = {(N, K, bits, gs) for *_, N, K, bits, gs in config_shards()}
    largest = {}
    for N, K, bits, gs in shapes:
        if K < 8192 and N > largest.get((bits, gs, K), 0):
            largest[(bits, gs, K)] = N
    return sorted({s for s in shapes if s[1] >= 8192} | {(N, K, b, g) for (b, g, K), N in largest.items()})


def grouped_calls():
    """The distinct q|k|v and gate|up calls of layers 0 and 1 (model x strategy x tp): tuples of
    (N, K, bits, gs, with_bias) segments.  Layer 0 of bpw-2.2 mixes group sizes in q|k|v; bpw-4.0 mixes 2- and 4-bit
    in gate|up and swaps them between layers 0 and 1; Qwen2 carries q/k/v biases."""
    layers = defaultdict(dict)
    for name, sname, tp, layer, proj, N, K, bits, gs in config_shards():
        if layer < 2:
            layers[(name, sname, tp, layer)][proj] = (N, K, bits, gs, W.MODELS[name].qkv_bias and proj in GROUPS[0])
    return sorted({tuple(projs[p] for p in group) for projs in layers.values() for group in GROUPS})


def _triple_id(t):
    return "b{}g{}K{}".format(*t)


def _shape_id(s):
    return "N{}K{}b{}g{}".format(*s)


def _group_id(segs):
    return "K{}-".format(segs[0][1]) + "|".join(f"{n}b{b}g{g}" + ("+bias" if bias else "") for n, _, b, g, bias in segs)


# ---------------------------------------------------------------------------------- the enumeration itself (CPU)
def test_config_enumeration_reaches_the_long_rows_and_shards():
    """A change to workloads must not silently shrink the sweep: the 70B down_proj row of 2-bit codes, the 8B 3-bit
    down_proj, the Qwen2.5-32B tp4 down_proj shard (K/gs = 4 mod 8) and the 3B 6-bit v_proj stay in it."""
    triples = config_triples()
    for t in ((2, 128, 28672), (3, 64, 14336), (4, 64, 6912), (6, 64, 3072)):
        assert t in triples, t
    assert len(triples) >= 79
    assert max(K for _, _, K in triples) == 28672
    # every triple is checked at the size of a real layer too, and every grouped call has its segments on one K
    assert {(b, g, K) for _, K, b, g in real_layer_shapes()} == set(triples)
    groups = grouped_calls()
    assert all(len({s[1] for s in segs}) == 1 for segs in groups)
    assert any(len({s[3] for s in segs}) > 1 for segs in groups)  # bpw-2.2 layer 0: q|k|v at gs 128 | 128 | 64
    assert any(s[4] for segs in groups for s in segs)  # Qwen2 q/k/v biases


# ---------------------------------------------------------------------------------- helpers (GPU)
class _Seg:
    """QuantizedLinear-like holder of device tensors (what quantized_matmul_grouped takes)."""

    def __init__(self, qweight, scales, zeros, bias, bits, gs):
        self.qweight, self.scales, self.zeros, self.bias = qweight, scales, zeros, bias
        self.bits, self.group_size = bits, gs


_LAYERS = {}


def _device_layer(dev, N, K, bits, gs, salt=0, with_bias=False) -> _Seg:
    """A layer drawn on the device by the recipe of oracle.mlx_affine.synth_layer (a host generator is too slow for
    28672 x 8192): random words are valid codes at every width, the straddling 3- and 6-bit streams included.
    Cached by shape for the module; `salt` tells apart the segments of one grouped call that share a shape."""
    key = (N, K, bits, gs, salt, with_bias)
    if key not in _LAYERS:
        gen = torch.Generator(device=dev).manual_seed(zlib.crc32(repr(key).encode()))
        nb = (1 << bits) - 1
        qw = torch.randint(-(2**31), 2**31, (N, K * bits // 32), dtype=torch.int32, device=dev, generator=gen)
        s = ((torch.rand((N, K // gs), device=dev, generator=gen) + 0.5) * (2.0 / math.sqrt(K) / nb)).to(torch.bfloat16)
        eps = torch.rand((N, K // gs), device=dev, generator=gen) * 0.1 - 0.05
        z = (-s.float() * (nb / 2.0) * (1.0 + eps)).to(torch.bfloat16)
        bias = (torch.randn((N,), device=dev, generator=gen) * 0.02).to(torch.bfloat16) if with_bias else None
        _LAYERS[key] = _Seg(qw, s, z, bias, bits, gs)
    return _LAYERS[key]


def _sample_rows(N, K, gs, seed) -> np.ndarray:
    """64 rows of a layer: the first and the last, the rows either side of where one CTA's share of the rows ends when
    the grid is one CTA per SM (rows go out in units of 4 when K/gs = 4 mod 8), and random ones."""
    if N <= SAMPLED_ROWS:
        return np.arange(N)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    unit = 4 if (K // gs) % 8 else 1
    grid = max(1, min(sms, N // unit))
    base, rem = (N // unit) // grid * unit, (N // unit) % grid
    starts = [b * base + min(b, rem) * unit for b in range(1, grid)]
    pick = {0, N - 1}
    for r in starts[:: max(1, len(starts) // 12)] + starts[-1:] + [s for s in starts if s == rem * (base + unit)]:
        pick |= {r - 1, r}
    rest = np.setdiff1d(np.arange(N), sorted(pick))
    fill = np.random.default_rng(seed).choice(rest, SAMPLED_ROWS - len(pick), replace=False)
    return np.sort(np.concatenate([np.array(sorted(pick)), fill]))


def _host_rows(seg: _Seg, rows: np.ndarray):
    """Rows `rows` of a device layer as the oracle's numpy arrays (codes as uint32 words, bf16 as uint16 bits)."""
    r = torch.from_numpy(rows).to(seg.qweight.device)
    qw = seg.qweight[r].cpu().numpy().view(np.uint32)
    bias = bits_from_bf16(seg.bias[r]) if seg.bias is not None else None
    return qw, bits_from_bf16(seg.scales[r]), bits_from_bf16(seg.zeros[r]), bias


def _x(M, K, seed, dev):
    x = torch.randn((M, K), generator=torch.Generator().manual_seed(seed)).to(torch.bfloat16)
    return x.to(dev), bits_from_bf16(x)


def _every_kernel(x, seg: _Seg, bias, ref, rows=None, what=""):
    """Auto dispatch and every kernel that accepts the call, each (rows `rows` of it) against `ref`; the auto output
    must be bit for bit that of the kernel select_kernel names -- the dispatch ran the kernel it says it runs."""
    from gbx_lm_b200 import ops

    M, N, K = x.shape[0], seg.qweight.shape[0], x.shape[1]
    chosen = ops.select_kernel(M, N, K, seg.bits, seg.group_size)
    cols = None if rows is None else torch.from_numpy(rows).to(x.device)
    outs = {}
    for kern in ("auto",) + KERNELS + (() if chosen in KERNELS else (chosen,)):
        try:
            y = ops.quantized_matmul(x, seg.qweight, seg.scales, seg.zeros, True, seg.group_size, seg.bits, bias=bias,
                                     kernel=kern)
        except RuntimeError as e:
            assert kern != "auto" and "does not support" in str(e), (what, kern, str(e))
            continue
        assert y.shape == (M, N)
        tol = TOL.get(chosen if kern == "auto" else kern, 2.0 ** -7)
        assert_close_to_truth(y if cols is None else y[:, cols], ref, f"{what} {kern} M{M}", tol)
        outs[kern] = y
    assert chosen in outs, (what, M, chosen)
    assert torch.equal(outs["auto"], outs[chosen]), (what, M, chosen)


def _add_bias(y_ref, bias_bits):
    """The oracle's `+ bias`: a second, separately rounded add on the rounded product (mlx_affine.quantized_matmul)."""
    s = y_ref.astype(np.float64) + A.bf16_bits_to_f32(bias_bits).astype(np.float64)
    return A.bf16_bits_to_f32(A.f32_to_bf16_bits(s.astype(np.float32)))


# ---------------------------------------------------------------------------------- 1. every (bits, gs, K), N = 260
@pytest.mark.gpu
@pytest.mark.parametrize("bits,gs,K", config_triples(), ids=[_triple_id(t) for t in config_triples()])
def test_decode_kernels_at_config_k(cuda_device, bits, gs, K):
    """Every kernel at every M of a decode step on one (bits, group size, K) of the configs, against the fp64 truth
    (one oracle call for all M: rows of x are independent)."""
    N = N_SMALL
    seed = zlib.crc32(_triple_id((bits, gs, K)).encode())
    L = A.synth_layer(N, K, bits, gs, seed=seed, with_bias=True)
    d = layer_to_cuda(L, cuda_device)
    seg = _Seg(d["qweight"], d["scales"], d["zeros"], None, bits, gs)
    xs = A.synth_x(sum(DECODE_M), K, seed=seed + 1)
    ref = A.quantized_matmul(xs, L["qweight"], L["scales"], L["zeros"], gs, bits, "bf16", "f64")
    o = 0
    for M in DECODE_M:
        x = bf16_from_bits(xs[o:o + M], cuda_device)
        want = ref[o:o + M]
        bias = d["bias"] if M == BIAS_M else None
        if bias is not None:
            want = _add_bias(want, L["bias"])
        _every_kernel(x, seg, bias, want, what=_triple_id((bits, gs, K)))
        o += M


# ---------------------------------------------------------------------------------- 2. real-size layers
@pytest.mark.gpu
@pytest.mark.parametrize("N,K,bits,gs", real_layer_shapes(), ids=[_shape_id(s) for s in real_layer_shapes()])
def test_decode_kernels_real_layers(cuda_device, N, K, bits, gs):
    """Layers as tall as the configs' (up to 28672 rows, up to K = 28672): each CTA loops over many rows and refills
    its ring, the last CTA takes the row tail.  64 sampled rows against the fp64 truth at M = 1 and 2."""
    seg = _device_layer(cuda_device, N, K, bits, gs)
    seed = zlib.crc32(_shape_id((N, K, bits, gs)).encode())
    rows = _sample_rows(N, K, gs, seed)
    qw, s, z, _ = _host_rows(seg, rows)
    x, xb = _x(3, K, seed, cuda_device)
    ref = A.quantized_matmul(xb, qw, s, z, gs, bits, "bf16", "f64")
    _every_kernel(x[:1], seg, None, ref[:1], rows, _shape_id((N, K, bits, gs)))
    _every_kernel(x[1:], seg, None, ref[1:], rows, _shape_id((N, K, bits, gs)))


# ---------------------------------------------------------------------------------- 3. grouped calls
@pytest.mark.gpu
@pytest.mark.parametrize("segs", grouped_calls(), ids=_group_id)
def test_grouped_calls_at_config_shapes(cuda_device, segs):
    """q|k|v and gate|up of the configs as one quantized_matmul_grouped call at M = 1, 2, 4, 16: each segment equals
    its own quantized_matmul call and 64 sampled rows of it agree with the fp64 truth."""
    import gbx_lm_b200 as g
    from gbx_lm_b200 import ops

    K = segs[0][1]
    layers = [_device_layer(cuda_device, N, K, bits, gs, salt=i, with_bias=bias) for i, (N, _, bits, gs, bias) in enumerate(segs)]
    seed = zlib.crc32(_group_id(segs).encode())
    Ms = (1, 2, 4, 16)
    x, xb = _x(sum(Ms), K, seed, cuda_device)
    refs = []
    for i, seg in enumerate(layers):
        rows = _sample_rows(seg.qweight.shape[0], K, seg.group_size, seed + i)
        qw, s, z, bias = _host_rows(seg, rows)
        refs.append((rows, A.quantized_matmul(xb, qw, s, z, seg.group_size, seg.bits, "bf16", "f64", bias=bias)))
    mixed_gs = len({seg.group_size for seg in layers}) > 1
    o = 0
    for M in Ms:
        xm = x[o:o + M]
        n0 = ops.launch_count()
        ys = g.quantized_matmul_grouped(xm, layers)
        launches = ops.launch_count() - n0
        if mixed_gs:
            assert launches >= len(layers), (segs, M, launches)  # no shared launch: one call per segment
        # one launch of the TMEM-operand GEMM for all segments (M >= 9, one width): its split-K plan is that of the
        # padded sum of the segments, so it equals the single calls within fp32 summation noise, not bit for bit
        ts_grouped = M > 4 and launches == 1
        for i, (seg, y) in enumerate(zip(layers, ys)):
            single = g.quantized_matmul(xm, seg.qweight, seg.scales, seg.zeros, True, seg.group_size, seg.bits, bias=seg.bias)
            assert y.shape == single.shape == (M, seg.qweight.shape[0])
            what = f"{_group_id(segs)} segment {i} M{M}"
            if ts_grouped:
                assert (y.float() - single.float()).abs().max() <= 2.0 ** -6 * single.float().abs().max(), what
            else:
                assert torch.equal(y, single), what
            rows, ref = refs[i]
            tol = 1e-2 if M >= 9 else 2.0 ** -7  # from 9 rows the tensor-core GEMM serves the call (see TOL)
            assert_close_to_truth(y[:, torch.from_numpy(rows).to(cuda_device)], ref[o:o + M], what, tol)
        o += M
