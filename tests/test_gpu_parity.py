"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  Every call goes through the C ABI
(libgbxq.so via the torch custom ops); results are checked against the CPU oracle (oracle/), the
committed golden fixtures, and -- at BASELINE sizes -- size-independent properties."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import c_oracle as C
from oracle import mlx_affine as A
from tests.gpu_util import assert_close_to_truth, bf16_from_bits, bits_from_bf16, layer_to_cuda, u32_to_torch

pytestmark = pytest.mark.gpu

BITS = (2, 3, 4, 6, 8)
GS = (32, 64, 128)
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "affine_golden.json")))


def _ops():
    import gbx_lm_b200 as g

    return g


# ---------------------------------------------------------------------------------- dequantize
@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("gs", GS)
@pytest.mark.parametrize("dtype", ["bf16", "f16", "f32"])
def test_dequantize_bit_exact(cuda_device, bits, gs, dtype):
    g = _ops()
    N, K = 37, 384
    L = A.synth_layer(N, K, bits, gs, seed=bits * 100 + gs)
    s32, z32 = A.bf16_bits_to_f32(L["scales"]), A.bf16_bits_to_f32(L["zeros"])
    w = u32_to_torch(L["qweight"], cuda_device)
    if dtype == "bf16":
        s, z = bf16_from_bits(L["scales"], cuda_device), bf16_from_bits(L["zeros"], cuda_device)
        ref = A.dequantize(L["qweight"], L["scales"], L["zeros"], gs, bits, "bf16")
    elif dtype == "f16":
        s16, z16 = s32.astype(np.float16), z32.astype(np.float16)
        s, z = torch.from_numpy(s16).to(cuda_device), torch.from_numpy(z16).to(cuda_device)
        ref = A.dequantize(L["qweight"], s16, z16, gs, bits, "f16")
    else:
        s32 = (s32 * np.float32(1.000123)).astype(np.float32)  # use all 24 significand bits
        s, z = torch.from_numpy(s32).to(cuda_device), torch.from_numpy(z32).to(cuda_device)
        ref = A.dequantize(L["qweight"], s32, z32, gs, bits, "f32")
    out = g.dequantize(w, s, z, gs, bits)
    assert out.shape == (N, K) and out.dtype == s.dtype
    got = out.float().cpu().numpy()
    assert (got.view(np.uint32) == ref.astype(np.float32).view(np.uint32)).all()


@pytest.mark.parametrize("case", GOLD["dequant"], ids=lambda c: f"b{c['bits']}-{c['dtype']}")
def test_dequantize_golden(cuda_device, case):
    g = _ops()
    tdt = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}[case["dtype"]]
    w = u32_to_torch(np.array([case["qweight"]], dtype=np.uint32), cuda_device)
    s = torch.tensor([[0.0123]], dtype=tdt, device=cuda_device)
    b = torch.tensor([[-0.771]], dtype=tdt, device=cuda_device)
    out = g.dequantize(w, s, b, 32, case["bits"]).float().cpu().numpy()
    assert out.view(np.uint32)[0].tolist() == case["out_f32_hex"]


def test_dequantize_full_size_against_c_oracle(cuda_device):
    """Llama-3-8B k_proj (1024 x 4096, 4-bit gs64) and a 3-bit o_proj slice: checksum of the whole
    matrix + exact compare, oracle = C restatement (seconds)."""
    g = _ops()
    for bits, gs, N, K in ((4, 64, 1024, 4096), (3, 64, 512, 4096), (6, 64, 256, 14336), (2, 128, 512, 3584)):
        L = A.synth_layer(N, K, bits, gs, seed=bits)
        ref = C.dequantize(L["qweight"], L["scales"], L["zeros"], gs, bits, "bf16")
        d = layer_to_cuda(L, cuda_device)
        out = g.dequantize(d["qweight"], d["scales"], d["zeros"], gs, bits)
        assert (bits_from_bf16(out) == ref).all()


# ---------------------------------------------------------------------------------- quantized matmul
def _run_case(g, dev, kernel, bits, gs, M, N, K, seed, with_bias=False, tol=2.0 ** -7):
    L = A.synth_layer(N, K, bits, gs, seed=seed, with_bias=with_bias)
    x = A.synth_x(M, K, seed=seed + 1)
    d = layer_to_cuda(L, dev)
    y = g.quantized_matmul(bf16_from_bits(x, dev), d["qweight"], d["scales"], d["zeros"], True, gs, bits,
                           bias=d.get("bias"), kernel=kernel)
    ref = A.quantized_matmul(x, L["qweight"], L["scales"], L["zeros"], gs, bits, "bf16", "f64", bias=L.get("bias"))
    assert y.shape == (M, N) and y.dtype == torch.bfloat16
    return assert_close_to_truth(y, ref, f"{kernel} b{bits} g{gs} M{M} N{N} K{K}", tol)


def _skinny_ok(bits, gs):
    return bits in (2, 4, 8) and not (bits == 2 and gs == 32)


@pytest.mark.parametrize("kernel", ["generic", "gemv", "skinny"])
@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("gs", GS)
def test_qmm_vs_oracle_small(cuda_device, kernel, bits, gs):
    g = _ops()
    if kernel == "skinny" and not _skinny_ok(bits, gs):
        with pytest.raises(RuntimeError):  # forcing a kernel that cannot serve the arguments is an error, not a fallback
            _run_case(g, cuda_device, kernel, bits, gs, 1, 70, 1024, seed=1)
        return
    for M in (1, 2, 3) + ((8, 9, 13, 16, 17) if kernel == "skinny" else ()):  # 9..16: one 16-token pass; 17: 16 + 1
        _run_case(g, cuda_device, kernel, bits, gs, M, 70, 1024, seed=bits * 31 + gs + M)


def _mmv_ok(bits, gs, K=1024, kernel="mmv"):
    if kernel == "mmv8":  # every packing width; 2/3/6-bit need a whole word per thread chunk (gs >= 64)
        return not (bits in (2, 3, 6) and gs == 32) and (K // gs) % 8 == 0
    return bits in (2, 4, 8) and gs * bits // 32 in (4, 8, 16) and (K // gs) % 8 == 0


MMV_KERNELS = ("mmv", "mmv8")


@pytest.mark.parametrize("kernel", MMV_KERNELS)
@pytest.mark.parametrize("bits", (2, 3, 4, 6, 8))
@pytest.mark.parametrize("gs", GS)
def test_qmm_mmv_vs_oracle_small(cuda_device, kernel, bits, gs):
    """Tensor-pipe decode kernels ("slice" MMA layout; bf16 HMMA and integer IMMA) at M = 1..4, every supported packing."""
    g = _ops()
    if not _mmv_ok(bits, gs, kernel=kernel):
        with pytest.raises(RuntimeError):  # forced kernel that cannot serve the arguments: error, not fallback
            _run_case(g, cuda_device, kernel, bits, gs, 1, 70, 1024, seed=1)
        return
    for M in (1, 2, 3, 4):
        _run_case(g, cuda_device, kernel, bits, gs, M, 70, 1024, seed=bits * 31 + gs + M, with_bias=(M == 3))


@pytest.mark.parametrize("bits,gs,K", [(4, 128, 1536), (4, 64, 768), (2, 128, 3584), (3, 64, 1792), (8, 64, 256 + 512)])
def test_qmm_mmv8_rows_of_scales_only_8_byte_aligned(cuda_device, bits, gs, K):
    """K / group_size = 4 (mod 8): a row of scales is 8 bytes off the 16-byte grid the bulk copies need (the K shards of
    tensor parallelism: Qwen2.5-32B down_proj K/2 = 13824 at gs 128, Llama-3-8B down_proj K/8 = 1792).  The kernel then
    shares rows out in units of four; N % 4 != 0 is refused."""
    g = _ops()
    assert (K // gs) % 8 == 4
    for M in (1, 2, 4):
        for N in (72, 1028, 4):
            _run_case(g, cuda_device, "mmv8", bits, gs, M, N, K, seed=bits + gs + M + N, with_bias=(M == 2))
    with pytest.raises(RuntimeError):
        _run_case(g, cuda_device, "mmv8", bits, gs, 1, 70, K, seed=1)


@pytest.mark.parametrize("bits,gs,K", [(4, 128, 1280), (4, 128, 6912), (2, 128, 768), (8, 128, 256 + 512), (3, 128, 1792), (6, 128, 768)])
def test_qmm_mmv8_half_full_last_chunk_column(cuda_device, bits, gs, K):
    """K / group_size = 2 (mod 4): the row ends in the middle of a 4-group chunk column (Qwen2.5-32B at tp4: o_proj K/4 =
    1280 and down_proj K/4 = 6912 at gs 128).  Served by the one-call decode launches at group size 128 and <= 2 rows of
    x (a separate instantiation): the dead slices multiply zero activations and their scale reads, which would run into
    the next row or into stale shared memory behind the last row of a stage, are redirected to a live slice."""
    g = _ops()
    from gbx_lm_b200 import _lib

    assert (K // gs) % 4 == 2
    for M in (1, 2):
        for N in (72, 1028, 4):
            _run_case(g, cuda_device, "mmv8", bits, gs, M, N, K, seed=bits + gs + M + N, with_bias=(M == 2))
    assert _lib.get().gbxq_select_kernel(1, 1024, K, bits, gs, 0) == _lib.KERNEL_MMV8
    with pytest.raises(RuntimeError):  # 4 rows of x: no such instantiation; auto dispatch serves the call elsewhere
        _run_case(g, cuda_device, "mmv8", bits, gs, 4, 72, K, seed=1)
    _run_case(g, cuda_device, "auto", bits, gs, 4, 72, K, seed=1, tol=1e-2)
    # a grouped call on such a K falls back to one launch per segment: same results
    segs = []
    for i, N in enumerate((256, 64)):
        segs.append(_Seg(layer_to_cuda(A.synth_layer(N, K, bits, gs, seed=90 + i), cuda_device), bits, gs))
    x = bf16_from_bits(A.synth_x(1, K, seed=3), cuda_device)
    for sg, y in zip(segs, g.quantized_matmul_grouped(x, segs)):
        assert torch.equal(y, g.quantized_matmul(x, sg.qweight, sg.scales, sg.zeros, True, gs, bits))


def test_qmm_mmv8_block_fixed_point_ranges(cuda_device):
    """The integer kernel represents x per (token, group) as 15-bit block fixed point: check wide dynamic range inside a
    group (outlier channels), tiny and huge magnitudes, exact zeros, and that inf / nan poison only what they should."""
    g = _ops()
    N, K, bits, gs = 64, 1024, 4, 64
    L = A.synth_layer(N, K, bits, gs, seed=3)
    d = layer_to_cuda(L, cuda_device)
    rng = np.random.default_rng(5)
    measured = {}
    for case in ("outliers", "outliers_1000", "massive_3000", "tiny", "huge", "zeros", "mixed"):
        x = rng.standard_normal((1, K)).astype(np.float32)
        if case == "outliers":
            x[0, ::64] *= 300.0
        elif case == "outliers_1000":
            x[0, ::64] *= 1000.0
        elif case == "massive_3000":  # the Llama "massive activation" regime: two channels thousands of times the rest
            x[0, 7] = 3000.0
            x[0, 500] = -2200.0
        elif case == "tiny":
            x *= 1e-30
        elif case == "huge":
            x *= 1e30
        elif case == "zeros":
            x[0, 128:512] = 0.0
        else:
            x *= np.exp(rng.uniform(-8, 8, size=(1, K))).astype(np.float32)
        xb = A.f32_to_bf16_bits(x)
        y = g.quantized_matmul(bf16_from_bits(xb, cuda_device), d["qweight"], d["scales"], d["zeros"], True, gs, bits, kernel="mmv8")
        ref = A.quantized_matmul(xb, L["qweight"], L["scales"], L["zeros"], gs, bits, "bf16", "f64")
        measured[case] = float(assert_close_to_truth(y, ref, f"mmv8 {case}"))
    # measured max |err| / max |y| per case, kept next to the bound (1e-2) in DESIGN.md section 3.1
    print("mmv8 block fixed point, max |err| / max |y|:", json.dumps(measured))
    x = rng.standard_normal((1, K)).astype(np.float32)
    x[0, 5] = np.inf
    y = g.quantized_matmul(bf16_from_bits(A.f32_to_bf16_bits(x), cuda_device), d["qweight"], d["scales"], d["zeros"], True, gs, bits, kernel="mmv8")
    assert not torch.isfinite(y).any()  # every output row multiplies x[5] by a non-zero weight


@pytest.mark.parametrize("kernel", MMV_KERNELS)
@pytest.mark.parametrize("bits", (2, 4, 8))
@pytest.mark.parametrize("pdl", (0, 1, 2))
def test_qmm_mmv_model_shapes(cuda_device, kernel, bits, pdl):
    """Config shapes: long rows (14336: 2 rows per stage), TP shards (3584), N smaller than / not a multiple
    of the grid, single rows, the three launch modes (plain, PDL, PDL with early weight streaming)."""
    g = _ops()
    from gbx_lm_b200 import ops

    ops.set_pdl_mode(pdl)
    try:
        for (N, K) in ((300, 4096), (96, 14336), (150, 3584), (1, 2048), (147, 8192), (149, 3072), (5000, 512), (1031, 1024)):
            for M in (1, 2, 4):
                # rows too long for W = 2*MP of them in one ring stage are served by another kernel (auto dispatch)
                try:
                    _run_case(g, cuda_device, kernel, bits, 64, M, N, K, seed=N + K + bits + M, with_bias=(M == 2))
                except RuntimeError as e:
                    assert "does not support" in str(e)  # stage too large for this kernel: auto dispatch serves it
                    _run_case(g, cuda_device, "auto", bits, 64, M, N, K, seed=N + K + bits + M, with_bias=(M == 2))
    finally:
        ops.set_pdl_mode(2)


def test_qmm_mmv_back_to_back_dependency(cuda_device):
    """PDL: a chain y1 = W1 x, y2 = W2 y1, ... launched back to back must see its predecessor's output
    (griddepcontrol.wait before x is read), eagerly and from a CUDA graph; bitwise equal to plain launches."""
    g = _ops()
    from gbx_lm_b200 import ops

    K = 1024
    Ls = [layer_to_cuda(A.synth_layer(K, K, 4, 64, seed=50 + i), cuda_device) for i in range(6)]
    x = bf16_from_bits(A.synth_x(1, K, seed=60), cuda_device)

    def chain(x):
        h = x
        for d in Ls:
            h = g.quantized_matmul(h * 8, d["qweight"], d["scales"], d["zeros"], True, 64, 4, kernel="mmv")
            h = g.quantized_matmul(h * 8, d["qweight"], d["scales"], d["zeros"], True, 64, 4, kernel="mmv8")
        return h

    ops.set_pdl_mode(0)
    ref = chain(x)
    ops.set_pdl_mode(2)
    for _ in range(5):
        assert torch.equal(chain(x), ref)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        chain(x)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = chain(x)
    for _ in range(5):
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, ref)


@pytest.mark.parametrize("bits", (2, 4, 8))
def test_qmm_skinny_model_shapes(cuda_device, bits):
    """mma.sync skinny kernel on the config shapes: ragged k-tiles (3584/64 = 56 groups = 3.5 tiles),
    row counts that are not multiples of 16 or of the grid, every token count 1..8 and a 2-pass 13."""
    g = _ops()
    for (N, K) in ((300, 4096), (96, 14336), (150, 3584), (1, 2048), (147, 8192), (149, 3072), (5000, 512)):
        for M in (1, 4, 7, 8, 13):
            _run_case(g, cuda_device, "skinny", bits, 64, M, N, K, seed=N + K + bits + M, with_bias=(M == 7))


@pytest.mark.parametrize("bits", BITS)
def test_qmm_gemv_model_shapes(cuda_device, bits):
    """Shapes of the configs (SURVEY 8a): ragged K (14336 = 14 pieces, 3584 = TP shard of 28672),
    N smaller / not a multiple of the grid, M = 1 and 2."""
    g = _ops()
    for (N, K) in ((300, 4096), (96, 14336), (150, 3584), (1, 2048), (147, 8192), (149, 3072)):
        for M in (1, 2):
            if bits == 3 and K % 128:
                continue
            _run_case(g, cuda_device, "gemv", bits, 64, M, N, K, seed=N + K + bits)


@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("gs", GS)
def test_qmm_gemm_tcgen05_vs_oracle(cuda_device, bits, gs):
    """tcgen05/TMEM GEMM with in-kernel dequant: the weight operand is rounded once to bf16
    (RN(scale*q+bias)), accumulation is fp32 in TMEM; tolerance = the path's 1e-2 (north_star)."""
    g = _ops()
    # the TMA descriptors need 16-byte row pitches: K*bits/8 and (K/gs)*2 multiples of 16
    for (M, N, K) in ((17, 128, 1024), (64, 200, 1024), (100, 384, 2048), (300, 130, 4096)):
        _run_case(g, cuda_device, "gemm", bits, gs, M, N, K, seed=bits + gs + M, with_bias=(M == 100), tol=1e-2)


@pytest.mark.parametrize("M,N,K,bits,gs", [(32, 512, 4096, 4, 64), (64, 640, 6144, 4, 128), (17, 128, 8192, 2, 64), (256, 1024, 3072, 8, 64),
                                          (100, 384, 5120, 3, 64)])
def test_qmm_gemm_split_k(cuda_device, M, N, K, bits, gs):
    """Skinny batches on layers with few output tiles: the tcgen05 GEMM splits K over blockIdx.z (fp32 partial tiles in
    the workspace, last split to arrive reduces in split order).  Against the oracle, bitwise reproducible call after
    call (the tile counters are left zero), and within fp32 summation noise of the unsplit launch."""
    g = _ops()
    from gbx_lm_b200 import _lib

    assert _lib.get().gbxq_workspace_bytes(M, N, K, bits, gs, 0) > 16384, "shape does not exercise split-K"
    L = A.synth_layer(N, K, bits, gs, seed=M + N, with_bias=True)
    d = layer_to_cuda(L, cuda_device)
    xb = A.synth_x(M, K, seed=K)
    x = bf16_from_bits(xb, cuda_device)
    ys = [g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, gs, bits, bias=d["bias"], kernel="gemm") for _ in range(3)]
    y0 = g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, gs, bits, kernel="gemm")
    ref = A.quantized_matmul(xb, L["qweight"], L["scales"], L["zeros"], gs, bits, "bf16", "f64")
    assert_close_to_truth(y0, ref, f"gemm split-K M{M} N{N} K{K} b{bits}", 1e-2)
    # the bias is a second, separately rounded add on the rounded product (quantized_linear_gba.py:204-205): checked
    # exactly (against the truth two roundings can stack to 2 bf16 ulps = 1.6 % at the bottom of a binade)
    assert torch.equal(ys[0], (y0.float() + d["bias"].float()).to(torch.bfloat16))
    assert torch.equal(ys[0], ys[1]) and torch.equal(ys[0], ys[2])
    # auto dispatch prefers the TMEM-operand GEMM from 9 rows (K % 256 == 0) and falls back to this kernel otherwise
    ya = g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, gs, bits, bias=d["bias"])
    assert torch.equal(ya, ys[0]) or torch.equal(ya, g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, gs, bits, bias=d["bias"], kernel="gemm_ts"))


@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("gs", GS)
def test_qmm_gemm_ts_vs_oracle(cuda_device, bits, gs):
    """tcgen05 GEMM with the dequantised weights as the TMEM operand (gbxq_gemm_ts_sm100.cu): every token tile width
    (16 .. 256 accumulator columns, several token tiles), ragged N (rows past N are zero-filled by TMA), K a multiple of
    the 128-k stage; tolerance = the path's 1e-2 (north_star)."""
    g = _ops()
    for (M, N, K) in ((5, 128, 1024), (16, 200, 1024), (17, 130, 2048), (33, 384, 1024), (100, 256, 2048), (200, 128, 1024),
                      (300, 130, 4096)):
        _run_case(g, cuda_device, "gemm_ts", bits, gs, M, N, K, seed=bits + gs + M, with_bias=(M == 100), tol=1e-2)
    # shortest loops and thinnest tiles: one or two 256-k stages, fewer rows than a tile, a few rows of x
    # (where K / group_size is not a multiple of 8 a row of scales is no legal TMA row pitch: the dequant threads then
    # read their scales from global memory -- tensor-parallel K shards: 1280 = 10 and 6912 = 54 groups of 128)
    for (M, N, K) in ((9, 16, 256), (3, 24, 512), (40, 129, 512), (33, 200, 1280), (300, 136, 6912), (12, 512, 768)):
        _run_case(g, cuda_device, "gemm_ts", bits, gs, M, N, K, seed=bits + gs + N, with_bias=(M == 33), tol=1e-2)


@pytest.mark.parametrize("M,N,K,bits,gs", [(8, 512, 4096, 4, 64), (32, 512, 4096, 4, 64), (64, 640, 6144, 4, 128), (17, 128, 8192, 2, 64),
                                          (256, 1024, 3072, 8, 64), (100, 384, 5120, 3, 64), (48, 256, 4096, 6, 32)])
def test_qmm_gemm_ts_split_k(cuda_device, M, N, K, bits, gs):
    """Split-K of the TMEM-operand GEMM: against the oracle, bitwise reproducible call after call (tile counters left
    zero), bias as a separately rounded add, and equal to the shared-memory-operand GEMM within fp32 summation noise."""
    g = _ops()
    from gbx_lm_b200 import _lib

    assert _lib.get().gbxq_workspace_bytes(M, N, K, bits, gs, 0) > 16384, "shape does not exercise split-K"
    L = A.synth_layer(N, K, bits, gs, seed=M + N, with_bias=True)
    d = layer_to_cuda(L, cuda_device)
    xb = A.synth_x(M, K, seed=K)
    x = bf16_from_bits(xb, cuda_device)
    ys = [g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, gs, bits, bias=d["bias"], kernel="gemm_ts") for _ in range(3)]
    y0 = g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, gs, bits, kernel="gemm_ts")
    ref = A.quantized_matmul(xb, L["qweight"], L["scales"], L["zeros"], gs, bits, "bf16", "f64")
    assert_close_to_truth(y0, ref, f"gemm_ts split-K M{M} N{N} K{K} b{bits}", 1e-2)
    assert torch.equal(ys[0], (y0.float() + d["bias"].float()).to(torch.bfloat16))
    assert torch.equal(ys[0], ys[1]) and torch.equal(ys[0], ys[2])
    if M >= 9:  # what auto dispatch runs from 9 rows
        assert torch.equal(ys[0], g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, gs, bits, bias=d["bias"]))
    if M >= 17:
        y1 = g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, gs, bits, kernel="gemm")
        assert (y0.float() - y1.float()).abs().max() <= 2.0 ** -6 * y1.float().abs().max()


def test_qmm_gemm_ts_model_shapes_and_pdl(cuda_device):
    """Model-sized calls at decode batches (8B q/o, gate, down at 8 / 32 / 64 rows of x), launched back to back with and
    without programmatic dependent launch: y of one call is x of the next (the x producer waits for the previous kernel,
    the weight producer does not)."""
    g = _ops()
    from gbx_lm_b200 import ops

    try:
        for pdl in (0, 2):
            ops.set_pdl_mode(pdl)
            for (M, N, K, bits) in ((8, 4096, 4096, 4), (32, 14336, 4096, 2), (64, 4096, 14336, 4)):
                _run_case(g, cuda_device, "gemm_ts", bits, 64, M, N, K, seed=M + bits, tol=1e-2)
            # chain: x -> A (K -> K) -> B (K -> K), three times on one stream without synchronising in between
            K = 2048
            LA, LB = A.synth_layer(K, K, 4, 64, seed=5), A.synth_layer(K, K, 4, 64, seed=6)
            dA, dB = layer_to_cuda(LA, cuda_device), layer_to_cuda(LB, cuda_device)
            xb = A.synth_x(24, K, seed=7)
            x = bf16_from_bits(xb, cuda_device)
            outs = []
            for _ in range(3):
                h = g.quantized_matmul(x, dA["qweight"], dA["scales"], dA["zeros"], True, 64, 4, kernel="gemm_ts")
                outs.append(g.quantized_matmul(h, dB["qweight"], dB["scales"], dB["zeros"], True, 64, 4, kernel="gemm_ts"))
            torch.cuda.synchronize()
            h_ref = g.quantized_matmul(x, dA["qweight"], dA["scales"], dA["zeros"], True, 64, 4, kernel="generic")
            ref = A.quantized_matmul(bits_from_bf16(h), LB["qweight"], LB["scales"], LB["zeros"], 64, 4, "bf16", "f64")
            assert (h.float() - h_ref.float()).abs().max() <= 1e-2 * h_ref.float().abs().max()
            assert_close_to_truth(outs[0], ref, "gemm_ts chain", 1e-2)
            assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    finally:
        ops.set_pdl_mode(2)


def test_qmm_gemm_declines_unaligned_pitch(cuda_device):
    """K = 256 with gs = 128 gives a 4-byte scale row pitch: the forced tensor-core kernel refuses
    (no silent fallback), auto dispatch serves the call with another kernel."""
    g = _ops()
    with pytest.raises(RuntimeError):
        _run_case(g, cuda_device, "gemm", 4, 128, 20, 64, 256, seed=1)
    _run_case(g, cuda_device, "auto", 4, 128, 20, 64, 256, seed=1, tol=1e-2)


def test_qmm_gemm_prefill_shape_properties(cuda_device):
    """Prefill-sized call (M = 2048 tokens, Llama-3.2-3B q_proj 3072 x 3072, 4-bit gs64): sampled
    rows/tokens against the oracle, and agreement with x . dequantize()^T computed in fp32."""
    g = _ops()
    N = K = 3072
    M, bits, gs = 2048, 4, 64
    P = __import__("gbx_lm_b200.packing", fromlist=["x"])
    L = P.synth_layer(N, K, bits, gs, seed=31, with_bias=True)
    qw, s, z, b = (L[k].to(cuda_device) for k in ("qweight", "scales", "zeros", "bias"))
    x = torch.randn((M, K), generator=torch.Generator().manual_seed(32)).to(torch.bfloat16).to(cuda_device)
    y = g.quantized_matmul(x, qw, s, z, True, gs, bits, bias=b, kernel="gemm")
    assert y.shape == (M, N)
    Wd = g.dequantize(qw, s, z, gs, bits).float()
    ref = (x.float() @ Wd.t()).to(torch.bfloat16).float() + b.float()
    assert (y.float() - ref).abs().max() <= 1e-2 * ref.abs().max()
    rows = np.random.default_rng(1).choice(N, 16, replace=False)
    toks = np.random.default_rng(2).choice(M, 24, replace=False)
    o = A.quantized_matmul(bits_from_bf16(x[torch.from_numpy(toks).to(cuda_device)]),
                           L["qweight"][rows].view(torch.int32).numpy().view(np.uint32), bits_from_bf16(L["scales"][rows]),
                           bits_from_bf16(L["zeros"][rows]), gs, bits, "bf16", "f64", bias=bits_from_bf16(L["bias"][rows]))
    sub = y[torch.from_numpy(toks).to(cuda_device)][:, torch.from_numpy(rows).to(cuda_device)]
    assert_close_to_truth(sub, o, "prefill sample", tol=1e-2)
    # auto dispatch picks the TMEM-operand GEMM for prefill: same bounds, and bit for bit the forced gemm_ts launch
    ya = g.quantized_matmul(x, qw, s, z, True, gs, bits, bias=b)
    assert (ya.float() - ref).abs().max() <= 1e-2 * ref.abs().max()
    assert torch.equal(ya, g.quantized_matmul(x, qw, s, z, True, gs, bits, bias=b, kernel="gemm_ts"))


def test_qmm_auto_dispatch_and_bias(cuda_device):
    g = _ops()
    for M in (1, 2, 4, 5, 16, 17, 40, 200):
        _run_case(g, cuda_device, "auto", 4, 64, M, 512, 2048, seed=77 + M, with_bias=True, tol=1e-2 if M >= 9 else 2.0 ** -7)
    _run_case(g, cuda_device, "gemv", 2, 128, 1, 256, 2048, seed=5, with_bias=True)
    _run_case(g, cuda_device, "generic", 6, 32, 3, 33, 96 * 4, seed=6, with_bias=True)


@pytest.mark.parametrize("case", GOLD["qmm"], ids=lambda c: f"b{c['bits']}-g{c['group_size']}")
def test_qmm_golden_fixtures(cuda_device, case):
    """Committed fixtures: GPU output within one bf16 ulp of the fp64-truth rounded to bf16."""
    g = _ops()
    w = u32_to_torch(np.array(case["qweight"], dtype=np.uint32), cuda_device)
    s = bf16_from_bits(np.array(case["scales_bf16"], dtype=np.uint16), cuda_device)
    z = bf16_from_bits(np.array(case["zeros_bf16"], dtype=np.uint16), cuda_device)
    x = bf16_from_bits(np.array(case["x_bf16"], dtype=np.uint16), cuda_device)
    gold = A.bf16_bits_to_f32(np.array(case["y_bf16"], dtype=np.uint16))
    for kernel in ("generic", "gemv", "skinny", "mmv", "mmv8"):
        if kernel == "skinny" and not _skinny_ok(case["bits"], case["group_size"]):
            continue
        if kernel in MMV_KERNELS and not (_mmv_ok(case["bits"], case["group_size"], x.shape[-1], kernel) and x.shape[0] <= 4):
            continue
        y = g.quantized_matmul(x, w, s, z, True, case["group_size"], case["bits"], kernel=kernel).float().cpu().numpy()
        ulp = np.maximum(np.abs(gold) * 2.0 ** -7, np.abs(gold).max() * 2.0 ** -9)
        assert (np.abs(y - gold) <= ulp).all(), kernel


def test_qmm_generic_f16_f32(cuda_device):
    g = _ops()
    N, K, M, bits, gs = 40, 512, 3, 4, 64
    L = A.synth_layer(N, K, bits, gs, seed=8)
    x32 = A.bf16_bits_to_f32(A.synth_x(M, K, seed=9))
    s32, z32 = A.bf16_bits_to_f32(L["scales"]), A.bf16_bits_to_f32(L["zeros"])
    w = u32_to_torch(L["qweight"], cuda_device)
    for tdt, name in ((torch.float16, "f16"), (torch.float32, "f32")):
        npdt = np.float16 if name == "f16" else np.float32
        y = g.quantized_matmul(torch.from_numpy(x32.astype(npdt)).to(cuda_device), w,
                               torch.from_numpy(s32.astype(npdt)).to(cuda_device),
                               torch.from_numpy(z32.astype(npdt)).to(cuda_device), True, gs, bits)
        ref = A.quantized_matmul(x32.astype(npdt), L["qweight"], s32.astype(npdt), z32.astype(npdt), gs, bits, name, "f64")
        assert y.dtype == tdt
        tol = 2.0 ** -10 if name == "f16" else 1e-5
        assert np.abs(y.float().cpu().numpy() - ref).max() <= tol * np.abs(ref).max()


def test_edge_cases(cuda_device):
    g = _ops()
    L = A.synth_layer(16, 64, 4, 64, seed=1)
    d = layer_to_cuda(L, cuda_device)
    # empty batch
    y = g.quantized_matmul(torch.zeros((0, 64), dtype=torch.bfloat16, device=cuda_device), d["qweight"], d["scales"], d["zeros"], True, 64, 4)
    assert y.shape == (0, 16)
    # leading dims [B, L, K] and a non-contiguous x
    x = bf16_from_bits(A.synth_x(6, 128, seed=2), cuda_device)[:, ::2].reshape(2, 3, 64)
    y = g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, 64, 4)
    xb = bits_from_bf16(x.reshape(6, 64))
    ref = A.quantized_matmul(xb, L["qweight"], L["scales"], L["zeros"], 64, 4, "bf16", "f64")
    assert y.shape == (2, 3, 16)
    assert_close_to_truth(y.reshape(6, 16), ref, "3-D non-contiguous x")
    # int32-typed qweight (same bits) is accepted
    y2 = g.quantized_matmul(x, d["qweight"].view(torch.int32), d["scales"], d["zeros"], True, 64, 4)
    assert torch.equal(y, y2)
    # K = 32 (one word-block) with the smallest group
    _run_case(g, cuda_device, "auto", 8, 32, 1, 3, 32, seed=3)
    # errors: ValueError like MLX
    with pytest.raises(ValueError):
        g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, 64, 5)
    with pytest.raises(ValueError):
        g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, 32, 4)
    with pytest.raises(ValueError):
        g.quantized_matmul(x.float(), d["qweight"], d["scales"], d["zeros"], True, 64, 4)
    with pytest.raises(ValueError):
        g.quantized_matmul(x, d["qweight"].float(), d["scales"], d["zeros"], True, 64, 4)
    with pytest.raises(ValueError):  # transpose=False reads the same tensors as [K, N]: x's last dim no longer matches
        g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], False, 64, 4)
    from gbx_lm_b200 import ops

    with pytest.raises(ValueError):  # forced fast kernel on unsupported arguments surfaces, never falls back silently
        ops.quantized_matmul(torch.zeros((1, 32), dtype=torch.float16, device=cuda_device),
                             torch.zeros((4, 4), dtype=torch.uint32, device=cuda_device),
                             torch.ones((4, 1), dtype=torch.float16, device=cuda_device),
                             torch.ones((4, 1), dtype=torch.bfloat16, device=cuda_device), True, 32, 4)


# ---------------------------------------------------------------------------------- full-size properties
def test_full_size_8b_gate_proj_properties(cuda_device):
    """Llama-3-8B gate_proj (14336 x 4096, 4-bit gs64) at M=1/2: (a) sampled rows vs oracle,
    (b) consistency with x . dequantize()^T, (c) split-K additivity (the row-parallel TP identity)."""
    g = _ops()
    N, K, bits, gs = 14336, 4096, 4, 64
    P = __import__("gbx_lm_b200.packing", fromlist=["x"])
    L = P.synth_layer(N, K, bits, gs, seed=11)
    qw, s, z = L["qweight"].to(cuda_device), L["scales"].to(cuda_device), L["zeros"].to(cuda_device)
    x = torch.randn((2, K), generator=torch.Generator().manual_seed(12)).to(torch.bfloat16).to(cuda_device)
    y = g.quantized_matmul(x, qw, s, z, True, gs, bits, kernel="gemv")
    # (a) 64 sampled rows against the oracle
    rows = np.random.default_rng(0).choice(N, 64, replace=False)
    ref = A.quantized_matmul(bits_from_bf16(x), L["qweight"][rows].view(torch.int32).numpy().view(np.uint32),
                             bits_from_bf16(L["scales"][rows]), bits_from_bf16(L["zeros"][rows]), gs, bits, "bf16", "f64")
    assert_close_to_truth(y[:, torch.from_numpy(rows).to(cuda_device)], ref, "sampled rows")
    # (b) matmul against the GPU-dequantised matrix in fp32
    W = g.dequantize(qw, s, z, gs, bits).float()
    y_deq = x.float() @ W.t()
    assert (y.float() - y_deq).abs().max() <= 2.0 ** -6 * y_deq.abs().max()
    # (c) split-K additivity: y(W) == y(W[:, :K/2]) + y(W[:, K/2:]) up to bf16 rounding of the halves
    h = K // 2
    wh = h * bits // 32
    y0 = g.quantized_matmul(x[:, :h].contiguous(), qw[:, :wh].contiguous(), s[:, : h // gs].contiguous(), z[:, : h // gs].contiguous(), True, gs, bits)
    y1 = g.quantized_matmul(x[:, h:].contiguous(), qw[:, wh:].contiguous(), s[:, h // gs :].contiguous(), z[:, h // gs :].contiguous(), True, gs, bits)
    assert (y.float() - (y0.float() + y1.float())).abs().max() <= 2.0 ** -6 * y.float().abs().max()
    # M=1 equals the first row of the M=2 call (rows of x are independent; reductions are order-fixed)
    y_m1 = g.quantized_matmul(x[:1], qw, s, z, True, gs, bits, kernel="gemv")
    assert torch.equal(y_m1, y[:1])
    # the tensor-pipe skinny kernel agrees with the FMA-pipe GEMV to bf16 resolution, and with itself bit for bit
    ys = g.quantized_matmul(x, qw, s, z, True, gs, bits, kernel="skinny")
    assert (ys.float() - y.float()).abs().max() <= 2.0 ** -7 * y.float().abs().max()
    assert torch.equal(ys, g.quantized_matmul(x, qw, s, z, True, gs, bits, kernel="skinny"))
    assert torch.equal(ys[:1], g.quantized_matmul(x[:1], qw, s, z, True, gs, bits, kernel="skinny"))
    # so does the tensor-pipe decode kernel (auto dispatch at M <= 4), sampled rows against the oracle again
    for kern in MMV_KERNELS:
        ym = g.quantized_matmul(x, qw, s, z, True, gs, bits, kernel=kern)
        assert_close_to_truth(ym[:, torch.from_numpy(rows).to(cuda_device)], ref, kern + " sampled rows")
        assert (ym.float() - y.float()).abs().max() <= 2.0 ** -7 * y.float().abs().max()
        assert torch.equal(ym, g.quantized_matmul(x, qw, s, z, True, gs, bits, kernel=kern))  # run-to-run reproducible
        ym1 = g.quantized_matmul(x[:1], qw, s, z, True, gs, bits, kernel=kern)
        assert (ym1.float() - ym[:1].float()).abs().max() <= 2.0 ** -7 * y.float().abs().max()
    assert torch.equal(ym, g.quantized_matmul(x, qw, s, z, True, gs, bits))  # auto dispatch at M <= 4 = the integer kernel


def test_cuda_graph_capture(cuda_device):
    g = _ops()
    L = A.synth_layer(256, 1024, 4, 64, seed=21)
    d = layer_to_cuda(L, cuda_device)
    x = bf16_from_bits(A.synth_x(1, 1024, seed=22), cuda_device)
    eager = g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, 64, 4)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, 64, 4)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, 64, 4)
    x.copy_(bf16_from_bits(A.synth_x(1, 1024, seed=23), cuda_device))
    graph.replay()
    torch.cuda.synchronize()
    ref = g.quantized_matmul(x, d["qweight"], d["scales"], d["zeros"], True, 64, 4)
    assert torch.equal(out, ref) and not torch.equal(out, eager)


# ---------------------------------------------------------------------------------- grouped launch
class _Seg:
    """QuantizedLinear-like holder for quantized_matmul_grouped."""

    def __init__(self, d, bits, gs):
        self.qweight, self.scales, self.zeros = d["qweight"], d["scales"], d["zeros"]
        self.bias = d.get("bias")
        self.bits, self.group_size = bits, gs


@pytest.mark.parametrize("M", (1, 2, 4, 7))
@pytest.mark.parametrize("gs", (64, 128))
def test_qmm_grouped_matches_single_calls_and_oracle(cuda_device, M, gs):
    """q|k|v and gate|up as one gbxq_qmm_grouped call (layer-mix: different bits per segment, Qwen2 biases):
    bitwise equal to one gbxq_qmm call per segment, and within the path's tolerance of the oracle.
    M = 7 and the 3-bit segment exercise the per-segment fallback inside the same entry point."""
    g = _ops()
    from gbx_lm_b200 import ops

    K = 2048
    for combo in (((4, 512), (4, 128), (4, 128)), ((2, 1024), (4, 1024)), ((8, 96), (2, 300), (4, 1), (4, 149)),
                  ((4, 256), (3, 128)), ((4, 4096), (2, 4096)), ((2, 512), (2, 128), (6, 128)), ((3, 300), (6, 77))):
        segs, raw = [], []
        for i, (bits, N) in enumerate(combo):
            L = A.synth_layer(N, K, bits, gs, seed=7 * i + bits + N, with_bias=(i == 1))
            raw.append(L)
            segs.append(_Seg(layer_to_cuda(L, cuda_device), bits, gs))
        xb = A.synth_x(M, K, seed=5 + M)
        x = bf16_from_bits(xb, cuda_device)
        n0 = ops.launch_count()
        ys = g.quantized_matmul_grouped(x, segs)
        launches = ops.launch_count() - n0
        fusable = M <= 2  # every width shares one launch (3-/6-bit are realigned in registers); M >= 3: skinny kernel per segment
        # the per-segment fallback may tile M inside a segment (3-/6-bit GEMV: M tiles of 1/2), so only a lower bound there
        assert (launches == 1) if fusable else (launches >= len(combo)), (combo, M, launches)
        for sg, L, y, (bits, N) in zip(segs, raw, ys, combo):
            single = g.quantized_matmul(x, sg.qweight, sg.scales, sg.zeros, True, gs, bits, bias=sg.bias)
            assert y.shape == (M, N) and torch.equal(y, single), (combo, bits, N)
            ref = A.quantized_matmul(xb, L["qweight"], L["scales"], L["zeros"], gs, bits, "bf16", "f64", bias=L.get("bias"))
            assert_close_to_truth(y, ref, f"grouped b{bits} N{N} M{M}")


@pytest.mark.parametrize("bits,gs", [(4, 64), (2, 128), (8, 64), (3, 64)])
def test_qmm_grouped_tensor_core_launch(cuda_device, bits, gs):
    """Decode batches and prefill chunks of q|k|v / gate|up with one bit width: ONE launch of the TMEM-operand GEMM
    (gbxq_gemm_ts_grouped_sm100.cu) for all segments -- against the oracle, against one call per segment (fp32
    summation noise: the split-K plans differ), bitwise reproducible; mixed widths fall back to one call per segment."""
    g = _ops()
    from gbx_lm_b200 import ops

    K = 2048
    for M in (9, 40, 300):
        for combo in ((512, 128, 128), (1024, 1000), (130, 64, 3)):
            segs, raw = [], []
            for i, N in enumerate(combo):
                L = A.synth_layer(N, K, bits, gs, seed=11 * i + bits + N, with_bias=(i == 1))
                raw.append(L)
                segs.append(_Seg(layer_to_cuda(L, cuda_device), bits, gs))
            xb = A.synth_x(M, K, seed=5 + M)
            x = bf16_from_bits(xb, cuda_device)
            n0 = ops.launch_count()
            ys = g.quantized_matmul_grouped(x, segs)
            assert ops.launch_count() - n0 == 1, (combo, M)
            ys2 = g.quantized_matmul_grouped(x, segs)
            plain = []
            for sg in segs:  # the same segments without their bias
                c = _Seg({"qweight": sg.qweight, "scales": sg.scales, "zeros": sg.zeros}, bits, gs)
                plain.append(c)
            ys0 = g.quantized_matmul_grouped(x, plain)
            for sg, L, y, y2, y0, N in zip(segs, raw, ys, ys2, ys0, combo):
                ref = A.quantized_matmul(xb, L["qweight"], L["scales"], L["zeros"], gs, bits, "bf16", "f64")
                assert y.shape == (M, N) and torch.equal(y, y2)
                assert_close_to_truth(y0, ref, f"grouped gemm_ts b{bits} N{N} M{M}", 1e-2)
                # the bias is a second, separately rounded add on the rounded product (quantized_linear_gba.py:204-205):
                # checked exactly (against the truth two roundings can stack to 2 bf16 ulps)
                want = y0 if sg.bias is None else (y0.float() + sg.bias.float()).to(torch.bfloat16)
                assert torch.equal(y, want)
                single = g.quantized_matmul(x, sg.qweight, sg.scales, sg.zeros, True, gs, bits)
                assert (y0.float() - single.float()).abs().max() <= 2.0 ** -6 * single.float().abs().max()
    # mixed widths: per-segment launches, bitwise the single calls
    segs = [_Seg(layer_to_cuda(A.synth_layer(256, K, b, gs, seed=b), cuda_device), b, gs) for b in (bits, 8 if bits != 8 else 4)]
    x = bf16_from_bits(A.synth_x(20, K, seed=1), cuda_device)
    n0 = ops.launch_count()
    ys = g.quantized_matmul_grouped(x, segs)
    assert ops.launch_count() - n0 == 2
    for sg, y in zip(segs, ys):
        assert torch.equal(y, g.quantized_matmul(x, sg.qweight, sg.scales, sg.zeros, True, gs, sg.bits))


def test_qmm_grouped_validation(cuda_device):
    g = _ops()
    K = 256
    a = _Seg(layer_to_cuda(A.synth_layer(64, K, 4, 64, seed=1), cuda_device), 4, 64)
    b = _Seg(layer_to_cuda(A.synth_layer(64, 512, 4, 64, seed=2), cuda_device), 4, 64)
    x = bf16_from_bits(A.synth_x(1, K, seed=3), cuda_device)
    with pytest.raises(ValueError):
        g.quantized_matmul_grouped(x, [a, b])  # K mismatch
    with pytest.raises(ValueError):
        g.quantized_matmul_grouped(x, [a] * 5)  # too many segments
    assert g.quantized_matmul_grouped(x, []) == []


# ---------------------------------------------------------------------------------- chain launch (persistent kernel)
def _chain_layers(cuda_device, gs, spec):
    """spec: list of calls, each a list of (bits, N) segments; K of call i+1 = N of segment 0 of call i."""
    calls = []
    K = spec[0][0]
    for ci, segs in enumerate(spec[1:]):
        layers = []
        for si, (bits, N) in enumerate(segs):
            L = A.synth_layer(N, K, bits, gs, seed=100 * ci + 7 * si + bits, with_bias=(si == 1))
            layers.append(_Seg(layer_to_cuda(L, cuda_device), bits, gs))
        calls.append((K, layers))
        K = segs[0][1]
    return calls


@pytest.mark.parametrize("M", (1, 2, 4))
@pytest.mark.parametrize("gs", (64, 128))
def test_stream_chain_matches_stream_ordered_calls(cuda_device, M, gs):
    """gbxq_qmm_stream: a chain whose every call reads the y of the call before it (a true dependency, as o_proj on
    q|k|v and down_proj on gate|up) must be bitwise equal to issuing the calls one by one, launch after launch
    (counters reset in-kernel), eagerly and replayed from a CUDA graph."""
    g = _ops()
    from gbx_lm_b200 import ops

    K0 = 2048
    kbig = {1: 14336, 2: 8192, 4: 4096}[M]  # widest K the decode kernel takes at this M (stationary-fragment budget)
    spec = [(K0,), [(4, 4096), (2, 512), (8, 256)], [(4, 2048)], [(2, kbig), (4, kbig)], [(4, 1024), (4, 300)],
            [(8, 2048)], [(4, 1024), (4, 128), (4, 128)], [(2, 2048)]]
    calls = _chain_layers(cuda_device, gs, spec)
    x0 = bf16_from_bits(A.synth_x(M, K0, seed=40 + M), cuda_device)

    def sequential(x):
        outs = []
        for K, layers in calls:
            assert x.shape[1] == K
            # the chain runs the mmv8 body for every M <= 4; AUTO dispatch leaves it at M >= 3, so name the kernel
            # (grouped and single mmv8 launches are bitwise equal: test_qmm_grouped_matches_single_calls_and_oracle)
            ys = [g.quantized_matmul(x, l.qweight, l.scales, l.zeros, True, gs, l.bits, bias=l.bias, kernel="mmv8")
                  for l in layers]
            outs.append(ys)
            x = ys[0]
        return outs

    want = sequential(x0)
    chain = ops.StreamChain(M)
    xin = x0.clone()
    x, got = xin, []
    for K, layers in calls:
        ys = chain.add(x, layers)
        got.append(ys)
        x = ys[0]
    chain.finalize()
    n0 = ops.launch_count()
    chain.run()
    assert ops.launch_count() - n0 == 1
    torch.cuda.synchronize()
    assert not chain.timed_out()

    def check(tag):
        for ci, (w, h) in enumerate(zip(want, got)):
            for si, (a, b) in enumerate(zip(w, h)):
                assert torch.isfinite(b.float()).all(), (tag, ci, si)
                assert torch.equal(a, b), (tag, ci, si, (a.float() - b.float()).abs().max().item())

    check("eager")
    assert int(chain._counters.abs().sum().item()) == 0  # the kernel leaves its counters at zero
    for ys in got:
        for y in ys:
            y.zero_()
    for _ in range(3):
        chain.run()
    torch.cuda.synchronize()
    check("repeat")
    # new activations through a CUDA graph replay
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        chain.run()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        chain.run()
    x1 = bf16_from_bits(A.synth_x(M, K0, seed=77 + M), cuda_device)
    want = sequential(x1)
    xin.copy_(x1)
    graph.replay()
    graph.replay()
    torch.cuda.synchronize()
    check("graph")
    assert not chain.timed_out()


def test_stream_chain_against_oracle_and_validation(cuda_device):
    """First call of a chain against the fp64 truth of the oracle; unsupported chains are refused, not mis-run."""
    g = _ops()
    from gbx_lm_b200 import ops

    K, gs = 4096, 64
    raw = [A.synth_layer(N, K, bits, gs, seed=N + bits) for bits, N in ((4, 1024), (2, 768))]
    segs = [_Seg(layer_to_cuda(L, cuda_device), b, gs) for L, b in zip(raw, (4, 2))]
    xb = A.synth_x(1, K, seed=9)
    x = bf16_from_bits(xb, cuda_device)
    chain = ops.StreamChain(1)
    ys = chain.add(x, segs, dep=None)
    (y2,) = chain.add(x, [segs[0]], dep=None)
    chain.run()
    torch.cuda.synchronize()
    for L, y, b in zip(raw, ys, (4, 2)):
        ref = A.quantized_matmul(xb, L["qweight"], L["scales"], L["zeros"], gs, b, "bf16", "f64")
        assert_close_to_truth(y, ref, f"chain b{b}")
    assert torch.equal(y2, ys[0])
    bad = ops.StreamChain(1)
    L3 = A.synth_layer(64, K, 3, gs, seed=1)
    bad.add(x, [_Seg(layer_to_cuda(L3, cuda_device), 3, gs)])
    with pytest.raises(RuntimeError):
        bad.finalize()  # 3-bit rows are not served by the chain kernel: GBXQ_EUNSUPPORTED
