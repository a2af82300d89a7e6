"""GPU parity of the convolution hot path (SURVEY.md §8 rows a1-a11) through the C ABI (include/fcuda.h),
against the oracle restatement (oracle/feather_oracle.c) and outputs of the unmodified reference build stored under
tests/golden/.  Tolerances: 3xTF32 (default, fp32-equivalent) 2e-4 of max|ref| per layer — the reference's own
Winograd path is ~1e-5 from an fp64 convolution; plain TF32 is held to the north-star bar of 1e-3."""
import ctypes
from pathlib import Path

import numpy as np
import pytest

from conftest import digest, rel_err, sampled_rel_err

pytestmark = pytest.mark.gpu


# Split modes of the fp32-equivalent contraction (include/fcuda.h): 0 = 3xTF32 everywhere, 2 = the default (BF16x3 in the
# implicit GEMM, 3xTF32 in the TensorGEMM).  Both are held to the same 2e-4 bar.
@pytest.fixture(params=[0, 2], ids=["tf32x3", "fp32split"])
def mode(request):
    return request.param

# (name, oc, ic, h, w, k, stride, pad, group, bias, relu)
CASES = [
    ("config1_64x64_56", 64, 64, 56, 56, 3, 1, 1, 1, True, False),       # BASELINE.json configs[0]
    ("wino_nonsquare_relu", 64, 64, 57, 55, 3, 1, 1, 1, True, True),     # non-multiple-of-6, nBlocks%4 != 0
    ("wino_nobias_128", 128, 128, 28, 28, 3, 1, 1, 1, False, False),
    ("wino_pad0", 32, 16, 11, 13, 3, 1, 0, 1, True, False),
    ("wino_min_size", 8, 4, 9, 9, 3, 1, 1, 1, True, True),               # smallest Winograd-eligible input
    ("wino_oc_tail", 36, 20, 20, 20, 3, 1, 1, 1, True, False),           # OC, IC not multiples of 32
    ("im2col_oc62", 62, 64, 20, 20, 3, 1, 1, 1, True, False),            # OC%4 != 0 -> IM2COL
    ("im2col_small_hw", 64, 64, 7, 7, 3, 1, 1, 1, True, True),           # input_h <= 8 -> IM2COL
    ("im2col_1x1", 64, 256, 28, 28, 1, 1, 0, 1, False, False),
    ("im2col_1x1_s2", 128, 64, 28, 28, 1, 2, 0, 1, False, True),
    ("im2col_7x7_s2", 64, 3, 64, 64, 7, 2, 3, 1, True, False),           # K = 147 -> padded to 148
    ("im2col_3x3_ic3", 64, 3, 32, 32, 3, 1, 1, 1, True, True),           # VGG conv1_1 shape class (K = 27)
    ("im2col_3x3_s2", 32, 32, 17, 19, 3, 2, 1, 1, True, False),
    ("im2col_5x5", 24, 12, 15, 15, 5, 1, 2, 1, True, False),
    ("dw_s1", 64, 64, 28, 28, 3, 1, 1, 64, False, False),
    ("dw_s2_relu", 32, 32, 56, 56, 3, 2, 1, 32, False, True),
    ("dw_s1_wide", 16, 16, 40, 70, 3, 1, 1, 16, False, False),           # > 2 x-strips in the shuffle kernel
    ("dw_small_plane", 128, 128, 7, 7, 3, 1, 1, 128, False, False),      # one-warp-per-plane kernel
    ("dw_s2_odd", 24, 24, 15, 15, 3, 2, 1, 24, False, False),
    ("dw_14_bias_relu", 40, 40, 14, 14, 3, 1, 1, 40, True, True),        # plane kernel (MobileNet 14x14 stage)
    ("dw_14_s2", 40, 40, 14, 14, 3, 2, 1, 40, True, False),              # plane kernel, stride 2 -> 7x7
    ("dw_9_nopad", 12, 12, 9, 11, 3, 1, 0, 12, False, True),             # plane kernel without padding
    ("dw_cols_ragged", 20, 20, 11, 13, 3, 1, 1, 20, True, False),       # column-per-lane kernel, H != W, planes not a multiple of 2
    ("dw_5x5", 8, 8, 12, 12, 5, 1, 2, 8, False, False),
    ("dw_global", 32, 32, 7, 7, 7, 1, 0, 32, False, False),              # kernel == input: globalDwConv
]


def _data(oracle, case, batch, seed=0):
    name, oc, ic, h, w, k, s, pad, group, bias, relu = case
    p = oracle.ConvParam.make(oc, ic, h, w, k, stride=s, pad=pad, group=group, bias=bias, relu=relu)
    rng = np.random.default_rng(seed)
    x = rng.uniform(-0.5, 0.5, (batch, ic, h, w)).astype(np.float32)
    fan_in = (ic // group if group == 1 else 1) * k * k
    wt = (rng.standard_normal(p.weight_shape) * np.sqrt(2.0 / fan_in)).astype(np.float32)
    b = rng.uniform(-0.1, 0.1, p.output_channels).astype(np.float32) if bias else None
    return p, x, wt, b


def _gpu_conv(cuda, case, x, wt, b, algo=None):
    from feathercnn_b200 import booster
    name, oc, ic, h, w, k, s, pad, group, bias, relu = case
    p = booster.ConvParam.make(oc, ic, h, w, k, stride=s, pad=pad, group=group, bias=bias, relu=relu)
    xd = cuda.from_numpy(x).cuda()
    wd = cuda.from_numpy(wt).cuda()
    bd = cuda.from_numpy(b).cuda() if b is not None else None
    out, used = booster.conv_forward(p, xd, wd, bd, algo)
    cuda.cuda.synchronize()
    return out.cpu().numpy(), used


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("batch", [1, 3])
def test_conv_matches_oracle(cuda, oracle, restatement, case, batch):
    from feathercnn_b200 import booster
    booster.set_precision(booster.PRECISION_TF32X3)
    p, x, wt, b = _data(oracle, case, batch)
    got, used = _gpu_conv(cuda, case, x, wt, b)
    assert used == restatement.select_algo(p), "SelectAlgo must mirror avx/booster.cpp:283-310"
    for n in range(batch):
        want = restatement.conv(p, x[n], wt, b)
        assert rel_err(got[n], want) < 2e-4, (case[0], n)


# The unmodified reference segfaults on the smallest Winograd shape (IC=4, 2x2 tiles) — its AVX TensorGEMM
# assumes larger blocks — so that case is checked against the restatement only.
REF_CASES = [c for c in CASES[:14] if c[0] != "wino_min_size"]


@pytest.mark.parametrize("case", REF_CASES, ids=[c[0] for c in REF_CASES])
def test_conv_matches_reference_build(cuda, oracle, case):
    """Against a fixed sample of the reference's ConvBooster output (tests/golden/make_golden.py)."""
    from feathercnn_b200 import booster
    booster.set_precision(booster.PRECISION_TF32X3)
    gold = np.load(Path(__file__).resolve().parent / "golden" / "ref_gpu_conv.npz")
    p, x, wt, b = _data(oracle, case, 1, seed=7)
    assert digest(x, wt, b) == str(gold[case[0] + "/inputs"]), "inputs differ from those the stored outputs were made from"
    got, _ = _gpu_conv(cuda, case, x, wt, b)
    assert sampled_rel_err(got[0], gold, case[0]) < 2e-4, case[0]


@pytest.mark.parametrize("algo_name", ["NAIVE", "IM2COL", "SGECONV", "WINOGRADF63", "WINOGRADF23"])
def test_forced_algorithms_agree(cuda, oracle, restatement, algo_name, mode):
    """ForceSelectAlgo (avx/booster.cpp:313-317): every algorithm computes the same convolution."""
    from feathercnn_b200 import booster
    booster.set_precision(mode)
    case = ("forced", 48, 32, 21, 28, 3, 1, 1, 1, True, True)
    p, x, wt, b = _data(oracle, case, 2, seed=3)
    got, used = _gpu_conv(cuda, case, x, wt, b, algo=getattr(booster, algo_name))
    assert used == getattr(booster, algo_name)
    for n in range(2):
        want = restatement.conv(p, x[n], wt, b, f64=True)
        assert rel_err(got[n], want) < 2e-4, (algo_name, n)


def test_unsupported_algorithms_return_minus_one(cuda, oracle):
    from feathercnn_b200 import booster
    from feathercnn_b200._lib import fcuda
    p = booster.ConvParam.make(64, 64, 16, 16, 3, pad=1)
    s, k = ctypes.c_size_t(), ctypes.c_size_t()
    # unselected and crashing upstream, avx/booster.cpp:258,291-292
    assert fcuda().fcuda_conv_get_buffer_size(ctypes.byref(p), booster.WINOGRADF63FUSED, 1, ctypes.byref(s), ctypes.byref(k)) == -1
    # grouped (non-depthwise) convolution: -1 like upstream (avx/booster.cpp:304-308) for every algorithm but the grouped
    # implicit GEMM, this engine's extension (tests/test_gpu_ext.py)
    bad = booster.ConvParam.make(64, 64, 16, 16, 3, pad=1, group=4)
    assert fcuda().fcuda_conv_get_buffer_size(ctypes.byref(bad), booster.SGECONV, 1, ctypes.byref(s), ctypes.byref(k)) == 0
    for algo in (booster.IM2COL, booster.WINOGRADF63, booster.DEPTHWISE):
        assert fcuda().fcuda_conv_get_buffer_size(ctypes.byref(bad), algo, 1, ctypes.byref(s), ctypes.byref(k)) == -1
    pg = booster.ConvParam.make(64, 64, 16, 16, 3, pad=1, group=4)  # partial groups: avx/booster.cpp:304-308
    a = ctypes.c_int()
    assert fcuda().fcuda_conv_select_algo(ctypes.byref(pg), ctypes.byref(a)) == -1


SGECONV_CASES = [
    # oc, ic, h, w, k, stride, pad, bias, relu
    (64, 64, 56, 56, 3, 1, 1, True, True),      # VGG conv1_2 class (two boxes per row)
    (128, 64, 28, 28, 3, 1, 1, False, False),   # one 28-wide box per row, BN = 128
    (64, 256, 28, 28, 1, 1, 0, False, True),    # pointwise: addressed as one 784-long row
    (36, 20, 12, 17, 3, 1, 1, True, False),     # IC, OC not multiples of 32, odd width
    (16, 8, 5, 224, 3, 1, 1, True, True),       # 7 boxes per row, image wider than a tile
    (24, 12, 15, 20, 5, 1, 2, True, False),     # 5x5
    (32, 32, 9, 12, 3, 1, 0, True, False),      # no padding
    (200, 64, 14, 16, 1, 1, 0, True, False),    # OC > 128: two N tiles
    (64, 3, 64, 64, 7, 2, 3, True, False),      # ResNet conv1 class: 7x7 stride 2, IC = 3 (padded to 4)
    (32, 32, 17, 19, 3, 2, 1, True, True),      # 3x3 stride 2, odd sizes
    (128, 64, 28, 28, 1, 2, 0, False, False),   # strided pointwise (ResNet downsample)
    (16, 2048, 7, 7, 1, 1, 0, True, False),     # deep K (64 channel blocks), 49-pixel images
    (64, 64, 7, 7, 3, 1, 1, True, True),        # ResNet stage-5 3x3 class: W % 4 != 0 -> generic gather, flattened pixel boxes
    (160, 64, 14, 14, 1, 2, 0, False, True),    # strided pointwise onto 7x7 (flattened boxes, two N tiles)
    (32, 40, 9, 9, 3, 2, 1, True, False),       # table gather (IC % 32 != 0) + stride 2 + flattened boxes (5x5 output)
]


@pytest.mark.parametrize("geom", SGECONV_CASES)
@pytest.mark.parametrize("batch", [1, 3])
def test_sgeconv_implicit_gemm(cuda, oracle, restatement, geom, batch, mode):
    """FCUDA_SGECONV: implicit GEMM from NCHW (patches gathered inside the tcgen05 kernel), vs fp64 direct conv."""
    from feathercnn_b200 import booster
    booster.set_precision(mode)
    oc, ic, h, w, k, stride, pad, bias, relu = geom
    case = ("sgeconv", oc, ic, h, w, k, stride, pad, 1, bias, relu)
    p, x, wt, b = _data(oracle, case, batch, seed=13)
    got, used = _gpu_conv(cuda, case, x, wt, b, algo=booster.SGECONV)
    assert used == booster.SGECONV
    for n in range(batch):
        assert rel_err(got[n], restatement.conv(p, x[n], wt, b, f64=True)) < 2e-4, (geom, n)
    booster.set_precision(booster.PRECISION_TF32)
    try:
        got1, _ = _gpu_conv(cuda, case, x, wt, b, algo=booster.SGECONV)
    finally:
        booster.set_precision(booster.PRECISION_TF32X3)
    for n in range(batch):
        assert rel_err(got1[n], restatement.conv(p, x[n], wt, b, f64=True)) < 2e-3, (geom, n)


@pytest.mark.parametrize("algo_name,geom", [
    ("SGECONV", (64, 32, 14, 14, 1, 1, 0, True)),      # ResNet bottleneck exit: pointwise, fused in the epilogue
    ("SGECONV", (40, 24, 9, 13, 3, 1, 1, False)),      # OC tail (not a multiple of 32), no bias
    ("SGECONV", (160, 64, 7, 7, 1, 1, 0, True)),       # two N tiles
    ("WINOGRADF63", (32, 32, 12, 12, 3, 1, 1, True)),  # not SGECONV: convolution, then add_relu in place
    ("IM2COL", (16, 8, 10, 10, 3, 2, 1, True)),
])
@pytest.mark.parametrize("relu", [False, True])
def test_conv_forward_residual(cuda, oracle, restatement, algo_name, geom, relu, mode):
    """fcuda_conv_forward_residual == ConvLayer::Forward then EltwiseLayer::Forward (eltwise_layer.h:68-82)."""
    from feathercnn_b200 import booster
    booster.set_precision(mode)
    oc, ic, h, w, k, stride, pad, bias = geom
    case = ("residual", oc, ic, h, w, k, stride, pad, 1, bias, False)
    p, x, wt, b = _data(oracle, case, 2, seed=21)
    pp = booster.ConvParam.make(oc, ic, h, w, k, stride=stride, pad=pad, bias=bias)
    rng = np.random.default_rng(5)
    res = rng.uniform(-1, 1, (2, oc, pp.output_h, pp.output_w)).astype(np.float32)
    xd, wd = cuda.from_numpy(x).cuda(), cuda.from_numpy(wt).cuda()
    bd = cuda.from_numpy(b).cuda() if b is not None else None
    out, used = booster.conv_forward(pp, xd, wd, bd, getattr(booster, algo_name), residual=cuda.from_numpy(res).cuda(),
                                     relu_after_add=relu)
    cuda.cuda.synchronize()
    got = out.cpu().numpy()
    for n in range(2):
        want = restatement.conv(p, x[n], wt, b, f64=True) + res[n]
        if relu:
            want = np.maximum(want, 0)
        assert rel_err(got[n], want) < 2e-4, (algo_name, geom, n)


def test_plain_tf32_meets_north_star_bar_on_im2col(cuda, oracle, restatement):
    from feathercnn_b200 import booster
    case = CASES[8]
    p, x, wt, b = _data(oracle, case, 2, seed=5)
    booster.set_precision(booster.PRECISION_TF32)
    try:
        got, _ = _gpu_conv(cuda, case, x, wt, b)
    finally:
        booster.set_precision(booster.PRECISION_TF32X3)
    for n in range(2):
        assert rel_err(got[n], restatement.conv(p, x[n], wt, b)) < 1e-3


def test_l2_chunking_is_invisible(cuda, oracle, restatement):
    """Chunk size only changes how the intermediates are tiled through L2, never the result."""
    from feathercnn_b200 import booster
    case = ("chunk", 32, 32, 30, 30, 3, 1, 1, 1, True, False)
    p, x, wt, b = _data(oracle, case, 5, seed=9)
    outs = []
    from feathercnn_b200._lib import fcuda
    default = fcuda().fcuda_get_l2_chunk_bytes()
    for chunk in (default, 1 << 18, 0):  # default (one chunk), tiny (many chunks), unbounded
        booster.set_l2_chunk_bytes(chunk)
        try:
            for algo in (booster.WINOGRADF63, booster.IM2COL):
                got, _ = _gpu_conv(cuda, case, x, wt, b, algo=algo)
                outs.append(got)
        finally:
            booster.set_l2_chunk_bytes(default)
    for i in (2, 4):
        np.testing.assert_array_equal(outs[i], outs[0])      # Winograd, any chunking: bit-identical
        np.testing.assert_array_equal(outs[i + 1], outs[1])  # im2col, any chunking: bit-identical
    for n in range(5):
        assert rel_err(outs[0][n], restatement.conv(p, x[n], wt, b)) < 2e-4


def test_full_size_linearity_vgg_conv(cuda):
    """Size-independent property at a BASELINE-size layer (VGG conv3: 256->256 @56x56, batch 8):
    conv(a*x1 + x2) == a*conv(x1) + conv(x2) without bias."""
    from feathercnn_b200 import booster
    torch = cuda
    p = booster.ConvParam.make(256, 256, 56, 56, 3, pad=1, bias=False)
    g = torch.Generator(device="cuda").manual_seed(0)
    x1 = torch.rand((8, 256, 56, 56), device="cuda", generator=g) - 0.5
    x2 = torch.rand((8, 256, 56, 56), device="cuda", generator=g) - 0.5
    w = torch.randn((256, 256, 3, 3), device="cuda", generator=g) * 0.03
    y1, _ = booster.conv_forward(p, x1, w)
    y2, _ = booster.conv_forward(p, x2, w)
    y3, algo = booster.conv_forward(p, 2.0 * x1 + x2, w)
    assert algo == booster.WINOGRADF63
    want = (2.0 * y1 + y2)
    err = (y3 - want).abs().max().item() / want.abs().max().item()
    assert err < 2e-4


@pytest.mark.parametrize("algo_name,geom", [
    ("WINOGRADF63", (32, 16, 24, 24, 1)),      # whole tiles
    ("WINOGRADF63", (64, 32, 15, 13, 1)),      # odd output: clipped windows, partial tiles
    ("WINOGRADF63", (256, 128, 56, 56, 1)),    # VGG conv3-class, several tile rows
    ("WINOGRADF23", (16, 16, 10, 14, 1)),
    ("SGECONV", (64, 64, 64, 96, 1)),          # slab kernel, two issuers, several tiles per image
    ("SGECONV", (64, 32, 15, 12, 1)),          # odd output height, partial 4 x 32 patches (the slab TMA needs W % 4 == 0)
    ("SGECONV", (128, 64, 112, 112, 1)),       # BN = 128 (one issuer), VGG conv2_1 shape
    ("SGECONV", (32, 32, 30, 72, 0)),          # no padding
])
def test_conv_with_fused_max_pool(cuda, algo_name, geom, mode):
    """fcuda_conv_forward_pool == the convolution followed by PoolingLayer (2x2 / s2 / pad 0 / max, ceil mode,
    pooling_layer.h:38-91,129-130): max commutes exactly with the per-channel bias and with ReLU, so the fused result is
    bit-identical to pooling the unfused output."""
    from feathercnn_b200 import booster
    booster.set_precision(mode)
    oc, ic, h, w, pad = geom
    rng = np.random.default_rng(oc * 7 + h)
    x = cuda.from_numpy(rng.uniform(-0.5, 0.5, (3, ic, h, w)).astype(np.float32)).cuda()
    wt = cuda.from_numpy((rng.standard_normal((oc, ic, 3, 3)) * np.sqrt(2.0 / (ic * 9))).astype(np.float32)).cuda()
    b = cuda.from_numpy(rng.uniform(-0.1, 0.1, oc).astype(np.float32)).cuda()
    algo = getattr(booster, algo_name)
    for relu in (True, False):
        p = booster.ConvParam.make(oc, ic, h, w, 3, pad=pad, relu=relu)
        plain, _ = booster.conv_forward(p, x, wt, b, algo=algo)
        want = booster.pooling(plain, 0, 2, 2, 2, 2, 0, 0, 0, 0)
        got, _ = booster.conv_forward(p, x, wt, b, algo=algo, pool=True)
        cuda.cuda.synchronize()
        assert got.shape == want.shape
        np.testing.assert_array_equal(got.cpu().numpy(), want.cpu().numpy())
    # algorithms that cannot pool in their epilogue say so
    p = booster.ConvParam.make(oc, ic, h, w, 3, pad=pad)
    with pytest.raises(booster.FcudaError) as e:
        booster.conv_forward(p, x, wt, b, algo=booster.IM2COL, pool=True)
    assert e.value.code == -200


def test_fused_pool_is_refused_where_the_slab_kernel_does_not_apply(cuda):
    """SGECONV pools only in its 3x3 / stride-1 slab kernel (IC % 32 == 0, rows of whole 16-byte units for the TMA)."""
    from feathercnn_b200 import booster
    from feathercnn_b200._lib import fcuda
    ok = booster.ConvParam.make(64, 64, 16, 16, 3, pad=1)
    assert fcuda().fcuda_conv_can_pool(ctypes.byref(ok), booster.SGECONV) == 1
    assert fcuda().fcuda_conv_can_pool(ctypes.byref(ok), booster.WINOGRADF63) == 1
    assert fcuda().fcuda_conv_can_pool(ctypes.byref(ok), booster.IM2COL) == 0
    for bad in (booster.ConvParam.make(64, 64, 16, 13, 3, pad=1),   # W % 4 != 0
                booster.ConvParam.make(64, 48, 16, 16, 3, pad=1),   # IC % 32 != 0
                booster.ConvParam.make(64, 64, 16, 16, 3, pad=1, stride=2),
                booster.ConvParam.make(64, 64, 16, 16, 1)):
        assert fcuda().fcuda_conv_can_pool(ctypes.byref(bad), booster.SGECONV) == 0
