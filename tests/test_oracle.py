"""Pins the parity oracle (CPU only).

1. the C restatement (oracle/feather_oracle.c) and the NumPy net interpreter reproduce the committed golden
   fixtures, which are outputs of the UNMODIFIED reference (tests/golden/make_golden.py);
2. the restatement also agrees with the reference's outputs over the shape sweep used by the GPU tests, the
   reference's Forward of a second net, and its pixel staging (stored from the unmodified reference by
   tests/golden/make_golden.py: fixed samples of the float outputs, digests of the bit-exact ones);
3. both agree with an independent fp64 direct convolution, so an oracle bug cannot silently become the spec.
"""
from pathlib import Path

import numpy as np
import pytest

from conftest import digest, rel_err, sampled_rel_err

GOLD = Path(__file__).resolve().parent / "golden"


def _param(oracle, geom):
    oc, ic, h, w, k, s, pad, group, bias, relu = [int(v) for v in geom]
    return oracle.ConvParam.make(oc, ic, h, w, k, stride=s, pad=pad, group=group, bias=bool(bias), relu=bool(relu))


def test_restatement_reproduces_golden_conv_outputs(oracle, restatement):
    z = np.load(GOLD / "conv_cases.npz")
    names = sorted({k.split("/")[0] for k in z.files})
    assert len(names) >= 9
    for name in names:
        p = _param(oracle, z[name + "/geom"])
        b = z[name + "/b"] if p.bias_term else None
        got = restatement.conv(p, z[name + "/x"], z[name + "/w"], b)
        # Winograd: different fp32 summation order than the AVX kernels (~1e-5); direct paths ~1e-7
        tol = 5e-5 if restatement.select_algo(p) == oracle.ALGO_WINOGRADF63 else 2e-6
        assert rel_err(got, z[name + "/y"]) < tol, name


def test_select_algo_branches_in_golden_set(oracle, restatement):
    z = np.load(GOLD / "conv_cases.npz")
    algos = {restatement.select_algo(_param(oracle, z[k])) for k in z.files if k.endswith("/geom")}
    assert algos == {oracle.ALGO_WINOGRADF63, oracle.ALGO_IM2COL, oracle.ALGO_DEPTHWISE}


def test_net_interpreter_reproduces_golden_blobs(oracle):
    z = np.load(GOLD / "mini_net.npz")
    net = oracle.OracleNet(GOLD / "mini.param", GOLD / "mini.bin")
    net.forward(z["input"])
    blobs = [k[5:] for k in z.files if k.startswith("blob/")]
    assert len(blobs) >= 25
    for b in blobs:
        assert rel_err(net.extract(b), z["blob/" + b]) < 5e-5, b


def test_golden_model_files_match_generator():
    """The committed mini.param/.bin are what feathercnn_b200.tools.modelgen.mini(seed=0, size=20, ch=8) writes."""
    from feathercnn_b200.tools import modelgen
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        param, binf = modelgen.mini(seed=0, size=20, ch=8).save(Path(d) / "mini")
        assert Path(param).read_text() == (GOLD / "mini.param").read_text()
        assert Path(binf).read_bytes() == (GOLD / "mini.bin").read_bytes()


SWEEP = [
    # oc, ic, h, w, k, stride, pad, group, bias, relu
    (64, 64, 56, 56, 3, 1, 1, 1, True, False),
    (64, 64, 57, 55, 3, 1, 1, 1, True, True),
    (32, 16, 11, 13, 3, 1, 0, 1, True, False),
    (36, 20, 20, 20, 3, 1, 1, 1, True, False),
    (62, 64, 20, 20, 3, 1, 1, 1, True, False),
    (64, 64, 7, 7, 3, 1, 1, 1, True, True),
    (64, 256, 28, 28, 1, 1, 0, 1, False, False),
    (64, 3, 64, 64, 7, 2, 3, 1, True, False),
    (32, 32, 17, 19, 3, 2, 1, 1, True, False),
    (64, 64, 28, 28, 3, 1, 1, 64, False, False),
    (32, 32, 56, 56, 3, 2, 1, 32, False, True),
    (32, 32, 7, 7, 7, 1, 0, 32, False, False),
]


def sweep_data(oracle, geom):
    p = _param(oracle, geom)
    rng = np.random.default_rng(11)
    x = rng.uniform(-0.5, 0.5, (p.input_channels, p.input_h, p.input_w)).astype(np.float32)
    w = (rng.standard_normal(p.weight_shape) * 0.05).astype(np.float32)
    b = rng.uniform(-0.1, 0.1, p.output_channels).astype(np.float32) if p.bias_term else None
    return p, x, w, b


@pytest.mark.parametrize("geom", SWEEP)
def test_restatement_vs_live_reference_and_fp64(oracle, restatement, geom):
    """The restatement against the reference's ConvBooster output on the sweep, read from tests/golden/ref_conv_sweep.npz
    (a fixed sample of each output, stored by make_golden.py), and against the fp64 direct convolution in full; the
    reference's own NAIVE path, stored the same way, against fp64."""
    gold = np.load(GOLD / "ref_conv_sweep.npz")
    key = str(SWEEP.index(geom))
    p, x, w, b = sweep_data(oracle, geom)
    assert digest(x, w, b) == str(gold[key + "/inputs"]), "inputs differ from those the stored outputs were made from"
    got = restatement.conv(p, x, w, b)
    assert sampled_rel_err(got, gold, key + "/ref") < 5e-5
    if p.group == 1:
        f64 = restatement.conv(p, x, w, b, f64=True)
        assert sampled_rel_err(f64, gold, key + "/ref") < 5e-5 and rel_err(got, f64) < 5e-5
        if not p.activation:  # the authors' own oracle, avx/booster.cpp:28-61; NAIVE_Forward ignores the activation field
            assert sampled_rel_err(f64, gold, key + "/naive") < 5e-6


def mini3(tmp_path):
    """modelgen.mini(seed=3) and its synthetic image 5: the second net the interpreter is checked on."""
    from feathercnn_b200.tools import modelgen
    m = modelgen.mini(seed=3)
    param, binf = m.save(tmp_path / "mini")
    return m, param, binf, modelgen.synthetic_input(m.shape["data"], 5)


def test_net_interpreter_vs_live_reference_net(oracle, tmp_path):
    """Every blob of the interpreter's Forward of modelgen.mini(seed=3) against the reference's feather::Net::Forward,
    read from tests/golden/ref_mini_seed3.npz (a fixed sample of each blob, stored by make_golden.py)."""
    gold = np.load(GOLD / "ref_mini_seed3.npz")
    m, param, binf, x = mini3(tmp_path)
    assert digest(x, np.frombuffer(Path(param).read_bytes(), np.uint8), np.fromfile(binf, np.uint8)) == str(gold["inputs"])
    on = oracle.OracleNet(param, binf)
    on.forward(x)
    for b in sorted(m.blobs):
        assert sampled_rel_err(on.extract(b), gold, b) < 5e-5, b


def test_pooling_quirks(restatement):
    """ceil-mode output size (pooling_layer.h:129-130) and the double pad subtraction (:56,:67)."""
    assert restatement.lib.oracle_pool_out_dim(112, 0, 0, 3, 2) == 56
    assert restatement.lib.oracle_pool_out_dim(224, 0, 0, 2, 2) == 112
    x = np.arange(16, dtype=np.float32).reshape(1, 4, 4)
    # pad 1/1, k=3, s=2: window of output 0 starts at -2 (not -1) => covers only row/col 0
    out = restatement.pooling(x, 0, 3, 3, 2, 2, 1, 1, 1, 1, False)
    assert out.shape == (1, 3, 3) or out.shape == (1, 2, 2)
    assert out[0, 0, 0] == x[0, 0, 0]


PIXEL_TYPES = [(1, 3), (2, 3), (4, 1), (8, 4), (1 | (2 << 16), 3), (2 | (1 << 16), 3), (1 | (4 << 16), 3), (2 | (4 << 16), 3),
               (4 | (1 << 16), 1), (4 | (2 << 16), 1), (8 | (1 << 16), 4), (8 | (2 << 16), 4), (8 | (4 << 16), 4)]


PIXEL_SIZES = [(32, 48, 24, 24), (37, 53, 224, 224), (64, 64, 64, 64), (240, 320, 224, 224), (17, 9, 40, 31), (2, 2, 5, 7)]


def pixel_cases():
    """(h, w, tw, th, type, image) in the order the stored reference digests were made."""
    rng = np.random.default_rng(0)
    for (h, w, tw, th) in PIXEL_SIZES:
        for t, c in PIXEL_TYPES:
            yield h, w, tw, th, t, rng.integers(0, 256, (h, w, c), dtype=np.uint8)


def test_pixel_staging_restatement_is_bit_exact_with_the_reference(oracle):
    """Input staging (SURVEY.md §8f rank 3): the NumPy restatement of ncnn::Mat::from_pixels / from_pixels_resize
    (mat_pixel.cpp:1329-1410, mat_pixel_resize.cpp:26-278 — u8 fixed-point bilinear, byte work: bit-exact bar) against the
    unmodified reference, every pixel type, up- and down-scaling, degenerate 2x2 sources."""
    import json
    gold = json.loads((GOLD / "ref_from_pixels.json").read_text())
    cases = list(pixel_cases())
    assert len(cases) == len(gold["cases"]) == len(PIXEL_SIZES) * len(PIXEL_TYPES)
    for (h, w, tw, th, t, img), want in zip(cases, gold["cases"]):
        what = f"type {t:#x} {w}x{h}->{tw}x{th}"
        assert digest(img) == want["image"], what + ": input differs from the one the stored output was made from"
        got = oracle.from_pixels(img, t, tw, th)
        assert got is not None and list(got.shape) == want["shape"], what
        assert digest(got) == want["output"], what
    assert oracle.from_pixels(np.zeros((4, 4, 3), np.uint8), 3) is None          # unknown type: empty Mat upstream
    assert gold["unknown_type"] is None
