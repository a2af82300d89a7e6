"""Generates the committed golden fixtures from the UNMODIFIED reference build (oracle/_ref, compiled by
oracle/Makefile from the FeatherCNN sources at its REF):  python tests/golden/make_golden.py

The reference ships no golden vectors of its own (SURVEY.md §4), so these are outputs of the reference itself:
  conv_cases.npz   ConvBooster::Forward outputs for small layers covering every SelectAlgo branch
  mini_net.npz     every blob of feather::Net::Forward on the "mini" model (all layer types), seed-fixed input
Inputs and weights are stored too, so the fixtures do not depend on NumPy's RNG staying stable.

The tests that compare with the reference on larger data regenerate their seeded inputs and read what the reference
computed from them here; a digest of those inputs is stored beside it, so a changed input fails loudly:
  ref_conv_sweep.npz   test_oracle SWEEP: ConvBooster::Forward (SelectAlgo and NAIVE), fixed samples (conftest.sample_of)
  ref_mini_seed3.npz   test_oracle: every blob of feather::Net::Forward on modelgen.mini(seed=3), fixed samples
  ref_from_pixels.json test_oracle: sha256 of ncnn::Mat::from_pixels[_resize] outputs (a bit-exact comparison)
  ref_gpu_conv.npz     test_gpu_conv REF_CASES: ConvBooster::Forward, fixed samples
"""
import json
import sys
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from feathercnn_b200.tools import modelgen  # noqa: E402
from oracle import oracle as O  # noqa: E402

# name, oc, ic, h, w, k, stride, pad, group, bias, relu
CONV_CASES = [
    ("wino_16x16_12", 16, 16, 12, 12, 3, 1, 1, 1, True, False),
    ("wino_ragged_relu", 8, 12, 13, 10, 3, 1, 1, 1, True, True),
    ("im2col_1x1", 12, 16, 9, 9, 1, 1, 0, 1, False, False),
    ("im2col_7x7_s2", 8, 3, 20, 20, 7, 2, 3, 1, True, False),
    ("im2col_small_hw", 8, 8, 7, 7, 3, 1, 1, 1, True, True),
    ("im2col_oc_not4", 6, 8, 12, 12, 3, 1, 1, 1, True, False),
    ("dw_s1", 8, 8, 10, 10, 3, 1, 1, 8, False, False),
    ("dw_s2_relu", 8, 8, 11, 11, 3, 2, 1, 8, False, True),
    ("dw_global", 8, 8, 5, 5, 5, 1, 0, 8, False, False),
]


def main():
    out = Path(__file__).resolve().parent
    O.build(ref=True)
    ref = O.Reference()
    rng = np.random.default_rng(20260922)
    conv = {}
    for name, oc, ic, h, w, k, s, pad, group, bias, relu in CONV_CASES:
        p = O.ConvParam.make(oc, ic, h, w, k, stride=s, pad=pad, group=group, bias=bias, relu=relu)
        x = rng.uniform(-0.5, 0.5, (ic, h, w)).astype(np.float32)
        fan_in = (ic if group == 1 else 1) * k * k
        wt = (rng.standard_normal(p.weight_shape) * np.sqrt(2.0 / fan_in)).astype(np.float32)
        b = rng.uniform(-0.1, 0.1, p.output_channels).astype(np.float32)
        y = ref.conv(p, x, wt, b if bias else None)
        conv[name + "/x"], conv[name + "/w"], conv[name + "/b"], conv[name + "/y"] = x, wt, b, y
        conv[name + "/geom"] = np.array([oc, ic, h, w, k, s, pad, group, int(bias), int(relu)], np.int32)
    np.savez_compressed(out / "conv_cases.npz", **conv)

    m = modelgen.mini(seed=0, size=20, ch=8)
    param, binf = m.save(out / "mini")
    x = modelgen.synthetic_input(m.shape["data"], 0)
    net = O.ReferenceNet(param, binf)
    net.forward(x)
    blobs = {"input": x}
    for b in sorted(m.blobs):
        blobs["blob/" + b] = net.extract(b)
    np.savez_compressed(out / "mini_net.npz", **blobs)
    print("wrote", out / "conv_cases.npz", out / "mini_net.npz", out / "mini.param", out / "mini.bin")
    reference_samples(out, ref)


def _put(d: dict, key: str, a) -> None:
    from conftest import sample_of
    for k, v in sample_of(a).items():
        d[f"{key}/{k}"] = v


def reference_samples(out: Path, ref) -> None:
    import test_gpu_conv
    import test_oracle
    from conftest import digest

    d = {}
    for i, geom in enumerate(test_oracle.SWEEP):
        p, x, w, b = test_oracle.sweep_data(O, geom)
        d[f"{i}/inputs"] = np.array(digest(x, w, b))
        _put(d, f"{i}/ref", ref.conv(p, x, w, b))
        if p.group == 1:
            _put(d, f"{i}/naive", ref.conv(p, x, w, b, algo=O.ALGO_NAIVE))
    np.savez_compressed(out / "ref_conv_sweep.npz", **d)

    with tempfile.TemporaryDirectory() as tmp:
        m, param, binf, x = test_oracle.mini3(Path(tmp))
        d = {"inputs": np.array(digest(x, np.frombuffer(Path(param).read_bytes(), np.uint8), np.fromfile(binf, np.uint8)))}
        net = O.ReferenceNet(param, binf)
        net.forward(x)
        for b in sorted(m.blobs):
            _put(d, b, net.extract(b))
        del net
    np.savez_compressed(out / "ref_mini_seed3.npz", **d)

    cases = []
    for h, w, tw, th, t, img in test_oracle.pixel_cases():
        want = ref.from_pixels(img, t, tw, th)
        cases.append({"h": h, "w": w, "tw": tw, "th": th, "type": t, "image": digest(img), "shape": list(want.shape),
                      "output": digest(want)})
    unknown = ref.from_pixels(np.zeros((4, 4, 3), np.uint8), 3)
    (out / "ref_from_pixels.json").write_text(json.dumps({"cases": cases, "unknown_type": unknown}) + "\n")

    d = {}
    for case in test_gpu_conv.REF_CASES:
        p, x, wt, b = test_gpu_conv._data(O, case, 1, seed=7)
        d[case[0] + "/inputs"] = np.array(digest(x, wt, b))
        _put(d, case[0], ref.conv(p, x[0], wt, b))
    np.savez_compressed(out / "ref_gpu_conv.npz", **d)
    print("wrote", *(out / f for f in ("ref_conv_sweep.npz", "ref_mini_seed3.npz", "ref_from_pixels.json", "ref_gpu_conv.npz")))


if __name__ == "__main__":
    main()
