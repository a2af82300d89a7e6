"""TEST INFRASTRUCTURE ONLY — Python face of the parity oracle.

Two CPU implementations of the reference's conv/dense hot path, behind one interface:

* ``Restatement``  — oracle/feather_oracle.c (plain-C restatement, built into oracle/_build/liboracle.so)
  plus a NumPy interpreter for whole ``.param/.bin`` nets (``OracleNet``) that follows
  /root/reference/src/net.cpp:68-334 layer by layer.
* ``Reference``    — the UNMODIFIED reference compiled from /root/reference into
  oracle/_ref/libfeather_ref.so (oracle/Makefile + oracle/ref_shim.cpp).

Only tests/, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs may import this module.
The product package (feathercnn_b200/) never does.
"""
from __future__ import annotations

import ctypes
import os
import struct
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_ORACLE_SO = _HERE / "_build" / "liboracle.so"
_REF_SO = _HERE / "_ref" / "libfeather_ref.so"
_REF_CUDA_SO = _HERE / "_ref" / "libfeather_ref_cuda.so"  # the reference host on libfcuda.so (tests/integration/cuda_booster.cpp)

_f32p = ctypes.POINTER(ctypes.c_float)


def _fp(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_f32p)


class ConvParam(ctypes.Structure):
    """Mirror of OracleConvParam / booster::ConvParam (booster.h:59-77)."""

    _fields_ = [(n, ctypes.c_int) for n in (
        "output_channels input_channels input_h input_w kernel_h kernel_w output_h output_w "
        "stride_h stride_w pad_left pad_bottom pad_right pad_top group bias_term activation").split()]

    @classmethod
    def make(cls, oc, ic, h, w, kh, kw=None, stride=1, pad=0, group=1, bias=True, relu=False, stride_w=None):
        kw = kh if kw is None else kw
        sw = stride if stride_w is None else stride_w
        p = cls(oc, ic, h, w, kh, kw, 0, 0, stride, sw, pad, pad, pad, pad, group, int(bias), int(relu))
        restatement().lib.oracle_assign_output_dim(ctypes.byref(p))
        return p

    def as_ref_ints(self):
        return (ctypes.c_int * 15)(self.output_channels, self.input_channels, self.input_h, self.input_w,
                                   self.kernel_h, self.kernel_w, self.stride_h, self.stride_w, self.pad_left,
                                   self.pad_bottom, self.pad_right, self.pad_top, self.group, self.bias_term,
                                   self.activation)

    @property
    def weight_shape(self):
        if self.group == self.input_channels and self.group > 1:
            return (self.input_channels, 1, self.kernel_h, self.kernel_w)
        return (self.output_channels, self.input_channels, self.kernel_h, self.kernel_w)

    @property
    def out_shape(self):
        return (self.output_channels, self.output_h, self.output_w)


ALGO_NAIVE, ALGO_IM2COL, ALGO_SGECONV, ALGO_DEPTHWISE, ALGO_WINOGRADF63, ALGO_WINOGRADF63FUSED, ALGO_WINOGRADF23 = range(7)


def build(ref: bool = True) -> None:
    """Compile the oracle (and oracle/_ref, when oracle/Makefile finds the reference sources)."""
    subprocess.run(["make", "-C", str(_HERE), "oracle"], check=True, stdout=subprocess.DEVNULL)
    if ref:
        subprocess.run(["make", "-C", str(_HERE), "ref", "-j8"], check=True, stdout=subprocess.DEVNULL)


class Restatement:
    def __init__(self):
        if not _ORACLE_SO.exists():
            build(ref=False)
        self.lib = ctypes.CDLL(str(_ORACLE_SO))
        self.lib.oracle_pool_out_dim.restype = ctypes.c_int

    # ---- convolution -------------------------------------------------------------------------
    def select_algo(self, p: ConvParam) -> int:
        return self.lib.oracle_select_algo(ctypes.byref(p))

    def conv(self, p: ConvParam, x, w, b=None, algo: int | None = None, f64: bool = False):
        x = np.ascontiguousarray(x, np.float32)
        w = np.ascontiguousarray(w, np.float32)
        bias = np.ascontiguousarray(b, np.float32) if b is not None else None
        out = np.zeros(p.out_shape, np.float32)
        bp = _fp(bias) if bias is not None else None
        if f64:
            self.lib.oracle_conv_direct(ctypes.byref(p), _fp(x), _fp(w), bp, _fp(out), 1)
        elif algo is None:
            rc = self.lib.oracle_conv_forward(ctypes.byref(p), _fp(x), _fp(w), bp, _fp(out))
            if rc < 0:
                raise ValueError("oracle: unsupported conv (partial groups)")
        elif algo == ALGO_WINOGRADF63:
            self.lib.oracle_conv_winograd_f63(ctypes.byref(p), _fp(x), _fp(w), bp, _fp(out))
        elif algo == ALGO_DEPTHWISE:
            self.lib.oracle_conv_depthwise(ctypes.byref(p), _fp(x), _fp(w), bp, _fp(out))
        else:
            self.lib.oracle_conv_direct(ctypes.byref(p), _fp(x), _fp(w), bp, _fp(out), 0)
        return out

    # ---- other layers ------------------------------------------------------------------------
    def pooling(self, x, type_, kh, kw, sh, sw, pl, pr, pt, pb, global_pooling):
        x = np.ascontiguousarray(x, np.float32)
        c, h, w = x.shape
        if global_pooling:
            oh = ow = 1
        else:
            oh = self.lib.oracle_pool_out_dim(h, pt, pb, kh, sh)
            ow = self.lib.oracle_pool_out_dim(w, pl, pr, kw, sw)
        out = np.zeros((c, oh, ow), np.float32)
        self.lib.oracle_pooling(_fp(x), c, h, w, type_, kh, kw, sh, sw, pl, pr, pt, pb, int(global_pooling), _fp(out))
        return out

    def inner_product(self, x, w, b, relu=False):
        x = np.ascontiguousarray(x, np.float32).reshape(-1)
        w = np.ascontiguousarray(w, np.float32)
        out = np.zeros(w.shape[0], np.float32)
        bias = np.ascontiguousarray(b, np.float32) if b is not None else None
        self.lib.oracle_inner_product(_fp(x), _fp(w), _fp(bias) if bias is not None else None, x.size, w.shape[0],
                                      int(relu), _fp(out))
        return out

    def batchnorm(self, x, slope, mean, var, bias, eps):
        x = np.ascontiguousarray(x, np.float32)
        out = np.empty_like(x)
        c = x.shape[0]
        args = [np.ascontiguousarray(a, np.float32) for a in (slope, mean, var, bias)]
        self.lib.oracle_batchnorm(_fp(x), c, x.size // c, *[_fp(a) for a in args], ctypes.c_float(eps), _fp(out))
        return out

    def scale(self, x, scale, bias):
        x = np.ascontiguousarray(x, np.float32)
        out = np.empty_like(x)
        c = x.shape[0]
        s = np.ascontiguousarray(scale, np.float32)
        b = np.ascontiguousarray(bias, np.float32) if bias is not None else None
        self.lib.oracle_scale(_fp(x), c, x.size // c, _fp(s), _fp(b) if b is not None else None, _fp(out))
        return out

    def eltwise_add(self, a, b, relu=False):
        a = np.ascontiguousarray(a, np.float32)
        b = np.ascontiguousarray(b, np.float32)
        out = np.empty_like(a)
        self.lib.oracle_eltwise_add(_fp(a), _fp(b), ctypes.c_long(a.size), int(relu), _fp(out))
        return out

    def relu(self, x):
        x = np.ascontiguousarray(x, np.float32)
        out = np.empty_like(x)
        self.lib.oracle_relu(_fp(x), ctypes.c_long(x.size), _fp(out))
        return out

    def softmax(self, x):
        x = np.ascontiguousarray(x, np.float32)
        out = np.empty_like(x)
        self.lib.oracle_softmax(_fp(x), ctypes.c_long(x.size), _fp(out))
        return out

    def dropout(self, x, scale):
        x = np.ascontiguousarray(x, np.float32)
        out = np.empty_like(x)
        self.lib.oracle_dropout(_fp(x), ctypes.c_long(x.size), ctypes.c_float(scale), _fp(out))
        return out


_restatement = None


def restatement() -> Restatement:
    global _restatement
    if _restatement is None:
        _restatement = Restatement()
    return _restatement


def reference_available() -> bool:
    return _REF_SO.exists()


def reference_cuda_available() -> bool:
    return _REF_CUDA_SO.exists()


def reference_on_cuda() -> "Reference":
    """The unmodified reference host (feather::Net, ConvLayer, ...) with tests/integration/cuda_booster.cpp in place of
    src/booster/avx/booster.cpp: its ConvBooster function table points into libfcuda.so (INTEGRATION.md §1, compiled)."""
    return Reference(_REF_CUDA_SO)


class Reference:
    """The unmodified reference build (oracle/_ref)."""

    def __init__(self, so_path: Path | None = None):
        so_path = so_path or _REF_SO
        if not so_path.exists():
            raise FileNotFoundError(f"{so_path} missing: run `make -C oracle ref ref_cuda` where /root/reference exists")
        self.lib = ctypes.CDLL(str(so_path), mode=ctypes.RTLD_LOCAL)
        self.lib.ref_net_create.restype = ctypes.c_void_p
        self.lib.ref_net_time_forward.restype = ctypes.c_double
        if hasattr(self.lib, "ref_modelbin_load_mem"):
            self.lib.ref_modelbin_load_mem.restype = ctypes.c_long

    def modelbin_load_mem(self, blob: bytes, w: int, type_: int):
        """ncnn::ModelBinFromMemory::load of the reference (modelbin.cpp:204-293) -> (floats or None, bytes consumed)."""
        out = np.zeros(max(w, 1), np.float32)
        buf = ctypes.create_string_buffer(blob + b"\0" * 64, len(blob) + 64)
        n = self.lib.ref_modelbin_load_mem(ctypes.cast(buf, ctypes.POINTER(ctypes.c_ubyte)), w, type_, _fp(out))
        return (None, -1) if n < 0 else (out[:w].copy(), int(n))

    def from_pixels(self, pixels: np.ndarray, type_: int, target_w: int = 0, target_h: int = 0):
        """ncnn::Mat::from_pixels / from_pixels_resize of the reference on one (h, w[, c]) uint8 image -> (C, th, tw) or None."""
        pixels = np.ascontiguousarray(pixels, np.uint8)
        h, w = pixels.shape[:2]
        tw, th = target_w or w, target_h or h
        out = np.zeros((4, th, tw), np.float32)
        c = self.lib.ref_from_pixels(pixels.ctypes.data_as(ctypes.POINTER(ctypes.c_ubyte)), type_, w, h, tw, th, _fp(out))
        return None if c < 0 else out[:c].copy()

    def conv(self, p: ConvParam, x, w, b=None, algo: int = -1, repeat: int = 1):
        x = np.ascontiguousarray(x, np.float32)
        w = np.ascontiguousarray(w, np.float32)
        bias = np.ascontiguousarray(b if b is not None else np.zeros(p.output_channels), np.float32)
        out = np.zeros(p.out_shape, np.float32)
        dims = (ctypes.c_int * 3)()
        sec = ctypes.c_double(0)
        rc = self.lib.ref_conv_forward(p.as_ref_ints(), algo, _fp(x), _fp(w), _fp(bias), _fp(out), dims, repeat,
                                       ctypes.byref(sec))
        if rc != 0:
            raise RuntimeError(f"reference ConvBooster returned {rc}")
        assert tuple(dims) == p.out_shape, (tuple(dims), p.out_shape)
        return (out, sec.value) if repeat > 1 else out


class ReferenceNet:
    """feather::Net of the unmodified reference (LoadParam/LoadWeights/FeedInput/Forward/Extract)."""

    def __init__(self, param_path: str, bin_path: str, ref: "Reference | None" = None):
        self.ref = ref or Reference()
        self.h = ctypes.c_void_p(self.ref.lib.ref_net_create())
        rc = self.ref.lib.ref_net_load(self.h, str(param_path).encode(), str(bin_path).encode())
        if rc != 0:
            raise RuntimeError(f"reference Net load failed: {rc}")

    def forward(self, x: np.ndarray, input_name: str = "data"):
        x = np.ascontiguousarray(x, np.float32)
        c, h, w = x.shape
        rc = self.ref.lib.ref_net_forward(self.h, input_name.encode(), _fp(x), c, h, w)
        if rc != 0:
            raise RuntimeError(f"reference Net forward failed: {rc}")

    def extract(self, blob: str) -> np.ndarray:
        ptr = _f32p()
        n, c, h, w = (ctypes.c_int() for _ in range(4))
        rc = self.ref.lib.ref_net_extract(self.h, blob.encode(), ctypes.byref(ptr), ctypes.byref(n), ctypes.byref(c),
                                          ctypes.byref(h), ctypes.byref(w))
        if rc != 0:
            raise KeyError(blob)
        shape = (c.value, h.value, w.value)
        return np.ctypeslib.as_array(ptr, shape=(int(np.prod(shape)),)).reshape(shape).copy()

    def time_forward(self, x: np.ndarray, iters: int, input_name: str = "data") -> float:
        x = np.ascontiguousarray(x, np.float32)
        c, h, w = x.shape
        return self.ref.lib.ref_net_time_forward(self.h, input_name.encode(), _fp(x), c, h, w, iters)

    def __del__(self):
        try:
            self.ref.lib.ref_net_destroy(self.h)
        except Exception:
            pass


# --------------------------------------------------------------------------------------------------
# Input staging restatement (ncnn::Mat::from_pixels[_resize] + substract_mean_normalize), NumPy
# --------------------------------------------------------------------------------------------------
PIXEL_RGB, PIXEL_BGR, PIXEL_GRAY, PIXEL_RGBA = 1, 2, 4, 8  # mat.h:126-129; conversions = from | (to << 16)


def _pixel_plan(type_: int):
    """(source channels, gray?, channel map) following Mat::from_pixels, mat_pixel.cpp:1329-1367."""
    frm, to = type_ & 0xffff, type_ >> 16
    src_c = {PIXEL_RGB: 3, PIXEL_BGR: 3, PIXEL_GRAY: 1, PIXEL_RGBA: 4}.get(frm)
    if src_c is None:
        return None
    if to == 0:
        return src_c, False, list(range(src_c))
    if (frm, to) in ((PIXEL_RGB, PIXEL_BGR), (PIXEL_BGR, PIXEL_RGB), (PIXEL_RGBA, PIXEL_BGR)):
        return src_c, False, [2, 1, 0]
    if (frm, to) == (PIXEL_RGBA, PIXEL_RGB):
        return src_c, False, [0, 1, 2]
    if frm == PIXEL_GRAY and to in (PIXEL_RGB, PIXEL_BGR):
        return src_c, False, [0, 0, 0]
    if to == PIXEL_GRAY and frm in (PIXEL_RGB, PIXEL_RGBA):
        return src_c, True, [0, 1, 2]
    if to == PIXEL_GRAY and frm == PIXEL_BGR:
        return src_c, True, [2, 1, 0]
    return None


def _resize_coef(n_dst: int, n_src: int):
    """xofs / ialpha of resize_bilinear_c* (mat_pixel_resize.cpp:52-74): float coefficients -> 11-bit shorts."""
    scale = np.float64(n_src) / np.float64(n_dst)
    d = np.arange(n_dst, dtype=np.float64)
    f = ((d + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = (f - s.astype(np.float32)).astype(np.float32)
    lo = s < 0
    s[lo], f[lo] = 0, 0.0
    hi = s >= n_src - 1
    s[hi], f[hi] = n_src - 2, 1.0
    a0 = ((np.float32(1.0) - f) * np.float32(2048.0)).astype(np.float32)
    a1 = (f * np.float32(2048.0)).astype(np.float32)
    sat = lambda x: np.clip((x + np.where(x >= 0, np.float32(0.5), np.float32(-0.5))).astype(np.int64), -32768, 32767)
    return s, sat(a0), sat(a1)


def resize_bilinear_u8(img: np.ndarray, tw: int, th: int) -> np.ndarray:
    """resize_bilinear_c1/c3/c4 (mat_pixel_resize.cpp:26-278): (h, w, c) uint8 -> (th, tw, c) uint8, bit-exact."""
    h, w, c = img.shape
    sx, a0, a1 = _resize_coef(tw, w)
    sy, b0, b1 = _resize_coef(th, h)
    src = img.astype(np.int64)
    to_short = lambda v: ((v + 32768) % 65536) - 32768
    rows = to_short((src[:, sx, :] * a0[None, :, None] + src[:, sx + 1, :] * a1[None, :, None]) >> 4)  # (h, tw, c)
    r0, r1 = rows[sy], rows[sy + 1]
    v = (to_short((b0[:, None, None] * r0) >> 16) + to_short((b1[:, None, None] * r1) >> 16) + 2) >> 2
    return (v % 256).astype(np.uint8)


def from_pixels(img: np.ndarray, type_: int, target_w: int = 0, target_h: int = 0, mean=None, norm=None):
    """Mat::from_pixels[_resize] then Mat::substract_mean_normalize (mat.cpp:30-107) -> (C, H, W) float32, or None."""
    plan = _pixel_plan(type_)
    if plan is None:
        return None
    src_c, gray, cmap = plan
    img = np.ascontiguousarray(img, np.uint8).reshape(img.shape[0], img.shape[1], src_c)
    h, w = img.shape[:2]
    tw, th = target_w or w, target_h or h
    if (tw, th) != (w, h):
        img = resize_bilinear_u8(img, tw, th)
    p = img.astype(np.int64)
    if gray:  # mat_pixel.cpp:545-548,627
        out = ((p[..., cmap[0]] * 77 + p[..., cmap[1]] * 150 + p[..., cmap[2]] * 29) >> 8)[None].astype(np.float32)
    else:
        out = np.stack([p[..., i] for i in cmap]).astype(np.float32)
    if mean is not None and norm is None:
        out = out + (-np.asarray(mean, np.float32))[:, None, None]
    elif mean is None and norm is not None:
        out = out * np.asarray(norm, np.float32)[:, None, None]
    elif mean is not None:
        n32, m32 = np.asarray(norm, np.float32), np.asarray(mean, np.float32)
        out = out * n32[:, None, None] + (-m32 * n32)[:, None, None]
    return out.astype(np.float32)


# --------------------------------------------------------------------------------------------------
# ncnn .param/.bin reader (independent of the product's C++ loader) and whole-net interpreter
# --------------------------------------------------------------------------------------------------
def parse_param(path) -> list[dict]:
    """Restates Net::LoadParam (net.cpp:68-170) + ParamDict::load_param (paramdict.cpp:92-174)."""
    toks = Path(path).read_text().split()
    assert int(toks[0]) == 7767517, "param magic"
    layer_count, _blob_count = int(toks[1]), int(toks[2])
    i = 3
    layers = []
    for _ in range(layer_count):
        ltype, name, nb, nt = toks[i], toks[i + 1], int(toks[i + 2]), int(toks[i + 3])
        i += 4
        bottoms = toks[i:i + nb]
        i += nb
        tops = toks[i:i + nt]
        i += nt
        params = {}
        while i < len(toks) and "=" in toks[i]:
            k, v = toks[i].split("=", 1)
            k = int(k)
            if k <= -23300:
                vals = v.split(",")
                params[-k - 23300] = [float(t) if ("." in t or "e" in t.lower()) else int(t) for t in vals[1:]]
            else:
                params[k] = float(v) if ("." in v or "e" in v.lower()) else int(v)
            i += 1
        layers.append(dict(type=ltype, name=name, bottoms=bottoms, tops=tops, params=params))
    return layers


class _BinReader:
    """ModelBinFromStdio::load (modelbin.cpp:47-197): type 0 = 4-byte flag + data, type 1 = raw fp32."""

    def __init__(self, path):
        self.buf = Path(path).read_bytes()
        self.off = 0

    def load(self, n: int, type_: int) -> np.ndarray:
        if type_ == 0:
            flag = struct.unpack_from("<I", self.buf, self.off)[0]
            self.off += 4
            if flag == 0x01306B47:  # fp16
                a = np.frombuffer(self.buf, np.float16, n, self.off).astype(np.float32)
                self.off += (n * 2 + 3) // 4 * 4
                return a
            if flag != 0:
                fb = self.buf[self.off - 4:self.off]
                if sum(fb) != 0:  # 256-entry LUT quantised
                    table = np.frombuffer(self.buf, np.float32, 256, self.off)
                    self.off += 1024
                    idx = np.frombuffer(self.buf, np.uint8, n, self.off)
                    self.off += (n + 3) // 4 * 4
                    return table[idx].astype(np.float32)
        a = np.frombuffer(self.buf, np.float32, n, self.off).copy()
        self.off += 4 * n
        return a


class OracleNet:
    """NumPy/C interpreter of an ncnn-format net with the reference's per-layer semantics (batch 1)."""

    def __init__(self, param_path, bin_path):
        self.layers = parse_param(param_path)
        self.r = restatement()
        mb = _BinReader(bin_path)
        for L in self.layers:
            pd, t = L["params"], L["type"]
            if t in ("Convolution", "ConvolutionDepthWise"):  # conv_layer.h:39-139
                kw = pd.get(1, 0); kh = pd.get(11, kw)
                group = pd.get(7, 1)
                oc = pd.get(0, 0) // group
                ic = pd.get(6, 0) // oc // kh // kw
                L["w"] = mb.load(ic * oc * kh * kw, 0).reshape(oc, ic, kh, kw)
                L["b"] = mb.load(oc, 1) if pd.get(5, 0) else None
                L["geom"] = (oc, ic, kh, kw, group)
            elif t == "InnerProduct":  # inner_product_layer.h:105-150
                out = pd.get(0, 0); n = pd.get(2, 0)
                L["w"] = mb.load(n, 0).reshape(out, n // out)
                L["b"] = mb.load(out, 1) if pd.get(1, 0) else None
            elif t == "BatchNorm":  # batchnorm_layer.h:43-77
                c = pd.get(0, 0)
                L["bn"] = [mb.load(c, 1) for _ in range(4)]  # slope, mean, var, bias
            elif t == "Scale":  # scale_layer.h:45-73
                c = pd.get(0, 0)
                L["s"] = mb.load(c, 1)
                L["b"] = mb.load(c, 1) if pd.get(1, 0) else None
        self.blobs: dict[str, np.ndarray] = {}

    def forward(self, x: np.ndarray, input_name: str = "data") -> None:
        r = self.r
        blobs = self.blobs = {input_name: np.ascontiguousarray(x, np.float32)}
        for L in self.layers:
            t, pd = L["type"], L["params"]
            ins = [blobs[b] for b in L["bottoms"]]
            if t == "Input":
                continue
            if t in ("Convolution", "ConvolutionDepthWise"):
                oc, ic, kh, kw, group = L["geom"]
                xin = ins[0]
                pl = pd.get(4, 0); pt = pd.get(14, pl)
                p = ConvParam(oc, ic, xin.shape[1], xin.shape[2], kh, kw, 0, 0, pd.get(13, pd.get(3, 1)), pd.get(3, 1),
                              pl, pt, pl, pt, group, int(bool(pd.get(5, 0))), 0)
                r.lib.oracle_assign_output_dim(ctypes.byref(p))
                out = [r.conv(p, xin, L["w"], L["b"])]
            elif t == "ReLU":
                out = [r.relu(ins[0])]
            elif t == "Pooling":  # pooling_layer.h:93-110
                kw = pd.get(1, 0); kh = pd.get(11, kw)
                sw = pd.get(2, 1); sh = pd.get(12, sw)
                pl = pd.get(3, 0); pr = pd.get(14, pl); pt = pd.get(13, pl); pb = pd.get(15, pt)
                out = [r.pooling(ins[0], pd.get(0, 0), kh, kw, sh, sw, pl, pr, pt, pb, pd.get(4, 0))]
            elif t == "InnerProduct":
                out = [r.inner_product(ins[0], L["w"], L["b"]).reshape(-1, 1, 1)]
            elif t == "BatchNorm":
                out = [r.batchnorm(ins[0], *L["bn"], pd.get(1, 0.0))]
            elif t == "Scale":
                out = [r.scale(ins[0], L["s"], L["b"])]
            elif t == "Eltwise":
                out = [r.eltwise_add(ins[0], ins[1])]
            elif t == "Split":
                out = [ins[0].copy() for _ in L["tops"]]
            elif t == "Concat":
                out = [np.concatenate(ins, axis=0)]
            elif t == "Softmax":
                out = [r.softmax(ins[0])]
            elif t == "Dropout":
                out = [r.dropout(ins[0], pd.get(0, 1.0))]
            else:
                raise NotImplementedError(t)
            for name, o in zip(L["tops"], out):
                blobs[name] = o

    def extract(self, blob: str) -> np.ndarray:
        return self.blobs[blob]
