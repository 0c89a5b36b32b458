"""ctypes bindings to the CPU checkers (oracle/liblce_oracle.so and, when built,
oracle/_ref/liblce_ref.so) plus seeded case generators shared by the tests,
``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline leg.

TEST INFRASTRUCTURE ONLY: nothing under ``compute_engine_b200/`` imports this.
Generators follow the reference's op tests: signs i.i.d. Bernoulli(0.5),
post multiplier / bias ~ U(0.01, 1.5) (bconv2d_test.cc:574-581), int8 output
scale = 1/n with n in [1,20] and zero point in [-20,20] (tests/utils.h:60-65).
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
from dataclasses import dataclass, field

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(REPO, "oracle")

PADDING_SAME, PADDING_VALID = 0, 1
ACT_NONE, ACT_RELU, ACT_RELU_N1_TO_1, ACT_RELU6 = 0, 1, 2, 3
OUT_FLOAT, OUT_INT8, OUT_BITPACKED, OUT_RAW_ACC = 0, 1, 2, 3
T_FLOAT, T_INT8, T_BOOL = 0, 1, 2


class BconvDesc(C.Structure):
    """Mirror of ``lce_bconv2d_desc`` (include/lce_b200_types.h)."""

    _fields_ = [(n, C.c_int32) for n in (
        "batch", "in_h", "in_w", "channels_in", "filter_h", "filter_w",
        "channels_out", "groups", "stride_h", "stride_w", "dilation_h",
        "dilation_w", "padding", "pad_value", "activation", "out_type")] + [
        ("out_scale", C.c_float), ("out_zero_point", C.c_int32)]


class BMaxPoolDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "batch", "in_h", "in_w", "channels_packed", "filter_h", "filter_w",
        "stride_h", "stride_w", "padding")]


class BgemmEpilogue(C.Structure):
    _fields_ = [("out_type", C.c_int32), ("clamp_min", C.c_int32),
                ("clamp_max", C.c_int32), ("multiplier", C.c_void_p),
                ("bias", C.c_void_p), ("thresholds", C.c_void_p)]


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def build_oracle():
    """(Re)build the checker libraries if sources are newer. Building the
    checker is not using it."""
    subprocess.run(["make", "-s", "-C", ORACLE_DIR], check=True,
                   stdout=subprocess.DEVNULL)


_cache = {}


def load_oracle():
    if "oracle" not in _cache:
        path = os.path.join(ORACLE_DIR, "liblce_oracle.so")
        if not os.path.exists(path):
            build_oracle()
        _cache["oracle"] = C.CDLL(path)
    return _cache["oracle"]


def _cpu_flags():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    return set(line.split(":", 1)[1].split())
    except OSError:
        pass
    return set()


_V3 = {"avx", "avx2", "bmi1", "bmi2", "f16c", "fma", "abm", "movbe", "xsave"}
_V4 = {"avx512f", "avx512bw", "avx512cd", "avx512dq", "avx512vl"}


def ref_flavour(force=None):
    """Widest x86-64 level of oracle/_ref the host can run: 'v4', 'v3' or 'base'
    (LCE_REF_FLAVOUR overrides)."""
    want = force or os.environ.get("LCE_REF_FLAVOUR")
    if want:
        return want
    flags = _cpu_flags()
    if _V3 <= flags and _V4 <= flags:
        return "v4"
    if _V3 <= flags:
        return "v3"
    return "base"


def load_ref(flavour=None):
    """The reference's own headers compiled by oracle/Makefile; None if absent. The widest
    flavour the host CPU supports is picked unless `flavour` / LCE_REF_FLAVOUR says otherwise."""
    fl = ref_flavour(flavour)
    key = "ref" if flavour is None else "ref_" + fl
    if key not in _cache:
        lib = None
        for cand in ([fl, "base"] if fl != "base" else ["base"]):
            name = "liblce_ref.so" if cand == "base" else f"liblce_ref_{cand}.so"
            path = os.path.join(ORACLE_DIR, "_ref", name)
            if os.path.exists(path):
                lib = C.CDLL(path)
                _cache[key + "_name"] = name
                break
        _cache[key] = lib
    return _cache[key]


def ref_build_info():
    load_ref()
    return {"library": "oracle/_ref/" + str(_cache.get("ref_name")),
            "flags": "-O3 -ffp-contract=off -mpopcnt -msse4.2" +
                     {"liblce_ref_v3.so": " -march=x86-64-v3", "liblce_ref_v4.so": " -march=x86-64-v4"}.get(
                         _cache.get("ref_name"), "")}


def cdiv(a, b):
    return (a + b - 1) // b


# --------------------------------------------------------------------------- #
# generic wrappers: `impl` is "oracle" or "ref"
# --------------------------------------------------------------------------- #
def _lib(impl):
    lib = load_oracle() if impl == "oracle" else load_ref()
    if lib is None:
        raise RuntimeError("oracle/_ref/liblce_ref.so not built")
    return lib


def out_shape(desc: BconvDesc, impl="oracle"):
    lib = _lib(impl)
    oh, ow, ph, pw = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    rc = getattr(lib, f"lce_{impl}_bconv2d_out_shape")(
        C.byref(desc), C.byref(oh), C.byref(ow), C.byref(ph), C.byref(pw))
    if rc:
        raise ValueError("invalid bconv2d parameters")
    return oh.value, ow.value, ph.value, pw.value


def bconv2d(desc: BconvDesc, inp, filt, mul=None, bias=None, thr=None,
            impl="oracle", kind=0, threads=1):
    """Run LceBconv2d on the CPU checker. kind: 0 = the reference kernel's semantics
    (BConv2DReference; Register_BCONV_2D_REF), 1 = the optimised kernels' (ref: indirect
    BGEMM Kernel4x2Portable + zero_padding_correction; oracle: its restatement) -- they differ
    only under zero padding, where kind 1 adds a FLOAT correction after the output transform."""
    lib = _lib(impl)
    oh, ow, _, _ = out_shape(desc, impl)
    if desc.out_type == OUT_BITPACKED:
        out = np.empty((desc.batch, oh, ow, cdiv(desc.channels_out, 32)), np.int32)
    elif desc.out_type == OUT_INT8:
        out = np.empty((desc.batch, oh, ow, desc.channels_out), np.int8)
    else:
        out = np.empty((desc.batch, oh, ow, desc.channels_out), np.float32)
    inp = np.ascontiguousarray(inp, np.int32)
    filt = np.ascontiguousarray(filt, np.int32)
    if impl == "oracle":
        fn = lib.lce_oracle_bconv2d_opt_mt if kind == 1 else lib.lce_oracle_bconv2d_mt
        rc = fn(C.byref(desc), C.c_int(threads), _ptr(inp), _ptr(filt), _ptr(mul),
                _ptr(bias), _ptr(thr), _ptr(out))
    else:
        rc = lib.lce_ref_bconv2d_mt(C.byref(desc), C.c_int(kind),
                                    C.c_int(threads), _ptr(inp), _ptr(filt),
                                    _ptr(mul), _ptr(bias), _ptr(thr), _ptr(out))
    if rc:
        raise ValueError(f"{impl} bconv2d refused the parameters (rc={rc})")
    return out


def fold(desc: BconvDesc, mul, bias):
    lib = load_oracle()
    m = np.empty(desc.channels_out, np.float32)
    b = np.empty(desc.channels_out, np.float32)
    cmin, cmax = C.c_int32(), C.c_int32()
    lib.lce_oracle_fold_output_transform(C.byref(desc), _ptr(mul), _ptr(bias),
                                         _ptr(m), _ptr(b), C.byref(cmin),
                                         C.byref(cmax))
    return m, b, cmin.value, cmax.value


def bgemm(A, W, out_type=OUT_RAW_ACC, clamp=(0, 2**31 - 1), mul=None, bias=None,
          thr=None, threads=1):
    lib = load_oracle()
    A = np.ascontiguousarray(A, np.int32)
    W = np.ascontiguousarray(W, np.int32)
    M, Kw = A.shape
    N = W.shape[0]
    ep = BgemmEpilogue(out_type, clamp[0], clamp[1], _ptr(mul), _ptr(bias), _ptr(thr))
    if out_type == OUT_BITPACKED:
        out = np.empty((M, cdiv(N, 32)), np.int32)
    elif out_type == OUT_INT8:
        out = np.empty((M, N), np.int8)
    elif out_type == OUT_FLOAT:
        out = np.empty((M, N), np.float32)
    else:
        out = np.empty((M, N), np.int32)
    lib.lce_oracle_bgemm_mt(C.c_int(threads), C.c_int64(M), C.c_int(N),
                            C.c_int(Kw), _ptr(A), _ptr(W), C.byref(ep), _ptr(out))
    return out


_NP_T = {T_FLOAT: np.float32, T_INT8: np.int8, T_BOOL: np.uint8}


def quantize(x, zero_point=0, impl="oracle"):
    """LceQuantize over the last axis. x: float32 / int8 / bool ndarray."""
    lib = _lib(impl)
    if x.dtype == np.bool_:
        t, x = T_BOOL, x.view(np.uint8)
    elif x.dtype == np.int8:
        t = T_INT8
    else:
        t, x = T_FLOAT, x.astype(np.float32, copy=False)
    x = np.ascontiguousarray(x)
    cols = x.shape[-1]
    rows = x.size // cols if cols else 0
    out = np.empty(x.shape[:-1] + (cdiv(cols, 32),), np.int32)
    rc = getattr(lib, f"lce_{impl}_quantize")(
        C.c_int(t), _ptr(x), C.c_int64(rows), C.c_int64(cols),
        C.c_int32(zero_point), _ptr(out))
    assert rc == 0
    return out


def dequantize(packed, channels, out_type=T_FLOAT, scale=1.0, zero_point=0,
               impl="oracle"):
    lib = _lib(impl)
    packed = np.ascontiguousarray(packed, np.int32)
    rows = packed.size // packed.shape[-1]
    out = np.empty(packed.shape[:-1] + (channels,), _NP_T[out_type])
    rc = getattr(lib, f"lce_{impl}_dequantize")(
        C.c_int(out_type), _ptr(packed), C.c_int64(rows), C.c_int64(channels),
        C.c_float(scale), C.c_int32(zero_point), _ptr(out))
    assert rc == 0
    return out.view(np.bool_) if out_type == T_BOOL else out


def bmaxpool(desc: BMaxPoolDesc, x, impl="oracle"):
    lib = _lib(impl)
    oh, ow = C.c_int(), C.c_int()
    getattr(lib, f"lce_{impl}_bmaxpool_out_shape")(C.byref(desc), C.byref(oh),
                                                   C.byref(ow))
    x = np.ascontiguousarray(x, np.int32)
    out = np.empty((desc.batch, oh.value, ow.value, desc.channels_packed), np.int32)
    rc = getattr(lib, f"lce_{impl}_bmaxpool")(C.byref(desc), _ptr(x), _ptr(out))
    assert rc == 0
    return out


def compute_thresholds(cin_pg, fh, fw, mul, bias, activation):
    lib = load_oracle()
    thr = np.empty(len(mul), np.int32)
    lib.lce_oracle_compute_thresholds(C.c_int(cin_pg), C.c_int(fh), C.c_int(fw),
                                      C.c_int(len(mul)), _ptr(mul), _ptr(bias),
                                      C.c_int(activation), _ptr(thr))
    return thr


# --------------------------------------------------------------------------- #
# seeded case generation
# --------------------------------------------------------------------------- #
def pack_signs(signs):
    """numpy bitpack of a +-1 / float array along the last axis (bit = x < 0,
    LSB first, zero tail bits) -- independent of both checkers."""
    x = np.asarray(signs)
    c = x.shape[-1]
    cw = cdiv(c, 32)
    bits = np.zeros(x.shape[:-1] + (cw * 32,), np.uint32)
    bits[..., :c] = (x < 0)
    bits = bits.reshape(x.shape[:-1] + (cw, 32))
    weights = (np.uint32(1) << np.arange(32, dtype=np.uint32))
    return (bits * weights).sum(-1, dtype=np.uint64).astype(np.uint32).view(np.int32)


@dataclass
class BconvCase:
    desc: BconvDesc
    inp: np.ndarray          # packed NHWC int32
    filt: np.ndarray         # packed OHWI int32
    mul: np.ndarray | None
    bias: np.ndarray | None
    thr: np.ndarray | None
    meta: dict = field(default_factory=dict)


def make_bconv_case(seed, batch, in_h, in_w, cin, fh, fw, cout, groups=1,
                    stride=(1, 1), dilation=(1, 1), padding=PADDING_SAME,
                    pad_value=1, activation=ACT_NONE, out_type=OUT_FLOAT):
    rng = np.random.default_rng(seed)
    cin_pg = cin // groups
    x = rng.integers(0, 2, (batch, in_h, in_w, cin), dtype=np.int8) * 2 - 1
    w = rng.integers(0, 2, (cout, fh, fw, cin_pg), dtype=np.int8) * 2 - 1
    mul = rng.uniform(0.01, 1.5, cout).astype(np.float32)
    bias = rng.uniform(0.01, 1.5, cout).astype(np.float32)
    scale, zp = 1.0, 0
    if out_type == OUT_INT8:
        scale = np.float32(1.0) / np.float32(rng.integers(1, 21))
        zp = int(rng.integers(-20, 21))
    desc = BconvDesc(batch, in_h, in_w, cin, fh, fw, cout, groups, stride[0],
                     stride[1], dilation[0], dilation[1], padding, pad_value,
                     activation, out_type, float(scale), zp)
    thr = None
    if out_type == OUT_BITPACKED:
        thr = compute_thresholds(cin_pg, fh, fw, mul, bias, activation)
    return BconvCase(desc, pack_signs(x), pack_signs(w), mul, bias, thr,
                     {"seed": seed})


def golden_op_cases():
    """Yield (section, index entry, input) for the LceQuantize / LceDequantize / LceBMaxPool2d
    golden vectors in the order tests/golden/make_golden.py minted them. The inputs are drawn
    from one seeded stream, so only the reference's outputs are stored; this order is part of
    the golden data. Grids: bitpack_test.cc:102-109, quantization_test.cc:121-130,
    bmaxpool_test.cc:204-218 (pruned)."""
    rng = np.random.default_rng(7)
    # the special values the bit semantics hinge on (SURVEY 9.3-2)
    specials = np.array([-0.0, 0.0, np.nan, -np.nan, -1e-30, -1e-45, 1e-45, -np.inf, np.inf],
                        np.float32)
    n = 0
    for rows in (1, 2, 3, 8, 10, 15, 64):
        for cols in (1, 3, 16, 32, 33, 63, 64, 128):
            xf = rng.uniform(-1.5, 1.5, (rows, cols)).astype(np.float32)
            flat = xf.reshape(-1)
            flat[: min(flat.size, specials.size)] = specials[: flat.size]
            yield "quantize", {"key": f"q_f32_{n}", "type": "f32", "zero_point": 0}, xf
            for zp in (-1000, -1, 0, 23, 127, 128):
                xi = rng.integers(-128, 128, (rows, cols), dtype=np.int8)
                yield "quantize", {"key": f"q_i8_{n}_{zp}", "type": "i8", "zero_point": zp}, xi
            xb = rng.integers(0, 2, (rows, cols), dtype=np.uint8).astype(np.bool_)
            yield "quantize", {"key": f"q_b_{n}", "type": "bool", "zero_point": 1}, xb
            n += 1
    for n, (shape, ch) in enumerate([((1, 4, 4), 1), ((2, 3, 3), 31), ((1, 5, 2), 32),
                                     ((1, 2, 2), 33), ((3, 1, 1), 64), ((1, 3, 3), 68),
                                     ((1, 2, 3), 130), ((1, 1, 2), 200)]):
        packed = rng.integers(-2**31, 2**31, shape + (cdiv(ch, 32),),
                              dtype=np.int64).astype(np.int32)
        for t, scale, zp in ((T_FLOAT, 1.0, 0), (T_BOOL, 1.0, 0), (T_INT8, 1.0, 0),
                             (T_INT8, 0.05, 3), (T_INT8, 0.007, -100), (T_INT8, 0.3, 127)):
            yield "dequantize", {"key": f"dq_{n}_{t}_{zp}", "channels": ch, "type": t,
                                 "scale": scale, "zero_point": zp}, packed
    n = 0
    for (b, h, w, ch) in ((1, 7, 7, 1), (4, 8, 5, 2), (1, 12, 9, 3), (2, 56, 56, 2)):
        for (fh, fw) in ((1, 1), (2, 2), (3, 3), (2, 3)):
            for (sh, sw) in ((1, 1), (2, 2), (2, 3)):
                for pad in (PADDING_SAME, PADDING_VALID):
                    if pad == PADDING_VALID and (fh > h or fw > w):
                        continue
                    x = rng.integers(-2**31, 2**31, (b, h, w, ch), dtype=np.int64).astype(np.int32)
                    yield "bmaxpool", {"key": f"mp_{n}",
                                       "desc": [b, h, w, ch, fh, fw, sh, sw, pad]}, x
                    n += 1


def random_walk_cases():
    """Yield (n, case, optimised) for the seeded 300-step walk over LceBconv2d parameters that
    tests/test_oracle.py checks against the reference; `optimised` is True where the optimised
    kernels (kind 1) accept the case. Drawn from one stream: the order is part of the golden data."""
    rng = np.random.default_rng(99)
    for n in range(300):
        c = int(rng.choice([4, 32, 64, 96, 128, 192, 256]))
        g = int(rng.choice([1, 2])) if c % 64 == 0 else 1
        co = int(rng.choice([1, 2, 4, 6, 32, 34, 64])) * g
        fh, fw = int(rng.integers(1, 4)), int(rng.integers(1, 4))
        h, w = int(rng.integers(3, 10)), int(rng.integers(3, 10))
        st = (int(rng.integers(1, 3)), int(rng.integers(1, 4)))
        dl = (int(rng.integers(1, 3)), int(rng.integers(1, 3)))
        pad, pv = [(PADDING_VALID, 1), (PADDING_SAME, 0), (PADDING_SAME, 1)][n % 3]
        if pad == PADDING_VALID and ((fh - 1) * dl[0] + 1 > h or (fw - 1) * dl[1] + 1 > w):
            dl = (1, 1)
        if pad == PADDING_SAME and pv == 0 and c % 2:
            pv = 1
        ot = [OUT_FLOAT, OUT_INT8, OUT_BITPACKED][n % 3 if n % 2 else (n // 2) % 3]
        act = int(rng.integers(0, 4))
        case = make_bconv_case(n, int(rng.integers(1, 3)), h, w, c, fh, fw, co, g,
                               st, dl, pad, pv, act, ot)
        if ot == OUT_BITPACKED and act not in (ACT_NONE, ACT_RELU):
            continue
        optimised = g == 1 and not (pad == PADDING_SAME and pv == 0 and
                                    (ot != OUT_FLOAT or act != ACT_NONE))
        yield n, case, optimised


GOLDEN_DIR = os.path.join(REPO, "tests", "golden")
# The reference's outputs, split so that no committed file exceeds 1 MB.
GOLDEN_FILES = {"bconv": "lce_golden_bconv.npz", "ops": "lce_golden_ops.npz"}


def load_golden():
    """(index, arrays) of the golden vectors: the reference's outputs under their keys, and the
    regenerated input of every quantize / dequantize / bmaxpool vector under key + "_in"."""
    with open(os.path.join(GOLDEN_DIR, "lce_golden.json")) as f:
        index = json.load(f)["index"]
    arrays = {}
    for name in GOLDEN_FILES.values():
        with np.load(os.path.join(GOLDEN_DIR, name)) as z:
            arrays.update((k, z[k]) for k in z.files)
    arrays.update((e["key"] + "_in", x) for _, e, x in golden_op_cases())
    return index, arrays


def load_random_walk():
    """{str(n): {"kind0": sha256, "kind1": sha256 (where optimised)}} of random_walk_cases()."""
    with open(os.path.join(GOLDEN_DIR, "lce_random_walk.json")) as f:
        return json.load(f)["cases"]


def desc_to_dict(d: BconvDesc):
    return {n: getattr(d, n) for n, _ in d._fields_}


def desc_from_dict(m):
    return BconvDesc(**{k: (float(v) if k == "out_scale" else int(v))
                        for k, v in m.items()})
