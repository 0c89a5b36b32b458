"""GPU tests of every float builtin entry point (include/lce_b200_builtins.h) against plain
references written here, independently of the library, at the shapes, paths and edges where the
kernels differ.

Two kinds of data:

* exact: small integers (|x|, |w| <= 4, integer bias), scaled by a power of two so that the clamps of
  RELU6 and RELU_N1_TO_1 are reached. With K <= 5000 every partial sum is an integer multiple of the
  scale and below 2^24 times it: exact in fp32, and exact after the tf32 hi/lo split (lo = 0). The
  result then does not depend on the summation order, and every convolution kernel must equal the
  fp64 reference rounded to fp32 exactly.
* Gaussian: |out - ref| <= 2e-6 * (sum|a||w| + |b|) against fp64, which a kernel that silently
  computes in tf32 or drops the fma fails.

lce_b200_f32_conv_path_counts says which of the eight convolution kernels ran; every case asserts
the one it means to test. Pools, element-wise ops, MEAN, DEQUANTIZE and PAD repeat fixed-order
float32 arithmetic, so they are compared bit for bit with NumPy. Output buffers start as NaN (or a
sentinel word), so an element a kernel forgets to write fails the comparison.
"""
import ctypes as C
import math
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import lce_testlib as L

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAME, VALID = 0, 1
NONE, RELU, RELU_N1_TO_1, RELU6 = 0, 1, 2, 3
T_INT8, T_UINT8 = 1, 2
PW_TF32, STEM7, DIRECT16, GEMM_SMALL_M, GEMM128, IGEMM8X8, IGEMM8X4, GEMM = range(8)
# LCE_B200_IGEMM_8X4=1 (read once per process) sends every implicit-GEMM shape to the 8x4 kernel;
# test_igemm_8x4_variant_in_subprocess runs the igemm tests of this file that way
IGEMM = IGEMM8X4 if os.environ.get("LCE_B200_IGEMM_8X4") == "1" else IGEMM8X8
SENTINEL = 0x5A5A5A5A


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("batch", "in_h", "in_w", "in_c", "filter_h", "filter_w", "out_c",
                                         "stride_h", "stride_w", "dilation_h", "dilation_w", "padding",
                                         "activation")]


class PoolDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("batch", "in_h", "in_w", "channels", "filter_h", "filter_w",
                                         "stride_h", "stride_w", "padding", "activation")]


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module")
def lib(torch):
    from compute_engine_b200 import capi
    return capi.lib()


@pytest.fixture
def rng(request):
    return np.random.default_rng(zlib.crc32(request.node.name.encode()))


# --------------------------------------------------------------------------------------------- #
# helpers
# --------------------------------------------------------------------------------------------- #
def to_dev(torch, a, offset=0):
    """`a` on the device as a flat view `offset` elements past a 16-byte boundary (offset 1: the
    kernels' unaligned paths)."""
    a = np.ascontiguousarray(a)
    t = torch.from_numpy(a.reshape(-1))
    flat = torch.zeros(a.size + offset, dtype=t.dtype, device="cuda")
    flat[offset:] = t
    return flat[offset:]


def nan_dev(torch, shape, offset=0):
    return to_dev(torch, np.full(shape, np.nan, np.float32), offset)


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def host(torch, t, shape):
    torch.cuda.synchronize()
    return t.cpu().numpy().reshape(shape)


def check(lib, rc):
    assert rc == 0, lib.lce_b200_last_error().decode()


def conv_counts(lib):
    a = (C.c_uint64 * 8)()
    lib.lce_b200_f32_conv_path_counts(a)
    return [int(v) for v in a]


def tfl_out_pad(padding, n, k, s, d=1):
    """TFLite's output size and leading zero padding: SAME out = ceil(n / s),
    total = max((o - 1) * s + (k - 1) * d + 1 - n, 0), before = total // 2; VALID no padding."""
    if padding == SAME:
        o = (n + s - 1) // s
        total = max((o - 1) * s + (k - 1) * d + 1 - n, 0)
        return o, total // 2
    return max((n - (k - 1) * d - 1) // s + 1, 0), 0


def act_f64(x, act):
    if act == RELU:
        return np.maximum(x, 0)
    if act == RELU_N1_TO_1:
        return np.clip(x, -1, 1)
    if act == RELU6:
        return np.clip(x, 0, 6)
    return x


def act_f32(x, act):
    """the kernels' fmaxf / fminf sequence in float32"""
    f = np.float32
    if act == RELU:
        return np.maximum(x, f(0))
    if act == RELU_N1_TO_1:
        return np.minimum(np.maximum(x, f(-1)), f(1))
    if act == RELU6:
        return np.minimum(np.maximum(x, f(0)), f(6))
    return x


def exact_data(rng, shape, scale=1.0):
    return (rng.integers(-4, 5, shape) * scale).astype(np.float32)


def gauss_data(rng, shape, sigma=1.0):
    return (rng.standard_normal(shape) * sigma).astype(np.float32)


def exact_scale(k):
    """power of two that brings a sum of k products of integers in [-4, 4] (std ~6.7 sqrt(k))
    to a std of about 3: both clamps of RELU6 and RELU_N1_TO_1 are reached"""
    return 2.0 ** -max(0, round(math.log2(6.7 * math.sqrt(k) / 3)))


def windows(x, oh, ow, ky, kx, sy, sx, py, px, fill):
    """the (ky, kx) tap of every output pixel: x[:, oy*sy - py + ky, ox*sx - px + kx] (`fill` outside)
    and the [oh, ow] mask of taps inside the image"""
    B, H, W = x.shape[:3]
    ys = np.arange(oh) * sy - py + ky
    xs = np.arange(ow) * sx - px + kx
    my, mx = (ys >= 0) & (ys < H), (xs >= 0) & (xs < W)
    m = my[:, None] & mx[None, :]
    if m.size and m.all():   # a strided view: no copy of the large-K inputs
        return x[:, ys[0]:ys[-1] + 1:sy, xs[0]:xs[-1] + 1:sx], m
    t = x[:, np.clip(ys, 0, H - 1)][:, :, np.clip(xs, 0, W - 1)]
    return np.where(m[None, :, :, None], t, fill), m


def conv_ref(x, w, b, stride, dil, padding, depthwise=False):
    """fp64 CONV_2D / DEPTHWISE_CONV_2D (depth multiplier 1) without activation. x NHWC,
    w OHWI [Cout, KH, KW, Cin] (depthwise: [1, KH, KW, C])."""
    x = x.astype(np.float64)
    w = w.astype(np.float64)
    _, H, W, _ = x.shape
    _, KH, KW, _ = w.shape
    oh, ph = tfl_out_pad(padding, H, KH, stride[0], dil[0])
    ow, pw = tfl_out_pad(padding, W, KW, stride[1], dil[1])
    acc = 0.0
    for fy in range(KH):
        for fx in range(KW):
            t, _ = windows(x, oh, ow, fy * dil[0], fx * dil[1], stride[0], stride[1], ph, pw, 0.0)
            acc = acc + (t * w[0, fy, fx] if depthwise else t @ w[:, fy, fx, :].T)
    if b is not None:
        acc = acc + b.astype(np.float64)
    return acc + 0.0   # -0 -> +0: the kernels accumulate from +0


def assert_close(got, x, w, b, stride, dil, padding, act, exact, depthwise=False):
    ref = act_f64(conv_ref(x, w, b, stride, dil, padding, depthwise), act)
    assert got.shape == ref.shape
    if exact:
        want = ref.astype(np.float32)
        bad = got != want
        assert not bad.any(), f"{bad.sum()} of {bad.size} differ, e.g. {got[bad][:4]} vs {want[bad][:4]}"
        return ref
    mag = conv_ref(np.abs(x), np.abs(w), None if b is None else np.abs(b), stride, dil, padding, depthwise)
    err = np.abs(got.astype(np.float64) - ref)
    assert np.isfinite(got).all()
    assert (err <= 2e-6 * mag).all(), (err / np.maximum(mag, 1e-30)).max()
    return ref


# --------------------------------------------------------------------------------------------- #
# CONV_2D: every kernel conv2d_impl chooses from
# --------------------------------------------------------------------------------------------- #
def run_conv(torch, lib, x, w, b, stride=(1, 1), dil=(1, 1), padding=SAME, act=NONE, offset=0, packed=False):
    B, H, W, Cin = x.shape
    Cout, KH, KW, _ = w.shape
    d = ConvDesc(B, H, W, Cin, KH, KW, Cout, stride[0], stride[1], dil[0], dil[1], padding, act)
    oh, ow = C.c_int(), C.c_int()
    check(lib, lib.lce_b200_f32_conv_out_shape(C.byref(d), C.byref(oh), C.byref(ow)))
    oh, ow = oh.value, ow.value
    assert (oh, ow) == (tfl_out_pad(padding, H, KH, stride[0], dil[0])[0],
                        tfl_out_pad(padding, W, KW, stride[1], dil[1])[0])
    shape = (B, oh, ow, Cout)
    xd, wd = to_dev(torch, x, offset), to_dev(torch, w, offset)
    bd = None if b is None else to_dev(torch, b, offset)
    out = nan_dev(torch, shape, offset)
    pk = None
    before = conv_counts(lib)
    if packed:
        pk = to_dev(torch, np.full((B, oh, ow, L.cdiv(Cout, 32)), SENTINEL, np.int32))
        check(lib, lib.lce_b200_f32_conv2d_packed(C.byref(d), ptr(xd), ptr(wd), ptr(bd), ptr(out), ptr(pk), None))
    else:
        check(lib, lib.lce_b200_f32_conv2d(C.byref(d), ptr(xd), ptr(wd), ptr(bd), ptr(out), None))
    got = host(torch, out, shape)
    ran = [a - b0 for a, b0 in zip(conv_counts(lib), before)]
    words = host(torch, pk, (B, oh, ow, L.cdiv(Cout, 32))) if packed else None
    return got, words, ran


def one_hot(i):
    return [int(j == i) for j in range(8)]


# name, (B, H, W, Cin), (KH, KW, Cout), stride, dilation, padding, act, bias, kernel, packed, offset
CONV_CASES = [
    # direct16, generic instantiation (K <= 32): ragged channel groups, scalar stores
    ("direct16_1x1_20to40", (2, 7, 9, 20), (1, 1, 40), (1, 1), (1, 1), SAME, RELU6, True, DIRECT16, False, 0),
    ("direct16_3x3_2to24_s2", (2, 12, 14, 2), (3, 3, 24), (2, 2), (1, 1), SAME, RELU, False, DIRECT16, False, 0),
    ("direct16_5x5_1to8_d2", (1, 17, 15, 1), (5, 5, 8), (1, 1), (2, 2), VALID, RELU_N1_TO_1, True, DIRECT16, False, 0),
    ("direct16_3x3_2to64_packed", (2, 9, 10, 2), (3, 3, 64), (1, 1), (1, 1), SAME, NONE, True, DIRECT16, True, 0),
    # direct16, the 3x3x3 stem instantiation (fused pack at Cout 32)
    ("direct16_stem_s1", (2, 19, 23, 3), (3, 3, 16), (1, 1), (1, 1), SAME, RELU6, True, DIRECT16, False, 0),
    ("direct16_stem_s2_packed", (3, 32, 30, 3), (3, 3, 32), (2, 2), (1, 1), SAME, NONE, True, DIRECT16, True, 0),
    ("direct16_stem_s2_valid_24", (1, 20, 17, 3), (3, 3, 24), (2, 2), (1, 1), VALID, RELU, False, DIRECT16, False, 0),
    # direct16, the 1x1x16 -> 64 instantiation: an odd pixel count, so the tf32 pairs path refuses
    ("direct16_pw16_odd_packed", (3, 7, 9, 16), (1, 1, 64), (1, 1), (1, 1), SAME, RELU, True, DIRECT16, True, 0),
    # plain GEMMs (1x1, K % 32 != 0 so tf32 refuses): fewer than 74 tiles -> small-M kernel
    ("gemm_small_m_k36", (8, 5, 5, 36), (1, 1, 64), (1, 1), (1, 1), SAME, RELU_N1_TO_1, True, GEMM_SMALL_M, True, 0),
    ("gemm_small_m_k36_n50", (8, 5, 5, 36), (1, 1, 50), (1, 1), (1, 1), VALID, NONE, False, GEMM_SMALL_M, True, 0),
    ("gemm128_k36_n100", (4, 71, 71, 36), (1, 1, 100), (1, 1), (1, 1), SAME, RELU6, True, GEMM128, True, 0),
    ("gemm128_k36_n160", (1, 141, 143, 36), (1, 1, 160), (1, 1), (1, 1), SAME, NONE, False, GEMM128, True, 0),
    ("gemm128_k5000", (1, 1, 9480, 5000), (1, 1, 128), (1, 1), (1, 1), VALID, RELU, True, GEMM128, False, 0),
    # implicit GEMM (K <= 4096, not a plain GEMM)
    ("igemm_3x3_64to80_s2", (2, 28, 26, 64), (3, 3, 80), (2, 2), (1, 1), SAME, RELU, True, IGEMM, True, 0),
    ("igemm_3x3_64to80_d2", (1, 30, 30, 64), (3, 3, 80), (1, 1), (2, 2), VALID, RELU6, False, IGEMM, False, 0),
    ("igemm_2x2_k2944", (2, 36, 36, 736), (2, 2, 40), (1, 1), (1, 1), SAME, NONE, True, IGEMM, False, 0),
    ("igemm_3x3_k3456", (2, 40, 40, 384), (3, 3, 64), (1, 1), (1, 1), SAME, RELU_N1_TO_1, True, IGEMM, True, 0),
    ("igemm_5x5_k3200", (1, 48, 52, 128), (5, 5, 96), (1, 1), (1, 1), SAME, NONE, False, IGEMM, False, 0),
    ("igemm_1x1_k3001", (1, 40, 50, 3001), (1, 1, 40), (1, 1), (1, 1), SAME, RELU, True, IGEMM, False, 0),
    ("igemm_1x1_s2_k4096", (1, 59, 60, 4096), (1, 1, 33), (2, 2), (1, 1), SAME, NONE, True, IGEMM, False, 0),
    ("igemm_1x1_unaligned", (2, 9, 11, 24), (1, 1, 36), (1, 1), (1, 1), SAME, RELU6, True, IGEMM, True, 1),
    # K > 4096
    ("gemm_3x3_k4608", (2, 50, 50, 512), (3, 3, 70), (1, 1), (1, 1), SAME, RELU, True, GEMM, False, 0),
    # tensor cores
    ("pw_tf32_k64_n128_packed", (2, 21, 21, 64), (1, 1, 128), (1, 1), (1, 1), SAME, RELU, True, PW_TF32, True, 0),
    ("pw_tf32_pairs", (2, 8, 8, 16), (1, 1, 64), (1, 1), (1, 1), SAME, RELU6, False, PW_TF32, False, 0),
    ("stem7_tf32", (2, 44, 38, 3), (7, 7, 64), (2, 2), (1, 1), SAME, RELU, True, STEM7, False, 0),
]


@pytest.mark.parametrize("exact", [True, False], ids=["exact", "gauss"])
@pytest.mark.parametrize("case", CONV_CASES, ids=[c[0] for c in CONV_CASES])
def test_conv_matches_reference(torch, lib, rng, case, exact):
    _, xs, (KH, KW, Cout), stride, dil, padding, act, with_bias, kernel, packed, offset = case
    K = KH * KW * xs[3]
    if exact:
        s = exact_scale(K)
        x, w = exact_data(rng, xs, s), exact_data(rng, (Cout, KH, KW, xs[3]))
        b = exact_data(rng, Cout, s) if with_bias else None
    else:
        x, w = gauss_data(rng, xs, 1.5), gauss_data(rng, (Cout, KH, KW, xs[3]), 0.3)
        b = gauss_data(rng, Cout) if with_bias else None
    got, words, ran = run_conv(torch, lib, x, w, b, stride, dil, padding, act, offset, packed)
    assert ran == one_hot(kernel), ran
    ref = assert_close(got, x, w, b, stride, dil, padding, act, exact)
    if packed:
        assert np.array_equal(words, L.quantize(got)), "packed words differ from LceQuantize of the output"
        if exact:
            assert np.array_equal(words, L.pack_signs(ref.astype(np.float32)))


def test_fully_connected_rows_do_not_depend_on_the_batch(torch, lib, rng):
    """FULLY_CONNECTED (a 1x1 conv on [B, 1, 1, K]) with K % 32 != 0: the small-M kernel below 74
    tiles and the 128x128 kernel above accumulate the same fmaf chain, so an image's logits are the
    same bits at batch 256 and at batch 9600."""
    K, N = 100, 100
    w, b = gauss_data(rng, (N, 1, 1, K), 0.3), gauss_data(rng, N)
    x = gauss_data(rng, (9600, 1, 1, K), 1.5)
    small, _, ran_s = run_conv(torch, lib, x[:256], w, b, act=RELU6)
    large, _, ran_l = run_conv(torch, lib, x, w, b, act=RELU6)
    assert ran_s == one_hot(GEMM_SMALL_M) and ran_l == one_hot(GEMM128), (ran_s, ran_l)
    assert np.array_equal(small.view(np.int32), large[:256].view(np.int32))
    assert_close(small, x[:256], w, b, (1, 1), (1, 1), SAME, RELU6, exact=False)


@pytest.mark.parametrize("cin,k,cout,stride", [(3, 3, 24, 2), (2, 3, 20, 1), (20, 1, 40, 1)])
def test_direct16_and_igemm_give_the_same_bits(torch, lib, rng, cin, k, cout, stride):
    """K <= 32: the direct kernel (aligned) and the implicit GEMM (offset-by-one views) both add one
    fmaf per k in ascending k from +0, then the bias, then the activation."""
    x, w, b = gauss_data(rng, (2, 15, 13, cin)), gauss_data(rng, (cout, k, k, cin), 0.5), gauss_data(rng, cout)
    d16, _, ran_d = run_conv(torch, lib, x, w, b, (stride, stride), act=RELU)
    ig, _, ran_i = run_conv(torch, lib, x, w, b, (stride, stride), act=RELU, offset=1)
    assert ran_d == one_hot(DIRECT16) and ran_i == one_hot(IGEMM), (ran_d, ran_i)
    assert np.array_equal(d16.view(np.int32), ig.view(np.int32))


def test_igemm_8x4_variant_in_subprocess():
    """conv_igemm_kernel is chosen by LCE_B200_IGEMM_8X4=1, read once per process: run this file's
    implicit-GEMM tests in a process of their own with it set (they then expect index 6)."""
    if os.environ.get("LCE_B200_IGEMM_8X4") == "1":
        pytest.skip("already the 8x4 process")
    env = dict(os.environ, LCE_B200_IGEMM_8X4="1")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-k",
                        "igemm and not subprocess", os.path.abspath(__file__)],
                       cwd=REPO, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and " failed" not in r.stdout


# --------------------------------------------------------------------------------------------- #
# DEPTHWISE_CONV_2D
# --------------------------------------------------------------------------------------------- #
# name, (B, H, W, C), (KH, KW), stride, dilation, padding, act, bias, offset
DW_CASES = [
    ("v4_3x3_s1_same", (2, 15, 13, 32), (3, 3), (1, 1), (1, 1), SAME, RELU6, True, 0),
    ("v4_3x3_s2_valid_nobias", (1, 16, 17, 8), (3, 3), (2, 2), (1, 1), VALID, NONE, False, 0),
    ("v4_3x3_s3_d2", (2, 20, 19, 12), (3, 3), (3, 3), (2, 2), SAME, RELU, True, 0),
    ("v0_5x5_s2", (2, 17, 18, 16), (5, 5), (2, 2), (1, 1), SAME, RELU_N1_TO_1, True, 0),
    ("v0_1x3_s13_valid", (1, 9, 21, 8), (1, 3), (1, 3), (1, 1), VALID, NONE, False, 0),
    ("scalar_c6_s2", (2, 11, 12, 6), (3, 3), (2, 2), (1, 1), SAME, RELU, True, 0),
    ("scalar_c5_5x5_d2", (1, 14, 13, 5), (5, 5), (1, 1), (2, 2), VALID, RELU6, False, 0),
    ("scalar_unaligned_s3", (2, 10, 11, 8), (3, 3), (3, 3), (1, 1), SAME, NONE, True, 1),
]


@pytest.mark.parametrize("exact", [True, False], ids=["exact", "gauss"])
@pytest.mark.parametrize("case", DW_CASES, ids=[c[0] for c in DW_CASES])
def test_depthwise_matches_reference(torch, lib, rng, case, exact):
    _, (B, H, W, Cc), (KH, KW), stride, dil, padding, act, with_bias, offset = case
    if exact:
        s = exact_scale(KH * KW)
        x, w = exact_data(rng, (B, H, W, Cc), s), exact_data(rng, (1, KH, KW, Cc))
        b = exact_data(rng, Cc, s) if with_bias else None
    else:
        x, w = gauss_data(rng, (B, H, W, Cc)), gauss_data(rng, (1, KH, KW, Cc), 0.5)
        b = gauss_data(rng, Cc) if with_bias else None
    d = ConvDesc(B, H, W, Cc, KH, KW, Cc, stride[0], stride[1], dil[0], dil[1], padding, act)
    oh = tfl_out_pad(padding, H, KH, stride[0], dil[0])[0]
    ow = tfl_out_pad(padding, W, KW, stride[1], dil[1])[0]
    out = nan_dev(torch, (B, oh, ow, Cc), offset)
    xd, wd = to_dev(torch, x, offset), to_dev(torch, w, offset)
    bd = None if b is None else to_dev(torch, b, offset)
    check(lib, lib.lce_b200_f32_depthwise_conv2d(C.byref(d), ptr(xd), ptr(wd), ptr(bd), ptr(out), None))
    got = host(torch, out, (B, oh, ow, Cc))
    assert_close(got, x, w, b, stride, dil, padding, act, exact, depthwise=True)


# --------------------------------------------------------------------------------------------- #
# MAX_POOL_2D / AVERAGE_POOL_2D
# --------------------------------------------------------------------------------------------- #
def pool_ref(x, fh, fw, sh, sw, padding, act, is_max):
    """float32, in-bounds taps only in (fy, fx) order; average = one division by the in-bounds
    count (TFLite pooling.h at SAME borders)"""
    B, H, W, Cc = x.shape
    oh, ph = tfl_out_pad(padding, H, fh, sh)
    ow, pw = tfl_out_pad(padding, W, fw, sw)
    acc = np.full((B, oh, ow, Cc), -np.finfo(np.float32).max if is_max else 0, np.float32)
    cnt = np.zeros((oh, ow), np.int64)
    for fy in range(fh):
        for fx in range(fw):
            t, m = windows(x, oh, ow, fy, fx, sh, sw, ph, pw, 0)
            new = np.maximum(acc, t) if is_max else acc + t
            acc = np.where(m[None, :, :, None], new, acc)
            cnt += m
    if not is_max:
        acc = acc / np.maximum(cnt, 1).astype(np.float32)[None, :, :, None]
    return act_f32(acc, act)


# name, (B, H, W, C), (fh, fw), stride, padding, act, offset: pool_v4 f = 2, 3, runtime; scalar kernel
POOL_CASES = [
    ("v4_f2_s2_valid", (2, 15, 16, 8), (2, 2), (2, 2), VALID, NONE, 0),
    ("v4_f2_s1_same", (1, 9, 7, 12), (2, 2), (1, 1), SAME, RELU, 0),
    ("v4_f3_s2_same", (2, 17, 14, 16), (3, 3), (2, 2), SAME, RELU6, 0),
    ("v4_f3_s1_valid", (1, 8, 9, 4), (3, 3), (1, 1), VALID, RELU_N1_TO_1, 0),
    ("v4_f3x2_s12_same", (2, 11, 10, 8), (3, 2), (1, 2), SAME, NONE, 0),
    ("v4_f5_s3_same", (1, 13, 14, 20), (5, 5), (3, 3), SAME, RELU, 0),
    ("scalar_c6_f3_s2_same", (2, 11, 12, 6), (3, 3), (2, 2), SAME, NONE, 0),
    ("scalar_unaligned_f2_s2_same", (1, 9, 7, 8), (2, 2), (2, 2), SAME, RELU6, 1),
    ("scalar_c3_f5x4_s23_valid", (2, 12, 13, 3), (5, 4), (2, 3), VALID, RELU_N1_TO_1, 0),
]


@pytest.mark.parametrize("is_max", [True, False], ids=["max", "avg"])
@pytest.mark.parametrize("case", POOL_CASES, ids=[c[0] for c in POOL_CASES])
def test_pool_is_bit_exact(torch, lib, rng, case, is_max):
    _, (B, H, W, Cc), (fh, fw), (sh, sw), padding, act, offset = case
    x = gauss_data(rng, (B, H, W, Cc), 2.0)
    d = PoolDesc(B, H, W, Cc, fh, fw, sh, sw, padding, act)
    oh, ow = C.c_int(), C.c_int()
    check(lib, lib.lce_b200_f32_pool_out_shape(C.byref(d), C.byref(oh), C.byref(ow)))
    assert (oh.value, ow.value) == (tfl_out_pad(padding, H, fh, sh)[0], tfl_out_pad(padding, W, fw, sw)[0])
    shape = (B, oh.value, ow.value, Cc)
    out = nan_dev(torch, shape, offset)
    fn = lib.lce_b200_f32_max_pool if is_max else lib.lce_b200_f32_avg_pool
    xd = to_dev(torch, x, offset)
    check(lib, fn(C.byref(d), ptr(xd), ptr(out), None))
    got = host(torch, out, shape)
    want = pool_ref(x, fh, fw, sh, sw, padding, act, is_max)
    assert np.array_equal(got.view(np.int32), want.view(np.int32))


def test_pool_without_output_writes_nothing(torch, lib):
    """VALID with a filter larger than the input in both dimensions: shape (0, 0), no launch"""
    d = PoolDesc(1, 3, 3, 4, 5, 5, 1, 1, VALID, NONE)
    oh, ow = C.c_int(), C.c_int()
    check(lib, lib.lce_b200_f32_pool_out_shape(C.byref(d), C.byref(oh), C.byref(ow)))
    assert (oh.value, ow.value) == (0, 0)
    x = to_dev(torch, np.ones((1, 3, 3, 4), np.float32))
    out = to_dev(torch, np.full(64, SENTINEL, np.int32))
    for fn in (lib.lce_b200_f32_max_pool, lib.lce_b200_f32_avg_pool):
        check(lib, fn(C.byref(d), ptr(x), ptr(out), None))
    assert (host(torch, out, (64,)) == SENTINEL).all()


# --------------------------------------------------------------------------------------------- #
# fused MAX_POOL_2D(2x2, s1, VALID) -> DEPTHWISE_CONV_2D(3x3)
# --------------------------------------------------------------------------------------------- #
# (B, H, W, C, dw stride, dw padding, act, bias): odd sizes, inputs 3 and 4 wide / tall, and channel
# counts that put interior and border threads into one warp
FUSED_CASES = [
    (1, 3, 3, 4, 1, SAME, NONE, True),
    (2, 4, 4, 12, 2, SAME, RELU, False),
    (1, 3, 4, 68, 1, SAME, RELU6, True),
    (1, 4, 5, 260, 1, VALID, NONE, False),
    (2, 21, 70, 4, 1, SAME, RELU, True),
    (1, 19, 40, 12, 2, SAME, NONE, False),
    (2, 17, 15, 68, 1, VALID, RELU6, True),
    (1, 11, 9, 260, 2, SAME, RELU_N1_TO_1, False),
    (2, 9, 11, 12, 2, VALID, RELU, True),
    (1, 13, 7, 68, 2, SAME, NONE, True),
]


def _fused_descs(B, H, W, Cc, s, padding, act):
    pool = PoolDesc(B, H, W, Cc, 2, 2, 1, 1, VALID, NONE)
    dw = ConvDesc(B, H - 1, W - 1, Cc, 3, 3, Cc, s, s, 1, 1, padding, act)
    oh = tfl_out_pad(padding, H - 1, 3, s)[0]
    ow = tfl_out_pad(padding, W - 1, 3, s)[0]
    return pool, dw, (B, oh, ow, Cc)


@pytest.mark.parametrize("case", FUSED_CASES, ids=[f"{c[1]}x{c[2]}c{c[3]}s{c[4]}p{c[5]}" for c in FUSED_CASES])
def test_maxpool2x2_depthwise3x3(torch, lib, rng, case):
    B, H, W, Cc, s, padding, act, with_bias = case
    pool, dw, shape = _fused_descs(B, H, W, Cc, s, padding, act)
    assert shape[1] > 0 and shape[2] > 0
    for exact in (False, True):
        if exact:
            x, w = exact_data(rng, (B, H, W, Cc), 0.25), exact_data(rng, (1, 3, 3, Cc))
            b = exact_data(rng, Cc, 0.25) if with_bias else None
        else:
            x, w = gauss_data(rng, (B, H, W, Cc)), gauss_data(rng, (1, 3, 3, Cc), 0.5)
            b = gauss_data(rng, Cc) if with_bias else None
        xd, wd = to_dev(torch, x), to_dev(torch, w)
        bd = None if b is None else to_dev(torch, b)
        got = nan_dev(torch, shape)
        check(lib, lib.lce_b200_f32_maxpool2x2_depthwise3x3(C.byref(pool), C.byref(dw), ptr(xd), ptr(wd), ptr(bd),
                                                             ptr(got), None))
        got = host(torch, got, shape)
        if exact:
            pooled = pool_ref(x, 2, 2, 1, 1, VALID, NONE, True)
            assert_close(got, pooled, w, b, (s, s), (1, 1), padding, act, True, depthwise=True)
        else:   # the two kernels one after the other
            pooled = nan_dev(torch, (B, H - 1, W - 1, Cc))
            check(lib, lib.lce_b200_f32_max_pool(C.byref(pool), ptr(xd), ptr(pooled), None))
            want = nan_dev(torch, shape)
            check(lib, lib.lce_b200_f32_depthwise_conv2d(C.byref(dw), ptr(pooled), ptr(wd), ptr(bd), ptr(want), None))
            assert np.array_equal(got.view(np.int32), host(torch, want, shape).view(np.int32))


def test_maxpool2x2_depthwise3x3_refusals(torch, lib):
    x, w, out = to_dev(torch, np.zeros(2 * 9 * 9 * 8, np.float32), 1), to_dev(torch, np.zeros(9 * 8, np.float32)), \
        nan_dev(torch, 2 * 8 * 8 * 8, 1)
    pool, dw, _ = _fused_descs(2, 9, 9, 8, 1, SAME, NONE)
    xa, outa = x.clone(), out.clone()   # 16-byte aligned copies

    def call(p, d, xx=xa, oo=outa):
        return lib.lce_b200_f32_maxpool2x2_depthwise3x3(C.byref(p), C.byref(d), ptr(xx), ptr(w), None, ptr(oo), None)

    for bad in (PoolDesc(2, 9, 9, 8, 3, 3, 1, 1, VALID, NONE), PoolDesc(2, 9, 9, 8, 2, 2, 2, 2, VALID, NONE),
                PoolDesc(2, 9, 9, 8, 2, 2, 1, 1, SAME, NONE), PoolDesc(2, 9, 9, 8, 2, 2, 1, 1, VALID, RELU)):
        assert call(bad, dw) != 0 and b"the pool must be 2x2" in lib.lce_b200_last_error()
    pool6, dw6, _ = _fused_descs(2, 9, 9, 6, 1, SAME, NONE)
    assert call(pool6, dw6) != 0 and b"unsupported depthwise shape" in lib.lce_b200_last_error()
    assert call(pool, dw, xx=x) != 0 and b"unaligned" in lib.lce_b200_last_error()
    assert call(pool, dw, oo=out) != 0 and b"unaligned" in lib.lce_b200_last_error()
    check(lib, call(pool, dw))


# --------------------------------------------------------------------------------------------- #
# ADD / MUL / activation
# --------------------------------------------------------------------------------------------- #
# name: (n, b_len, offset). vec: the 128-bit path (n above 4 x the grid-stride cap of 1.2 M threads);
# the others take the scalar path: n % 4 != 0 above the cap, offset views, broadcasts
ELT_LAYOUTS = {
    "vec": (4 * 1_300_003, None, 0),
    "odd_n": (1_300_001, None, 0),
    "offset": (1003, None, 1),
    "bcast_last": (37 * 40_000, 37, 0),
    "bcast_1": (1_250_000, 1, 0),
}
ELT_CASES = [(op, lay, (i + j) % 4) for i, op in enumerate(("add", "mul")) for j, lay in enumerate(ELT_LAYOUTS)] + \
    [("act", "vec", RELU), ("act", "odd_n", RELU6), ("act", "offset", RELU_N1_TO_1)]


@pytest.mark.parametrize("op,layout,act", ELT_CASES)
def test_eltwise_is_bit_exact(torch, lib, rng, op, layout, act):
    n, b_len, offset = ELT_LAYOUTS[layout]
    b_len = b_len or n
    a = gauss_data(rng, n, 4.0)
    out = nan_dev(torch, n, offset)
    ad = to_dev(torch, a, offset)
    if op == "act":
        check(lib, lib.lce_b200_f32_activation(ptr(ad), ptr(out), C.c_int64(n), act, None))
        want = act_f32(a, act)
    else:
        b = gauss_data(rng, b_len, 2.0)
        fn = lib.lce_b200_f32_add if op == "add" else lib.lce_b200_f32_mul
        bd = to_dev(torch, b, offset)
        check(lib, fn(ptr(ad), ptr(bd), ptr(out), C.c_int64(n), C.c_int64(b_len), act, None))
        bb = np.tile(b, n // b_len)
        want = act_f32(a + bb if op == "add" else a * bb, act)
    assert np.array_equal(host(torch, out, n).view(np.int32), want.view(np.int32))


def test_eltwise_refuses_shapes_that_do_not_broadcast(torch, lib):
    a, out = to_dev(torch, np.ones(10, np.float32)), nan_dev(torch, 10)
    for fn, name in ((lib.lce_b200_f32_add, b"add"), (lib.lce_b200_f32_mul, b"mul")):
        for b_len in (3, 0, -1):
            assert fn(ptr(a), ptr(a), ptr(out), C.c_int64(10), C.c_int64(b_len), NONE, None) != 0
            assert name + b": operand shapes do not broadcast" in lib.lce_b200_last_error()


# --------------------------------------------------------------------------------------------- #
# MEAN over H, W
# --------------------------------------------------------------------------------------------- #
@pytest.mark.parametrize("hw", [1, 49, 3136])
@pytest.mark.parametrize("pre_act", [None, RELU, RELU6])
def test_mean_hw_is_bit_exact(torch, lib, rng, hw, pre_act):
    B, Cc = 3, 100      # B * C > 256: more than one block
    h = {1: 1, 49: 7, 3136: 56}[hw]
    x = gauss_data(rng, (B, h, hw // h, Cc), 3.0)
    out = nan_dev(torch, (B, Cc))
    xd = to_dev(torch, x)
    if pre_act is None:
        check(lib, lib.lce_b200_f32_mean_hw(ptr(xd), ptr(out), B, h, hw // h, Cc, None))
    else:
        check(lib, lib.lce_b200_f32_mean_hw_act(ptr(xd), ptr(out), B, h, hw // h, Cc, pre_act, None))
    a = act_f32(x.reshape(B, hw, Cc), pre_act or NONE)
    want = np.add.accumulate(a, axis=1, dtype=np.float32)[:, -1] / np.float32(hw)
    assert np.array_equal(host(torch, out, (B, Cc)).view(np.int32), want.view(np.int32))


# --------------------------------------------------------------------------------------------- #
# SOFTMAX
# --------------------------------------------------------------------------------------------- #
@pytest.mark.parametrize("beta", [1.0, 0.5, 3.0])
@pytest.mark.parametrize("cols", [1, 5, 1000, 1024, 1025, 4099])
def test_softmax_matches_fp64(torch, lib, rng, cols, beta):
    """Bound, with u = 2^-24: t = beta (x - max) is rounded twice (relative error <= 2u |t| in
    exp(t)); expf is within 2 ulp (4u); the row sum (cols / 128 sequential adds per thread, then a
    tree of 7) adds <= (cols + 8) u of the sum; the division u. Subnormal results are within a few
    ulp of 2^-149."""
    rows = 7
    x = rng.uniform(-80, 80, (rows, cols)).astype(np.float32)
    x[0, :] = x[0, 0]   # one row of equal logits
    out = nan_dev(torch, (rows, cols))
    xd = to_dev(torch, x)
    check(lib, lib.lce_b200_f32_softmax(ptr(xd), ptr(out), C.c_int64(rows), cols, C.c_float(beta), None))
    got = host(torch, out, (rows, cols)).astype(np.float64)
    u = 2.0 ** -24
    t = beta * (x.astype(np.float64) - x.max(axis=1, keepdims=True))
    e = np.exp(t)
    S = e.sum(axis=1, keepdims=True)
    ref = e / S
    term = 2 * u * np.abs(t) + 4 * u
    sum_rel = (e * term).sum(axis=1, keepdims=True) / S + (cols + 8) * u
    bound = ref * (term + sum_rel + u) + 2.0 ** -146
    err = np.abs(got - ref)
    assert (err <= bound).all(), (err / bound).max()
    assert (np.abs(got.sum(axis=1) - 1) <= bound.sum(axis=1) + cols * 2.0 ** -53).all()


# --------------------------------------------------------------------------------------------- #
# DEQUANTIZE (int8 / uint8 -> float)
# --------------------------------------------------------------------------------------------- #
@pytest.mark.parametrize("n", [1024, 1025, 1039, 2368 * 256 * 16 + 1615])   # n % 16 = 0, 1, 15; grid-stride
@pytest.mark.parametrize("in_type", [T_INT8, T_UINT8], ids=["int8", "uint8"])
def test_dequantize_affine_is_bit_exact(torch, lib, in_type, n):
    lo, dt = (-128, np.int8) if in_type == T_INT8 else (0, np.uint8)
    q = ((np.arange(n) % 256) + lo).astype(dt)   # every code
    qd = to_dev(torch, q)
    for scale in (1 / 255, 4 / 127, 0.5):
        for zp in (lo, lo + 255, 3):
            out = nan_dev(torch, n)
            check(lib, lib.lce_b200_dequantize_affine(in_type, ptr(qd), ptr(out), C.c_int64(n), C.c_double(scale),
                                                      C.c_int32(zp), None))
            want = (np.float64(scale) * (q.astype(np.int64) - zp).astype(np.float64)).astype(np.float32)
            assert np.array_equal(host(torch, out, n).view(np.int32), want.view(np.int32)), (scale, zp)


def test_dequantize_affine_refuses_unaligned_buffers(torch, lib):
    q, out = to_dev(torch, np.zeros(64, np.int8), 1), nan_dev(torch, 64, 1)
    qa, outa = to_dev(torch, np.zeros(64, np.int8)), nan_dev(torch, 64)
    for qq, oo in ((q, outa), (qa, out)):
        assert lib.lce_b200_dequantize_affine(T_INT8, ptr(qq), ptr(oo), C.c_int64(64), C.c_double(1.0), C.c_int32(0),
                                              None) != 0
        assert b"16-byte aligned" in lib.lce_b200_last_error()


# --------------------------------------------------------------------------------------------- #
# PAD / PADV2 of 32-bit elements
# --------------------------------------------------------------------------------------------- #
PAD_CASES = [
    ((2, 3, 4, 5), (1, 0, 0, 0), (0, 0, 0, 0)),
    ((2, 3, 4, 5), (0, 2, 0, 0), (0, 1, 0, 0)),
    ((2, 3, 4, 5), (0, 0, 1, 3), (0, 0, 2, 0)),
    ((2, 3, 4, 5), (0, 0, 0, 0), (0, 0, 0, 2)),
    ((2, 3, 4, 5), (1, 2, 3, 4), (4, 3, 2, 1)),
    ((3, 7, 5, 33), (0, 0, 0, 0), (0, 0, 0, 0)),
    ((2, 0, 4, 5), (0, 1, 0, 0), (0, 2, 0, 0)),    # empty input axis, padded
    ((1, 6, 9, 70), (0, 1, 1, 0), (0, 1, 1, 0)),   # QuickNet-like spatial pad
]


@pytest.mark.parametrize("fill", [0xFFFFFFFF, 0xBF800000, 0], ids=["ones", "minus1f", "zero"])
@pytest.mark.parametrize("dtype", [np.float32, np.int32], ids=["float", "int32"])
@pytest.mark.parametrize("dims,before,after", PAD_CASES)
def test_pad4d_32_matches_numpy(torch, lib, rng, dims, before, after, dtype, fill):
    if dtype is np.float32:
        x = gauss_data(rng, dims)
    else:
        x = rng.integers(-2**31, 2**31, dims, dtype=np.int64).astype(np.int32)
    out_dims = tuple(d + a + b for d, a, b in zip(dims, before, after))
    want = np.pad(x.view(np.uint32), list(zip(before, after)), constant_values=fill)
    out = to_dev(torch, np.full(out_dims, SENTINEL, np.int32))
    a4 = lambda v: (C.c_int32 * 4)(*v)   # noqa: E731
    xd = to_dev(torch, x)
    check(lib, lib.lce_b200_pad4d_32(ptr(xd), ptr(out), a4(dims), a4(before), a4(after),
                                     C.c_uint32(fill), None))
    assert np.array_equal(host(torch, out, out_dims).view(np.uint32), want)


def test_pad4d_32_empty_output_writes_nothing(torch, lib):
    out = to_dev(torch, np.full(16, SENTINEL, np.int32))
    a4 = lambda v: (C.c_int32 * 4)(*v)   # noqa: E731
    check(lib, lib.lce_b200_pad4d_32(None, ptr(out), a4((2, 0, 4, 5)), a4((1, 0, 0, 0)), a4((0, 0, 1, 0)),
                                     C.c_uint32(0), None))
    assert (host(torch, out, 16) == SENTINEL).all()
