"""CPU tests of the checker itself: the plain-C oracle (oracle/lce_oracle.c) is
pinned against (1) the known-answer vectors in the reference's own tests, (2) the
committed golden vectors minted from the compiled reference headers
(tests/golden/make_golden.py), and (3) the reference's results on a 300-case random walk
(stored digests; live as well when oracle/_ref/liblce_ref.so is built)."""
import hashlib

import numpy as np
import pytest

import lce_testlib as L


@pytest.fixture(scope="module")
def golden():
    return L.load_golden()


def case_from_spec(entry):
    (b, h, w, c, fh, fw, co, g, st, dl, pad, pv, act, ot) = entry["spec"]
    return L.make_bconv_case(entry["seed"], b, h, w, c, fh, fw, co, g, tuple(st),
                             tuple(dl), pad, pv, act, ot)


# ---- (1) known answers held by the reference's own tests ------------------- #
def test_kat_bitpack_constant_folds():
    # LCE/mlir/tests/const-fold.mlir:4-27
    assert L.quantize(np.full((1, 32), 0.5, np.float32)).tolist() == [[0]]
    assert L.quantize(np.full((1, 32), -0.5, np.float32)).tolist() == [[-1]]
    assert np.all(L.dequantize(np.array([[0]], np.int32), 32) == 1.0)
    assert np.all(L.dequantize(np.array([[-1]], np.int32), 32) == -1.0)
    # LCE/mlir/tests/bitpack-weights.mlir:5-10: all +1 filter 16x3x3x3 -> zeros 16x3x3x1
    assert not L.quantize(np.ones((16, 3, 3, 3), np.float32)).any()
    assert L.quantize(np.ones((16, 3, 3, 3), np.float32)).shape == (16, 3, 3, 1)


def test_kat_bit_order_one_hot():
    # LCE/core/bitpacking/tests/bitpack_aarch64_test.cc:17-56: one-hot input i sets bit i
    for i in range(128):
        x = np.ones((1, 128), np.float32)
        x[0, i] = -1
        out = L.quantize(x).view(np.uint32)[0]
        expect = np.zeros(4, np.uint32)
        expect[i // 32] = np.uint32(1) << np.uint32(i % 32)
        assert np.array_equal(out, expect)


def test_kat_bit_semantics_special_values():
    # SURVEY 9.3-2 (values observed from the compiled reference)
    x = np.array([[-0.0, np.nan, -1e-30]], np.float32)
    assert L.quantize(x).tolist() == [[0x4]]
    i8 = np.array([[-128, -1, 0, 1, 127]], np.int8)
    assert L.quantize(i8, 0).tolist() == [[0x3]]
    assert L.quantize(i8, 1).tolist() == [[0x7]]
    assert L.quantize(i8, 128).tolist() == [[0x1F]]   # padding bits stay 0
    assert L.quantize(i8, -1000).tolist() == [[0]]


def test_kat_converter_thresholds():
    # LCE/mlir/tests/optimize.mlir:217-241
    import ctypes as C
    mul = np.array([-4, -3, -2, -1, 0, 1, 2, 3], np.float32)
    bias = np.array([-10, 8, 0.4, 1, -0.01, 0.5, -1, 2.71], np.float32)
    thr = np.empty(8, np.int32)
    L.load_oracle().lce_oracle_converter_thresholds(
        C.c_int(1), C.c_int(2), C.c_int(2), C.c_int(8), L._ptr(mul), L._ptr(bias),
        C.c_int(L.ACT_NONE), L._ptr(thr))
    assert thr.tolist() == [0, 3, 2, 2, -2**31, 2, 1, 2]


def test_bitpack_property_grid():
    # LCE/core/bitpacking/tests/bitpack_test.cc:19-109: every bit == (x < zp), pad bits 0
    rng = np.random.default_rng(0)
    for rows in (1, 2, 3, 8, 10, 15, 64):
        for cols in (1, 3, 16, 32, 33, 63, 64, 128):
            x = rng.uniform(-1.5, 1.5, (rows, cols)).astype(np.float32)
            assert np.array_equal(L.quantize(x), L.pack_signs(x))
            for zp in (-1000, -1, 0, 23, 127, 128):
                xi = rng.integers(-128, 128, (rows, cols), dtype=np.int8)
                assert np.array_equal(L.quantize(xi, zp),
                                      L.pack_signs(xi.astype(np.int32) - zp))


def test_quantize_dequantize_roundtrip():
    # LCE/tflite/tests/quantization_test.cc:76-111
    rng = np.random.default_rng(1)
    for c in (1, 2, 31, 32, 33, 64, 68, 130, 200):
        s = (rng.integers(0, 2, (2, 3, 3, c)) * 2 - 1).astype(np.float32)
        assert np.array_equal(L.dequantize(L.quantize(s), c), s)
        bl = s > 0
        assert np.array_equal(L.dequantize(L.quantize(bl), c, L.T_BOOL), bl)


def test_bmaxpool_is_float_maxpool_on_signs():
    # LCE/tflite/tests/bmaxpool_test.cc:144-201
    rng = np.random.default_rng(2)
    b, h, w, c, f, s = 2, 9, 7, 40, 3, 2
    x = (rng.integers(0, 2, (b, h, w, c)) * 2 - 1).astype(np.float32)
    d = L.BMaxPoolDesc(b, h, w, L.cdiv(c, 32), f, f, s, s, L.PADDING_SAME)
    out = L.dequantize(L.bmaxpool(d, L.quantize(x)), c)
    oh, ow = -(-h // s), -(-w // s)
    ph = max(0, (oh - 1) * s + f - h) // 2
    pw = max(0, (ow - 1) * s + f - w) // 2
    for oy in range(oh):
        for ox in range(ow):
            ys = slice(max(0, oy * s - ph), min(h, oy * s - ph + f))
            xs = slice(max(0, ox * s - pw), min(w, ox * s - pw + f))
            assert np.array_equal(out[:, oy, ox], x[:, ys, xs].max((1, 2)))


def test_bconv_matches_float_convolution():
    """The op test's own definition (bconv2d_test.cc:649-742): +-1 float conv,
    fused activation, then post multiply / bias."""
    rng_cases = [(3, 2, 6, 5, 40, 3, 3, 8, L.PADDING_SAME, 1, L.ACT_RELU),
                 (4, 1, 5, 5, 64, 2, 3, 5, L.PADDING_VALID, 1, L.ACT_NONE),
                 (5, 1, 6, 6, 32, 3, 3, 4, L.PADDING_SAME, 0, L.ACT_NONE)]
    for seed, b, h, w, c, fh, fw, co, pad, pv, act in rng_cases:
        case = L.make_bconv_case(seed, b, h, w, c, fh, fw, co, padding=pad,
                                 pad_value=pv, activation=act)
        out = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias)
        x = L.dequantize(case.inp, c).astype(np.float64)
        wt = L.dequantize(case.filt, c).astype(np.float64)
        oh, ow, ph, pw = L.out_shape(case.desc)
        fill = 1.0 if pv == 1 else 0.0
        xp = np.full((b, h + fh, w + fw, c), fill)
        xp[:, ph:ph + h, pw:pw + w] = x
        ref = np.zeros((b, oh, ow, co))
        for oy in range(oh):
            for ox in range(ow):
                patch = xp[:, oy:oy + fh, ox:ox + fw]
                ref[:, oy, ox] = np.einsum("bhwc,ohwc->bo", patch, wt)
        if act == L.ACT_RELU:
            ref = np.maximum(ref, 0)
        ref = ref * case.mul + case.bias
        assert np.allclose(out, ref, atol=1e-3)


# ---- (2) committed golden vectors minted from the reference --------------- #
def test_golden_bconv(golden):
    index, arrays = golden
    assert len(index["bconv"]) > 100
    for e in index["bconv"]:
        case = case_from_spec(e)
        out = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, case.thr)
        want = arrays[e["key"]]
        assert out.dtype == want.dtype and out.shape == want.shape, e
        assert np.array_equal(out.view(np.uint8), want.view(np.uint8)), e


def test_golden_bconv_config1_digests(golden):
    index, _ = golden
    for e in index["bconv_full"]:
        case = L.make_bconv_case(e["seed"], 1, 56, 56, 256, 3, 3, 256, 1, (1, 1),
                                 (1, 1), L.PADDING_SAME, e["pad_value"],
                                 e["activation"], e["out_type"])
        out = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias,
                        case.thr, threads=1)
        assert hashlib.sha256(out.tobytes()).hexdigest() == e["sha256_reference_kernel"], e


def zpc_case(e):
    b, h, w, c, fh, fw, co, st, dl = e["spec"]
    return L.make_bconv_case(e["seed"], b, h, w, c, fh, fw, co, 1, tuple(st), tuple(dl),
                             L.PADDING_SAME, 0, L.ACT_NONE, L.OUT_FLOAT)


def test_golden_zero_padding_correction(golden):
    """The optimised kernels' zero padding (the reference's DEFAULT registration): the oracle's
    restatement of zero_padding_correction.h equals the vectors minted from the reference's own
    Kernel4x2Portable + ApplyCorrection, bit for bit; the reference kernel's integer result on the
    same inputs differs (the two are different float computations), which is why both exist."""
    index, arrays = golden
    assert len(index["bconv_zpc"]) == 10
    differs = 0
    for e in index["bconv_zpc"]:
        case = zpc_case(e)
        out = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, None, kind=1)
        want = arrays[e["key"]]
        assert out.dtype == want.dtype and out.shape == want.shape, e
        assert np.array_equal(out.view(np.uint8), want.view(np.uint8)), e
        if case.desc.channels_in % 2 == 0:
            ref_kernel = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, None, kind=0)
            assert np.allclose(ref_kernel, want, rtol=1e-3, atol=1e-3)      # bconv2d_test.cc:396-405
            differs += int(not np.array_equal(ref_kernel.view(np.uint8), want.view(np.uint8)))
    assert differs > 0
    # config 1 with zero padding: the committed digest of the reference's optimised kernel
    for e in index["bconv_full"]:
        if e["pad_value"] == 0 and "sha256_indirect_kernel" in e:
            case = L.make_bconv_case(e["seed"], 1, 56, 56, 256, 3, 3, 256, 1, (1, 1), (1, 1),
                                     L.PADDING_SAME, 0, e["activation"], e["out_type"])
            out = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, None, kind=1)
            assert hashlib.sha256(out.tobytes()).hexdigest() == e["sha256_indirect_kernel"], e


def test_optimised_semantics_refusals():
    """bconv2d.cc:188-200, optimised branch: zero padding needs float output, no activation."""
    for act, ot in ((L.ACT_RELU, L.OUT_FLOAT), (L.ACT_NONE, L.OUT_INT8), (L.ACT_NONE, L.OUT_BITPACKED)):
        case = L.make_bconv_case(1, 1, 6, 6, 64, 3, 3, 8, pad_value=0, activation=act, out_type=ot)
        with pytest.raises(ValueError):
            L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, case.thr, kind=1)
    # everywhere else the optimised kernels compute the reference kernel's integers
    case = L.make_bconv_case(2, 2, 7, 5, 96, 3, 2, 24, pad_value=1, activation=L.ACT_RELU)
    a = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, None, kind=1)
    b = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, None, kind=0)
    assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


def test_golden_quantize_dequantize_bmaxpool(golden):
    index, arrays = golden
    for e in index["quantize"]:
        x = arrays[e["key"] + "_in"]
        assert np.array_equal(L.quantize(x, e["zero_point"]), arrays[e["key"]]), e
    for e in index["dequantize"]:
        out = L.dequantize(arrays[e["key"] + "_in"], e["channels"], e["type"],
                           e["scale"], e["zero_point"])
        assert np.array_equal(out.view(np.uint8), arrays[e["key"]].view(np.uint8)), e
    for e in index["bmaxpool"]:
        d = L.BMaxPoolDesc(*e["desc"])
        assert np.array_equal(L.bmaxpool(d, arrays[e["key"] + "_in"]), arrays[e["key"]]), e


# ---- (3) against the compiled reference: stored digests, and live where oracle/_ref exists -- #
def test_live_reference_random_walk():
    """300 seeded LceBconv2d cases (lce_testlib.random_walk_cases): the oracle's reference-kernel
    result (kind 0) and, where legal, its optimised-kernel result (kind 1) equal the reference's,
    held as digests in tests/golden/lce_random_walk.json; with oracle/_ref built, also compared
    with the compiled reference live."""
    stored = L.load_random_walk()
    ref = L.load_ref()
    seen = 0
    for n, case, optimised in L.random_walk_cases():
        e, where = stored[str(n)], L.desc_to_dict(case.desc)
        args = (case.desc, case.inp, case.filt, case.mul, case.bias, case.thr)
        for kind in (0, 1) if optimised else (0,):
            a = L.bconv2d(*args, kind=kind)
            assert hashlib.sha256(a.tobytes()).hexdigest() == e[f"kind{kind}"], (n, kind, where)
            if ref is not None:
                b = L.bconv2d(*args, impl="ref", kind=kind)
                assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), (n, kind, where)
        assert optimised == ("kind1" in e), (n, where)
        seen += 1
    assert seen == len(stored)


def test_oracle_bgemm_equals_1x1_bconv():
    """The BGEMM orientation (optimized_bgemm.h:126-151): a 1x1 s1 conv is a plain
    BGEMM over [M=B*H*W, Kw] x [N, Kw]."""
    case = L.make_bconv_case(11, 2, 5, 4, 96, 1, 1, 40, padding=L.PADDING_VALID,
                             out_type=L.OUT_FLOAT, activation=L.ACT_RELU)
    conv = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias)
    m, b, cmin, cmax = L.fold(case.desc, case.mul, case.bias)
    A = case.inp.reshape(-1, 3)
    W = case.filt.reshape(40, 3)
    out = L.bgemm(A, W, L.OUT_FLOAT, (cmin, cmax), m, b)
    assert np.array_equal(out.view(np.uint8).ravel(), conv.view(np.uint8).ravel())
    raw = L.bgemm(A, W)
    assert raw.min() >= 0 and raw.max() <= 96
