"""CPU test: the C-ABI shared library builds, loads, and exports every symbol that
include/lce_b200.h declares (no compute calls without a GPU), and refuses to run
without a device instead of falling back to a CPU path."""
import ctypes as C
import os
import re

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from compute_engine_b200 import build
    path = build.build_cuda()
    return C.CDLL(path)


def declared_symbols(header):
    text = open(os.path.join(REPO, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(lce_b200_[a-z0-9_]+)\s*\(", text)))


def test_every_declared_symbol_is_exported(lib):
    names = declared_symbols("lce_b200.h")
    assert len(names) >= 19
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/lce_b200.h but not exported"


def test_binding_lists_the_same_symbols():
    from compute_engine_b200 import capi
    assert sorted(capi.EXPORTS) == declared_symbols("lce_b200.h")


def test_abi_version_and_shape_inference_without_gpu(lib):
    from compute_engine_b200 import capi
    assert lib.lce_b200_abi_version() == 1
    # shape inference is host logic: usable without a device
    d = capi.BconvDesc(1, 56, 56, 256, 3, 3, 256, 1, 1, 1, 1, 1, capi.PADDING_SAME, 1,
                       capi.ACT_NONE, capi.OUT_FLOAT, 1.0, 0)
    oh, ow, ph, pw = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    assert lib.lce_b200_bconv2d_out_shape(C.byref(d), C.byref(oh), C.byref(ow), C.byref(ph),
                                          C.byref(pw)) == 0
    assert (oh.value, ow.value, ph.value, pw.value) == (56, 56, 1, 1)
    d.pad_value = 2   # bconv2d.cc:113-116
    assert lib.lce_b200_bconv2d_out_shape(C.byref(d), C.byref(oh), C.byref(ow), C.byref(ph),
                                          C.byref(pw)) != 0
    lib.lce_b200_last_error.restype = C.c_char_p
    assert b"pad_values must be 0 or 1" in lib.lce_b200_last_error()


def test_shape_inference_matches_oracle(lib):
    import lce_testlib as L
    from compute_engine_b200 import capi
    for (h, w, fh, fw, sh, sw, dh, dw, pad) in [
            (7, 7, 3, 3, 1, 1, 1, 1, 0), (8, 5, 2, 3, 2, 3, 3, 2, 0), (8, 5, 2, 3, 2, 3, 1, 1, 1),
            (56, 56, 3, 3, 2, 2, 1, 1, 0), (6, 6, 5, 5, 1, 1, 1, 1, 1), (9, 4, 1, 1, 3, 2, 1, 1, 0)]:
        d = capi.BconvDesc(2, h, w, 64, fh, fw, 32, 1, sh, sw, dh, dw, pad, 1, 0, 0, 1.0, 0)
        o = [C.c_int() for _ in range(4)]
        assert lib.lce_b200_bconv2d_out_shape(C.byref(d), *[C.byref(x) for x in o]) == 0
        want = L.out_shape(L.BconvDesc(2, h, w, 64, fh, fw, 32, 1, sh, sw, dh, dw, pad, 1, 0, 0,
                                       1.0, 0))
        assert tuple(x.value for x in o) == want


def test_float_shape_inference_matches_tflite(lib):
    """lce_b200_f32_conv_out_shape / _pool_out_shape against TFLite's rule: SAME out = ceil(in / s),
    VALID out = max(floor((in - (k - 1) d - 1) / s) + 1, 0)."""
    from test_gpu_float_kernels import ConvDesc, PoolDesc, tfl_out_pad
    oh, ow = C.c_int(), C.c_int()
    for n in (1, 2, 3, 4, 7, 8, 56):
        for k in (1, 2, 3, 5, 7):
            for s in (1, 2, 3):
                for d in (1, 2):
                    for pad in (0, 1):
                        want = tfl_out_pad(pad, n, k, s, d)[0]
                        desc = ConvDesc(2, n, n + 1, 3, k, 1, 4, s, 1, d, 1, pad, 0)
                        assert lib.lce_b200_f32_conv_out_shape(C.byref(desc), C.byref(oh), C.byref(ow)) == 0
                        assert (oh.value, ow.value) == (want, tfl_out_pad(pad, n + 1, 1, 1)[0]), (n, k, s, d, pad)
                        if d == 1:
                            p = PoolDesc(2, n + 1, n, 4, 1, k, 1, s, pad, 0)
                            assert lib.lce_b200_f32_pool_out_shape(C.byref(p), C.byref(oh), C.byref(ow)) == 0
                            assert (oh.value, ow.value) == (tfl_out_pad(pad, n + 1, 1, 1)[0], want), (n, k, s, pad)


def test_no_cpu_fallback_without_device(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    from compute_engine_b200 import capi
    import numpy as np
    d = capi.BconvDesc(1, 4, 4, 32, 1, 1, 8, 1, 1, 1, 1, 1, 1, 1, 0, 0, 1.0, 0)
    with pytest.raises(capi.LceError, match="no CUDA device"):
        capi.BConv2d(d, np.zeros((8, 1, 1, 1), np.int32), np.ones(8, np.float32),
                     np.ones(8, np.float32))


def test_builtin_kernels_header_symbols_are_exported(lib):
    names = declared_symbols("lce_b200_builtins.h")
    assert len(names) == 18
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/lce_b200_builtins.h but not exported"
