"""The stand-alone ABI mirror (include/lce_b200_tflite.h) must lay out the TFLite C
structs exactly like the reference's vendored tensorflow/lite/core/c/common.h. The
proof is a compile of oracle/abi_check.cc (static_asserts on every size / offset)
against that header, so it runs where REF names a larq/compute-engine checkout (the
variable oracle/Makefile reads)."""
import os
import subprocess

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TF = os.path.join(os.environ.get("REF", ""), "third_party", "tensorflow")


@pytest.mark.skipif(not os.environ.get("REF") or not os.path.isdir(TF),
                    reason="needs REF=<larq/compute-engine checkout> for TFLite's common.h")
def test_abi_mirror_matches_vendored_tflite_header():
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-I", TF,
                        os.path.join(REPO, "oracle", "abi_check.cc")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]


def test_registration_factories_are_exported():
    import ctypes as C
    import re
    from compute_engine_b200 import build
    lib = C.CDLL(build.host_lib_path())
    text = open(os.path.join(REPO, "include", "lce_b200_tflite.h")).read()
    names = sorted(set(re.findall(r"\b(lce_b200_Register_[A-Z0-9_]+|lce_b200_[sg]et_stream)\s*\(", text)))
    assert len(names) == 9
    for n in names:
        assert hasattr(lib, n), n
    # C++ names identical to the reference's (lce_ops_register.h:16-21)
    out = subprocess.run(["nm", "-D", "--defined-only", build.host_lib_path()],
                         capture_output=True, text=True).stdout
    for sym in ("_ZN14compute_engine6tflite17Register_BCONV_2DEv",
                "_ZN14compute_engine6tflite21Register_BCONV_2D_REFEv",
                "_ZN14compute_engine6tflite36Register_BCONV_2D_OPT_INDIRECT_BGEMMEv",
                "_ZN14compute_engine6tflite17Register_QUANTIZEEv",
                "_ZN14compute_engine6tflite19Register_DEQUANTIZEEv",
                "_ZN14compute_engine6tflite20Register_BMAXPOOL_2DEv"):
        assert sym in out, sym
    # every registration carries the four callbacks the reference fills
    class Reg(C.Structure):
        _fields_ = [("init", C.c_void_p), ("free", C.c_void_p), ("prepare", C.c_void_p),
                    ("invoke", C.c_void_p)]
    for n in names:
        if "Register" not in n:
            continue
        f = getattr(lib, n)
        f.restype = C.POINTER(Reg)
        r = f().contents
        assert r.prepare and r.invoke
        if "QUANTIZE" in n:   # quantization.cc:149-159: init = free = nullptr
            assert not r.init and not r.free
        else:
            assert r.init and r.free
