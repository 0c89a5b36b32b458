#!/usr/bin/env python
"""Mint the golden vectors under tests/golden/ from the REFERENCE ITSELF.

Needs oracle/_ref/liblce_ref.so: the reference's own headers, compiled by
oracle/Makefile from a larq/compute-engine checkout (`make -C oracle REF=<dir>`).
The resulting ``lce_golden_bconv.npz``, ``lce_golden_ops.npz`` and ``lce_golden.json``
are committed; the test-suite only reads them (``lce_testlib.load_golden``).
Inputs are regenerated from the recorded seeds by ``lce_testlib.make_bconv_case``
and ``lce_testlib.golden_op_cases``, so only outputs (or, for the full-size
config-1 case, SHA-256 digests of the outputs) are stored, split over two files
so that neither exceeds 1 MB. ``lce_random_walk.json`` holds the digests of the
reference's results on ``lce_testlib.random_walk_cases()``.

The case list re-runs the parameter grids of the reference's own op tests with
fixed seeds (they use std::random_device): bconv2d_test.cc:790-856 (SmallTest /
BigTest shapes), bmaxpool_test.cc:204-218, quantization_test.cc:121-130,
bitpack_test.cc:102-109.

Usage:  python tests/golden/make_golden.py
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import lce_testlib as L  # noqa: E402


def bconv_specs():
    """(batch,h,w,cin, fh,fw,cout, groups, stride, dilation, padding, pad_value,
    activation, out_type) -- a pruned walk of the reference's BigTest grid plus
    SmallTest shapes, the 16-bit-overflow shape and QuickNet-like shapes."""
    specs = []
    S, V = L.PADDING_SAME, L.PADDING_VALID
    shapes = [(1, 7, 7, 4), (3, 8, 5, 64), (2, 7, 7, 96), (1, 8, 5, 128),
              (1, 7, 7, 192), (1, 8, 5, 256), (1, 7, 7, 512), (1, 4, 4, 64)]
    filters = [(1, 1, 1), (3, 3, 1), (2, 3, 2), (1, 1, 3), (3, 3, 4), (2, 3, 5),
               (1, 1, 6), (3, 3, 7), (2, 3, 32), (3, 3, 64)]
    i = 0
    for shape in shapes:
        for filt in filters:
            for groups in (1, 2, 4):
                b, h, w, c = shape
                fh, fw, co = filt
                if groups > 1 and (c % groups or co % groups or (c // groups) % 32):
                    continue
                # rotate through the remaining axes instead of the full product
                stride = ((1, 1), (2, 3))[i % 2]
                dil = ((1, 1), (3, 2))[(i // 2) % 2]
                pad, pv = ((V, 1), (S, 0), (S, 1))[i % 3]
                act = (L.ACT_NONE, L.ACT_RELU)[(i // 3) % 2]
                ot = (L.OUT_FLOAT, L.OUT_INT8, L.OUT_BITPACKED)[(i // 5) % 3]
                i += 1
                if pad == S and pv == 0 and c % 2:
                    pv = 1
                if pad == V and ((fh - 1) * dil[0] + 1 > h or (fw - 1) * dil[1] + 1 > w):
                    dil = (1, 1)
                specs.append((b, h, w, c, fh, fw, co, groups, stride, dil, pad,
                              pv, act, ot))
    # other activations
    for act in (L.ACT_RELU6, L.ACT_RELU_N1_TO_1):
        for ot in (L.OUT_FLOAT, L.OUT_INT8):
            specs.append((2, 6, 6, 64, 3, 3, 32, 1, (1, 1), (1, 1), S, 1, act, ot))
    # 16-bit accumulator overflow shape (bconv2d_test.cc:818-833)
    for ot in (L.OUT_FLOAT, L.OUT_BITPACKED):
        specs.append((1, 6, 6, 3072, 5, 5, 4, 1, (1, 1), (1, 1), S, 1,
                      L.ACT_RELU, ot))
    # QuickNet / Bi-RealNet-like layers at reduced spatial size (SURVEY 8d table)
    for c, hw in ((64, 14), (128, 10), (256, 7), (512, 7)):
        specs.append((2, hw, hw, c, 3, 3, c, 1, (1, 1), (1, 1), S, 1, L.ACT_RELU,
                      L.OUT_FLOAT))
        specs.append((2, hw, hw, c, 3, 3, c, 1, (1, 1), (1, 1), S, 0, L.ACT_NONE,
                      L.OUT_FLOAT))
    specs.append((1, 14, 14, 64, 3, 3, 128, 1, (2, 2), (1, 1), S, 0, L.ACT_NONE,
                  L.OUT_FLOAT))
    return specs


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def write_random_walk(impl, source):
    """lce_random_walk.json: SHA-256 digests of the `impl` checker's outputs on
    lce_testlib.random_walk_cases(), kind 0 (the reference kernel) always and kind 1 (the
    optimised kernels) where they accept the case. `source` records where they came from."""
    cases = {}
    for n, case, optimised in L.random_walk_cases():
        args = (case.desc, case.inp, case.filt, case.mul, case.bias, case.thr)
        cases[str(n)] = {"kind0": digest(L.bconv2d(*args, impl=impl, kind=0))}
        if optimised:
            cases[str(n)]["kind1"] = digest(L.bconv2d(*args, impl=impl, kind=1))
    with open(os.path.join(HERE, "lce_random_walk.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_golden.py", "source": source,
                   "cases": cases}, f, indent=0)
    return len(cases)


def main():
    if L.load_ref() is None:
        sys.exit("oracle/_ref/liblce_ref.so missing: run `make -C oracle` here")
    arrays, index = {}, {"bconv": [], "bconv_full": [], "bconv_zpc": [], "quantize": [],
                         "dequantize": [], "bmaxpool": []}

    for n, s in enumerate(bconv_specs()):
        (b, h, w, c, fh, fw, co, g, st, dl, pad, pv, act, ot) = s
        seed = 1000 + n
        case = L.make_bconv_case(seed, b, h, w, c, fh, fw, co, g, st, dl, pad, pv,
                                 act, ot)
        out = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias,
                        case.thr, impl="ref", kind=0)
        key = f"bconv_{n}"
        arrays[key] = out
        index["bconv"].append({"key": key, "seed": seed, "spec": list(s)})

    # Zero padding as the OPTIMISED kernels compute it -- what the reference's default
    # registration returns: Kernel4x2Portable with one-padding, OutputTransform, then
    # zero_padding_correction::ApplyCorrection (kind 1 of oracle/ref_shim.cc). Float output, no
    # activation (bconv2d.cc:188-200), odd channel counts included.
    for n, (b, h, w, c, fh, fw, co, st, dl) in enumerate([
            (2, 8, 8, 64, 3, 3, 32, (1, 1), (1, 1)), (1, 16, 16, 128, 3, 3, 64, (2, 2), (1, 1)),
            (2, 7, 7, 96, 3, 3, 16, (1, 1), (1, 1)), (1, 12, 12, 32, 5, 5, 8, (1, 1), (2, 2)),
            (1, 9, 11, 64, 3, 3, 8, (2, 1), (1, 1)), (1, 5, 5, 33, 3, 3, 8, (1, 1), (1, 1)),
            (1, 6, 6, 64, 5, 5, 8, (2, 2), (1, 1)), (3, 7, 7, 512, 3, 3, 64, (1, 1), (1, 1)),
            (1, 14, 14, 256, 3, 3, 128, (2, 2), (1, 1)), (1, 10, 7, 100, 2, 3, 12, (1, 2), (1, 1))]):
        seed = 5000 + n
        case = L.make_bconv_case(seed, b, h, w, c, fh, fw, co, 1, st, dl, L.PADDING_SAME, 0,
                                 L.ACT_NONE, L.OUT_FLOAT)
        key = f"bconv_zpc_{n}"
        arrays[key] = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, None,
                                impl="ref", kind=1)
        index["bconv_zpc"].append({"key": key, "seed": seed,
                                   "spec": [b, h, w, c, fh, fw, co, list(st), list(dl)]})

    # config 1 (BASELINE.json configs[0]): 56x56x256 -> 256, k3 s1 SAME.
    # Outputs are 0.1-3.2 MB each, so only digests are stored.
    n = 0
    for pv in (1, 0):
        for act in (L.ACT_NONE, L.ACT_RELU):
            for ot in (L.OUT_FLOAT, L.OUT_INT8, L.OUT_BITPACKED):
                seed = n % 4
                case = L.make_bconv_case(seed, 1, 56, 56, 256, 3, 3, 256, 1,
                                         (1, 1), (1, 1), L.PADDING_SAME, pv, act,
                                         ot)
                ref0 = L.bconv2d(case.desc, case.inp, case.filt, case.mul,
                                 case.bias, case.thr, impl="ref", kind=0)
                entry = {"seed": seed, "pad_value": pv, "activation": act,
                         "out_type": ot, "sha256_reference_kernel": digest(ref0)}
                legal_opt = not (pv == 0 and (ot != L.OUT_FLOAT or act != L.ACT_NONE))
                if legal_opt:
                    ref1 = L.bconv2d(case.desc, case.inp, case.filt, case.mul,
                                     case.bias, case.thr, impl="ref", kind=1)
                    if pv == 1:
                        assert digest(ref1) == digest(ref0)
                    entry["sha256_indirect_kernel"] = digest(ref1)
                index["bconv_full"].append(entry)
                n += 1

    # LceQuantize / LceDequantize / LceBMaxPool2d grids: the inputs come from one seeded stream
    # (lce_testlib.golden_op_cases), so only the outputs are stored.
    for section, e, x in L.golden_op_cases():
        if section == "quantize":
            out = L.quantize(x, zero_point=e["zero_point"] if e["type"] == "i8" else 0, impl="ref")
        elif section == "dequantize":
            t = e["type"]
            out = L.dequantize(x, e["channels"], t, e["scale"], e["zero_point"], impl="ref").view(
                np.uint8 if t == L.T_BOOL else L._NP_T[t])
        else:
            out = L.bmaxpool(L.BMaxPoolDesc(*e["desc"]), x, impl="ref")
        arrays[e["key"]] = out
        index[section].append(e)

    sizes = {}
    for part, name in L.GOLDEN_FILES.items():
        path = os.path.join(HERE, name)
        np.savez_compressed(path, **{k: v for k, v in arrays.items()
                                     if k.startswith("bconv_") == (part == "bconv")})
        sizes[name] = os.path.getsize(path)
    with open(os.path.join(HERE, "lce_golden.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_golden.py",
                   "reference": "larq/compute-engine e6860fcf core headers via "
                                "oracle/ref_shim.cc (kReference kernel unless "
                                "stated)", "index": index}, f, indent=1)
    assert all(sz < 1e6 for sz in sizes.values()), sizes
    write_random_walk("ref", "larq/compute-engine e6860fcf core headers via oracle/ref_shim.cc")
    print(f"wrote {len(arrays)} arrays,", {k: f"{v/1e6:.2f} MB" for k, v in sizes.items()},
          {k: len(v) for k, v in index.items()})


if __name__ == "__main__":
    main()
