"""GPU parity tests (run on the B200 box): the CUDA path, called through the C-ABI
(compute_engine_b200.capi -> liblce_b200.so), against the CPU oracle on the same
seeded inputs and against the committed golden vectors minted from the reference.
Bar: bit-exact for bitpacked / int8 / int32 results AND for float results (the
epilogue reproduces the reference's two-rounding multiply-add)."""
import hashlib

import numpy as np
import pytest
import torch

import lce_testlib as L

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi():
    from compute_engine_b200 import capi as m
    m.lib()
    return m


@pytest.fixture(scope="module")
def golden():
    return L.load_golden()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def gpu_desc(capi, d: L.BconvDesc):
    return capi.BconvDesc(*[getattr(d, n) for n, _ in d._fields_])


def run_gpu_bconv(capi, case, float_input=None):
    plan = capi.BConv2d(gpu_desc(capi, case.desc), case.filt, case.mul, case.bias, case.thr)
    x = dev(case.inp) if float_input is None else dev(float_input)
    out = plan(x)
    torch.cuda.synchronize()
    res = out.cpu().numpy()
    plan.close()
    return res


def assert_same_bits(a, b, msg=""):
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape, msg)
    if not np.array_equal(a.view(np.uint8), b.view(np.uint8)):
        bad = np.argwhere(a != b)
        raise AssertionError(f"{msg}: {len(bad)} mismatches, first at {bad[:3].tolist()} "
                             f"got {a[tuple(bad[0])]} want {b[tuple(bad[0])]}")


# ------------------------------ LceQuantize ------------------------------- #
def test_quantize_golden(capi, golden):
    index, arrays = golden
    for e in index["quantize"]:
        x = arrays[e["key"] + "_in"]
        got = capi.quantize(dev(x), e["zero_point"]).cpu().numpy()
        assert_same_bits(got, arrays[e["key"]], str(e))


def test_quantize_fast_path_and_special_values(capi):
    rng = np.random.default_rng(3)
    for shape in [(1, 32), (5, 7, 64), (2, 56, 56, 64), (3, 9, 9, 256), (1000, 32), (1, 33, 96)]:
        x = rng.standard_normal(shape).astype(np.float32)
        flat = x.reshape(-1)
        sp = np.array([-0.0, 0.0, np.nan, -np.nan, -1e-30, -1e-45, 1e-45, -np.inf, np.inf,
                       -1.17e-38, np.float32(-1e-40)], np.float32)
        pos = rng.choice(flat.size, size=min(flat.size, 4 * sp.size), replace=False)
        flat[pos] = np.resize(sp, pos.size)
        assert_same_bits(capi.quantize(dev(x)).cpu().numpy(), L.quantize(x), str(shape))
    # empty tensors (ragged edge case)
    assert capi.quantize(torch.empty((0, 64), device="cuda")).shape == (0, 2)


def test_quantize_large_is_idempotent_under_roundtrip(capi):
    # full-size property: Quantize(Dequantize(Quantize(x))) == Quantize(x), and the
    # checksum of words equals the oracle's on a strided sample.
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn((256, 56, 56, 64), device="cuda", generator=g)
    q = capi.quantize(x)
    back = capi.dequantize(q, 64)
    assert torch.equal(back, torch.where(x < 0, -1.0, 1.0))
    assert torch.equal(capi.quantize(back), q)
    sample = x[::37].cpu().numpy()
    assert_same_bits(q[::37].cpu().numpy(), L.quantize(sample))


# ----------------------------- LceDequantize ------------------------------ #
def test_dequantize_golden(capi, golden):
    index, arrays = golden
    tmap = {L.T_FLOAT: torch.float32, L.T_INT8: torch.int8, L.T_BOOL: torch.bool}
    for e in index["dequantize"]:
        got = capi.dequantize(dev(arrays[e["key"] + "_in"]), e["channels"], tmap[e["type"]],
                              e["scale"], e["zero_point"]).cpu().numpy()
        assert np.array_equal(got.view(np.uint8), arrays[e["key"]].view(np.uint8)), e


# ----------------------------- LceBMaxPool2d ------------------------------ #
def test_bmaxpool_golden(capi, golden):
    index, arrays = golden
    for e in index["bmaxpool"]:
        b, h, w, c, fh, fw, sh, sw, pad = e["desc"]
        got = capi.bmaxpool(dev(arrays[e["key"] + "_in"]), (fh, fw), (sh, sw), pad).cpu().numpy()
        assert_same_bits(got, arrays[e["key"]], str(e))


# ------------------------------- LceBconv2d ------------------------------- #
def test_bconv_golden(capi, golden):
    index, arrays = golden
    for e in index["bconv"]:
        (b, h, w, c, fh, fw, co, g, st, dl, pad, pv, act, ot) = e["spec"]
        case = L.make_bconv_case(e["seed"], b, h, w, c, fh, fw, co, g, tuple(st), tuple(dl),
                                 pad, pv, act, ot)
        assert_same_bits(run_gpu_bconv(capi, case), arrays[e["key"]], str(e["spec"]))


def test_bconv_golden_zero_padding_correction(capi, golden):
    """Vectors minted from the reference's optimised kernel + zero_padding_correction."""
    index, arrays = golden
    for e in index["bconv_zpc"]:
        b, h, w, c, fh, fw, co, st, dl = e["spec"]
        case = L.make_bconv_case(e["seed"], b, h, w, c, fh, fw, co, 1, tuple(st), tuple(dl),
                                 L.PADDING_SAME, 0, L.ACT_NONE, L.OUT_FLOAT)
        plan = capi.BConv2d(gpu_desc(capi, case.desc), case.filt, case.mul, case.bias)
        plan.set_zero_padding_mode(1)
        got = plan(dev(case.inp)).cpu().numpy()
        plan.close()
        assert_same_bits(got, arrays[e["key"]], str(e["spec"]))


def test_bconv_config1_digests(capi, golden):
    """BASELINE.json configs[0]: 56x56x256 -> 256, k3 s1 SAME; digests minted from the
    reference's BConv2DReference (and equal to its indirect-BGEMM kernel for one-padding)."""
    index, _ = golden
    for e in index["bconv_full"]:
        case = L.make_bconv_case(e["seed"], 1, 56, 56, 256, 3, 3, 256, 1, (1, 1), (1, 1),
                                 L.PADDING_SAME, e["pad_value"], e["activation"], e["out_type"])
        out = run_gpu_bconv(capi, case)
        assert hashlib.sha256(out.tobytes()).hexdigest() == e["sha256_reference_kernel"], e


def test_bconv_random_walk_vs_oracle(capi):
    rng = np.random.default_rng(2024)
    n_done = 0
    for n in range(400):
        c = int(rng.choice([1, 3, 4, 31, 32, 33, 64, 96, 128, 192, 256, 288]))
        g = int(rng.choice([1, 2, 3])) if c % 96 == 0 or c % 64 == 0 else 1
        if g > 1 and (c % g or (c // g) % 32):
            g = 1
        co = int(rng.choice([1, 2, 3, 8, 31, 32, 33, 64, 65, 72, 130])) * g
        fh, fw = int(rng.integers(1, 4)), int(rng.integers(1, 5))
        h, w = int(rng.integers(1, 12)), int(rng.integers(1, 12))
        st = (int(rng.integers(1, 3)), int(rng.integers(1, 4)))
        dl = (int(rng.integers(1, 3)), int(rng.integers(1, 3)))
        pad, pv = [(L.PADDING_VALID, 1), (L.PADDING_SAME, 0), (L.PADDING_SAME, 1)][n % 3]
        if pad == L.PADDING_VALID and ((fh - 1) * dl[0] + 1 > h or (fw - 1) * dl[1] + 1 > w):
            continue
        if pad == L.PADDING_SAME and pv == 0 and c % 2:
            pv = 1
        ot = [L.OUT_FLOAT, L.OUT_INT8, L.OUT_BITPACKED][int(rng.integers(0, 3))]
        act = int(rng.integers(0, 4))
        if ot == L.OUT_BITPACKED and act not in (L.ACT_NONE, L.ACT_RELU):
            act = L.ACT_NONE
        case = L.make_bconv_case(5000 + n, int(rng.integers(1, 4)), h, w, c, fh, fw, co, g, st,
                                 dl, pad, pv, act, ot)
        want = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, case.thr)
        assert_same_bits(run_gpu_bconv(capi, case), want, str(L.desc_to_dict(case.desc)))
        n_done += 1
    assert n_done > 300


def test_bconv_negative_and_zero_multipliers(capi):
    # multipliers of either sign / zero, biases of either sign (the converter emits these)
    case = L.make_bconv_case(77, 2, 9, 9, 128, 3, 3, 64, activation=L.ACT_RELU)
    rng = np.random.default_rng(77)
    case.mul = rng.uniform(-2, 2, 64).astype(np.float32)
    case.mul[::7] = 0.0
    case.bias = rng.uniform(-3, 3, 64).astype(np.float32)
    for ot in (L.OUT_FLOAT, L.OUT_INT8):
        case.desc.out_type = ot
        case.desc.out_scale, case.desc.out_zero_point = 0.25, -3
        want = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias)
        assert_same_bits(run_gpu_bconv(capi, case), want)


def test_bconv_float_input_prologue(capi):
    """LceQuantize fused in front of LceBconv2d: float NHWC input."""
    rng = np.random.default_rng(8)
    for (b, h, w, c, co) in [(2, 14, 14, 64, 64), (1, 7, 7, 512, 96), (3, 5, 6, 96, 40)]:
        xf = rng.standard_normal((b, h, w, c)).astype(np.float32)
        xf.reshape(-1)[::13] = -0.0
        case = L.make_bconv_case(9, b, h, w, c, 3, 3, co, activation=L.ACT_RELU)
        case.inp = L.quantize(xf)
        want = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias)
        assert_same_bits(run_gpu_bconv(capi, case, float_input=xf), want)


def test_bconv_resize_and_empty_batch(capi):
    case = L.make_bconv_case(21, 2, 8, 8, 64, 3, 3, 32)
    plan = capi.BConv2d(gpu_desc(capi, case.desc), case.filt, case.mul, case.bias)
    out = plan(dev(case.inp)).cpu().numpy()
    assert_same_bits(out, L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias))
    # Prepare again after a resize (bconv2d.cc:295-297): new batch and spatial size
    big = L.make_bconv_case(22, 5, 11, 6, 64, 3, 3, 32)
    big.filt, big.mul, big.bias = case.filt, case.mul, case.bias
    out = plan(dev(big.inp)).cpu().numpy()
    assert out.shape == (5, 11, 6, 32)
    assert_same_bits(out, L.bconv2d(big.desc, big.inp, big.filt, big.mul, big.bias))
    empty = plan(torch.empty((0, 11, 6, 2), dtype=torch.int32, device="cuda"))
    assert empty.shape == (0, 11, 6, 32)
    plan.close()


def test_bconv_host_buffer_call(capi):
    case = L.make_bconv_case(31, 3, 10, 10, 96, 3, 3, 48, out_type=L.OUT_BITPACKED)
    plan = capi.BConv2d(gpu_desc(capi, case.desc), case.filt, None, None, case.thr)
    out = np.empty(plan.out_shape(), np.int32)
    plan.run_host(np.ascontiguousarray(case.inp), out)
    assert_same_bits(out, L.bconv2d(case.desc, case.inp, case.filt, thr=case.thr))
    plan.close()


def test_bconv_refusals_match_reference(capi):
    # zero padding (bconv2d.cc:188-200): an odd channel count AND a fused activation satisfies
    # neither the reference kernel's rule nor the optimised kernels'
    d = capi.BconvDesc(1, 8, 8, 33, 3, 3, 8, 1, 1, 1, 1, 1, capi.PADDING_SAME, 0, 1, 0, 1.0, 0)
    with pytest.raises(capi.LceError, match="Zero-padding is only supported"):
        capi.BConv2d(d, np.zeros((8, 3, 3, 2), np.int32), np.ones(8, np.float32),
                     np.ones(8, np.float32))
    # odd channel count, float output, no activation: only the optimised kernels' result exists
    d = capi.BconvDesc(1, 8, 8, 33, 3, 3, 8, 1, 1, 1, 1, 1, capi.PADDING_SAME, 0, 0, 0, 1.0, 0)
    plan = capi.BConv2d(d, np.zeros((8, 3, 3, 2), np.int32), np.ones(8, np.float32), np.ones(8, np.float32))
    with pytest.raises(capi.LceError, match="Zero-padding is only supported"):
        plan.set_zero_padding_mode(0)
    plan.close()
    # even channel count with a fused activation: only the reference kernel's result exists
    d = capi.BconvDesc(1, 8, 8, 64, 3, 3, 8, 1, 1, 1, 1, 1, capi.PADDING_SAME, 0, 1, 0, 1.0, 0)
    plan = capi.BConv2d(d, np.zeros((8, 3, 3, 2), np.int32), np.ones(8, np.float32), np.ones(8, np.float32))
    with pytest.raises(capi.LceError, match="Zero-padding is only supported"):
        plan.set_zero_padding_mode(1)
    plan.close()
    d = capi.BconvDesc(1, 8, 8, 64, 3, 3, 8, 1, 1, 1, 1, 1, capi.PADDING_SAME, 3, 0, 0, 1.0, 0)
    with pytest.raises(capi.LceError, match="pad_values must be 0 or 1"):
        capi.BConv2d(d, np.zeros((8, 3, 3, 2), np.int32), np.ones(8, np.float32),
                     np.ones(8, np.float32))
    d = capi.BconvDesc(1, 8, 8, 96, 3, 3, 8, 2, 1, 1, 1, 1, capi.PADDING_SAME, 1, 0, 0, 1.0, 0)
    with pytest.raises(capi.LceError, match="grouped"):
        capi.BConv2d(d, np.zeros((8, 3, 3, 2), np.int32), np.ones(8, np.float32),
                     np.ones(8, np.float32))


def test_bconv_full_size_batch_properties(capi):
    """QuickNet stage shapes at batch 32: (a) a strided sample of images equals the
    oracle bit for bit; (b) batch independence: out[b] does not depend on the other
    images (the property multi-GPU sharding relies on)."""
    for (hw, c) in [(56, 64), (28, 128), (14, 256), (7, 512)]:
        B = 32
        case = L.make_bconv_case(hw, B, hw, hw, c, 3, 3, c, activation=L.ACT_RELU)
        plan = capi.BConv2d(gpu_desc(capi, case.desc), case.filt, case.mul, case.bias)
        x = dev(case.inp)
        full = plan(x)
        sel = [0, 13, 31]
        sub = L.make_bconv_case(hw, len(sel), hw, hw, c, 3, 3, c, activation=L.ACT_RELU)
        sub.inp = case.inp[sel]
        want = L.bconv2d(sub.desc, sub.inp, case.filt, case.mul, case.bias, threads=4)
        assert_same_bits(full[sel].cpu().numpy(), want, f"stage {hw}x{hw}x{c}")
        alone = plan(x[5:6].contiguous())
        assert torch.equal(alone[0], full[5])
        plan.close()


# --------------------------------- BGEMM ---------------------------------- #
def test_bgemm_sweep_vs_oracle(capi):
    rng = np.random.default_rng(11)
    for (M, N, Kw) in [(256, 256, 8), (300, 70, 5), (128, 64, 1), (1, 1, 1), (513, 129, 18),
                       (256, 512, 64), (1024, 256, 256), (77, 33, 130)]:
        A = rng.integers(-2**31, 2**31, (M, Kw), dtype=np.int64).astype(np.int32)
        W = rng.integers(-2**31, 2**31, (N, Kw), dtype=np.int64).astype(np.int32)
        raw = capi.BGemm(W)(dev(A)).cpu().numpy()
        assert_same_bits(raw, L.bgemm(A, W, threads=4), f"raw {M}x{N}x{Kw}")
        mul = rng.uniform(-1.5, 1.5, N).astype(np.float32)
        bias = rng.uniform(-1.5, 1.5, N).astype(np.float32)
        K = Kw * 32
        clamp = (K - min(6, K), K)
        got = capi.BGemm(W, capi.OUT_FLOAT, clamp, mul, bias)(dev(A)).cpu().numpy()
        assert_same_bits(got, L.bgemm(A, W, L.OUT_FLOAT, clamp, mul, bias, threads=4))
        got = capi.BGemm(W, capi.OUT_INT8, clamp, mul, bias)(dev(A)).cpu().numpy()
        assert_same_bits(got, L.bgemm(A, W, L.OUT_INT8, clamp, mul, bias, threads=4))
        thr = rng.integers(K // 2 - 8, K // 2 + 8, N).astype(np.int32)
        got = capi.BGemm(W, capi.OUT_BITPACKED, thresholds=thr)(dev(A)).cpu().numpy()
        assert_same_bits(got, L.bgemm(A, W, L.OUT_BITPACKED, thr=thr, threads=4))


def test_bgemm_large_linearity_properties(capi):
    """Size-independent properties at sweep sizes the oracle cannot finish quickly:
    acc(A, W) + acc(~A, W) == K_bits, acc(A, A) diagonal == 0, symmetry."""
    g = torch.Generator(device="cuda").manual_seed(1)
    M = N = 2048
    Kw = 256
    A = torch.randint(-2**31, 2**31 - 1, (M, Kw), device="cuda", generator=g, dtype=torch.int64).to(torch.int32)
    W = torch.randint(-2**31, 2**31 - 1, (N, Kw), device="cuda", generator=g, dtype=torch.int64).to(torch.int32)
    gemm = capi.BGemm(W)
    acc = gemm(A)
    acc_not = gemm(~A)
    assert torch.all(acc + acc_not == Kw * 32)
    self_gemm = capi.BGemm(A)
    s = self_gemm(A)
    assert torch.all(torch.diagonal(s) == 0) and torch.equal(s, s.T)
    rows = [0, 1, 1023, 2047]
    want = L.bgemm(A[rows].cpu().numpy(), W.cpu().numpy(), threads=4)
    assert np.array_equal(acc[rows].cpu().numpy(), want)


def test_bconv_fused_residual_and_pack_entry_point(capi):
    """lce_b200_bconv2d_run_fused == LceBconv2d -> ADD(shortcut) -> LceQuantize, bit for bit."""
    import ctypes as C
    rng = np.random.default_rng(5)
    for (b, hw, c, co, act_add) in [(2, 14, 64, 64, L.ACT_NONE), (1, 7, 512, 128, L.ACT_RELU),
                                    (3, 9, 96, 72, L.ACT_NONE)]:
        case = L.make_bconv_case(60 + c, b, hw, hw, c, 3, 3, co, activation=L.ACT_RELU)
        res = rng.standard_normal((b, hw, hw, co)).astype(np.float32)
        plan = capi.BConv2d(gpu_desc(capi, case.desc), case.filt, case.mul, case.bias)
        out = torch.empty((b, hw, hw, co), device="cuda")
        packed = torch.empty((b, hw, hw, L.cdiv(co, 32)), dtype=torch.int32, device="cuda")
        d_in, d_res = dev(case.inp), dev(res)          # keep the device tensors alive
        rc = capi.lib().lce_b200_bconv2d_run_fused(
            plan._h, C.c_void_p(d_in.data_ptr()), C.c_void_p(d_res.data_ptr()),
            C.c_int(act_add), C.c_void_p(out.data_ptr()), C.c_void_p(packed.data_ptr()),
            C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, capi.lib().lce_b200_last_error()
        y = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias)
        want = (y + res).astype(np.float32)
        if act_add == L.ACT_RELU:
            want = np.maximum(want, 0)
        torch.cuda.synchronize()
        assert_same_bits(out.cpu().numpy(), want, "fused sum")
        assert_same_bits(packed.cpu().numpy(), L.quantize(want), "fused packed signs")
        plan.close()


KERNEL_ENV = {"xor": {"LCE_B200_BCONV_TC": "0", "LCE_B200_BCONV_IMMA": "0"},
              "imma": {"LCE_B200_BCONV_TC": "0", "LCE_B200_BCONV_IMMA": "1"},
              "tc": {"LCE_B200_BCONV_TC": "1", "LCE_B200_BCONV_IMMA": "1"}}
PATH_INDEX = {"tc": 0, "imma": 1, "xor": 2}


def path_counts(capi):
    import ctypes as C
    a = (C.c_uint64 * 3)()
    capi.lib().lce_b200_path_counts(a)
    return list(a)


@pytest.mark.parametrize("imma", ["xor", "imma", "tc"])
def test_bconv_both_inner_products_vs_oracle(capi, imma, monkeypatch):
    """The three inner products -- XOR+POPC (north_star's), int8 mma.sync, and tcgen05 kind::i8
    with TMEM accumulators (the default wherever a plan is eligible) -- produce the reference's
    integers: ones / zero padding, stride, dilation, groups, multi-chunk K, ragged M, fused tail.
    lce_b200_path_counts proves which kernel ran."""
    import ctypes as C
    for k, v in KERNEL_ENV[imma].items():
        monkeypatch.setenv(k, v)
    before = path_counts(capi)
    rng = np.random.default_rng(77)
    grid = [
        # b, h, w, cin, fh, fw, cout, groups, stride, dilation, padding, pad_value, act
        (2, 14, 14, 64, 3, 3, 64, 1, (1, 1), (1, 1), L.PADDING_SAME, 1, L.ACT_RELU),
        (1, 7, 7, 512, 3, 3, 128, 1, (1, 1), (1, 1), L.PADDING_SAME, 1, L.ACT_NONE),
        (3, 9, 11, 64, 3, 3, 64, 1, (1, 1), (1, 1), L.PADDING_SAME, 0, L.ACT_NONE),
        (2, 13, 9, 128, 3, 3, 192, 1, (2, 2), (1, 1), L.PADDING_SAME, 0, L.ACT_NONE),
        (2, 12, 12, 96, 3, 2, 64, 1, (1, 2), (2, 1), L.PADDING_VALID, 1, L.ACT_RELU6),
        (2, 10, 10, 128, 3, 3, 128, 2, (1, 1), (1, 1), L.PADDING_SAME, 1, L.ACT_RELU),
        (1, 5, 5, 1024, 5, 5, 64, 1, (1, 1), (1, 1), L.PADDING_SAME, 1, L.ACT_NONE),   # K = 800 words
        (5, 6, 6, 32, 1, 1, 64, 1, (1, 1), (1, 1), L.PADDING_VALID, 1, L.ACT_RELU_N1_TO_1),
    ]
    for n, (b, h, w, cin, fh, fw, co, g, st, dl, pad, pv, act) in enumerate(grid):
        case = L.make_bconv_case(9000 + n, b, h, w, cin, fh, fw, co, g, st, dl, pad, pv, act,
                                 L.OUT_FLOAT)
        want = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, case.thr)
        assert_same_bits(run_gpu_bconv(capi, case), want, f"kernel={imma} case {n}")
        # fused tail on the same plan shape
        plan = capi.BConv2d(gpu_desc(capi, case.desc), case.filt, case.mul, case.bias)
        res = rng.standard_normal(want.shape).astype(np.float32)
        out = torch.empty(want.shape, device="cuda")
        packed = torch.empty(want.shape[:3] + (L.cdiv(co, 32),), dtype=torch.int32, device="cuda")
        d_in, d_res = dev(case.inp), dev(res)
        rc = capi.lib().lce_b200_bconv2d_run_fused(
            plan._h, C.c_void_p(d_in.data_ptr()), C.c_void_p(d_res.data_ptr()),
            C.c_int(L.ACT_RELU if n % 2 else L.ACT_NONE), C.c_void_p(out.data_ptr()),
            C.c_void_p(packed.data_ptr() if g == 1 else 0),
            C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, capi.lib().lce_b200_last_error()
        torch.cuda.synchronize()
        ws = (want + res).astype(np.float32)
        if n % 2:
            ws = np.maximum(ws, 0)
        assert_same_bits(out.cpu().numpy(), ws, f"kernel={imma} fused sum {n}")
        if g == 1:
            assert_same_bits(packed.cpu().numpy(), L.quantize(ws), f"kernel={imma} fused signs {n}")
        plan.close()
    # plain BGEMM, raw accumulators
    A = rng.integers(-2**31, 2**31 - 1, (333, 24), dtype=np.int64).astype(np.int32)
    W = rng.integers(-2**31, 2**31 - 1, (128, 24), dtype=np.int64).astype(np.int32)
    gemm = capi.BGemm(dev(W))
    got = gemm(dev(A)).cpu().numpy()
    gemm.close()
    assert np.array_equal(got, L.bgemm(A, W, threads=4))
    ran = [b - a for a, b in zip(before, path_counts(capi))]
    # 8 plain + 8 fused convolutions + 1 BGEMM; the grouped case (2 launches) is outside the
    # tcgen05 and (64-channel groups) inside the mma.sync kernel's reach
    want_main = 17 if imma != "tc" else 15
    assert ran[PATH_INDEX[imma]] == want_main, (imma, ran)
    assert sum(ran) == 17, (imma, ran)


# ---- zero padding: both results the reference has (include/lce_b200_types.h) ---------------- #
BIREALNET_LAYERS = [  # (in hw, cin, cout, stride) of Bi-RealNet-18's 16 binary 3x3 convolutions
    (56, 64, 64, 1), (56, 64, 64, 1), (56, 64, 64, 1), (56, 64, 64, 1),
    (56, 64, 128, 2), (28, 128, 128, 1), (28, 128, 128, 1), (28, 128, 128, 1),
    (28, 128, 256, 2), (14, 256, 256, 1), (14, 256, 256, 1), (14, 256, 256, 1),
    (14, 256, 512, 2), (7, 512, 512, 1), (7, 512, 512, 1), (7, 512, 512, 1)]


def ulp_distance(a, b):
    ai = a.view(np.int32).astype(np.int64)
    bi = b.view(np.int32).astype(np.int64)
    ai = np.where(ai < 0, -(ai & 0x7FFFFFFF), ai)
    bi = np.where(bi < 0, -(bi & 0x7FFFFFFF), bi)
    return np.abs(ai - bi)


@pytest.mark.parametrize("kernel", ["tc", "imma"])
def test_zero_padding_matches_the_default_registration_within_1_ulp(capi, kernel, monkeypatch):
    """Bi-RealNet-18's 16 layer shapes (SAME, pad_values 0, float output, no activation): the
    result the reference's DEFAULT registration computes there is one-padding + OutputTransform +
    the float correction of zero_padding_correction.h, not the reference kernel's integers (the
    two differ by up to ~1e5 ULP near cancellation). north_star allows 1 ULP on the float
    post-transform; LCE_ZERO_PADDING_CORRECTION reproduces the optimised kernels bit for bit
    (0 ULP) -- against the reference's own headers compiled in oracle/_ref when that library
    travelled with the snapshot, else against the oracle's restatement (pinned to it in
    tests/test_oracle.py)."""
    for k, v in KERNEL_ENV[kernel].items():
        monkeypatch.setenv(k, v)
    impl = "ref" if L.load_ref() is not None else "oracle"
    worst = 0
    for n, (hw, cin, cout, stride) in enumerate(BIREALNET_LAYERS):
        case = L.make_bconv_case(4000 + n, 2, hw, hw, cin, 3, 3, cout, stride=(stride, stride),
                                 pad_value=0, activation=L.ACT_NONE)
        plan = capi.BConv2d(gpu_desc(capi, case.desc), case.filt, case.mul, case.bias)
        plan.set_zero_padding_mode(1)
        got = plan(dev(case.inp)).cpu().numpy()
        want = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, impl=impl, kind=1, threads=4)
        worst = max(worst, int(ulp_distance(got, want).max()))
        assert worst <= 1, (n, hw, cin, cout, stride, worst)
        assert_same_bits(got, want, f"layer {n}")
        # and the reference kernel's result on the same plan shape (Register_BCONV_2D_REF)
        plan.set_zero_padding_mode(0)
        got0 = plan(dev(case.inp)).cpu().numpy()
        assert_same_bits(got0, L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, threads=4),
                         f"layer {n} reference kernel")
        plan.close()


def test_zero_padding_correction_fused_tail_and_odd_channels(capi):
    """CORRECTION mode with the fused shortcut + sign-pack tail (Bi-RealNet's residual block), and
    an odd channels_in, which only the optimised kernels accept (bconv2d.cc:188-200)."""
    import ctypes as C
    rng = np.random.default_rng(9)
    for (b, hw, cin, cout) in [(2, 14, 256, 256), (3, 7, 64, 64), (1, 9, 33, 32)]:
        case = L.make_bconv_case(77 + cin, b, hw, hw, cin, 3, 3, cout, pad_value=0)
        plan = capi.BConv2d(gpu_desc(capi, case.desc), case.filt, case.mul, case.bias)
        plan.set_zero_padding_mode(1)
        if cin % 2:
            with pytest.raises(capi.LceError, match="Zero-padding is only supported"):
                plan.set_zero_padding_mode(0)
        res = rng.standard_normal((b, hw, hw, cout)).astype(np.float32)
        out = torch.empty((b, hw, hw, cout), device="cuda")
        packed = torch.empty((b, hw, hw, L.cdiv(cout, 32)), dtype=torch.int32, device="cuda")
        d_in, d_res = dev(case.inp), dev(res)
        rc = capi.lib().lce_b200_bconv2d_run_fused(
            plan._h, C.c_void_p(d_in.data_ptr()), C.c_void_p(d_res.data_ptr()), C.c_int(L.ACT_NONE),
            C.c_void_p(out.data_ptr()), C.c_void_p(packed.data_ptr()),
            C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, capi.lib().lce_b200_last_error()
        torch.cuda.synchronize()
        y = L.bconv2d(case.desc, case.inp, case.filt, case.mul, case.bias, kind=1)
        want = (y + res).astype(np.float32)
        assert_same_bits(out.cpu().numpy(), want, "fused sum, float correction")
        assert_same_bits(packed.cpu().numpy(), L.quantize(want), "fused signs, float correction")
        plan.close()
