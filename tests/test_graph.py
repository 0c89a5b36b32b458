"""Graph-host tests on synthesised `.tflite` models (the three model families of
BASELINE.json; topology from the public descriptions, random weights).

CPU: the flatbuffer writer against an independent pure-Python reader; the C++ reader
against that reader (and against TFLite's own fixtures when REF names a
larq/compute-engine checkout); shape inference / resize of every op through prepare.
GPU: whole graphs through the device-arena host; every LCE custom op is checked BIT
EXACT against the oracle on the tensors the device itself produced (op-by-op parity),
the float builtins against a PyTorch fp32 CPU reference within a stated tolerance.
"""
import os

import numpy as np
import pytest

import lce_testlib as L
import tflite_ref as R
from compute_engine_b200 import host as H
from compute_engine_b200 import zoo
from compute_engine_b200 import tflite_writer as W

TF_TESTDATA = os.path.join(os.environ.get("REF", ""), "third_party", "tensorflow", "tensorflow",
                           "lite", "testdata")


@pytest.fixture(scope="module")
def quicknet_small():
    return zoo.quicknet(batch=1, image=64, seed=3)


def test_writer_roundtrips_through_independent_reader(quicknet_small):
    m = R.parse(quicknet_small)
    assert m["version"] == 3 and m["description"] == "QuickNet"
    kinds = [(o["code"], o["custom"]) for o in m["ops"]]
    assert kinds.count((32, "LceBconv2d")) == 16 and kinds.count((32, "LceQuantize")) == 16
    assert kinds.count((0, "")) == 16            # residual ADDs
    assert kinds.count((3, "")) == 5             # stem conv, stem pointwise, 3 transitions
    assert kinds.count((4, "")) == 4             # stem depthwise + 3 blur-pools
    assert m["tensors"][m["inputs"][0]]["shape"] == (1, 64, 64, 3)
    assert m["tensors"][m["outputs"][0]]["shape"] == (1, 1000)
    bconvs = [o for o in m["ops"] if o["custom"] == "LceBconv2d"]
    a = R._flex_ints(bconvs[0]["custom_options"])
    assert a == {"channels_in": 64, "dilation_height_factor": 1, "dilation_width_factor": 1,
                 "fused_activation_function": 1, "pad_values": 1, "padding": 0,
                 "stride_height": 1, "stride_width": 1}
    assert bconvs[0]["inputs"][4] == -1          # optional thresholds absent
    filt = m["tensors"][bconvs[-1]["inputs"][1]]
    assert filt["shape"] == (512, 3, 3, 16) and filt["dtype"] == np.int32
    # buffers are 16-byte aligned inside the file (schema.fbs:1562)
    off = quicknet_small.find(filt["data"].tobytes()[:64])
    assert off > 0 and off % 16 == 0


def test_cpp_reader_matches_python_reader(quicknet_small):
    m = R.parse(quicknet_small)
    g = H.HostGraph.from_tflite(quicknet_small, device_arena=False)
    assert g.num_nodes() == len(m["ops"])
    assert H.lib().lce_host_num_tensors(g._g) == len(m["tensors"])
    g.allocate_tensors()                         # every prepare runs on the CPU
    for i, t in enumerate(m["tensors"]):
        assert g.shape(i) == t["shape"], (i, t["name"])
        assert g.dtype(i) == t["dtype"]
    assert [g.shape(t) for t in g.outputs()] == [(1, 1000)]
    # batch is pinned to 1 by the converter: resizing re-prepares every op
    g.resize_input(g.inputs()[0], (5, 64, 64, 3))
    g.allocate_tensors()
    assert [g.shape(t) for t in g.outputs()] == [(5, 1000)]
    g.close()


def test_all_three_families_build_and_prepare():
    for name, fn, n_bconv in (("quicknet", zoo.quicknet, 16),
                              ("quicknet_large", zoo.quicknet_large, 32),
                              ("birealnet18", zoo.birealnet18, 16)):
        blob = fn(batch=2)
        m = R.parse(blob)
        assert sum(o["custom"] == "LceBconv2d" for o in m["ops"]) == n_bconv
        g = H.HostGraph.from_tflite(blob, device_arena=False)
        g.allocate_tensors()
        assert [g.shape(t) for t in g.outputs()] == [(2, 1000)], name
        g.close()


def test_unknown_custom_op_is_reported():
    from compute_engine_b200.tflite_writer import TFLiteModel
    m = TFLiteModel()
    a = m.add_tensor("a", (1, 4))
    b = m.add_tensor("b", (1, 4))
    m.add_op("NotAnLceOp", [a], [b], custom_options=b"")
    m.inputs, m.outputs = [a], [b]
    with pytest.raises(H.HostError, match="unresolved custom op: NotAnLceOp"):
        H.HostGraph.from_tflite(m.serialize(), device_arena=False)
    with pytest.raises(H.HostError, match="not a TFL3 flatbuffer"):
        H.HostGraph.from_tflite(b"garbage-bytes-here", device_arena=False)


def test_malformed_tensor_indices_are_rejected():
    """A .tflite whose operators or graph inputs / outputs point outside the tensor table is
    refused by the reader (the op shells index context->tensors unchecked afterwards)."""
    from compute_engine_b200.tflite_writer import TFLiteModel

    def model(op_in, op_out, g_in, g_out):
        m = TFLiteModel()
        a = m.add_tensor("a", (1, 4, 4, 32))
        b = m.add_tensor("b", (1, 4, 4, 1), np.int32)
        m.add_op("LceQuantize", [a if op_in is None else op_in], [b if op_out is None else op_out],
                 custom_options=b"")
        m.inputs = [a if g_in is None else g_in]
        m.outputs = [b if g_out is None else g_out]
        return m.serialize()

    H.HostGraph.from_tflite(model(None, None, None, None), device_arena=False).close()
    for bad, what in ((model(7, None, None, None), "operator 0 input"),
                      (model(-3, None, None, None), "operator 0 input"),
                      (model(None, 2, None, None), "operator 0 output"),
                      (model(None, -1, None, None), "operator 0 output"),
                      (model(None, None, 5, None), "graph input"),
                      (model(None, None, None, -1), "graph output")):
        with pytest.raises(H.HostError, match=what + " refers to a missing tensor"):
            H.HostGraph.from_tflite(bad, device_arena=False)


def test_residual_fusion_skips_what_the_fused_kernel_cannot_do():
    """A grouped LceBconv2d, or an ADD whose other operand only broadcasts onto the convolution's
    output, stays unfused (ADVICE r01: the rewrite used to happen first and fail in Prepare)."""
    from compute_engine_b200.tflite_writer import TFLiteModel, bconv2d_options
    rng = np.random.default_rng(0)
    for groups, res_shape in ((2, (1, 6, 6, 64)), (1, (64,))):
        m = TFLiteModel()
        x = m.add_tensor("x", (1, 6, 6, 128))
        xq = m.add_tensor("xq", (1, 6, 6, 4), np.int32)
        f = m.add_tensor("f", None, np.int32,
                         data=rng.integers(-2**31, 2**31 - 1, (64, 3, 3, 4 // groups), dtype=np.int64).astype(np.int32))
        mul = m.add_tensor("mul", None, np.float32, data=rng.uniform(0.1, 1, 64))
        bias = m.add_tensor("bias", None, np.float32, data=rng.uniform(0.1, 1, 64))
        y = m.add_tensor("y", (1, 6, 6, 64))
        r = m.add_tensor("r", res_shape)
        z = m.add_tensor("z", (1, 6, 6, 64))
        m.add_op("LceQuantize", [x], [xq], custom_options=b"")
        m.add_op("LceBconv2d", [xq, f, mul, bias, -1], [y], custom_options=bconv2d_options(128))
        m.add_op("ADD", [y, r], [z])
        m.inputs, m.outputs = [x, r], [z]
        g = H.HostGraph.from_tflite(m.serialize(), device_arena=True)
        assert g.fuse_residual_blocks() == 0 and g.num_nodes() == 3
        g.close()
        g = H.HostGraph.from_tflite(m.serialize(), device_arena=False)   # and it prepares unfused
        g.allocate_tensors()
        g.close()


@pytest.mark.skipif(not os.environ.get("REF") or not os.path.isdir(TF_TESTDATA),
                    reason="needs REF=<larq/compute-engine checkout> for TFLite's test fixtures")
def test_readers_on_tflite_own_fixtures():
    for name, n_ops in (("add.bin", 2), ("multi_add.bin", 3)):
        blob = open(os.path.join(TF_TESTDATA, name), "rb").read()
        m = R.parse(blob)
        assert len(m["ops"]) == n_ops, name
        g = H.HostGraph.from_tflite(blob, device_arena=False)
        assert g.num_nodes() == n_ops
        for i, t in enumerate(m["tensors"]):
            assert g.shape(i) == t["shape"]
        g.close()
    blob = open(os.path.join(TF_TESTDATA, "conv_huge_im2col.bin"), "rb").read()
    assert [o["code"] for o in R.parse(blob)["ops"]] == [2, 3, 0]     # CONCATENATION, CONV_2D, ADD
    g = H.HostGraph.from_tflite(blob, device_arena=False)
    assert g.num_nodes() == 3
    g.close()
    blob = open(os.path.join(TF_TESTDATA, "custom_sinh.bin"), "rb").read()
    assert R.parse(blob)["ops"][0]["custom"] == "Sinh"
    with pytest.raises(H.HostError, match="unresolved custom op: Sinh"):
        H.HostGraph.from_tflite(blob, device_arena=False)


# ------------------------------- GPU ------------------------------------- #
def _check_graph_on_gpu(blob, batch, image, seed, final_atol):
    m = R.parse(blob)
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((batch, image, image, 3)).astype(np.float32)
    g = H.HostGraph.from_tflite(blob, device_arena=True)
    g.preserve_all_tensors(True)
    g.resize_input(g.inputs()[0], x.shape)
    g.allocate_tensors()
    g.write(g.inputs()[0], x)
    g.invoke()
    want_out, _ = R.run(m, [x])
    got_out = g.read(g.outputs()[0])
    # (1) op-by-op: each LCE op, fed with the DEVICE's own input tensor, is bit exact
    n_lce = 0
    for op in m["ops"]:
        if op["code"] != 32:
            continue
        sub = {"tensors": m["tensors"], "ops": [op], "inputs": [op["inputs"][0]],
               "outputs": [op["outputs"][0]]}
        dev_in = g.read(op["inputs"][0])
        want, _ = R.run(sub, [dev_in])
        got = g.read(op["outputs"][0])
        assert got.shape == want[0].shape
        assert np.array_equal(got.view(np.uint8), want[0].view(np.uint8)), op["custom"]
        n_lce += 1
    # (2) float builtins vs the torch fp32 CPU reference, op by op on device inputs
    for op in m["ops"]:
        if op["code"] == 32:
            continue
        act_inputs = [i for i in op["inputs"] if i >= 0 and m["tensors"][i]["data"] is None]
        sub = {"tensors": m["tensors"], "ops": [op], "inputs": act_inputs,
               "outputs": [op["outputs"][0]]}
        want, _ = R.run(sub, [g.read(i) for i in act_inputs])
        got = g.read(op["outputs"][0])
        scale = max(1.0, float(np.abs(want[0]).max()))
        assert np.allclose(got, want[0], rtol=1e-4, atol=1e-5 * scale), (op["code"], np.abs(got - want[0]).max())
    # (3) end to end: class probabilities against the CPU graph
    assert got_out.shape == want_out[0].shape
    assert np.abs(got_out - want_out[0]).max() <= final_atol
    assert np.allclose(got_out.sum(-1), 1.0, atol=1e-4)
    g.close()
    return n_lce


@pytest.mark.gpu
def test_gpu_quicknet_graph_parity():
    assert _check_graph_on_gpu(zoo.quicknet(batch=1, image=64, seed=5), 3, 64, 0, 2e-4) == 32


@pytest.mark.gpu
def test_gpu_birealnet18_graph_parity():
    assert _check_graph_on_gpu(zoo.birealnet18(batch=1, image=64, seed=6), 2, 64, 1, 2e-4) == 32


@pytest.mark.gpu
def test_gpu_interpreter_predict_true_batching():
    from compute_engine_b200.interpreter import Interpreter
    blob = zoo.quicknet(batch=1, image=64, seed=7)
    it = Interpreter(blob, batch_size=4)
    assert it.input_shapes == [(1, 64, 64, 3)] and it.output_shapes == [(1, 1000)]
    assert it.input_types == [np.float32] and it.input_scales == [None]
    x = np.random.default_rng(2).standard_normal((10, 64, 64, 3)).astype(np.float32)
    y = it.predict(x)                      # mini-batches 4, 4, 2; CUDA graph re-captured on resize
    assert y.shape == (10, 1000)
    y1 = np.concatenate([it.predict(x[i:i + 1]) for i in range(10)])   # the reference's batch-1 loop
    assert np.allclose(y, y1, atol=1e-6)
    want, _ = R.run(R.parse(blob), [x])
    assert np.abs(y - want[0]).max() < 2e-4
    it.close()


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["quicknet", "quicknet_large", "birealnet18"])
def test_gpu_graph_parity_at_the_benched_shape(family):
    """224 x 224 images, batch 64 -- the shape bench.py times (M up to 200 k pixels per layer,
    thousands of tiles per binary convolution), not the 64 x 64 toys above:
    (1) unfused graph: every LCE op, fed with the device's own input tensor, is bit exact on a
        sample of images against the CPU checker;
    (2) the FUSED graph under CUDA-graph replay (what is benchmarked) gives bit-identical class
        probabilities for all 64 images;
    (3) the sampled images' probabilities match the CPU graph to 2e-4."""
    B, sel = 64, [0, 29, 63]
    blob = zoo.MODELS[family](batch=1, image=224, seed=21)
    m = R.parse(blob)
    x = np.random.default_rng(8).standard_normal((B, 224, 224, 3)).astype(np.float32)
    g = H.HostGraph.from_tflite(blob, device_arena=True)
    g.preserve_all_tensors(True)
    g.resize_input(g.inputs()[0], x.shape)
    g.allocate_tensors()
    g.write(g.inputs()[0], x)
    g.invoke()
    n_lce = 0
    for op in m["ops"]:
        if op["code"] != 32:
            continue
        sub = {"tensors": m["tensors"], "ops": [op], "inputs": [op["inputs"][0]],
               "outputs": [op["outputs"][0]]}
        want, _ = R.run(sub, [g.read(op["inputs"][0])[sel]])
        got = g.read(op["outputs"][0])[sel]
        assert got.shape == want[0].shape
        assert np.array_equal(got.view(np.uint8), want[0].view(np.uint8)), (op["custom"], n_lce)
        n_lce += 1
    assert n_lce >= 32
    unfused = g.read(g.outputs()[0])
    g.close()
    g = H.HostGraph.from_tflite(blob, device_arena=True)
    assert g.fuse_all() > 0
    g.resize_input(g.inputs()[0], x.shape)
    g.allocate_tensors()
    g.enable_cuda_graph(True)
    for _ in range(3):                                   # eager, capture, replay
        g.write(g.inputs()[0], x)
        g.invoke()
    fused = g.read(g.outputs()[0])
    g.close()
    assert np.array_equal(fused.view(np.uint8), unfused.view(np.uint8))
    want_out, _ = R.run(m, [x[sel]])
    assert np.abs(fused[sel] - want_out[0]).max() <= 2e-4
    assert np.allclose(fused.sum(-1), 1.0, atol=1e-4)


@pytest.mark.gpu
def test_gpu_interpreter_selectors_and_devices():
    """use_reference_bconv picks the reference kernel's zero-padding integers, the default the
    optimised kernels' float correction (Bi-RealNet differs between them; QuickNet does not);
    devices=[0, 0] shards every mini-batch over two graphs and returns the outputs in order."""
    from compute_engine_b200.interpreter import Interpreter
    blob = zoo.birealnet18(batch=1, image=64, seed=13)
    x = np.random.default_rng(3).standard_normal((6, 64, 64, 3)).astype(np.float32)
    m = R.parse(blob)
    outs = {}
    for name, kw, kind in (("default", {}, 1), ("ref", {"use_reference_bconv": True}, 0),
                           ("indirect", {"use_indirect_bgemm": True}, 1)):
        it = Interpreter(blob, **kw)
        outs[name] = it.predict(x)
        want, _ = R.run(m, [x], bconv_kind=kind)
        assert np.abs(outs[name] - want[0]).max() < 2e-4, name
        it.close()
    assert np.array_equal(outs["default"], outs["indirect"])
    assert not np.array_equal(outs["default"], outs["ref"])     # two different float computations
    it2 = Interpreter(blob, devices=[0, 0], batch_size=5)
    y2 = it2.predict(x)                                         # mini-batches 5 (3 + 2) and 1
    it2.close()
    assert np.array_equal(y2, outs["default"])


@pytest.mark.gpu
def test_gpu_benchmark_cli_flags():
    """tools/lce_benchmark_model.py runs, and its --use_reference_bconv / --use_indirect_bgemm flags
    reach the op resolver (lce_benchmark_tflite_model.cc:41-71)."""
    import json as _json
    import subprocess
    import sys as _sys
    tool = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools",
                        "lce_benchmark_model.py")
    for flags, reg in (([], "Register_BCONV_2D"),
                       (["--use_reference_bconv=true"], "Register_BCONV_2D_REF"),
                       (["--use_indirect_bgemm=true"], "Register_BCONV_2D_OPT_INDIRECT_BGEMM")):
        out = subprocess.run([_sys.executable, tool, "--zoo=birealnet18", "--batch=2", "--num_runs=3",
                              "--warmup_runs=2"] + flags, capture_output=True, text=True, timeout=600,
                             check=True).stdout
        d = _json.loads(out)
        assert d["bconv_registration"] == reg and d["images_per_s"] > 0 and d["nodes"] > 0


def test_residual_block_fusion_rewrites_the_graph():
    """Structure of the graph-level fusion (pure host logic; no device needed):
    LceBconv2d -> ADD [-> LceQuantize] collapses into one node."""
    g = H.HostGraph.from_tflite(zoo.quicknet(batch=1, image=64, seed=3), device_arena=True)
    assert g.num_nodes() == 64
    removed = g.fuse_residual_blocks()
    # 16 ADDs + the 12 LceQuantize ops that read an ADD's output (3 per stage)
    assert removed == 28 and g.num_nodes() == 36
    names = [g.node_name(i) for i in range(g.num_nodes())]
    assert names.count("LceBconv2d+ADD+LceQuantize") == 12
    assert names.count("LceBconv2d+ADD") == 4          # last block of each stage
    assert names.count("LceQuantize") == 4             # first block of each stage
    assert "builtin:0" not in names and "LceBconv2d" not in names
    assert g.fuse_residual_blocks() == 0               # idempotent
    # float glue: the stem's conv 3x3 s2 -> depthwise 3x3 s2 pair (1 node removed), the four
    # CONV_2D -> LceQuantize pairs (stem pointwise + three transitions) and the three
    # (max-pool 2x2 s1 -> blur depthwise 3x3 s2) pairs of the transitions, and the head's RELU -> MEAN
    assert g.fuse_float_glue() == 1 + 4 + 3 + 1 and g.num_nodes() == 27
    names = [g.node_name(i) for i in range(g.num_nodes())]
    assert names.count("MAX_POOL_2D+DEPTHWISE_CONV_2D") == 3 and "builtin:17" not in names
    assert names[0] == "CONV_2D+DEPTHWISE_CONV_2D" and "builtin:4" not in names
    assert names.count("CONV_2D+LceQuantize") == 4 and "LceQuantize" not in names
    assert names.count("RELU+MEAN") == 1 and "builtin:19" not in names
    assert g.fuse_float_glue() == 0                    # idempotent
    g.close()


def test_fusion_switches_and_dequantize_folding(monkeypatch):
    """An int8-input model: the DEQUANTIZE in front of the stem is folded into the fused stem node
    (the kernel reads the quantised image). LCE_B200_FUSE_STEM=0 / LCE_B200_FUSE_CONV_QUANT=0
    switch the two fusions off."""
    blob = zoo.quicknet(batch=1, image=64, seed=3, input_type="int8")
    g = H.HostGraph.from_tflite(blob, device_arena=True)
    assert g.num_nodes() == 65
    assert g.fuse_all() == 28 + 2 + 4 + 3 + 1 and g.num_nodes() == 27
    names = [g.node_name(i) for i in range(g.num_nodes())]
    assert names[0] == "DEQUANTIZE+CONV_2D+DEPTHWISE_CONV_2D" and "builtin:6" not in names
    g.close()
    monkeypatch.setenv("LCE_B200_FUSE_STEM", "0")
    monkeypatch.setenv("LCE_B200_FUSE_CONV_QUANT", "0")
    g = H.HostGraph.from_tflite(blob, device_arena=True)
    assert g.fuse_all() == 28 + 3 + 1 and g.num_nodes() == 33
    names = [g.node_name(i) for i in range(g.num_nodes())]
    assert names[0] == "builtin:6" and names.count("builtin:4") == 1 and names.count("LceQuantize") == 4
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("family,image,input_type",
                         [("quicknet", 64, "float32"), ("quicknet", 88, "float32"), ("quicknet", 64, "int8"),
                          ("quicknet", 224, "int8"), ("quicknet", 100, "int8"), ("birealnet18", 64, "float32")])
def test_gpu_fused_graph_is_bit_identical_to_unfused(family, image, input_type):
    blob = zoo.MODELS[family](batch=1, image=image, seed=11, input_type=input_type)
    if input_type == "int8":
        x = np.random.default_rng(4).integers(-128, 128, (5, image, image, 3)).astype(np.int8)
    else:
        x = np.random.default_rng(4).standard_normal((5, image, image, 3)).astype(np.float32)
    outs = []
    for fuse in (False, True):
        g = H.HostGraph.from_tflite(blob, device_arena=True)
        if fuse:
            assert g.fuse_residual_blocks() > 0
            want = 0 if family != "quicknet" else (1 + 4 + 3 + 1 + (1 if input_type == "int8" else 0))
            assert g.fuse_float_glue() == want
        g.resize_input(g.inputs()[0], x.shape)
        g.allocate_tensors()
        g.enable_cuda_graph(True)
        for _ in range(3):                               # eager, capture, replay
            g.write(g.inputs()[0], x)
            g.invoke()
        outs.append(g.read(g.outputs()[0]))
        g.close()
    assert np.array_equal(outs[0].view(np.uint8), outs[1].view(np.uint8))


# ---- PAD / PADV2 / CONCATENATION: the glue the converter leaves around LceBconv2d ---- #
def _pad_concat_model(batch=2, hw=9, cin=64, cout=32, seed=5):
    """float x -> LceQuantize -> PADV2(bitpacked words, border word -1 = thirty-two -1 values)
    -> LceBconv2d VALID -> float PAD (channels) -> CONCATENATION(axis 3) with x."""
    rng = np.random.default_rng(seed)
    m = W.TFLiteModel()
    x = m.add_tensor("x", (batch, hw, hw, cin))
    xq = m.add_tensor("xq", (batch, hw, hw, cin // 32), np.int32)
    pads = m.add_tensor("pads", None, np.int32, data=np.array([[0, 0], [1, 1], [1, 1], [0, 0]]))
    fillv = m.add_tensor("fill", None, np.int32, data=np.array([-1], np.int32).reshape(()))
    xp = m.add_tensor("xp", (batch, hw + 2, hw + 2, cin // 32), np.int32)
    filt = rng.integers(-2**31, 2**31 - 1, size=(cout, 3, 3, cin // 32), dtype=np.int64).astype(np.int32)
    f = m.add_tensor("filter", None, np.int32, data=filt)
    mul = m.add_tensor("mul", None, np.float32, data=rng.uniform(0.01, 1.5, cout))
    bias = m.add_tensor("bias", None, np.float32, data=rng.uniform(0.01, 1.5, cout))
    y = m.add_tensor("y", (batch, hw, hw, cout))
    m.add_op("LceQuantize", [x], [xq], custom_options=b"")
    m.add_op("PADV2", [xq, pads, fillv], [xp])
    m.add_op("LceBconv2d", [xp, f, mul, bias, -1], [y],
             custom_options=H.bconv2d_options(cin, (1, 1), (1, 1), 1, 1, 0))
    pads2 = m.add_tensor("pads2", None, np.int32,
                         data=np.array([[0, 0], [0, 0], [0, 0], [3, 5]]))
    yp = m.add_tensor("yp", (batch, hw, hw, cout + 8))
    m.add_op("PAD", [y, pads2], [yp])
    z = m.add_tensor("z", (batch, hw, hw, cin + cout + 8))
    m.add_op("CONCATENATION", [x, yp], [z], axis=3)
    m.inputs, m.outputs = [x], [z]
    return m.serialize()


def test_pad_concat_graph_builds_and_infers_shapes():
    blob = _pad_concat_model()
    g = H.HostGraph.from_tflite(blob, device_arena=False)
    g.allocate_tensors()
    assert g.shape(g.outputs()[0]) == (2, 9, 9, 64 + 32 + 8)
    g.close()


@pytest.mark.gpu
def test_gpu_pad_concat_graph_matches_reference():
    blob = _pad_concat_model()
    m = R.parse(blob)
    x = np.random.default_rng(11).standard_normal((2, 9, 9, 64)).astype(np.float32)
    want, _ = R.run(m, [x])
    g = H.HostGraph.from_tflite(blob, device_arena=True)
    g.allocate_tensors()
    g.write(g.inputs()[0], x)
    g.invoke()
    got = g.read(g.outputs()[0])
    g.close()
    assert got.shape == want[0].shape and np.array_equal(got, want[0])


def test_float_glue_fusions_respect_their_preconditions():
    """Pure host logic: RELU -> MEAN folds only when the RELU's output has no other reader; the stem
    fusion needs CONSTANT filters (the kernel takes them by value) and a 3-channel 3x3/s2 conv."""
    from compute_engine_b200.tflite_writer import TFLiteModel
    rng = np.random.default_rng(0)
    axes = np.array([1, 2], np.int32)

    def head(relu_also_an_output):
        m = TFLiteModel()
        x = m.add_tensor("x", (2, 7, 7, 32))
        r = m.add_tensor("r", (2, 7, 7, 32))
        p = m.add_tensor("p", (2, 32))
        ax = m.add_tensor("axes", None, np.int32, data=axes)
        m.add_op("RELU", [x], [r])
        m.add_op("MEAN", [r, ax], [p], keep_dims=False)
        m.inputs, m.outputs = [x], ([p, r] if relu_also_an_output else [p])
        return m.serialize()

    g = H.HostGraph.from_tflite(head(False), device_arena=True)
    assert g.fuse_float_glue() == 1 and [g.node_name(i) for i in range(g.num_nodes())] == ["RELU+MEAN"]
    g.close()
    g = H.HostGraph.from_tflite(head(True), device_arena=True)      # the RELU's output is also a graph output
    assert g.fuse_float_glue() == 0 and g.num_nodes() == 2
    g.close()

    def stem(cin, const_filter):
        m = TFLiteModel()
        x = m.add_tensor("x", (1, 32, 32, cin))
        w1d = (rng.standard_normal((16, 3, 3, cin)) * 0.2).astype(np.float32)
        w1 = m.add_tensor("w1", None, np.float32, data=w1d) if const_filter else m.add_tensor("w1", (16, 3, 3, cin))
        b1 = m.add_tensor("b1", None, np.float32, data=np.zeros(16, np.float32))
        y = m.add_tensor("y", (1, 16, 16, 16))
        w2 = m.add_tensor("w2", None, np.float32, data=(rng.standard_normal((1, 3, 3, 16)) * 0.3).astype(np.float32))
        b2 = m.add_tensor("b2", None, np.float32, data=np.zeros(16, np.float32))
        z = m.add_tensor("z", (1, 8, 8, 16))
        m.add_op("CONV_2D", [x, w1, b1], [y], padding="SAME", stride=(2, 2), activation="RELU")
        m.add_op("DEPTHWISE_CONV_2D", [y, w2, b2], [z], padding="SAME", stride=(2, 2), depth_multiplier=1)
        m.inputs, m.outputs = ([x] if const_filter else [x, w1]), [z]
        return m.serialize()

    for cin, const_filter, fused in ((3, True, True), (4, True, False), (3, False, False)):
        g = H.HostGraph.from_tflite(stem(cin, const_filter), device_arena=True)
        removed = g.fuse_float_glue()
        names = [g.node_name(i) for i in range(g.num_nodes())]
        assert (removed == 1 and names == ["CONV_2D+DEPTHWISE_CONV_2D"]) if fused else (removed == 0 and len(names) == 2), \
            (cin, const_filter, names)
        g.close()
