#!/usr/bin/env python
"""bench.py -- the measurement contract.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload W]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the workload over one batch of synthetic input; rank 0 prints ONE JSON
line. Every field is explained in DESIGN.md section 6.

Workloads (config.workload):
  quicknet         (default; BASELINE.json configs[1]) the full QuickNet `.tflite` graph, batch 256
                   per GPU, through the graph host + custom-op registrations
  quicknet_large   configs[2] (batch 1024 sharded over the GPUs: --batch 128 --gpus 8)
  birealnet18      configs[3] (--batch 512)
  bconv_stack      the 16 LceQuantize -> LceBconv2d layers of QuickNet alone
  bgemm_sweep      configs[4]: prints one extra JSON object per (M, N, K, epilogue) to stderr
The graph workloads take `--input-type int8` (default: the model the converter emits with
inference_input_type=int8 -- int8 images + DEQUANTIZE in the graph, a quarter of the host-link
bytes) or `float32`; at N = 1 the default run reports both (`f32_input`), Bi-RealNet-18 b512 and
QuickNetLarge b128 (`other_configs`), the same graph on the two older inner products
(`legacy_paths`), and checks the GPU against the CPU checker on 4 images before it times anything.
Inputs and weights are seeded, so `--dump-outputs DIR` (the outputs of the last timed step) lets
two builds be compared output for output.

`--impl reference` times the reference's own CPU kernels (oracle/_ref: its headers compiled by
oracle/Makefile; LCE ops: bitpack_matrix + Kernel4x2Portable indirect BGEMM + zero-padding
correction) with PyTorch-CPU fp32 standing in for TFLite's float builtins, on the same model bytes
and batch. It imports nothing from compute_engine_b200 (the model is synthesised by loading
zoo.py / tflite_writer.py, pure Python, as stand-alone files).
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

STAGES = [(56, 64), (28, 128), (14, 256), (7, 512)]   # (H=W, C) of QuickNet's 4 sections
LAYERS_PER_STAGE = 4
DEFAULT_BATCH = {"quicknet": 256, "quicknet_large": 128, "birealnet18": 512, "bconv_stack": 256,
                 "bgemm_sweep": 1}
METRIC = {"quicknet": "quicknet_images_per_sec", "quicknet_large": "quicknet_large_images_per_sec",
          "birealnet18": "birealnet18_images_per_sec",
          "bconv_stack": "quicknet_binary_conv_stack_images_per_sec",
          "bgemm_sweep": "bgemm_binary_tops"}
GRAPHS = ("quicknet", "quicknet_large", "birealnet18")

# Libraries (NCCL's version banner, ...) may write to fd 1; the contract is ONE JSON line on
# stdout, so fd 1 is pointed at stderr for the whole run and the result goes to the saved fd.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(obj):
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="quicknet", choices=sorted(DEFAULT_BATCH))
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (0 = workload default)")
    ap.add_argument("--input-type", default="int8", choices=["int8", "float32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip f32_input / other_configs / legacy_paths / parity check")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as "
                         "DIR/<name>.npy (rank 0; float32, or float64 for integer results)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.workload == "bgemm_sweep"):
        ap.error("--dump-outputs applies to --impl b200 and the graph / bconv_stack workloads")
    if a.batch <= 0:
        a.batch = DEFAULT_BATCH[a.workload]
    return a


DUMP_MAX_ELEMENTS = 1 << 21      # per array: 8 MB as float32; larger outputs are sampled
DUMP_MAX_BYTES = 64 * 10**6


def dump_array(a):
    """An output as --dump-outputs stores it: float32, or float64 for integers (exact for int32),
    and, above DUMP_MAX_ELEMENTS, the flattened elements at a fixed seeded set of sorted indices,
    the same in every run."""
    a = np.asarray(a)
    a = a.astype(np.float64 if a.dtype.kind in "iub" or a.dtype == np.float64 else np.float32)
    if a.size > DUMP_MAX_ELEMENTS:
        idx = np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMENTS, replace=False)
        a = a.reshape(-1)[np.sort(idx)]
    return a


def write_dump(out_dir, arrays):
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peaks():
    """(hbm GB/s, source, sm max MHz, bf16 TFLOP/s burst, bf16 sustained) from the driver's file."""
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return (float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(p.get("sm_max_mhz", 1965.0)),
                float(p.get("bf16_tflops", 1590.0)), float(p.get("bf16_tflops_sustained", 1400.0)))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0, 1590.0, 1400.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            time.sleep(0.25)          # let the first samples arrive before the timed region
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if t0 is not None and not (t0 - 0.05 <= ts <= t1 + 0.05):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "power_w_max": float(max(pw)) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- #
# synthetic model / data (seeded; identical for both arms)
# --------------------------------------------------------------------------- #
_ZOO = None


def zoo_module():
    """compute_engine_b200/zoo.py + tflite_writer.py loaded as stand-alone files (pure Python):
    the reference arm builds the same model bytes without importing the product package."""
    global _ZOO
    if _ZOO is None:
        pkg = os.path.join(REPO, "compute_engine_b200")
        for name in ("tflite_writer", "zoo"):
            spec = importlib.util.spec_from_file_location(name, os.path.join(pkg, name + ".py"))
            mod = importlib.util.module_from_spec(spec)
            sys.modules[name] = mod
            spec.loader.exec_module(mod)
        _ZOO = sys.modules["zoo"]
    return _ZOO


def build_model_bytes(workload, input_type="float32"):
    z = zoo_module()
    return z.MODELS[workload](batch=1, seed=0, input_type=input_type)


def make_images(batch, seed, input_type="float32"):
    x = np.random.default_rng(seed).standard_normal((batch, 224, 224, 3), dtype=np.float32)
    return zoo_module().quantize_images(x) if input_type == "int8" else x


def make_stack_weights(seed=0):
    rng = np.random.default_rng(seed)
    layers = []
    for (hw, c) in STAGES:
        for _ in range(LAYERS_PER_STAGE):
            filt = rng.integers(-2**31, 2**31, (c, 3, 3, c // 32), dtype=np.int64).astype(np.int32)
            mul = rng.uniform(0.01, 1.5, c).astype(np.float32) / np.float32(9 * c)
            bias = rng.uniform(-1.0, 1.0, c).astype(np.float32)
            layers.append({"filter": filt, "mul": mul, "bias": bias})
    return layers


def make_stage_inputs(batch, seed):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal((batch, hw, hw, c), dtype=np.float32) for (hw, c) in STAGES]


def ncu_traffic_per_launch(fname, kernel_substr=None):
    """Mean dram__bytes_read + dram__bytes_write per launch from a committed `ncu --set full`
    summary under profiles/ (rows of the binary-convolution kernel), or None."""
    import csv
    path = os.path.join(REPO, "profiles", fname)
    try:
        rows = list(csv.reader(open(path)))
        hdr, units = rows[0], rows[1]
        ir, iw = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
        ik = hdr.index("Kernel Name") if "Kernel Name" in hdr else None
        scale = {"Mbyte": 1e6, "Kbyte": 1e3, "Gbyte": 1e9, "byte": 1.0}
        tot = [float(r[ir]) * scale.get(units[ir], 1.0) + float(r[iw]) * scale.get(units[iw], 1.0)
               for r in rows[2:] if kernel_substr is None or ik is None or kernel_substr in r[ik]]
        return sum(tot) / len(tot) if tot else None
    except Exception:
        return None


def bconv_alg_bytes(in_shape, filt_shape, out_shape, out_itemsize=4):
    """SURVEY 8(d): packed input + packed filter + output + multiplier/bias."""
    return (int(np.prod(in_shape)) * 4 + int(np.prod(filt_shape)) * 4 +
            int(np.prod(out_shape)) * out_itemsize + 8 * filt_shape[0])


def bconv_word_ops(out_shape, filt_shape):
    return int(np.prod(out_shape[:3])) * filt_shape[0] * int(np.prod(filt_shape[1:]))


# --------------------------------------------------------------------------- #
# reference arm: the reference's own CPU kernels on the host cores
# --------------------------------------------------------------------------- #
def run_reference(workload, n_img, steps, warmup, input_type):
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import lce_testlib as L          # the cpu-baseline leg is where bench.py may use oracle/
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    impl = "ref" if L.load_ref() is not None else "oracle"
    kind = "reference" if impl == "ref" else "port"
    build = L.ref_build_info() if impl == "ref" else {"library": "oracle/liblce_oracle.so",
                                                       "flags": "-O3 -mpopcnt -msse4.2 -ffp-contract=off"}
    if workload == "bconv_stack":
        layers = make_stack_weights(0)
        inputs = [x[:n_img] for x in make_stage_inputs(n_img, 1)]

        def one_step():
            li = 0
            for s, (hw, c) in enumerate(STAGES):
                x = inputs[s]
                for _ in range(LAYERS_PER_STAGE):
                    lay = layers[li]; li += 1
                    d = L.BconvDesc(n_img, hw, hw, c, 3, 3, c, 1, 1, 1, 1, 1, L.PADDING_SAME, 1,
                                    L.ACT_RELU, L.OUT_FLOAT, 1.0, 0)
                    x = L.bconv2d(d, L.quantize(x, impl=impl), lay["filter"], lay["mul"],
                                  lay["bias"], impl=impl, kind=1, threads=cores)
        what = "16 layers (bitpack + Kernel4x2Portable indirect BGEMM)"
    else:
        import tflite_ref as R
        model = R.parse(build_model_bytes(workload, input_type))
        x = make_images(n_img, 1, input_type)

        def one_step():
            R.run(model, [x], threads=cores, lce_impl=impl, bconv_kind=1)
        what = ("full graph: LCE ops = reference bitpack + Kernel4x2Portable indirect BGEMM (+ zero-"
                "padding correction), float builtins = PyTorch CPU fp32 (TFLite's own builtins cannot "
                "be built offline)")
    for _ in range(warmup):
        one_step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        one_step()
        ts.append(time.perf_counter() - t0)
    dt = sum(ts) / max(steps, 1)
    return {"images_per_s": n_img / dt, "ms_per_step": dt * 1e3, "kind": kind, "cores": cores,
            "build": build, "step_ms": [round(t * 1e3, 1) for t in ts],
            "sample": f"{n_img} images per step, {steps} timed steps after {warmup} warm-up, "
                      f"{what}, one image per task on {cores} host threads"}


def cpu_baseline_subprocess(workload, batch, input_type):
    """The reference arm in its own process (its OpenMP settings must be in place before torch is
    imported; this process has long since imported it): bounded sample, 2 timed steps."""
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference",
                              "--workload", workload, "--batch", str(batch), "--steps", "2",
                              "--warmup", "1", "--input-type", input_type], env=env,
                             capture_output=True, text=True, timeout=900,
                             check=True).stdout.strip().splitlines()[-1]
        ref = json.loads(out)
        cb = dict(ref["cpu_baseline"])
        cb["value"], cb["unit"] = ref["value"], ref["unit"]
        return cb
    except Exception as e:  # never lose the GPU line over the baseline
        return {"value": None, "unit": "images/s", "error": str(e)[:200]}


def graph_config(workload, batch, world, input_type):
    return {"workload": workload, "batch_per_gpu": batch, "global_batch": batch * world,
            "model": f"{workload}: synthesised .tflite (random weights, seed 0)",
            "input": ("int8 images [B,224,224,3] + DEQUANTIZE in the graph (converter's "
                      "inference_input_type=int8)") if input_type == "int8" else "float32 images [B,224,224,3]"}


def main_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    # The LCE kernels run on a pthread pool, the float builtins on torch's OpenMP pool. With the
    # default active wait policy torch's idle workers spin on every core and starve the LCE
    # threads (measured on the 128-core box: 15.7 -> 134.8 images/s just from this setting).
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
    os.environ.setdefault("KMP_BLOCKTIME", "0")
    if args.workload == "bgemm_sweep":
        emit({"impl": "reference", "unavailable": "bgemm_sweep has no reference arm"})
        return
    steps = args.steps
    warm = min(args.warmup, 1)
    n_img = args.batch                          # the GPU arm's batch: same config on both arms
    r = run_reference(args.workload, n_img, steps, warm, args.input_type)
    cfg = (graph_config(args.workload, n_img, 1, args.input_type) if args.workload in GRAPHS
           else {"workload": args.workload, "batch_per_gpu": n_img, "global_batch": n_img})
    cfg["note"] = "reference CPU kernels on the host cores; rank 0 only"
    emit({
        "impl": "reference", "metric": METRIC[args.workload], "value": r["images_per_s"],
        "unit": "images/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32 xor-popcount + f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": r["images_per_s"], "unit": "images/s", "cores": r["cores"],
                         "kind": r["kind"], "sample": r["sample"], "build": r["build"],
                         "step_ms": r["step_ms"]},
        "e2e": {"value": r["images_per_s"], "unit": "images/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0})


# --------------------------------------------------------------------------- #
# B200 arm
# --------------------------------------------------------------------------- #
def bind_to_gpu_numa_node(torch, index):
    """Pin this rank (and so the pinned host buffers it allocates next: first touch) to the CPUs
    of the NUMA node its GPU hangs off. Without it 8 ranks pull their images across the socket
    link and end-to-end scaling bends (SCALE_r01: 0.76 at N = 8). Returns a description."""
    try:
        p = torch.cuda.get_device_properties(index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        base = f"/sys/bus/pci/devices/{bdf}"
        node = int(open(base + "/numa_node").read().strip())
        cpus = set()
        for part in open(base + "/local_cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"pci": bdf, "numa_node": node, "cpus_bound": len(cpus)}
    except Exception as e:  # containers without sysfs access: run unbound
        return {"error": str(e)[:120]}


class Dist:
    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.numa = bind_to_gpu_numa_node(torch, self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_ms(self, ms):
        t = self.torch.tensor([ms], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum(self, v):
        t = self.torch.tensor([float(v)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t)
        return float(t.item())

    def timed(self, fn, steps, sync, stream=None):
        """K steps bracketed by barrier + synchronize; device time from CUDA events on the
        launching stream; max over ranks."""
        torch = self.torch
        self.barrier()
        sync()
        stream = stream or torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        wall0 = time.time()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        sync()
        self.barrier()
        return self.max_ms(e0.elapsed_time(e1)), wall0, time.time()


def broadcast_model_bytes(D, workload, input_type):
    """Rank 0 owns the model file; ONE broadcast of the flatbuffer (packed weights + graph): the
    only collective of the whole run."""
    torch = D.torch
    if D.rank == 0:
        blob = np.frombuffer(build_model_bytes(workload, input_type), np.uint8)
        n = torch.tensor([blob.size], device=D.dev, dtype=torch.int64)
    else:
        n = torch.zeros(1, device=D.dev, dtype=torch.int64)
    if D.world > 1:
        D.dist.broadcast(n, src=0)
    model = torch.empty(int(n.item()), dtype=torch.uint8, device=D.dev)
    if D.rank == 0:
        model.copy_(torch.from_numpy(blob.copy()))
    if D.world > 1:
        D.dist.broadcast(model, src=0)
    return model.cpu().numpy().tobytes()


def parity_check(model_bytes, input_type, n_img=4):
    """Before anything is timed: n_img images through the UNFUSED graph with every tensor kept;
    each LCE op, fed with the device's own input, must equal the CPU checker bit for bit, and the
    FUSED graph's class probabilities (what is timed) must be bit-identical to the unfused graph's
    and within 2e-4 of the CPU graph's. The checker is oracle/_ref (the reference's own headers)
    when that library is present, else the oracle port."""
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import lce_testlib as L
    import tflite_ref as R
    from compute_engine_b200 import host as H
    impl = "ref" if L.load_ref() is not None else "oracle"
    m = R.parse(model_bytes)
    x = make_images(n_img, 7, input_type)
    g = H.HostGraph.from_tflite(model_bytes, device_arena=True)
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
        want, _ = R.run(sub, [g.read(op["inputs"][0])], lce_impl=impl, bconv_kind=1)
        got = g.read(op["outputs"][0])
        if got.shape != want[0].shape or not np.array_equal(got.view(np.uint8), want[0].view(np.uint8)):
            raise SystemExit(f"parity check FAILED at LCE op {n_lce} ({op['custom']}): GPU != {impl}")
        n_lce += 1
    unfused = g.read(g.outputs()[0])
    g.close()
    g = H.HostGraph.from_tflite(model_bytes, device_arena=True)
    g.fuse_all()
    g.resize_input(g.inputs()[0], x.shape)
    g.allocate_tensors()
    g.write(g.inputs()[0], x)
    g.invoke()
    fused = g.read(g.outputs()[0])
    g.close()
    if not np.array_equal(fused.view(np.uint8), unfused.view(np.uint8)):
        raise SystemExit("parity check FAILED: fused graph != unfused graph")
    want_out, _ = R.run(m, [x], lce_impl=impl, bconv_kind=1)
    err = float(np.abs(fused - want_out[0]).max())
    if err > 2e-4:
        raise SystemExit(f"parity check FAILED: probabilities differ from the CPU graph by {err}")
    return {"images": n_img, "lce_ops_bit_exact": n_lce, "checker": "oracle/_ref (reference headers)"
            if impl == "ref" else "oracle port", "fused_equals_unfused": True, "max_prob_err": err}


def graph_workload(D, workload, B, input_type, steps, warmup, want_e2e=True, want_profile=True,
                   model_bytes=None, env=None, want_outputs=False):
    """Full `.tflite` graph through the graph host (custom-op registrations). want_outputs: also
    return the graph outputs of the last timed step (res["outputs"], for --dump-outputs)."""
    torch = D.torch
    from compute_engine_b200 import capi, host as H
    saved = {}
    for k, v in (env or {}).items():
        saved[k] = os.environ.get(k)
        os.environ[k] = v
    try:
        if model_bytes is None:
            model_bytes = broadcast_model_bytes(D, workload, input_type)
        g = H.HostGraph.from_tflite(model_bytes, device_arena=True)
        fused = 0 if os.environ.get("LCE_NO_FUSION") else g.fuse_all()
        t_in, t_out = g.inputs()[0], g.outputs()[0]
        g.resize_input(t_in, (B, 224, 224, 3))
        g.allocate_tensors()
        gs = torch.cuda.ExternalStream(g.stream())
        host_in = torch.from_numpy(make_images(B, 100 + D.rank, input_type)).pin_memory()
        host_out = torch.empty(g.shape(t_out), dtype=torch.float32).pin_memory()
        in_bytes = host_in.numel() * host_in.element_size()
        out_bytes = host_out.numel() * 4
        g.write_ptr(t_in, host_in.data_ptr(), in_bytes)          # inputs resident in HBM
        g.synchronize()
        sync = g.synchronize

        # ---- (1) value: CUDA-graph replay, inputs resident -----------------------------
        g.invoke()                                               # eager: plans (weight images) are built
        g.synchronize()
        launches0 = capi.launch_count()
        g.invoke()                                               # eager again: exactly one step's kernels
        g.synchronize()
        per_step_launches = capi.launch_count() - launches0
        g.enable_cuda_graph(True)
        g.invoke()                                               # the eager pass before the capture
        g.synchronize()
        W = max(warmup, 3)
        for _ in range(W):                                       # capture happens on the first
            g.invoke()
        sampler = ClockSampler(D.local)
        if D.rank == 0:
            sampler.start()
        total_ms, w0, w1 = D.timed(g.invoke, steps, sync, gs)
        clocks = sampler.stop(w0, w1) if D.rank == 0 else None
        res = {"total_ms": total_ms, "clocks": clocks, "launches": per_step_launches * steps,
               "in_bytes": in_bytes, "out_bytes": out_bytes, "fused_nodes_removed": fused,
               "graph_nodes": g.num_nodes(), "arena_bytes": g.arena_bytes(),
               "model_bytes": len(model_bytes), "e2e_ms": None}
        if want_outputs:
            res["outputs"] = {f"output{i}": dump_array(g.read(t)) for i, t in enumerate(g.outputs())}

        # ---- (2) per-node device times: eager pass with CUDA events on the graph's stream
        if want_profile:
            g.enable_cuda_graph(False)
            g.enable_profiling(True)
            g.invoke(); g.synchronize(); g.reset_profile()
            prof_ms, _, _ = D.timed(g.invoke, steps, sync, gs)
            node_ms = g.node_times_ms()
            g.enable_profiling(False)
            if os.environ.get("LCE_BENCH_VERBOSE") and D.rank == 0:
                for i in range(g.num_nodes()):
                    ins, outs = g.node_io(i)
                    print(f"node {i:3d} {g.node_name(i):28s} {node_ms[i] / steps:8.4f} ms  "
                          f"{g.shape(ins[0])} -> {g.shape(outs[0])}", file=sys.stderr)
            conv_ms = conv_bytes = conv_words = 0
            n_conv = 0
            glue_bytes = 0      # float / byte builtins: every operand read once, the result written once
            by_op = {}
            for i in range(g.num_nodes()):
                name = g.node_name(i)
                by_op[name] = by_op.get(name, 0.0) + node_ms[i]
                if not name.startswith("LceBconv2d"):
                    ins, outs = g.node_io(i)
                    glue_bytes += sum(g.nbytes(t) for t in ins if t >= 0) + g.nbytes(outs[0])
                    if "+LceQuantize" in name:
                        glue_bytes += int(np.prod(g.shape(outs[0]))) // 8
                    continue
                ins, outs = g.node_io(i)
                conv_ms += node_ms[i]
                conv_bytes += bconv_alg_bytes(g.shape(ins[0]), g.shape(ins[1]), g.shape(outs[0]))
                if "+ADD" in name:            # fused shortcut read (+ packed signs written)
                    conv_bytes += int(np.prod(g.shape(outs[0]))) * 4
                if "+LceQuantize" in name:
                    conv_bytes += int(np.prod(g.shape(outs[0]))) // 8
                conv_words += bconv_word_ops(g.shape(outs[0]), g.shape(ins[1]))
                n_conv += 1
            res.update({"step_alg_bytes": conv_bytes + glue_bytes,
                        "conv_s_per_step": conv_ms * 1e-3 / steps, "conv_bytes": conv_bytes,
                        "conv_words": conv_words, "n_conv": n_conv * steps,
                        "conv_share": conv_ms / prof_ms if prof_ms else None,
                        "eager_ms_per_step": prof_ms / steps,
                        "by_op_ms_per_step": {k: round(v / steps, 4) for k, v in
                                              sorted(by_op.items(), key=lambda kv: -kv[1])}})

        # ---- (3) e2e: pinned host input -> H2D -> graph -> D2H of the result, every step,
        #      double-buffered so the copy of step i+1 overlaps the compute of step i
        if want_e2e:
            g.enable_cuda_graph(True)
            g.invoke(); g.invoke(); g.synchronize()
            copy_stream = torch.cuda.Stream()
            staging = [torch.empty(host_in.shape, dtype=host_in.dtype, device=D.dev) for _ in range(2)]
            copied = [torch.cuda.Event() for _ in range(2)]
            consumed = [torch.cuda.Event() for _ in range(2)]
            state = {"i": 0}

            def issue_copy(i):
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(consumed[i & 1])
                    staging[i & 1].copy_(host_in, non_blocking=True)
                    copied[i & 1].record(copy_stream)

            for ev in consumed:
                ev.record(gs)
            issue_copy(0)

            def step_e2e():
                i = state["i"]
                issue_copy(i + 1)                                # prefetch the next step's input
                gs.wait_event(copied[i & 1])
                g.write_ptr(t_in, staging[i & 1].data_ptr(), in_bytes)   # D2D into the arena
                consumed[i & 1].record(gs)
                g.invoke()
                g.read_ptr_async(t_out, host_out.data_ptr(), out_bytes)
                state["i"] = i + 1

            def sync_all():
                g.synchronize()
                copy_stream.synchronize()

            for _ in range(2):
                step_e2e()
            res["e2e_ms"], _, _ = D.timed(step_e2e, steps, sync_all, gs)
        g.close()
        return res
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def stack_workload(args, D):
    torch = D.torch
    from compute_engine_b200 import capi, parallel
    B = args.batch
    layers = make_stack_weights(0) if D.rank == 0 else None
    dev_layers, _ = parallel.broadcast_model(layers, D.dev)    # the only collective
    shapes = [(c, hw) for (hw, c) in STAGES for _ in range(LAYERS_PER_STAGE)]
    plans = []
    for (c, hw), lay in zip(shapes, dev_layers):
        d = capi.BconvDesc(B, hw, hw, c, 3, 3, c, 1, 1, 1, 1, 1, capi.PADDING_SAME, 1,
                           capi.ACT_RELU, capi.OUT_FLOAT, 1.0, 0)
        plans.append(capi.BConv2d(d, lay["filter"], lay["mul"], lay["bias"]))
    host_in = [torch.from_numpy(x).pin_memory() for x in make_stage_inputs(B, 100 + D.rank)]
    dev_in = [x.to(D.dev, non_blocking=True) for x in host_in]
    bufs = [[torch.empty((B, hw, hw, c), device=D.dev) for _ in range(2)] for (hw, c) in STAGES]
    packed = [torch.empty((B, hw, hw, c // 32), dtype=torch.int32, device=D.dev) for (hw, c) in STAGES]
    host_out = [torch.empty((B, hw, hw, c), dtype=torch.float32).pin_memory() for (hw, c) in STAGES]
    ev_pairs = []

    def step(record=False):
        li, outs = 0, []
        for s in range(len(STAGES)):
            x = dev_in[s]
            for k in range(LAYERS_PER_STAGE):
                capi.quantize(x, out=packed[s])
                y = bufs[s][k & 1]
                if record:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); plans[li](packed[s], out=y); e1.record()
                    ev_pairs.append((e0, e1))
                else:
                    plans[li](packed[s], out=y)
                x = y
                li += 1
            outs.append(x)
        return outs

    def step_e2e():
        for d, h in zip(dev_in, host_in):
            d.copy_(h, non_blocking=True)
        for h, o in zip(host_out, step()):
            h.copy_(o, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(D.local)
    if D.rank == 0:
        sampler.start()
    last = []

    def timed_step():
        last[:] = step(True)

    l0 = capi.launch_count()
    total_ms, w0, w1 = D.timed(timed_step, args.steps, torch.cuda.synchronize)
    launches = capi.launch_count() - l0
    clocks = sampler.stop(w0, w1) if D.rank == 0 else None
    torch.cuda.synchronize()
    outputs = ({f"stage{s}": dump_array(x.cpu().numpy()) for s, x in enumerate(last)}
               if args.dump_outputs and D.rank == 0 else None)
    conv_ms = sum(a.elapsed_time(b) for a, b in ev_pairs)
    e2e_ms = None
    if not args.no_e2e:
        step_e2e()
        e2e_ms, _, _ = D.timed(step_e2e, args.steps, torch.cuda.synchronize)
    conv_bytes = sum(bconv_alg_bytes((B, hw, hw, c // 32), (c, 3, 3, c // 32), (B, hw, hw, c))
                     for hw, c in STAGES) * LAYERS_PER_STAGE
    conv_words = sum(bconv_word_ops((B, hw, hw, c), (c, 3, 3, c // 32))
                     for hw, c in STAGES) * LAYERS_PER_STAGE
    return {"total_ms": total_ms, "e2e_ms": e2e_ms, "clocks": clocks, "launches": launches,
            "conv_s_per_step": conv_ms * 1e-3 / args.steps, "conv_bytes": conv_bytes,
            "conv_words": conv_words, "n_conv": len(ev_pairs), "conv_share": conv_ms / total_ms,
            "in_bytes": sum(x.numel() * 4 for x in host_in),
            "out_bytes": sum(x.numel() * 4 for x in host_out), "outputs": outputs}


SWEEP_MN = (256, 512, 1024, 2048, 4096)
SWEEP_K = (256, 512, 1024, 2048, 4096, 8192)


def bgemm_sweep(args, D):
    """BASELINE.json configs[4] / SURVEY 8(d) config 5: M, N in {256..4096}, K_bits in {256..8192},
    epilogues raw int32 / float / bitpacked; rows of A sharded over the ranks (W replicated).
    One JSON object per point on stderr."""
    torch = D.torch
    from compute_engine_b200 import capi
    hbm_peak, _, sm_max, bf16_peak, _ = measured_peaks()
    g = torch.Generator(device=D.dev).manual_seed(D.rank)
    flush = torch.empty(192 << 20, dtype=torch.uint8, device=D.dev)
    rows = []
    quick = os.environ.get("LCE_SWEEP_QUICK")
    for ep in ("raw", "float", "bitpacked"):
        for M in SWEEP_MN:
            for N in SWEEP_MN:
                for Kb in SWEEP_K:
                    if quick and not (M == N and Kb in (256, 2048, 8192)):
                        continue
                    if ep != "raw" and not (M == N or (M, N) in ((4096, 256), (256, 4096))):
                        continue        # raw: the full 150-point grid; float / bitpacked: the diagonal + corners
                    Kw, Ml = Kb // 32, max(M // D.world, 1)
                    A = torch.randint(-2**31, 2**31 - 1, (Ml, Kw), device=D.dev, generator=g,
                                      dtype=torch.int64).to(torch.int32)
                    Wt = torch.randint(-2**31, 2**31 - 1, (N, Kw), device=D.dev, generator=g,
                                       dtype=torch.int64).to(torch.int32)
                    if ep == "raw":
                        gemm, s_out = capi.BGemm(Wt), 4.0
                        out = torch.empty((Ml, N), dtype=torch.int32, device=D.dev)
                    elif ep == "float":
                        mul = np.random.default_rng(1).uniform(0.01, 1.5, N).astype(np.float32)
                        gemm, s_out = capi.BGemm(Wt, capi.OUT_FLOAT, (0, 2 * Kb), mul, mul), 4.0
                        out = torch.empty((Ml, N), dtype=torch.float32, device=D.dev)
                    else:
                        thr = np.full(N, Kb // 2, np.int32)
                        gemm, s_out = capi.BGemm(Wt, capi.OUT_BITPACKED, thresholds=thr), 1.0 / 8
                        out = torch.empty((Ml, (N + 31) // 32), dtype=torch.int32, device=D.dev)
                    for _ in range(3):
                        gemm(A, out)
                    ts = []
                    for _ in range(args.steps):
                        flush.zero_()                       # L2 flush between timed launches
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(); gemm(A, out); e1.record()
                        torch.cuda.synchronize()
                        ts.append(e0.elapsed_time(e1))
                    ms = D.max_ms(float(np.median(ts)))
                    alg = (M + N * D.world) * Kw * 4 + M * N * s_out
                    tops = 2 * M * N * Kb / ms / 1e9
                    rows.append({"epilogue": ep, "M": M, "N": N, "K_bits": Kb, "n_gpus": D.world,
                                 "ms": round(ms, 5), "binary_TOPS": round(tops, 2),
                                 "alg_GBps": round(alg / ms / 1e6, 1),
                                 "hbm_frac": round(alg / ms / 1e6 / (hbm_peak * D.world), 4),
                                 "tensor_frac": round(tops / (2 * bf16_peak * D.world), 4)})
                    gemm.close()
                    if D.rank == 0:
                        print(json.dumps(rows[-1]), file=sys.stderr)
    return rows


def tensor_block(conv_words, conv_s, bf16_peak, sm_max):
    tops = 2 * 32 * conv_words / conv_s / 1e12
    peak = 2.0 * bf16_peak
    return {"achieved": tops, "unit": "TOP/s (int8 MAC x 2)", "peak": peak, "frac": tops / peak,
            "peak_source": "2 x MEASURED_PEAKS.json bf16_tflops (kind::i8 issues at twice the bf16 "
                           "rate; tools/tc_probe.cu measures 7708 MAC/clk/SM at N = 256)",
            "legacy_mma_sync_peak": 148 * 2046.5 * sm_max * 1e6 * 2 / 1e12}


def main_b200(args):
    D = Dist()
    from compute_engine_b200 import capi
    capi.lib()
    hbm_peak, peak_src, sm_max, bf16_peak, _ = measured_peaks()
    if args.workload == "bgemm_sweep":
        rows = bgemm_sweep(args, D)
        if D.rank == 0:
            best = max(rows, key=lambda r: r["binary_TOPS"])
            best_hbm = max(rows, key=lambda r: r["hbm_frac"])
            emit({"metric": METRIC["bgemm_sweep"], "value": best["binary_TOPS"],
                  "unit": "binary TOPS", "n_gpus": D.world, "steps": args.steps, "warmup": 3,
                  "ms_per_step": best["ms"], "higher_is_better": True,
                  "scaling": "strong", "vs_baseline": None,
                  "dtype": "s8 x s8 -> s32 on tcgen05 kind::i8 (== xor-popcount, bit-exact)",
                  "data": "synthetic",
                  "roofline": {"bound": "hbm", "achieved": best_hbm["alg_GBps"], "peak": hbm_peak * D.world,
                               "unit": "GB/s", "frac": best_hbm["hbm_frac"], "traffic": None,
                               "point": best_hbm,
                               "points_at_or_above_0.40": sum(r["hbm_frac"] >= 0.40 for r in rows)},
                  "config": {"workload": "bgemm_sweep", "best_point": best, "points": len(rows),
                             "l2": "192 MiB flush between launches"}})
        if D.world > 1:
            D.dist.destroy_process_group()
        return

    B, K = args.batch, args.steps
    extras = D.world == 1 and not args.no_extras and args.workload in GRAPHS
    parity = None
    if args.workload == "bconv_stack":
        r = stack_workload(args, D)
        input_type = None
    else:
        input_type = args.input_type
        model_bytes = broadcast_model_bytes(D, args.workload, input_type)
        if extras:
            parity = parity_check(model_bytes, input_type)
        r = graph_workload(D, args.workload, B, input_type, K, args.warmup, want_e2e=not args.no_e2e,
                           model_bytes=model_bytes, want_outputs=bool(args.dump_outputs) and D.rank == 0)
    launches = int(D.sum(r["launches"]))
    multi_extra = None
    if D.world > 1 and args.workload == "quicknet" and not args.no_extras:
        # BASELINE.json configs[2] next to configs[1]: QuickNetLarge, batch 128 per GPU (1024 at N = 8)
        multi_extra = graph_workload(D, "quicknet_large", 128, input_type, K, 3,
                                     want_e2e=not args.no_e2e)
    if D.rank != 0:
        if D.world > 1:
            D.dist.destroy_process_group()
        return
    ms_per_step = r["total_ms"] / K
    n_launch = max(r["n_conv"] // K, 1)
    achieved = r["conv_bytes"] / r["conv_s_per_step"] / 1e9
    cfg = (graph_config(args.workload, B, D.world, input_type) if args.workload in GRAPHS
           else {"workload": args.workload, "batch_per_gpu": B, "global_batch": B * D.world})
    cfg.update({"parallelism": f"dp{D.world}: batch-sharded, one NCCL broadcast of the model at load, "
                               "no collective per step",
                "l2": "activations per step exceed the 126 MB L2 (largest tensor 205 MB)",
                "numa": D.numa})
    line = {
        "metric": METRIC[args.workload], "value": B * D.world / (ms_per_step * 1e-3),
        "unit": "images/s", "n_gpus": D.world, "steps": K, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None,
        "dtype": "s8 x s8 -> s32 (binary convs on tcgen05 kind::i8, bit-exact with xor-popcount) + "
                 "f32 (builtins, epilogue)",
        "data": "synthetic", "config": cfg, "clocks": r["clocks"], "gpu_launches": launches,
        "roofline": {
            "kernel": "lce::tc::bconv_tc_kernel (LceBconv2d [+ADD +LceQuantize]: TMA-staged packed "
                      "activations -> bits->bytes in TMEM -> tcgen05.mma kind::i8 -> fused "
                      "OutputTransform epilogue -> TMA store)",
            "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
            "frac": achieved / hbm_peak, "peak_source": peak_src,
            "traffic": ncu_traffic_per_launch("r02_ncu_bconv_tc_summary.csv", "bconv_tc")
            if args.workload == "quicknet" else None,
            "traffic_unit": "bytes per launch (mean over the binary-conv launches of one step, "
                            "ncu --set full, profiles/r02_ncu_bconv_tc_summary.csv)",
            "alg_bytes_per_launch": r["conv_bytes"] / n_launch,
            "launches_timed": r["n_conv"],
            "avg_launch_ms": r["conv_s_per_step"] * 1e3 / n_launch,
            "share_of_step": r["conv_share"],
            "timing": "separate eager pass of the same K steps with CUDA events around every node on "
                      "the graph's stream (events cannot sit inside a replayed CUDA graph)",
            "tensor": tensor_block(r["conv_words"], r["conv_s_per_step"], bf16_peak, sm_max)},
    }
    if r.get("step_alg_bytes"):
        floor_ms = r["step_alg_bytes"] / (hbm_peak * 1e9) * 1e3
        line["step_roofline"] = {"alg_bytes_per_step": r["step_alg_bytes"], "hbm_ms": floor_ms,
                                 "frac": floor_ms / (r["total_ms"] / K),
                                 "note": "all kernels of one step: operands read once + results written once "
                                         "(binary layers: SURVEY 8d bytes) at the measured HBM rate, against "
                                         "ms_per_step"}
    if r.get("e2e_ms") is not None:
        line["e2e"] = {"value": B * D.world / (r["e2e_ms"] / K * 1e-3), "unit": "images/s",
                       "h2d_bytes_per_step": r["in_bytes"], "d2h_bytes_per_step": r["out_bytes"],
                       "ms_per_step": r["e2e_ms"] / K,
                       "note": "pinned host input -> H2D -> graph -> D2H result every step; the copy of "
                               "step i+1 overlaps the compute of step i"}
    for k in ("by_op_ms_per_step", "eager_ms_per_step", "arena_bytes", "model_bytes",
              "fused_nodes_removed", "graph_nodes"):
        if k in r:
            line["config"][k] = r[k]
    if parity is not None:
        line["parity_checked"] = True
        line["parity"] = parity
    if extras:
        other_in = "float32" if input_type == "int8" else "int8"
        f = graph_workload(D, args.workload, B, other_in, K, 3, want_e2e=not args.no_e2e,
                           want_profile=False)
        line[f"{'f32' if other_in == 'float32' else 'int8'}_input"] = {
            "value": B / (f["total_ms"] / K * 1e-3), "ms_per_step": f["total_ms"] / K,
            "e2e": {"value": B / (f["e2e_ms"] / K * 1e-3), "h2d_bytes_per_step": f["in_bytes"],
                    "d2h_bytes_per_step": f["out_bytes"]} if f["e2e_ms"] else None,
            "unit": "images/s", "steps": K,
            "note": "the same graph with the other input type, same run"}
        line["legacy_paths"] = {}
        for name, env in (("mma_sync_int8", {"LCE_B200_BCONV_TC": "0"}),
                          ("xor_popc", {"LCE_B200_BCONV_TC": "0", "LCE_B200_BCONV_IMMA": "0"})):
            x = graph_workload(D, args.workload, B, input_type, K, 3, want_e2e=False,
                               want_profile=False, model_bytes=model_bytes, env=env)
            line["legacy_paths"][name] = {"value": B / (x["total_ms"] / K * 1e-3), "unit": "images/s",
                                          "ms_per_step": x["total_ms"] / K, "env": env}
        line["legacy_paths"]["note"] = ("same graph, same run, every LceBconv2d on the round-1 kernels: "
                                        "int8 mma.sync (lce_b200_imma.cuh) and the XOR + POPC kernel "
                                        "north_star describes (lce_b200_kernels.cuh)")
        line["other_configs"] = {}
        for wl, b in (("birealnet18", 512), ("quicknet_large", 128)):
            if wl == args.workload:
                continue
            o = graph_workload(D, wl, b, input_type, K, 3, want_e2e=not args.no_e2e)
            ach = o["conv_bytes"] / o["conv_s_per_step"] / 1e9
            line["other_configs"][wl] = {
                "batch": b, "value": b / (o["total_ms"] / K * 1e-3), "unit": "images/s",
                "ms_per_step": o["total_ms"] / K, "steps": K,
                "e2e": b / (o["e2e_ms"] / K * 1e-3) if o["e2e_ms"] else None,
                "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                             "frac": ach / hbm_peak, "share_of_step": o["conv_share"]},
                "by_op_ms_per_step": o["by_op_ms_per_step"]}
    if multi_extra is not None:
        o = multi_extra
        ach = o["conv_bytes"] / o["conv_s_per_step"] / 1e9
        line["other_configs"] = {"quicknet_large": {
            "batch_per_gpu": 128, "global_batch": 128 * D.world,
            "value": 128 * D.world / (o["total_ms"] / K * 1e-3), "unit": "images/s",
            "ms_per_step": o["total_ms"] / K, "steps": K,
            "e2e": 128 * D.world / (o["e2e_ms"] / K * 1e-3) if o["e2e_ms"] else None,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                         "frac": ach / hbm_peak, "share_of_step": o["conv_share"]}}}
    if not args.no_cpu_baseline and D.world == 1:
        line["cpu_baseline"] = cpu_baseline_subprocess(args.workload, B, input_type or "float32")
    if args.dump_outputs:
        write_dump(args.dump_outputs, r["outputs"])
    emit(line)
    if D.world > 1:
        D.dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        main_reference(a)
    else:
        main_b200(a)
