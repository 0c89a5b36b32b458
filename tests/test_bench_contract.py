"""bench.py's reference arm is CPU-only, so its side of the measurement contract can be checked
without a GPU: ONE JSON line on stdout with the agreed keys (DESIGN.md section 6). The
--dump-outputs test runs the B200 arm."""
import json
import os
import subprocess
import sys
import textwrap

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference",
                          "--batch", "4", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, check=True).stdout
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, out
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "quicknet_images_per_sec"
    assert d["unit"] == "images/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}


def _bench(*args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *args],
                          capture_output=True, text=True, timeout=timeout)


def test_reference_arm_times_exactly_the_requested_steps():
    r = _bench("--impl", "reference", "--batch", "2", "--steps", "6", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout)
    assert d["steps"] == 6 and len(d["cpu_baseline"]["step_ms"]) == 6


def test_bad_arguments_are_refused():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"],
                 ["--workload", "bgemm_sweep", "--dump-outputs", "unused"]):
        r = _bench(*args, timeout=120)
        assert r.returncode == 2 and "error:" in r.stderr, (args, r.stderr[-500:])


def test_dump_sampling_is_fixed_and_bounded():
    """Outputs above DUMP_MAX_ELEMENTS are reduced to the same sorted flat indices in every run,
    in float32 (float64 for integers), and a dump over DUMP_MAX_BYTES is refused. bench.py redirects
    fd 1 when imported, so this runs in a child process."""
    code = textwrap.dedent("""
        import numpy as np
        import bench
        n = bench.DUMP_MAX_ELEMENTS
        x = np.arange(7 * (n // 2 + 1), dtype=np.int32).reshape(-1, 7)
        a, b = bench.dump_array(x), bench.dump_array(x.copy())
        assert a.shape == (n,) and a.dtype == np.float64 and np.array_equal(a, b)
        assert np.all(np.diff(a) > 0) and a[0] >= 0 and a[-1] < x.size   # distinct, sorted indices
        f = bench.dump_array(np.linspace(-1, 1, 2 * n + 1, dtype=np.float32))
        assert f.shape == (n,) and f.dtype == np.float32
        small = np.ones((4, 5), np.int8)
        assert np.array_equal(bench.dump_array(small), small) and bench.dump_array(small).shape == (4, 5)
        parts = {f"o{i}": a for i in range(bench.DUMP_MAX_BYTES // a.nbytes + 1)}
        try:
            bench.write_dump("unused", parts)
        except SystemExit as e:
            assert "limit" in str(e)
        else:
            raise AssertionError("an oversized dump was written")
        print("ok")
        """)
    r = subprocess.run([sys.executable, "-c", code], cwd=REPO, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0 and "ok" in r.stderr, r.stderr[-2000:]


@pytest.mark.gpu
def test_dump_outputs_repeat_from_run_to_run(tmp_path):
    """--dump-outputs writes the last timed step's outputs; inputs are seeded, so two runs with
    the same arguments write the same arrays."""
    import numpy as np
    common = ["--steps", "2", "--warmup", "1", "--no-extras", "--no-cpu-baseline", "--no-e2e"]
    for run in ("a", "b"):
        for wl, batch in (("quicknet", "8"), ("bconv_stack", "2")):
            r = _bench("--workload", wl, "--batch", batch, *common, "--dump-outputs",
                       str(tmp_path / run / wl))
            assert r.returncode == 0, r.stderr[-2000:]
    a = np.load(tmp_path / "a" / "quicknet" / "output0.npy")
    assert a.shape == (8, 1000) and a.dtype == np.float32
    assert np.array_equal(a, np.load(tmp_path / "b" / "quicknet" / "output0.npy"))
    assert np.allclose(a.sum(1), 1.0, atol=1e-3)                      # softmax probabilities
    for s, (hw, c) in enumerate([(56, 64), (28, 128), (14, 256), (7, 512)]):
        x = np.load(tmp_path / "a" / "bconv_stack" / f"stage{s}.npy")
        assert x.shape == (2, hw, hw, c) and x.dtype == np.float32 and np.isfinite(x).all()
        assert np.array_equal(x, np.load(tmp_path / "b" / "bconv_stack" / f"stage{s}.npy"))
