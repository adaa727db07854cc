"""bench.py contract on the CPU: the reference arm (`--impl reference`) runs without a GPU and prints ONE JSON line
with the keys the driver reads; the GPU arm refuses to run without a GPU (no CPU fallback)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--workload", "small"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "csx_spmv_gflops" and d["unit"] == "GFLOP/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["value"] > 0 and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_dump_outputs_is_bounded_and_repeatable(tmp_path):
    """--dump-outputs: float64 .npy files, a long vector sampled on the same rows every time, a short one whole."""
    import numpy as np
    import torch
    import bench
    v = torch.arange(bench.DUMP_MAX_ENTRIES + 1000, dtype=torch.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"y": v, "short": v[:10]})
    a, b = np.load(str(tmp_path / "a" / "y.npy")), np.load(str(tmp_path / "b" / "y.npy"))
    assert a.dtype == np.float64 and a.size == bench.DUMP_MAX_ENTRIES and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0)   # distinct rows in increasing order (the values are the row indices)
    assert np.array_equal(np.load(str(tmp_path / "a" / "short.npy")), v[:10].numpy())


def test_refused_arguments(tmp_path):
    """No timed step at all, and a dump where it is not implemented, are refused before any work."""
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "out")]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "small"] + args,
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 2 and "error:" in r.stderr, (args, r.stderr[-2000:])
    assert not os.path.exists(str(tmp_path / "out"))


def test_gpu_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        return   # covered by the -m gpu tests and the bench itself
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "small", "--steps", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "needs a GPU" in (r.stderr + r.stdout)
