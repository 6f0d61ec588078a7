"""bench.py's output contract on the CPU box: the reference arm prints exactly ONE JSON line on stdout
(also under torch.distributed.run with two ranks, where rank 0 alone works), and the product arm refuses
to run without a CUDA device instead of falling back to anything."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline", "impl"}


def _run(cmd, timeout=600):
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    return subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)


def _check_line(stdout, n_gpus):
    lines = [l for l in stdout.splitlines() if l.strip()]
    assert len(lines) == 1, stdout
    j = json.loads(lines[0])
    assert KEYS <= set(j), KEYS - set(j)
    assert j["impl"] == "reference" and j["metric"] == "M points/s forward" and j["unit"] == "Mpoints/s"
    assert j["n_gpus"] == n_gpus and j["higher_is_better"] is True and j["vs_baseline"] is None
    assert j["value"] > 0 and j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0
    assert j["e2e"]["value"] == j["value"] and "workload" in j["config"]


def test_reference_arm_prints_one_json_line():
    r = _run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0"])
    assert r.returncode == 0, r.stderr[-2000:]
    _check_line(r.stdout, 1)


def test_reference_arm_dumps_the_outputs_of_its_last_step(tmp_path):
    r = _run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0",
              "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    _check_line(r.stdout, 1)
    assert sorted(os.listdir(tmp_path)) == ["logits.npy"]
    a = np.load(tmp_path / "logits.npy")
    assert a.dtype == np.float32 and a.shape == (1, 45056, 19) and np.isfinite(a).all()


def test_dumped_outputs_are_a_fixed_sample_under_64_mb():
    import torch
    import bench
    outs = (torch.arange(12_000_000, dtype=torch.float32), torch.arange(6_000_000, dtype=torch.float32).view(1000, 6000))
    a = bench.take_outputs(("x", "y"), outs)
    assert sorted(a) == ["x", "x.index", "y", "y.index"]
    assert sum(v.nbytes for v in a.values()) < 64e6
    for k in ("x", "y"):
        assert a[k].dtype == np.float32 and a[k + ".index"].dtype == np.float64
        assert np.array_equal(a[k], a[k + ".index"])            # arange: every kept value is its own index
    b = bench.take_outputs(("x", "y"), outs)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    small = bench.take_outputs(("z",), torch.ones(3, 4))
    assert list(small) == ["z"] and small["z"].shape == (3, 4)


def test_reference_arm_under_torchrun_rank0_only():
    r = _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
              "--master-addr", "127.0.0.1", "--master-port", "29533", "bench.py", "--gpus", "2", "--impl",
              "reference", "--steps", "1", "--warmup", "0"])
    assert r.returncode == 0, r.stderr[-2000:]
    _check_line(r.stdout, 2)


def test_product_arm_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("CUDA present: the product arm runs")
    r = _run([sys.executable, "bench.py", "--steps", "1"])
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")], "no bench line may be printed on a CPU box"
    assert "CUDA" in r.stderr or "NVIDIA" in r.stderr
