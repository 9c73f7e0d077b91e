"""bench.py's driver contract, as far as it can be checked without a GPU: the reference arm prints
one JSON line with the agreed keys (the b200 arm needs a device and is exercised on the GPU box)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from path_optimizer_2_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-sample", "16", *extra], capture_output=True, text=True, check=True, cwd=ROOT).stdout
    lines = [ln for ln in out.splitlines() if ln.strip()]
    assert len(lines) == 1, out
    return json.loads(lines[0])


def test_reference_arm_json_line():
    d = _run()
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "solves/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["vs_baseline"] is None and d["gpu_launches"] == 0 and "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_is_float_and_repeats_run_to_run(tmp_path):
    dumps = []
    for run in range(2):
        d = tmp_path / ("run%d" % run)
        line = _run("--steps", "2", "--dump-outputs", str(d))
        assert line["steps"] == 2
        dumps.append({p.stem: np.load(p) for p in sorted(d.glob("*.npy"))})
    a, b = dumps
    assert sorted(a) == ["cost", "instance", "iters", "sol", "status"]
    assert a["sol"].shape == (16, 4, 240) and a["cost"].shape == (16,) and np.array_equal(a["instance"], np.arange(16))
    for name in a:
        assert a[name].dtype == np.float64 and np.array_equal(a[name], b[name]), name
    assert np.all(a["status"] == abi.PQP_SOLVED) and np.all(a["iters"] > 0)


def test_dump_outputs_samples_instances_under_the_size_limit(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 100_000)
    batch = 100
    arrays = {"sol": np.arange(batch * 4 * 60, dtype=np.float64).reshape(batch, 4, 60), "cost": np.arange(batch) + 0.5,
              "status": np.zeros(batch, dtype=np.int32), "iters": np.arange(batch, dtype=np.int32)}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    files = sorted((tmp_path / "a").glob("*.npy"))
    assert sum(p.stat().st_size for p in files) <= 100_000
    idx = np.load(tmp_path / "a" / "instance.npy").astype(np.int64)
    assert 0 < len(idx) < batch and np.all(np.diff(idx) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "sol.npy"), arrays["sol"][idx])
    assert np.array_equal(np.load(tmp_path / "a" / "iters.npy"), idx)
    for p in files:
        assert np.array_equal(np.load(p), np.load(tmp_path / "b" / p.name))


@pytest.mark.gpu
def test_dump_outputs_of_the_gpu_workloads(tmp_path):
    """The device-resident cold loop (measure_cold) and the receding-horizon loop (run_receding): float64 arrays of the
    last timed step, the ones the printed line summarises, identical from run to run."""
    def run(workload, d):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--batch", "64",
                              "--steps", "2", "--warmup", "3", "--no-secondary", "--no-cpu", "--dump-outputs", str(d)],
                             capture_output=True, text=True, check=True, cwd=ROOT).stdout
        line = json.loads([ln for ln in out.splitlines() if ln.strip()][-1])
        dump = {p.stem: np.load(p) for p in sorted(d.glob("*.npy"))}
        assert sorted(dump) == ["cost", "instance", "iters", "sol", "status"]
        assert dump["sol"].shape == (64, 4, 240) and np.array_equal(dump["instance"], np.arange(64))
        assert all(a.dtype == np.float64 and len(a) == 64 for a in dump.values())
        assert line["steps"] == 2
        assert np.mean(dump["status"] == abi.PQP_SOLVED) == line["config"]["solved_fraction"] > 0
        assert np.mean(dump["iters"]) == line["config"]["mean_admm_iters"]
        return dump

    a, b = run("cold", tmp_path / "cold0"), run("cold", tmp_path / "cold1")
    for name in a:
        assert np.array_equal(a[name], b[name]), name
    r = run("receding", tmp_path / "receding")
    assert np.all(r["iters"] <= 50)


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_b200_arm_refuses_to_run_without_a_device():
    try:
        import torch
        if torch.cuda.is_available():
            return
    except ImportError:
        pass
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, cwd=ROOT)
    assert p.returncode != 0 and "no CPU path" in (p.stderr + p.stdout)


def test_numa_binding_is_a_no_op_without_a_device():
    """bench.py binds each rank to its GPU's NUMA node when N > 1; without a device (or without sysfs topology) it
    must leave the process where it is and report None."""
    import os
    import bench
    before = os.sched_getaffinity(0)
    assert bench.bind_to_gpu_numa_node(0) is None
    assert os.sched_getaffinity(0) == before
