"""
bench.py's contract on a CPU box: the reference arm prints one JSON line with the
keys the driver reads (and times the CPU port on a bounded sample); the GPU arm
refuses to run without a CUDA device instead of falling back.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--ref-sample", "200"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "investor-steps/sec (leverage sweep)"
    assert d["unit"] == "investor-steps/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["steps"] == 1 and d["warmup"] == 0 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT,
                         env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def _bench_gpu(args, cwd):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--no-e2e", "--no-secondary",
                          "--no-cpu-baseline"] + args, capture_output=True, text=True, timeout=900, cwd=cwd)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


@pytest.mark.gpu
@pytest.mark.parametrize("workload, size", [("dice", ["--investors", "20000"]), ("gbm", ["--gbm-investors", "100000"])])
def test_gpu_arm_runs_the_asked_steps_and_dumps_its_outputs(tmp_path, workload, size):
    """--steps K times exactly K steps; --dump-outputs writes the last step's results, the same on every run."""
    dumps = []
    for k in (2, 3):
        d = _bench_gpu(["--workload", workload, "--steps", str(k), "--warmup", "1", "--dump-outputs",
                        str(tmp_path / f"k{k}")] + size, cwd=tmp_path)
        assert d["steps"] == k and d["n_gpus"] == 1
        files = {f[:-4]: np.load(tmp_path / f"k{k}" / f) for f in sorted(os.listdir(tmp_path / f"k{k}"))}
        names = ["growth", "stats"] if workload == "gbm" else ["stats"]
        assert sorted(files) == sorted(names + [n + "_nonfinite" for n in names])
        assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in files.values())
        got = {}
        for n in names:      # the values back: 0 finite, 1 +inf, 2 -inf, 3 nan
            code = files[n + "_nonfinite"]
            assert set(np.unique(code)) <= {0.0, 1.0, 2.0, 3.0} and (files[n][code != 0] == 0).all()
            got[n] = np.select([code == 1, code == 2, code == 3], [np.inf, -np.inf, np.nan], files[n])
        g = 10 if workload == "gbm" else 20
        assert got["stats"].shape == (g, 12)
        if workload == "gbm":
            assert np.array_equal(got["stats"][:, 9], d["check"]["median_wealth"], equal_nan=True)
            assert got["growth"].shape[0] == g and got["growth"][:, 0].tolist() == d["check"]["valid_runs"]
        else:
            assert d["gpu_launches"] == 3 * k
            assert got["stats"][0, 9] == d["check"]["median_wealth_lev0"]
        dumps.append(got)
    # same inputs on every run: order statistics exact, fp64 moments up to the order of their atomic sums
    a, b = dumps
    assert np.array_equal(a["stats"][:, 9:12], b["stats"][:, 9:12], equal_nan=True)
    for name in a:
        assert np.allclose(a[name], b[name], rtol=1e-12, atol=0, equal_nan=True), name


@pytest.mark.skipif(torch.cuda.is_available(), reason="GPU present")
def test_gpu_arm_fails_loudly_without_a_device():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0
    assert "no CUDA device" in (out.stderr + out.stdout)
