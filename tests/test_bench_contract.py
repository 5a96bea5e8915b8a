"""CPU: the parts of bench.py's contract that need no GPU -- the reference arm (`--impl reference`: the CPU oracle on the
bounded sample of the bench workload) prints ONE JSON line with the keys the driver reads, and marks its number as what
it is (a port, extrapolated from the sample)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from conftest import ROOT


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["metric"] == "Sim3 LM iterations/s" and d["unit"] == "LM iterations/s" and d["dtype"] == "f64"
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 0
    assert d["config"]["workload"].startswith("s1m")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["extrapolated"] is True and cb["cores"] >= 1 and "sample" in cb
    assert abs(cb["value"] - d["value"]) <= 1e-12 * d["value"]
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0 and e["unit"] == d["unit"]
    assert abs(e["value"] - d["value"]) <= 1e-12 * d["value"]


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun (N > 1) rank 0 alone runs the CPU arm; the other ranks exit 0 without output."""
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_caps_the_estimates_with_a_fixed_sample(tmp_path):
    """--dump-outputs stores at most bench.DUMP_ROWS estimate rows, always the same ones, as float64 .npy files."""
    est = np.arange(8.0 * (bench.DUMP_ROWS + 10)).reshape(-1, 8)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), est, 2.5, 0.1, np.ones((1, 5)))
    names = sorted(f for f in os.listdir(tmp_path / "a"))
    assert names == ["chi2.npy", "estimate_rows.npy", "estimates.npy", "lambda.npy", "lm_history.npy"]
    for f in names:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and np.array_equal(a, b)
    rows = np.load(tmp_path / "a" / "estimate_rows.npy").astype(np.int64)
    assert len(rows) == bench.DUMP_ROWS and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "estimates.npy"), est[rows])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= 64e6


def test_bench_rejects_arguments_it_cannot_honour():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                           timeout=300, cwd=ROOT)
        assert r.returncode != 0 and "error" in r.stderr


@pytest.mark.gpu
def test_bench_runs_exactly_the_steps_asked_for_and_dumps_the_last_one(tmp_path):
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "s10k", "--steps", "5", "--warmup", "2",
                        "--no-configs", "--no-cpu-baseline", "--no-parity", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == 5 and len(d["step_ms"]) == 5 and len(d["step_trace"]) == 5
    est = np.load(out / "estimates.npy")
    assert est.shape == (10000, 8) and np.array_equal(np.load(out / "estimate_rows.npy"), np.arange(10000.0))
    assert np.allclose(np.linalg.norm(est[:, :4], axis=1), 1.0)
    # the dump is the last timed step: its chi2 and lambda close that step's trace row
    last = d["step_trace"][-1]
    assert np.load(out / "chi2.npy")[0] == last[0] and np.load(out / "lm_history.npy")[-1].tolist() == last
    assert np.load(out / "lambda.npy")[0] > 0
