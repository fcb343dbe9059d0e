"""bench.py prints exactly one JSON line with the contract's keys (checked on the CPU-runnable
reference arm; the CUDA arm prints the same structure and is exercised on the GPU box)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--imagesets", "6",
                        "--steps", "1", "--warmup", "0", "--cpu-budget", "2"], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    # every step is a COMPLETE iteration: the reported time is the measured time, not an extrapolation
    assert d["steps"] >= 1 and len(d["attempts_per_step"]) == d["steps"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and d["value"] > 0


def _bench_with_dump(out_dir, *extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--imagesets", "6", "--steps", "2", "--warmup",
                        "0", "--dump-outputs", str(out_dir), *extra], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout)
    arrays = {f[:-4]: np.load(out_dir / f) for f in os.listdir(out_dir)}
    assert sorted(arrays) == d["dump_outputs"]["arrays"]
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(os.path.getsize(out_dir / f) for f in os.listdir(out_dir)) <= 64 * 2 ** 20
    return d, arrays


def test_reference_arm_dumps_the_same_outputs_on_every_run(tmp_path):
    runs = [_bench_with_dump(tmp_path / f"run{i}", "--impl", "reference", "--config", "1", "--cpu-budget", "600")
            for i in range(2)]
    (d, a), (_, b) = runs
    assert d["steps"] == 2 and float(a["final_cost"]) == d["costs"][-1]
    assert a["points"].shape == (d["config"]["n_points"], 3) and a["rig_tr_global"].shape == (6, 7)
    assert a["last_projection"].shape == (d["config"]["n_obs"], 2)
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)


@pytest.mark.gpu
def test_cuda_arm_dumps_its_last_step(tmp_path):
    d, a = _bench_with_dump(tmp_path, "--no-cpu-baseline", "--no-library-comparison")
    assert d["steps"] == 2 and len(d["step_ms"]) == 2
    assert float(a["final_cost"]) == d["final_cost"] and float(a["rmse"]) == d["rmse_px"]
    assert a["points"].shape == (d["config"]["n_points"], 3) and np.isfinite(a["points"]).all()
    assert a["last_projection"].shape == (d["config"]["n_obs"], 2)


def test_dump_samples_last_projection_beyond_the_size_limit(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    from camera_calibration_b200 import cabi
    n = bench.DUMP_LIMIT_BYTES // 16 + 1000
    st = cabi.FlatState(np.zeros((10, 3)), np.zeros((4, 7)), np.zeros((1, 7)), [np.zeros(12)],
                        np.arange(2 * n, dtype=np.float64).reshape(n, 2))
    info = bench.dump_outputs(str(tmp_path), st, cabi.Report())
    assert info["last_projection_sampled"] and info["bytes"] <= bench.DUMP_LIMIT_BYTES
    rows = np.load(tmp_path / "last_projection_rows.npy")
    lp = np.load(tmp_path / "last_projection.npy")
    assert len(rows) == len(lp) and np.all(np.diff(rows) > 0)
    assert np.array_equal(lp, st.last_projection[rows.astype(np.int64)])
    bench.dump_outputs(str(tmp_path / "again"), st, cabi.Report())
    assert np.array_equal(np.load(tmp_path / "again" / "last_projection_rows.npy"), rows)


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
