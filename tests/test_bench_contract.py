"""bench.py's stdout contract: exactly ONE JSON line, whatever native libraries print.

CPU legs only (the reference arm runs the oracle port on host cores); the GPU arm's line is
checked by the driver and by profiles/r01*_bench*.json.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]

REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
            "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline", "impl"}


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--horizon", "2"], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    out = json.loads(lines[0])
    assert REQUIRED <= set(out), REQUIRED - set(out)
    assert out["impl"] == "reference" and out["value"] > 0
    assert out["e2e"]["h2d_bytes_per_step"] == 0 and out["e2e"]["d2h_bytes_per_step"] == 0
    assert out["cpu_baseline"]["kind"] == "port" and out["cpu_baseline"]["cores"] >= 1


def test_native_stdout_is_diverted(tmp_path):
    code = ("import bench, ctypes\n"
            "bench.claim_stdout()\n"
            "c = ctypes.CDLL(None); c.printf(b'NCCL version x\\n'); c.fflush(None)\n"
            "print('stray python print')\n"
            "bench.emit({'ok': 1})\n")
    p = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stderr
    assert p.stdout == '{"ok": 1}\n'
    assert "NCCL version x" in p.stderr and "stray python print" in p.stderr


def test_gpu_arm_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        return
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "0"], cwd=ROOT,
                       capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and p.stdout.strip() == ""
    assert "no CPU fallback" in p.stderr


def test_every_config_builds_rows_that_are_a_pure_function_of_the_global_id():
    """--config c2|c3|c4|c5: the sweep row of a replica depends on its global id only, every rank's contiguous id
    range covers the whole grid (equal work per rank), and SweepSpec accepts the columns."""
    import numpy as np

    import bench
    from asyncflow_b200 import SweepSpec, flatten
    for key in ("c2", "c3", "c4", "c5"):
        w = bench.make_workload(key, horizon=5, replicas=4000)
        flat = flatten(w.payload)
        ids = np.arange(0, 4000, dtype=np.int64)
        a = SweepSpec(flat, 4000, w.columns(flat, ids, 4000))
        b = SweepSpec(flat, 4000, w.columns(flat, ids + 3 * 4000, 4000))      # rank 3 of a larger job: same grid
        assert np.array_equal(a.values, b.values) and a.n_columns >= 1, key
        sub = SweepSpec(flat, 7, w.columns(flat, ids[100:107], 4000))
        assert np.array_equal(sub.values, a.values[100:107]), key
        assert w.bytes_per_completion == 96.0 * w.events_per_completion + 8.0
        p = a.payload_for(w.payload, 1234)                                    # the reference-side view of one row
        assert p["sim_settings"]["total_simulation_time"] == 5


def test_effective_cores_respects_affinity_and_quota():
    import bench
    n, info = bench.effective_cores()
    assert 1 <= n <= (info["os_cpu_count"] or 1) and n <= info["affinity"]
    if info["cgroup_quota_cpus"]:
        assert n <= max(1, round(info["cgroup_quota_cpus"]))


def test_dump_outputs_writes_the_results_as_float64_within_the_budget(tmp_path, monkeypatch):
    """--dump-outputs on results of the twin-backed SweepRunner: every array float64, the per-replica ones
    whole while they fit, one fixed sample of rows (the same in every run) once they do not."""
    import numpy as np
    from twin_engine import TwinEngine

    import asyncflow_b200.runner as R
    import bench
    from asyncflow_b200 import flatten
    from asyncflow_b200.distributed import all_gather_summary, summary_block
    monkeypatch.setattr(R, "Engine", TwinEngine)
    w = bench.make_workload("c3", horizon=3, replicas=40)
    flat = flatten(w.payload)
    sw = R.SweepRunner(flat, 40, w.columns(flat, np.arange(40), 40), seed=bench.SEED, pinned=False)
    res = sw.run()
    res.global_summary = all_gather_summary(*summary_block(res.stats, None))

    bench.dump_outputs(str(tmp_path / "all"), res)
    got = {p.stem: np.load(p) for p in (tmp_path / "all").glob("*.npy")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert np.array_equal(got["replica_rows"], np.arange(40))
    assert np.array_equal(got["stats_completed"], res.stats["completed"])
    assert np.array_equal(got["sampled_sum"], res.samp_sum) and np.array_equal(got["edge_dropped"], res.edge_dropped)
    assert got["summary_counts"][0] == res.stats["completed"].sum()

    monkeypatch.setattr(bench, "DUMP_BYTES", 48 << 10)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), res)
        assert sum(p.stat().st_size for p in (tmp_path / run).glob("*.npy")) <= bench.DUMP_BYTES
    rows = np.load(tmp_path / "a" / "replica_rows.npy").astype(np.int64)
    assert 0 < len(rows) < 40 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "stats_lat_sum.npy"), res.stats["lat_sum"][rows])
    for p in (tmp_path / "a").glob("*.npy"):
        assert p.read_bytes() == (tmp_path / "b" / p.name).read_bytes(), p.name
