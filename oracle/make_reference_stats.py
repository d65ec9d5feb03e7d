"""Statistics of the UNMODIFIED reference with its OWN RNG (numpy PCG64) -> tests/golden/.

    ASYNCFLOW_REFERENCE_SRC=<reference>/src python oracle/make_reference_stats.py

The bit-exact parity chain (ref_harness -> des_port -> engine) injects AF-RNG through the
reference's seeding seam.  This script is the independent, statistical leg: the reference runs
exactly as upstream would run it -- ``SimulationRunner`` with ``numpy.random.default_rng(seed)`` in
``runner.rng`` (the documented seam, reference tests/integration/single_server/
test_int_single_server.py:36) and libm's ``math.log`` -- for N seeds, and the per-replica latency
statistics / counts are summarised (mean and standard error over replicas).  The engine's sweep
over the same scenario has to land inside those intervals (tests/test_statistical_parity.py):
BASELINE.json's "p50/p95/p99 latency within 2 % vs the SimPy reference".
"""

from __future__ import annotations

import json
import sys
from pathlib import Path

import numpy as np
import yaml

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "oracle"))
import ref_harness  # noqa: E402

CASES = {"c1_my_service.yml": (60, 96), "c3_lb_two_servers.yml": (60, 96), "mixed_lc.yml": (30, 160)}


def one(payload_dict: dict, seed: int) -> dict:
    ref_harness._ensure_paths()
    import simpy
    from asyncflow.runtime.simulation_runner import SimulationRunner
    from asyncflow.schemas.payload import SimulationPayload
    runner = SimulationRunner(env=simpy.Environment(), simulation_input=SimulationPayload.model_validate(payload_dict))
    runner.rng = np.random.default_rng(seed)
    an = runner.run()
    st = {k.value: float(v) for k, v in an.get_latency_stats().items()}
    _, rps = an.get_throughput_series()
    st["rps_mean"] = float(np.mean(rps))
    st["generated"] = float(next(iter(runner._rqs_runtime.values())).id_counter)
    sampled = an.get_sampled_metrics()
    st["ram_mean_first_server"] = float(np.mean(next(iter(sampled["ram_in_use"].values()))))
    st["io_mean_first_server"] = float(np.mean(next(iter(sampled["event_loop_io_sleep"].values()))))
    return st


def main() -> None:
    if not ref_harness.reference_available():
        sys.exit("set ASYNCFLOW_REFERENCE_SRC to the src/ directory of a reference checkout")
    out = {}
    for name, (horizon, n) in CASES.items():
        payload = yaml.safe_load((ROOT / "tests" / "scenarios" / name).read_text())
        payload["sim_settings"]["total_simulation_time"] = horizon
        rows = [one(payload, 1000 + s) for s in range(n)]
        keys = sorted(rows[0])
        arr = {k: np.array([r[k] for r in rows]) for k in keys}
        out[name] = {"horizon": horizon, "replicas": n, "rng": "numpy.random.default_rng(1000 + i)",
                     "mean": {k: float(v.mean()) for k, v in arr.items()},
                     "sem": {k: float(v.std(ddof=1) / np.sqrt(n)) for k, v in arr.items()}}
        print(name, {k: round(out[name]["mean"][k], 5) for k in ("mean", "median", "p95", "p99", "total_requests", "rps_mean")})
    (ROOT / "tests" / "golden" / "reference_numpy_stats.json").write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
