"""Generate tests/golden/*.json from the UNMODIFIED reference actors.

Needs a checkout of the reference:

    ASYNCFLOW_REFERENCE_SRC=<reference>/src python oracle/make_golden.py

Every vector is one replica of a scenario under tests/scenarios, simulated by
``oracle/ref_harness.run_reference`` -- the reference's own ``SimulationRunner``
and actors on the oracle kernel with AF-RNG injected.  Floats are stored as
``float.hex()`` so the fixtures pin BITS, not decimal renderings.  Large clock
lists are pinned by a SHA-256 over their little-endian f64 bytes plus the first
and last 32 entries.
"""

from __future__ import annotations

import hashlib
import json
import sys
from pathlib import Path

import numpy as np
import yaml

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "oracle"))
import ref_harness  # noqa: E402

SEED = 0xA5F10
#: scenario file -> (horizon override or None, replicas)
CASES = {
    "c1_my_service.yml": (20, [0, 1, 7]),
    "c3_lb_two_servers.yml": (30, [0, 3]),
    "c4_lb8_events.yml": (250, [2]),
    "ev_spikes_outages.yml": (None, [0, 5]),
    "mixed_lc.yml": (None, [0, 5, 11]),
    "overload_single.yml": (None, [0, 5]),
    "chain_two_servers.yml": (None, [0, 4]),
    "poisson_ties.yml": (None, [0, 5]),
    "tie_cpu_io.yml": (None, [1, 6]),
    "c5_multihop32.yml": (8, [1]),
}
#: the BASELINE shapes at their BASELINE horizons (README my_service.yml: 60 s; the LB example's YAML: 600 s) -- long-run
#: queue growth, u32 counters, trace capacity; hash-only, one replica each (VERDICT r1 item 10)
FULL_CASES = {
    "c1_my_service.yml": (60, [0]),
    "c3_lb_two_servers.yml": (600, [0]),
}
FULL_CLOCKS_MAX = 1500


def sha(arr: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()


def vector(payload: dict, replica: int) -> dict:
    r = ref_harness.run_reference(payload, seed=SEED, replica=replica)
    clocks = np.array(r["clocks"], dtype="<f8").reshape(-1, 2)
    T = payload["sim_settings"]["total_simulation_time"]
    lat = clocks[:, 1] - clocks[:, 0]
    thr = np.zeros(T, dtype=np.int64)
    for f in clocks[:, 1]:
        thr[int(np.ceil(f)) - 1] += 1
    # cross-check the bucket rule against the reference analyzer itself
    _, rps = r["analyzer"].get_throughput_series()
    assert [int(round(x)) for x in rps] == thr.tolist()
    stats = r["analyzer"].get_latency_stats()
    out = {
        "replica": replica, "generated": r["generated"], "completed": r["completed"],
        "edge_sent": r["edge_sent"], "edge_dropped": r["edge_dropped"],
        "clocks_sha256": sha(clocks), "throughput": thr.tolist(),
        "lat_sum_seq": float(sum(lat.tolist())).hex(),
        "latency_stats": {k.value: float(v).hex() for k, v in stats.items()},
        "clocks_head": [[a.hex(), b.hex()] for a, b in clocks[:32].tolist()],
        "clocks_tail": [[a.hex(), b.hex()] for a, b in clocks[-32:].tolist()],
        "server_series": {}, "edge_series": {},
    }
    if len(clocks) <= FULL_CLOCKS_MAX:
        out["clocks"] = [[a.hex(), b.hex()] for a, b in clocks.tolist()]
    for sid, ser in r["server_series"].items():
        out["server_series"][sid] = {
            k: {"n": len(v), "sum": int(sum(v)), "max": int(max(v)) if v else 0,
                "sha256": sha(np.array(v, dtype="<u4"))} for k, v in ser.items()}
    for eid, ser in r["edge_series"].items():
        out["edge_series"][eid] = {
            k: {"n": len(v), "sum": int(sum(v)), "max": int(max(v)) if v else 0,
                "sha256": sha(np.array(v, dtype="<u4"))} for k, v in ser.items()}
    return out


def main(only_full: bool = False) -> None:
    if not ref_harness.reference_available():
        sys.exit("set ASYNCFLOW_REFERENCE_SRC to the src/ directory of a reference checkout")
    gold = ROOT / "tests" / "golden"
    gold.mkdir(exist_ok=True)
    for name, (horizon, replicas) in ({} if only_full else CASES).items():
        payload = yaml.safe_load((ROOT / "tests" / "scenarios" / name).read_text())
        if horizon is not None:
            payload["sim_settings"]["total_simulation_time"] = horizon
        doc = {"scenario": name, "horizon": payload["sim_settings"]["total_simulation_time"],
               "seed": SEED, "generator": "oracle/make_golden.py (reference actors @ /root/reference)",
               "vectors": [vector(payload, rep) for rep in replicas]}
        path = gold / (Path(name).stem + ".json")
        path.write_text(json.dumps(doc, indent=0, separators=(",", ":")))
        print(path.name, path.stat().st_size, [v["completed"] for v in doc["vectors"]])
    for name, (horizon, replicas) in FULL_CASES.items():
        payload = yaml.safe_load((ROOT / "tests" / "scenarios" / name).read_text())
        payload["sim_settings"]["total_simulation_time"] = horizon
        doc = {"scenario": name, "horizon": horizon, "seed": SEED,
               "generator": "oracle/make_golden.py (reference actors @ /root/reference), BASELINE horizon",
               "vectors": [vector(payload, rep) for rep in replicas]}
        path = gold / (Path(name).stem + "_full.json")
        path.write_text(json.dumps(doc, indent=0, separators=(",", ":")))
        print(path.name, path.stat().st_size, [v["completed"] for v in doc["vectors"]])


if __name__ == "__main__":
    main(only_full="--full-only" in sys.argv)
