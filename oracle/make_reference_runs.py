"""Generate tests/golden/reference_runs.json: what the UNMODIFIED reference computes for every case
the reference-comparison tests check (tests/test_oracle.py, tests/test_flatten.py,
tests/test_integration_reference.py), so those tests run without the reference.

Needs a checkout of the reference (AsyncFlow 0.1.1):

    ASYNCFLOW_REFERENCE_SRC=<reference>/src python oracle/make_reference_runs.py

Runs come from ``oracle/ref_harness.run_reference`` (the reference's own ``SimulationRunner`` and actors
on the oracle kernel with AF-RNG injected).  Clock lists and sampled series are pinned by SHA-256
digests of their little-endian f64 bytes (``tests/helpers.py: f64_digest``), counters and analyzer
statistics are stored as they are.  The reference's example scenario files are stored as the payloads
the tests simulate (horizon cut to 40 s, event timeline compressed into it).
"""

from __future__ import annotations

import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "oracle", ROOT / "tests"):
    sys.path.insert(0, str(p))
import fuzz  # noqa: E402
import ref_harness  # noqa: E402
import yaml  # noqa: E402
from helpers import PARITY_CASES, SEED, f64_digest, load_scenario, pod_tables  # noqa: E402

from asyncflow_b200.flatten import SweepSpec, flatten  # noqa: E402

#: test_oracle.py::test_port_equals_unmodified_reference_actors: horizon overrides, replicas (c4: the first only)
ACTOR_HORIZONS = {"c1_my_service.yml": 12, "c3_lb_two_servers.yml": 15, "c4_lb8_events.yml": 245, "c5_multihop32.yml": 5}
ACTOR_REPLICAS = (1, 9)
TIE_PRONE_SEEDS = range(100, 130)
BIG_SEEDS = range(0, 8)
DASHBOARD = ("c3_lb_two_servers.yml", 120, 0)
ANALYZER_CASES = [("c1_my_service.yml", 15), ("ev_spikes_outages.yml", None), ("mixed_lc.yml", None)]
ANALYZER_REPLICA = 4
SWEEP_SEEDS = (301, 305, 312, 327)
SWEEP_ROWS = 2
SHIPPED_YAMLS = ["examples/yaml_input/data/two_servers_lb.yml", "examples/yaml_input/data/event_inj_single_server.yml",
                 "examples/yaml_input/data/heavy_inj_single_server.yml", "examples/yaml_input/data/single_server.yml",
                 "examples/yaml_input/data/event_inj_lb.yml", "tests/integration/single_server/data/single_server.yml"]
SHIPPED_HORIZON = 40
SHIPPED_REPLICA = 2
VALIDATED = ["c1_my_service.yml", "c4_lb8_events.yml", "mixed_lc.yml", "ev_spikes_outages.yml"]


def run_record(r: dict) -> dict:
    """Counters, clock digest and per-series digests of one reference run."""
    return {
        "generated": r["generated"], "completed": r["completed"],
        "edge_sent": r["edge_sent"], "edge_dropped": r["edge_dropped"],
        "clocks_sha256": f64_digest(r["clocks"]),
        "server_series": {sid: {k: f64_digest(v) for k, v in ser.items()} for sid, ser in r["server_series"].items()},
        "edge_series": {eid: {k: f64_digest(v) for k, v in ser.items()} for eid, ser in r["edge_series"].items()},
    }


def sampled_record(analyzer) -> dict:
    return {m: {ent: f64_digest(v) for ent, v in per.items()} for m, per in analyzer.get_sampled_metrics().items()}


def analyzer_record(r: dict) -> dict:
    ra = r["analyzer"]
    sid = ra.list_server_ids()[0]
    t, v = ra.get_series("ram_in_use", sid)
    return {
        "latency_stats": {k.value: float(x) for k, x in ra.get_latency_stats().items()},
        "throughput": [list(map(float, s)) for s in ra.get_throughput_series()],
        "throughput_2_5": [list(map(float, s)) for s in ra.get_throughput_series(window_s=2.5)],
        "sampled": sampled_record(ra),
        "server_ids": ra.list_server_ids(),
        "ram_in_use_series": {"server": sid, "t": f64_digest(t), "v": f64_digest(v)},
        "format_latency_stats": ra.format_latency_stats(),
    }


def shipped_payload(rel: str) -> dict:
    payload = yaml.safe_load((ref_harness.REFERENCE_SRC.parent / rel).read_text())
    full = int(payload["sim_settings"].get("total_simulation_time", 3600))
    horizon = min(full, SHIPPED_HORIZON)
    payload["sim_settings"]["total_simulation_time"] = horizon
    for ev in payload.get("events") or []:
        ev["start"]["t_start"] = float(ev["start"]["t_start"]) * horizon / full
        ev["end"]["t_end"] = float(ev["end"]["t_end"]) * horizon / full
    return payload


def main() -> None:
    if not ref_harness.reference_available():
        sys.exit("set ASYNCFLOW_REFERENCE_SRC to the src/ directory of a reference checkout")
    doc: dict = {"seed": SEED, "generator": "oracle/make_reference_runs.py (reference AsyncFlow 0.1.1)"}

    doc["actors"] = {}
    for name in sorted(PARITY_CASES):
        payload = load_scenario(name, ACTOR_HORIZONS.get(name))
        for rep in ACTOR_REPLICAS[:1] if name.startswith("c4") else ACTOR_REPLICAS:
            doc["actors"][f"{name}@{rep}"] = run_record(ref_harness.run_reference(payload, seed=SEED, replica=rep))

    doc["tie_prone"] = {str(s): run_record(ref_harness.run_reference(fuzz.scenario(s), seed=SEED, replica=s))
                        for s in TIE_PRONE_SEEDS}
    doc["big_topologies"] = {str(s): run_record(ref_harness.run_reference(fuzz.big_scenario(s), seed=SEED, replica=s))
                             for s in BIG_SEEDS}

    name, horizon, rep = DASHBOARD
    r = ref_harness.run_reference(load_scenario(name, horizon), seed=SEED, replica=rep)
    doc["dashboard"] = {"scenario": name, "horizon": horizon, "replica": rep, **run_record(r),
                        "latency_stats": {k.value: float(x) for k, x in r["analyzer"].get_latency_stats().items()}}

    doc["analyzer"] = {}
    for name, horizon in ANALYZER_CASES:
        r = ref_harness.run_reference(load_scenario(name, horizon), seed=SEED, replica=ANALYZER_REPLICA)
        doc["analyzer"][name] = {"clocks_sha256": f64_digest(r["clocks"]), **analyzer_record(r)}

    doc["sweep_rows"] = {}
    for seed in SWEEP_SEEDS:
        payload = fuzz.scenario(seed)
        spec = SweepSpec(flatten(payload), SWEEP_ROWS, fuzz.sweep_columns(seed, payload, SWEEP_ROWS))
        doc["sweep_rows"][str(seed)] = [run_record(ref_harness.run_reference(spec.payload_for(payload, i), seed=SEED,
                                                                             replica=i)) for i in range(SWEEP_ROWS)]

    doc["shipped_scenarios"] = {}
    for rel in SHIPPED_YAMLS:
        payload = shipped_payload(rel)
        r = ref_harness.run_reference(payload, seed=SEED, replica=SHIPPED_REPLICA)
        doc["shipped_scenarios"][rel] = {"payload": payload, **run_record(r), "sampled": sampled_record(r["analyzer"])}

    ref_harness._ensure_paths()
    from asyncflow.schemas.payload import SimulationPayload  # noqa: PLC0415
    doc["validated_payloads"] = {}
    for name in VALIDATED:
        model = SimulationPayload.model_validate(load_scenario(name))
        dumped = model.model_dump(mode="json")
        assert pod_tables(flatten(dumped)) == pod_tables(flatten(model)), name
        doc["validated_payloads"][name] = dumped

    path = ROOT / "tests" / "golden" / "reference_runs.json"
    path.write_text(json.dumps(doc, indent=0, separators=(",", ":")) + "\n")
    print(path.name, path.stat().st_size)


if __name__ == "__main__":
    main()
