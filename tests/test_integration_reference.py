"""The OUT seam: engine results against what the reference's REAL ResultsAnalyzer computed.

The reference side is tests/golden/reference_runs.json (oracle/make_reference_runs.py: the unmodified
reference actors and analyzer), the engine side comes from the CPU debugging twin; the object under
test is the product's `ReplicaResults` (holders, getters).  On the GPU the same class is exercised with
real engine output by tests/test_gpu_parity.py::test_runner_api_mirrors_the_reference."""

from __future__ import annotations

import des_port
import pytest
import twin
from helpers import SEED, assert_matches_reference_run, f64_digest, load_reference_runs, load_scenario

from asyncflow_b200.flatten import flatten
from asyncflow_b200.results import ReplicaResults

REFERENCE_RUNS = load_reference_runs()


def twin_results(payload, replica) -> ReplicaResults:
    flat = flatten(payload)
    r = twin.run(flat, seed=SEED, replica_begin=replica, n=1, trace=1, clock_cap=100000)
    st = r["stats"][0]
    n, nt = int(st["completed"]), int(st["n_ticks"])
    return ReplicaResults(flat=flat, clocks=r["trace_clocks"][0, :n].copy(), series=r["trace_series"][0][:, :nt].copy(),
                          generated=int(st["generated"]), edge_sent=dict(zip(flat.edge_ids, map(int, r["sent"][0]))),
                          edge_dropped=dict(zip(flat.edge_ids, map(int, r["dropped"][0]))),
                          n_events=int(st["n_events"]), flags=int(st["flags"]))


def assert_sampled(rec: dict, got: dict) -> None:
    """Every series the reference analyzer holds, bit for bit (``rec``: {metric: {entity: digest}})."""
    assert set(rec) == set(got)
    for metric in rec:
        assert set(rec[metric]) == set(got[metric])
        for ent, dig in rec[metric].items():
            assert f64_digest(got[metric][ent]) == dig, (metric, ent)


@pytest.mark.parametrize("name,horizon", [("c1_my_service.yml", 15), ("ev_spikes_outages.yml", None), ("mixed_lc.yml", None)])
def test_reference_analyzer_on_engine_results_equals_reference_run(name, horizon):
    rec = REFERENCE_RUNS["analyzer"][name]
    mine = twin_results(load_scenario(name, horizon), 4)
    assert f64_digest(mine.clocks) == rec["clocks_sha256"]
    # what ResultsAnalyzer reads through its duck-typed seam
    h = mine.holders()
    assert f64_digest([(c.start, c.finish) for c in h["client"].rqs_clock]) == rec["clocks_sha256"]
    held: dict = {}
    for s in h["servers"]:
        for k, v in s.enabled_metrics.items():
            held.setdefault(k.value, {})[s.server_config.id] = v
    for e in h["edges"]:
        for k, v in e.enabled_metrics.items():
            held.setdefault(k.value, {})[e.edge_config.id] = v
    assert_sampled(rec["sampled"], held)
    assert (h["settings"].total_simulation_time, h["settings"].sample_period_s) == (mine.flat.horizon_s, mine.flat.sample_period)
    # and the product's own getters agree with the reference analyzer's
    assert mine.get_latency_stats() == rec["latency_stats"]
    assert [list(x) for x in mine.get_throughput_series()] == rec["throughput"]
    assert [list(x) for x in mine.get_throughput_series(window_s=2.5)] == rec["throughput_2_5"]
    assert_sampled(rec["sampled"], mine.get_sampled_metrics())
    assert mine.list_server_ids() == rec["server_ids"]
    ser = rec["ram_in_use_series"]
    t, v = mine.get_series("ram_in_use", ser["server"])
    assert (f64_digest(t), f64_digest(v)) == (ser["t"], ser["v"])
    assert mine.format_latency_stats() == rec["format_latency_stats"]


@pytest.mark.parametrize("seed", [301, 305, 312, 327])
def test_sweep_row_equals_unmodified_reference_on_payload_for(seed):
    """A sweep point handed back to the reference: the UNMODIFIED reference actors, run on
    SweepSpec.payload_for(i), produced the clocks the engine produces for row i of the sweep; the port
    (pinned to those actors by tests/test_oracle.py) reproduces them from today's payload_for(i)."""
    import fuzz

    from asyncflow_b200.flatten import SweepSpec

    payload = fuzz.scenario(seed)
    flat = flatten(payload)
    n = 2
    spec = SweepSpec(flat, n, fuzz.sweep_columns(seed, payload, n))
    r = twin.run(flat, seed=SEED, replica_begin=0, n=n, sweep=spec, trace=n, clock_cap=100000, request_capacity=200000)
    for i in range(n):
        ref = REFERENCE_RUNS["sweep_rows"][str(seed)][i]
        k = int(r["stats"][i]["completed"])
        assert f64_digest(r["trace_clocks"][i, :k]) == ref["clocks_sha256"]
        assert dict(zip(flat.edge_ids, map(int, r["dropped"][i]))) == ref["edge_dropped"]
        o = des_port.simulate(spec.payload_for(payload, i), seed=SEED, replica=i)
        assert_matches_reference_run(ref, generated=o["generated"], completed=o["completed"], clocks=o["clocks"],
                                     edge_sent=o["edge_sent"], edge_dropped=o["edge_dropped"])


REFERENCE_YAMLS = ["examples/yaml_input/data/two_servers_lb.yml", "examples/yaml_input/data/event_inj_single_server.yml",
                   "examples/yaml_input/data/heavy_inj_single_server.yml", "examples/yaml_input/data/single_server.yml",
                   "examples/yaml_input/data/event_inj_lb.yml", "tests/integration/single_server/data/single_server.yml"]


@pytest.mark.parametrize("rel", REFERENCE_YAMLS)
def test_every_scenario_file_the_reference_ships_runs_identically(rel):
    """The reference's own example / test YAMLs (stored as the payloads run: horizon cut to 40 s, event
    timeline compressed into it): unmodified reference actors == engine state machine, clock for clock
    and series for series."""
    rec = REFERENCE_RUNS["shipped_scenarios"][rel]
    mine = twin_results(rec["payload"], 2)
    assert f64_digest(mine.clocks) == rec["clocks_sha256"]
    assert mine.generated == rec["generated"] and mine.edge_dropped == rec["edge_dropped"]
    got = mine.get_sampled_metrics()
    for metric, per in rec["sampled"].items():
        for ent, dig in per.items():
            assert f64_digest(got[metric][ent]) == dig, (metric, ent)
