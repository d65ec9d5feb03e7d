"""The oracle port against what the UNMODIFIED reference actors computed: (a) the golden vectors
of tests/golden/<scenario>.json, (b) the runs of tests/golden/reference_runs.json."""

from __future__ import annotations

import des_port
import numpy as np
import pytest
from helpers import (PARITY_CASES, SEED, assert_matches_reference_run, check_against_golden, load_golden,
                     load_reference_runs, load_scenario)

from asyncflow_b200.flatten import flatten

REFERENCE_RUNS = load_reference_runs()


@pytest.mark.parametrize("name", sorted(PARITY_CASES) + ["c1_my_service_full.yml", "c3_lb_two_servers_full.yml"])
def test_port_reproduces_golden_vectors(name):
    gold = load_golden(name)                       # (*_full: the BASELINE horizons, 60 s / 600 s)
    payload = load_scenario(gold["scenario"], gold["horizon"])
    flat = flatten(payload)
    vectors = gold["vectors"] if gold["horizon"] <= 60 else gold["vectors"][:1]
    for vec in vectors:
        o = des_port.simulate(payload, seed=gold["seed"], replica=vec["replica"])
        oc = np.array(o["clocks"], dtype=np.float64).reshape(-1, 2)
        thr = np.zeros(gold["horizon"], dtype=np.int64)
        for f in oc[:, 1]:
            thr[int(np.ceil(f)) - 1] += 1
        from helpers import oracle_series_matrix
        check_against_golden(vec, generated=o["generated"], completed=o["completed"], clocks=oc,
                             edge_sent=o["edge_sent"], edge_dropped=o["edge_dropped"], throughput=thr,
                             series=oracle_series_matrix(o, flat), flat=flat)


def test_python_and_c_rng_backends_give_identical_runs():
    payload = load_scenario("mixed_lc.yml")
    a = des_port.simulate(payload, seed=SEED, replica=2, backend="py")
    b = des_port.simulate(payload, seed=SEED, replica=2, backend="c")
    assert a["clocks"] == b["clocks"] and a["edge_dropped"] == b["edge_dropped"]


def _port_equals_reference(payload, replica, rec):
    o = des_port.simulate(payload, seed=SEED, replica=replica)
    assert_matches_reference_run(rec, generated=o["generated"], completed=o["completed"], clocks=o["clocks"],
                                 edge_sent=o["edge_sent"], edge_dropped=o["edge_dropped"],
                                 server_series=o["server_series"], edge_series=o["edge_series"])


@pytest.mark.parametrize("name", sorted(PARITY_CASES))
def test_port_equals_unmodified_reference_actors(name):
    horizon = {"c1_my_service.yml": 12, "c3_lb_two_servers.yml": 15, "c4_lb8_events.yml": 245,
               "c5_multihop32.yml": 5}.get(name)
    payload = load_scenario(name, horizon)
    for rep in (1, 9):
        _port_equals_reference(payload, rep, REFERENCE_RUNS["actors"][f"{name}@{rep}"])
        if name.startswith("c4"):
            break


def test_reference_statistics_match_published_dashboard():
    """BASELINE.md: README LB example reads mean 0.024 / p95 0.034 / p99 0.040 s.  The reference's
    statistics of that run are stored; the port reproduces the run they were computed from."""
    rec = REFERENCE_RUNS["dashboard"]
    st = rec["latency_stats"]
    assert abs(st["mean"] - 0.024) < 0.001
    assert abs(st["p95"] - 0.034) < 0.002
    assert abs(st["p99"] - 0.040) < 0.003
    payload = load_scenario(rec["scenario"], rec["horizon"])
    _port_equals_reference(payload, rec["replica"], rec)


@pytest.mark.parametrize("seed", range(100, 130))
def test_port_equals_reference_on_random_tie_prone_scenarios(seed):
    """tests/fuzz.py scenarios (deterministic ties, queueing, every distribution, events): the port
    must reproduce the unmodified reference actors bit for bit -- the fuzz tests then compare the
    engine with the port."""
    import fuzz
    _port_equals_reference(fuzz.scenario(seed), seed, REFERENCE_RUNS["tie_prone"][str(seed)])


@pytest.mark.parametrize("seed", range(0, 8))
def test_port_equals_reference_on_big_topologies(seed):
    """C5-shaped random topologies (fuzz.big_scenario): LB over many front ends, shared back ends."""
    import fuzz
    _port_equals_reference(fuzz.big_scenario(seed), seed, REFERENCE_RUNS["big_topologies"][str(seed)])
