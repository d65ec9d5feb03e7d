"""Helpers shared by the CPU-tier and GPU-tier tests."""

from __future__ import annotations

import hashlib
import json
from pathlib import Path

import numpy as np
import yaml

from asyncflow_b200 import _capi as K

ROOT = Path(__file__).resolve().parent.parent
SCEN = ROOT / "tests" / "scenarios"
GOLD = ROOT / "tests" / "golden"
SEED = 0xA5F10
SERVER_SERIES = ("ready_queue_len", "event_loop_io_sleep", "ram_in_use")

#: scenario -> horizon used in the oracle-vs-engine parity tests (None = as written)
PARITY_CASES = {
    "c1_my_service.yml": 20, "c3_lb_two_servers.yml": 30, "c4_lb8_events.yml": 250,
    "ev_spikes_outages.yml": None, "mixed_lc.yml": None, "overload_single.yml": None,
    "chain_two_servers.yml": None, "poisson_ties.yml": None, "tie_cpu_io.yml": None,
    "c5_multihop32.yml": 8,
}


def load_scenario(name: str, horizon: int | None = None) -> dict:
    d = yaml.safe_load((SCEN / name).read_text())
    if horizon is not None:
        d["sim_settings"]["total_simulation_time"] = horizon
    return d


def load_golden(name: str) -> dict:
    return json.loads((GOLD / (Path(name).stem + ".json")).read_text())


def sha(arr: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()


def f64_digest(values) -> str:
    """SHA-256 of ``values`` as little-endian f64: how tests/golden/reference_runs.json pins clock lists
    and sampled series."""
    return sha(np.asarray(values, dtype="<f8"))


def load_reference_runs() -> dict:
    """What the unmodified reference computed for the reference-comparison tests
    (oracle/make_reference_runs.py)."""
    return json.loads((GOLD / "reference_runs.json").read_text())


def assert_matches_reference_run(rec: dict, *, generated, completed, clocks, edge_sent, edge_dropped,
                                 server_series=None, edge_series=None) -> None:
    """One run against one record of reference_runs.json, bit for bit; every series the reference
    sampled must be there (``*_series``: {entity id: {metric: list}})."""
    assert generated == rec["generated"]
    assert completed == rec["completed"]
    assert dict(edge_sent) == rec["edge_sent"]
    assert dict(edge_dropped) == rec["edge_dropped"]
    assert f64_digest(clocks) == rec["clocks_sha256"]
    for got, key in ((server_series, "server_series"), (edge_series, "edge_series")):
        if got is None:
            continue
        for ent, per in rec[key].items():
            for m, dig in per.items():
                assert f64_digest(got[ent][m]) == dig, (ent, m)


def pod_tables(flat) -> list[bytes]:
    """The flattened scenario as bytes, pointers left out: the header and every table row."""
    p = flat.pod
    out = [bytes(p)[: K.AfScenario.edges.offset]]
    for arr, n in (("edges", p.n_edges), ("servers", p.n_servers), ("endpoints", p.n_endpoints),
                   ("steps", p.n_steps), ("spike_marks", p.n_spike_marks), ("outage_marks", p.n_outage_marks)):
        out += [bytes(getattr(p, arr)[i]) for i in range(n)]
    out.append(np.array([p.lb_edges[i] for i in range(p.n_lb_edges)], dtype="<i4").tobytes())
    return out


def unhex(pairs) -> np.ndarray:
    return np.array([[float.fromhex(a), float.fromhex(b)] for a, b in pairs], dtype=np.float64).reshape(-1, 2)


def check_against_golden(vec: dict, *, generated, completed, clocks, edge_sent, edge_dropped,
                         throughput=None, series=None, flat=None) -> None:
    """`clocks` is an [n,2] f64 array in completion order; `series` [n_series, n_ticks] u32."""
    assert generated == vec["generated"]
    assert completed == vec["completed"]
    assert dict(edge_sent) == vec["edge_sent"]
    assert dict(edge_dropped) == vec["edge_dropped"]
    clocks = np.ascontiguousarray(clocks, dtype="<f8").reshape(-1, 2)
    assert clocks.shape[0] == vec["completed"]
    np.testing.assert_array_equal(clocks[:32], unhex(vec["clocks_head"]))
    np.testing.assert_array_equal(clocks[-32:], unhex(vec["clocks_tail"]))
    assert sha(clocks) == vec["clocks_sha256"]
    if "clocks" in vec:
        np.testing.assert_array_equal(clocks, unhex(vec["clocks"]))
    if throughput is not None:
        assert [int(x) for x in throughput] == vec["throughput"]
    if series is not None:
        for si, sid in enumerate(flat.server_ids):
            for mi, m in enumerate(SERVER_SERIES):
                g = vec["server_series"][sid].get(m)
                if g is None:
                    continue
                row = np.ascontiguousarray(series[3 * si + mi], dtype="<u4")
                assert len(row) == g["n"] and int(row.sum()) == g["sum"] and sha(row) == g["sha256"], (sid, m)
        for ei, eid in enumerate(flat.edge_ids):
            g = vec["edge_series"][eid].get("edge_concurrent_connection")
            if g is None:
                continue
            row = np.ascontiguousarray(series[3 * flat.n_servers + ei], dtype="<u4")
            assert len(row) == g["n"] and int(row.sum()) == g["sum"] and sha(row) == g["sha256"], eid


def oracle_series_matrix(o: dict, flat) -> np.ndarray:
    """Oracle sampled series in the engine's row order, [n_series, n_ticks]."""
    rows = []
    for sid in flat.server_ids:
        for m in SERVER_SERIES:
            rows.append(o["server_series"][sid].get(m, []))
    for eid in flat.edge_ids:
        rows.append(o["edge_series"][eid].get("edge_concurrent_connection", []))
    n = max((len(r) for r in rows), default=0)
    out = np.zeros((len(rows), n), dtype=np.uint32)
    for i, r in enumerate(rows):
        out[i, : len(r)] = r
    return out


def assert_matches_oracle(o: dict, flat, *, stats, clocks, sent, dropped, series=None,
                          throughput=None, hist=None) -> None:
    """Bit-exact comparison of one engine replica with one oracle replica."""
    assert int(stats["generated"]) == o["generated"]
    assert int(stats["completed"]) == o["completed"]
    assert [int(x) for x in sent] == [o["edge_sent"][e] for e in flat.edge_ids]
    assert [int(x) for x in dropped] == [o["edge_dropped"][e] for e in flat.edge_ids]
    oc = np.array(o["clocks"], dtype=np.float64).reshape(-1, 2)
    if clocks is not None:
        np.testing.assert_array_equal(np.asarray(clocks).reshape(-1, 2), oc)
    lat = oc[:, 1] - oc[:, 0]
    # sequential sums in completion order: the engine accumulates in the same order
    s = 0.0
    s2 = 0.0
    for x in lat.tolist():
        s += x
        s2 += x * x
    assert float(stats["lat_sum"]) == s
    assert float(stats["lat_sumsq"]) == s2
    if len(lat):
        assert float(stats["lat_min"]) == float(lat.min())
        assert float(stats["lat_max"]) == float(lat.max())
    if series is not None:
        np.testing.assert_array_equal(np.asarray(series), oracle_series_matrix(o, flat))
    if throughput is not None:
        thr = np.zeros(flat.horizon_s, dtype=np.int64)
        for f in oc[:, 1]:
            thr[int(np.ceil(f)) - 1] += 1
        np.testing.assert_array_equal(np.asarray(throughput, dtype=np.int64), thr)
    if hist is not None:
        assert int(np.asarray(hist).sum()) == o["completed"]
        if len(lat):
            # percentiles read off the histogram (128 bins per octave: <= 0.78 % wide) are within 1 % of numpy's exact
            # ones -- half of the 2 % the north star allows
            for q, key in ((50, "p50"), (95, "p95"), (99, "p99")):
                exact = float(np.percentile(lat, q))
                assert abs(float(stats[key]) - exact) <= 0.01 * exact, (key, float(stats[key]), exact)
