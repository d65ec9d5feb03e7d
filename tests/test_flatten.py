"""Payload -> POD flattening (host logic)."""

from __future__ import annotations

import numpy as np
import pytest
from helpers import load_reference_runs, load_scenario, pod_tables

from asyncflow_b200 import _capi as K
from asyncflow_b200.flatten import SweepSpec, flatten


def test_c4_tables():
    f = flatten(load_scenario("c4_lb8_events.yml"))
    p = f.pod
    assert (p.n_edges, p.n_servers, p.n_endpoints, p.n_steps, p.n_lb_edges) == (18, 8, 8, 16, 8)
    assert p.lb_algo == K.LB_ROUND_ROBIN and p.horizon_s == 300
    assert f.edge_ids[p.gen_edge] == "gen-client" and f.edge_ids[p.client_edge] == "client-lb"
    assert [f.edge_ids[p.lb_edges[i]] for i in range(8)] == [f"lb-srv{i}" for i in range(1, 9)]
    assert p.edges[0].dropout == 0.01 and p.edges[0].dist == K.DIST["exponential"]
    assert p.endpoints[0].total_ram == 128 and p.endpoints[0].n_steps == 2   # RAM step folded away
    assert [p.steps[i].kind for i in range(2)] == [K.STEP_CPU, K.STEP_IO]
    assert p.rate_per_user == 20 / 60
    assert p.n_spike_marks == 2 and p.n_outage_marks == 2
    assert (p.spike_marks[0].fire_time, p.spike_marks[0].delta) == (100.0, 0.030)
    assert (p.spike_marks[1].fire_time, p.spike_marks[1].delta) == (160.0, -0.030)
    assert f.edge_ids[p.outage_marks[0].lb_edge] == "lb-srv3" and p.outage_marks[0].down == 1
    assert p.outage_marks[1].fire_time == 240.0 and p.outage_marks[1].down == 0


def test_timeline_sort_and_fire_times():
    f = flatten(load_scenario("ev_spikes_outages.yml"))
    p = f.pod
    fires = [p.spike_marks[i].fire_time for i in range(p.n_spike_marks)]
    assert fires == sorted(fires)
    # END sorts before START at t=20 (ev-b ends, ev-c starts): injection.py:142-151
    at20 = [(f.spike_mark_events[i]) for i in range(p.n_spike_marks) if p.spike_marks[i].fire_time == 20.0]
    assert at20 == [("ev-b", "end"), ("ev-c", "start")]
    # a mark at t=0 fires at 0.0 (applied before the first event)
    assert p.spike_marks[0].fire_time == 0.0 and f.spike_mark_events[0] == ("ev-d", "start")


def test_defaults_follow_the_schema():
    d = load_scenario("chain_two_servers.yml")
    del d["sim_settings"]["sample_period_s"]
    del d["rqs_input"]["user_sampling_window"]
    f = flatten(d)
    assert f.pod.sample_period == 0.01 and f.pod.window_s == 60
    assert f.pod.metrics_mask == 15
    assert f.pod.users_dist == K.DIST["poisson"]          # RVConfig default distribution
    assert f.pod.lb_algo == K.LB_NONE and f.pod.n_lb_edges == 0
    # normal/log_normal without variance: variance = mean
    m = flatten(load_scenario("mixed_lc.yml"))
    e = m.pod.edges[m.edge_ids.index("srv1-client")]
    assert e.dist == K.DIST["normal"] and e.sigma == e.mean == 0.002


def test_explicitly_empty_metric_set_disables_sampling():
    d = load_scenario("c1_my_service.yml")
    d["sim_settings"]["enabled_sample_metrics"] = []
    assert flatten(d).pod.metrics_mask == 0
    d["sim_settings"]["enabled_sample_metrics"] = ["ram_in_use", "edge_concurrent_connection"]
    f = flatten(d)
    assert f.pod.metrics_mask == 4 | 8


def test_sweep_spec_columns():
    f = flatten(load_scenario("c3_lb_two_servers.yml"))
    n = 5
    spec = SweepSpec(f, n, {("users_mean",): np.linspace(10, 50, n), ("edge_mean", "client-lb"): 0.02,
                            ("server_ram_mb", "srv-2"): [256, 512, 768, 1024, 2048]})
    assert spec.values.shape == (n, 3)
    assert spec.columns == [(K.FIELDS["users_mean"], 0), (K.FIELDS["edge_mean"], 1), (K.FIELDS["server_ram_mb"], 1)]
    sw, rows = spec.pod(2, 2)
    assert sw.n_rows == 2 and rows[0, 0] == 30.0 and rows[1, 2] == 1024.0
    with pytest.raises(KeyError):
        SweepSpec(f, n, {("bogus",): 1.0})


def test_payload_for_spells_out_one_sweep_row():
    base = load_scenario("c4_lb8_events.yml")
    f = flatten(base)
    ev = next(e["event_id"] for e in base["events"] if "spike_s" in e["start"])
    spec = SweepSpec(f, 3, {("users_mean",): [10, 20, 30], ("rate_per_user",): [0.5, 1.0, 2.0],
                            ("edge_mean", "client-lb"): [0.001, 0.002, 0.003], ("edge_dropout", "client-lb"): 0.0,
                            ("server_cpu_cores", "srv-3"): [1, 2, 4], ("endpoint_ram", "srv-3", 0): [64, 0, 512],
                            ("step_duration", "srv-3", 0, 0): [0.001, 0.002, 0.004], ("spike_delta", ev): [0.1, 0.2, 0.3]})
    p = spec.payload_for(base, 2)
    assert base["rqs_input"]["avg_active_users"]["mean"] != 30          # the base is not touched
    g = flatten(p)
    assert g.pod.users_mean == 30 and g.pod.rate_per_user == 2.0
    e = f.edge_ids.index("client-lb")
    assert g.pod.edges[e].mean == 0.003 and g.pod.edges[e].dropout == 0.0
    s = f.server_ids.index("srv-3")
    assert g.pod.servers[s].cpu_cores == 4
    assert g.pod.endpoints[f.endpoint_index[("srv-3", 0)]].total_ram == 512
    assert g.pod.steps[f.step_index[("srv-3", 0, 0)]].duration == 0.004
    amps = sorted(abs(g.pod.spike_marks[i].delta) for i in range(g.pod.n_spike_marks))
    assert amps[-1] == 0.3
    # a zero-RAM row drops the RAM step altogether
    assert flatten(spec.payload_for(base, 1)).pod.endpoints[f.endpoint_index[("srv-3", 0)]].total_ram == 0
    # everything the sweep did not name is unchanged
    assert bytes(g.pod.servers[0]) == bytes(f.pod.servers[0])


def test_sweep_runner_hands_out_payloads_without_a_device():
    from asyncflow_b200 import SweepRunner
    base = load_scenario("c1_my_service.yml")
    sw = SweepRunner(base, 4, {("users_mean",): [10, 20, 30, 40]}, pinned=False)
    assert sw.payload_for(3)["rqs_input"]["avg_active_users"]["mean"] == 40
    r = sw.replica_runner(2)
    assert (r.seed, r.replica) == (sw.seed, 2) and r.simulation_input["rqs_input"]["avg_active_users"]["mean"] == 30
    with pytest.raises(IndexError):
        sw.payload_for(4)
    with pytest.raises(ValueError):
        SweepRunner(flatten(base), 2, pinned=False).payload_for(0)


@pytest.mark.parametrize("name", ["c1_my_service.yml", "c4_lb8_events.yml", "mixed_lc.yml", "ev_spikes_outages.yml"])
def test_validated_payload_flattens_like_the_raw_dict(name):
    """The schema defaults flatten() fills in are the reference's: the raw YAML dict flattens like the
    reference's own SimulationPayload validation of it (stored as its model_dump)."""
    d = load_scenario(name)
    validated = load_reference_runs()["validated_payloads"][name]
    assert pod_tables(flatten(d)) == pod_tables(flatten(validated))
