"""CPU oracle: a restatement of AsyncFlow's actor layer on the oracle kernel.

ORACLE / TEST INFRASTRUCTURE ONLY (importers: ``tests/``, ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs, ``__graft_entry__.smoke()``).
The product path is the CUDA engine; nothing under ``asyncflow_b200/`` imports
this module.

Unlike ``oracle/ref_harness.py`` this file does not need ``/root/reference``,
so it travels to the GPU box.  It keeps the reference's *execution model* --
one Python generator per actor / per in-flight message, driven by a simpy-style
heap (``oracle/simpy_shim``) -- so that timing it is a fair statement of "the
reference's CPU path", and it follows the reference function by function:

===========================  ==================================================
here                         reference (``/root/reference/src/asyncflow``)
===========================  ==================================================
``normalise_payload``        schemas/** defaults (constants.py:137, 23-40, ...)
``_Generator.run``           runtime/actors/rqs_generator.py:97-119 +
                             samplers/poisson_poisson.py:39-82 /
                             samplers/gaussian_poisson.py:64-94
``_Edge.deliver``            runtime/actors/edge.py:73-116
``_Client.run``              runtime/actors/client.py:43-71
``_LoadBalancer.run``        runtime/actors/load_balancer.py:60-72,
                             routing/lb_algorithms.py:10-36
``_Server.dispatch/handle``  runtime/actors/server.py:79-276, 303-313
``_Injection``               runtime/events/injection.py:35-226
``_collector``               metrics/collector.py:50-66
``simulate`` (start order)   runtime/simulation_runner.py:349-376, 301-342
===========================  ==================================================

Parity pin: ``tests/test_oracle.py`` (against the stored reference runs) requires
this port to reproduce ``ref_harness.run_reference`` -- the unmodified
reference actors -- bit for bit (every (start, finish) clock, every counter,
every sampled series) on all scenarios under ``tests/scenarios``; the golden
vectors under ``tests/golden`` were produced by the reference harness and are
checked against this port on every box.
"""

from __future__ import annotations

import sys
from collections import OrderedDict
from pathlib import Path

_HERE = Path(__file__).resolve().parent
for _p in (str(_HERE), str(_HERE / "simpy_shim")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import afrng  # noqa: E402
import simpy  # noqa: E402  (oracle/simpy_shim)

CPU_KINDS = {"initial_parsing", "cpu_bound_operation"}
IO_KINDS = {"io_task_spawn", "io_llm", "io_wait", "io_db", "io_cache"}
RAM_KINDS = {"ram"}
ALL_SAMPLED = ("ready_queue_len", "event_loop_io_sleep", "ram_in_use",
               "edge_concurrent_connection")


# --------------------------------------------------------------------------- #
# payload defaults                                                            #
# --------------------------------------------------------------------------- #
def _rv(d: dict) -> dict:
    dist = d.get("distribution", "poisson")          # RVConfig default
    var = d.get("variance")
    if var is None and dist in ("normal", "log_normal"):
        var = d["mean"]                                # default_variance validator
    return {"mean": float(d["mean"]), "distribution": dist,
            "variance": None if var is None else float(var)}


def normalise_payload(p: dict) -> dict:
    """Fill the schema defaults into a YAML-shaped payload dict."""
    g = p["rqs_input"]
    nodes = p["topology_graph"]["nodes"]
    ss = p.get("sim_settings", {}) or {}
    out = {
        "rqs_input": {
            "id": g["id"],
            "avg_active_users": _rv(g["avg_active_users"]),
            "avg_request_per_minute_per_user": _rv(g["avg_request_per_minute_per_user"]),
            "user_sampling_window": int(g.get("user_sampling_window", 60)),
        },
        "client": {"id": nodes["client"]["id"]},
        "load_balancer": None,
        "servers": [],
        "edges": [],
        "sim_settings": {
            "total_simulation_time": int(ss.get("total_simulation_time", 3600)),
            "sample_period_s": float(ss.get("sample_period_s", 0.01)),
            "enabled_sample_metrics": list(ss.get("enabled_sample_metrics", ALL_SAMPLED)),
        },
        "events": [],
    }
    lb = nodes.get("load_balancer")
    if lb is not None:
        out["load_balancer"] = {
            "id": lb["id"],
            "algorithms": lb.get("algorithms", "round_robin"),
            "server_covered": list(lb.get("server_covered", [])),
        }
    for s in nodes["servers"]:
        res = s.get("server_resources", {}) or {}
        eps = []
        for ep in s["endpoints"]:
            steps = []
            for st in ep["steps"]:
                (op, val), = st["step_operation"].items()
                steps.append({"kind": str(st["kind"]), "op": str(op), "value": val})
            eps.append({"endpoint_name": ep["endpoint_name"].lower(), "steps": steps})
        out["servers"].append({
            "id": s["id"],
            "cpu_cores": int(res.get("cpu_cores", 1)),
            "ram_mb": int(res.get("ram_mb", 1024)),
            "endpoints": eps,
        })
    for e in p["topology_graph"]["edges"]:
        out["edges"].append({
            "id": e["id"], "source": e["source"], "target": e["target"],
            "latency": _rv(e["latency"]),
            "dropout_rate": float(e.get("dropout_rate", 0.01)),
        })
    for ev in p.get("events") or []:
        out["events"].append({
            "event_id": ev["event_id"], "target_id": ev["target_id"],
            "t_start": float(ev["start"]["t_start"]), "t_end": float(ev["end"]["t_end"]),
            "start_kind": str(ev["start"]["kind"]),
            "spike_s": ev["start"].get("spike_s"),
        })
    return out


# --------------------------------------------------------------------------- #
# RNG back-ends (same numbers; the C one only removes interpreter overhead)   #
# --------------------------------------------------------------------------- #
class PyRng:
    """AF-RNG through the normative pure-Python spec (``oracle/afrng.py``)."""

    def __init__(self, seed: int, replica: int) -> None:
        self.seed, self.replica = seed, replica
        self.gen = afrng.GenStream(seed, replica)

    def gen_uniform(self) -> float:
        return self.gen.next53()

    def gen_poisson(self, lam: float) -> int:
        return afrng.poisson(lam, self.gen)

    def gen_normal(self, mean: float, sigma: float) -> float:
        return mean + sigma * afrng.std_normal(self.gen)

    def edge(self, rid: int, hop: int, dist: int, mean: float, sigma: float):
        d = afrng.RequestDraw(self.seed, self.replica, afrng.P_EDGE, rid, hop)
        return d.head53(), afrng.sample_rv(dist, mean, sigma, d)

    def endpoint(self, rid: int, hop: int, n: int) -> int:
        return afrng.pick_endpoint(self.seed, self.replica, rid, hop, n)


def make_rng(seed: int, replica: int, backend: str = "auto"):
    if backend in ("auto", "c"):
        try:
            import afrng_c
            return afrng_c.CRng(seed, replica)
        except (ImportError, OSError):
            if backend == "c":
                raise
    return PyRng(seed, replica)


# --------------------------------------------------------------------------- #
# actors                                                                      #
# --------------------------------------------------------------------------- #
class _Request:
    __slots__ = ("rid", "t0", "hops", "finish")

    def __init__(self, rid: int, t0: float) -> None:
        self.rid = rid
        self.t0 = t0
        self.hops = 0          # == len(RequestState.history), rqs_state.py:38-40
        self.finish = None


class _Edge:
    def __init__(self, sim: "_Sim", cfg: dict) -> None:
        self.sim = sim
        self.id = cfg["id"]
        lat = cfg["latency"]
        self.dist = afrng.DIST_CODE[lat["distribution"]]
        self.mean = lat["mean"]
        self.sigma = 0.0 if lat["variance"] is None else lat["variance"]
        self.dropout = cfg["dropout_rate"]
        self.target_box = None
        self.conn = 0
        self.sent = 0
        self.dropped = 0
        self.series = [] if "edge_concurrent_connection" in sim.enabled else None

    def transport(self, req: _Request):
        return self.sim.env.process(self.deliver(req))

    def deliver(self, req: _Request):
        sim = self.sim
        u, transit = sim.rng.edge(req.rid, req.hops, self.dist, self.mean, self.sigma)
        self.sent += 1
        if u < self.dropout:                       # edge.py:78-86
            req.finish = sim.env.now
            req.hops += 1
            self.dropped += 1
            return
        self.conn += 1
        spike = 0.0                                 # edge.py:94-100
        if sim.edges_spike and sim.edges_affected and self.id in sim.edges_affected:
            spike = sim.edges_spike.get(self.id, 0.0)
        effective = transit + spike
        yield sim.env.timeout(effective)
        req.hops += 1
        self.conn -= 1
        yield self.target_box.put(req)


class _Client:
    def __init__(self, sim: "_Sim", cid: str) -> None:
        self.sim = sim
        self.id = cid
        self.box = simpy.Store(sim.env)
        self.done_box = simpy.Store(sim.env)
        self.out_edge = None
        self.clocks: list = []

    def run(self):
        env = self.sim.env
        while True:
            req = yield self.box.get()
            req.hops += 1
            if req.hops > 3:                        # client.py:62
                req.finish = env.now
                self.clocks.append((req.t0, req.finish))
                yield self.done_box.put(req)
            else:
                self.out_edge.transport(req)


class _LoadBalancer:
    def __init__(self, sim: "_Sim", cfg: dict) -> None:
        self.sim = sim
        self.id = cfg["id"]
        self.algo = cfg["algorithms"]
        self.box = simpy.Store(sim.env)
        self.out_edges: OrderedDict = OrderedDict()

    def run(self):
        while True:
            req = yield self.box.get()
            req.hops += 1
            edges = self.out_edges
            if self.algo == "round_robin":          # lb_algorithms.py:22-36
                key, edge = next(iter(edges.items()))
                edges.move_to_end(key)
            else:                                   # least_connection, :10-20
                key = min(edges, key=lambda k: edges[k].conn)
                edge = edges[key]
            edge.transport(req)


class _Server:
    def __init__(self, sim: "_Sim", cfg: dict) -> None:
        self.sim = sim
        self.id = cfg["id"]
        self.endpoints = cfg["endpoints"]
        env = sim.env
        self.cpu = simpy.Container(env, capacity=cfg["cpu_cores"], init=cfg["cpu_cores"])
        self.ram = simpy.Container(env, capacity=cfg["ram_mb"], init=cfg["ram_mb"])
        self.box = simpy.Store(env)
        self.out_edge = None
        self.ready_q = 0
        self.io_q = 0
        self.ram_in_use = 0
        en = sim.enabled
        self.series = {k: [] for k in ("ready_queue_len", "event_loop_io_sleep", "ram_in_use")
                       if k in en}

    def dispatch(self):
        env = self.sim.env
        while True:
            req = yield self.box.get()
            env.process(self.handle(req))

    def handle(self, req: _Request):
        env = self.sim.env
        req.hops += 1
        ep = self.endpoints[self.sim.rng.endpoint(req.rid, req.hops, len(self.endpoints))]
        steps = ep["steps"]
        total_ram = sum(s["value"] for s in steps if s["kind"] in RAM_KINDS)
        if total_ram:                               # server.py:147-149
            yield self.ram.get(total_ram)
            self.ram_in_use += total_ram
        core_locked = False
        in_io = False
        waiting = False
        for s in steps:
            kind = s["kind"]
            if kind in CPU_KINDS:                   # server.py:199-231
                if in_io:
                    in_io = False
                    self.io_q -= 1
                if not core_locked:
                    cpu_req = self.cpu.get(1)
                    if not cpu_req.triggered:
                        waiting = True
                        self.ready_q += 1
                    yield cpu_req
                    if waiting:
                        waiting = False
                        self.ready_q -= 1
                    core_locked = True
                yield env.timeout(s["value"])
            elif kind in IO_KINDS:                  # server.py:235-255
                if core_locked:
                    yield self.cpu.put(1)
                    core_locked = False
                    if not in_io:
                        in_io = True
                        self.io_q += 1
                elif not in_io:
                    in_io = True
                    self.io_q += 1
                yield env.timeout(s["value"])
        if core_locked:                             # server.py:257-273
            yield self.cpu.put(1)
        if in_io:
            self.io_q -= 1
        if waiting:
            self.ready_q -= 1
        if total_ram:
            self.ram_in_use -= total_ram
            yield self.ram.put(total_ram)
        self.out_edge.transport(req)


class _Generator:
    def __init__(self, sim: "_Sim", cfg: dict, horizon: int) -> None:
        self.sim = sim
        self.id = cfg["id"]
        self.users = cfg["avg_active_users"]
        self.rate = float(cfg["avg_request_per_minute_per_user"]["mean"]) / 60
        self.window = cfg["user_sampling_window"]
        self.horizon = horizon
        self.out_edge = None
        self.count = 0

    def gaps(self):
        """The sampler's virtual clock (poisson_poisson.py:52-82)."""
        rng = self.sim.rng
        mean_u = float(self.users["mean"])
        gaussian = self.users["distribution"] == "normal"
        sigma_u = float(self.users["variance"]) if gaussian else 0.0
        now = 0.0
        window_end = 0.0
        lam = 0.0
        T = self.horizon
        while now < T:
            if now >= window_end:
                window_end = now + float(self.window)
                if gaussian:
                    users = max(0.0, rng.gen_normal(mean_u, sigma_u))
                else:
                    users = rng.gen_poisson(mean_u)
                lam = users * self.rate
            if lam <= 0.0:
                now = window_end
                continue
            u = max(rng.gen_uniform(), 1e-15)
            dt = -afrng.af_log(1.0 - u) / lam
            if now + dt > T:
                break
            if now + dt >= window_end:
                now = window_end
                continue
            now += dt
            yield dt

    def run(self):
        env = self.sim.env
        for gap in self.gaps():
            yield env.timeout(gap)                  # the SIMULATION clock: rqs_generator.py:103-104
            self.count += 1
            req = _Request(self.count, env.now)
            req.hops = 1
            self.out_edge.transport(req)


class _Sim:
    """Everything one replica owns."""

    def __init__(self, payload: dict, seed: int, replica: int, backend: str) -> None:
        self.p = payload
        self.env = simpy.Environment()
        self.rng = make_rng(seed, replica, backend)
        self.enabled = set(payload["sim_settings"]["enabled_sample_metrics"])
        self.edges_spike: dict = {}
        self.edges_affected: set = set()


def _injection_timelines(sim: _Sim, lb: "_LoadBalancer | None", edges: dict):
    """injection.py:112-164 -- returns the two generator functions (or None)."""
    events = sim.p["events"]
    if not events:
        return None
    edge_ids = {e["id"] for e in sim.p["edges"]}
    server_ids = {s["id"] for s in sim.p["servers"]}
    edges_events: dict = {}
    e_tl, s_tl = [], []
    for ev in events:
        st = (ev["t_start"], ev["event_id"], ev["target_id"], "start")
        en = (ev["t_end"], ev["event_id"], ev["target_id"], "end")
        if ev["target_id"] in edge_ids:
            edges_events.setdefault(ev["event_id"], {})[ev["target_id"]] = ev["spike_s"]
            e_tl += [st, en]
            sim.edges_affected.add(ev["target_id"])
        elif ev["target_id"] in server_ids:
            s_tl += [st, en]
    key = lambda e: (e[0], e[3] == "start", e[1], e[2])  # noqa: E731
    e_tl.sort(key=key)
    s_tl.sort(key=key)
    edge_by_server = {}
    if lb is not None:
        for eid, er in lb.out_edges.items():
            edge_by_server[er.target_id] = (eid, er)
    env = sim.env

    def spikes():
        last_t = float(env.now)
        for t, event_id, edge_id, mark in e_tl:
            dt = t - last_t
            if dt > 0.0:
                yield env.timeout(dt)
            last_t = t
            cur = sim.edges_spike.get(edge_id, 0.0)
            delta = edges_events[event_id][edge_id]
            sim.edges_spike[edge_id] = cur + delta if mark == "start" else cur - delta

    def outages():
        last_t = float(env.now)
        for t, _eid, server_id, mark in s_tl:
            dt = t - last_t
            if dt > 0.0:
                yield env.timeout(dt)
            last_t = t
            info = edge_by_server.get(server_id)
            if not info:
                continue
            edge_id, er = info
            if mark == "start":
                lb.out_edges.pop(edge_id, None)
            else:
                lb.out_edges[edge_id] = er
                lb.out_edges.move_to_end(edge_id)

    return spikes, outages


def _collector(sim: _Sim, edges: list, servers: list, period: float):
    env = sim.env
    while True:                                      # collector.py:50-66
        yield env.timeout(period)
        for e in edges:
            if e.series is not None:
                e.series.append(e.conn)
        for s in servers:
            if len(s.series) == 3:
                s.series["ram_in_use"].append(s.ram_in_use)
                s.series["event_loop_io_sleep"].append(s.io_q)
                s.series["ready_queue_len"].append(s.ready_q)


def simulate(payload: dict, *, seed: int, replica: int, backend: str = "auto",
             normalised: bool = False) -> dict:
    """One replica, start to horizon.  Returns raw per-replica results."""
    p = payload if normalised else normalise_payload(payload)
    sim = _Sim(p, seed, replica, backend)
    env = sim.env
    T = p["sim_settings"]["total_simulation_time"]

    gen = _Generator(sim, p["rqs_input"], T)
    client = _Client(sim, p["client"]["id"])
    servers = [_Server(sim, s) for s in p["servers"]]
    lb = _LoadBalancer(sim, p["load_balancer"]) if p["load_balancer"] else None

    nodes = {s.id: s for s in servers}
    nodes[client.id] = client
    nodes[gen.id] = gen
    if lb is not None:
        nodes[lb.id] = lb
    edges = []
    for cfg in p["edges"]:                           # simulation_runner.py:205-260
        e = _Edge(sim, cfg)
        e.target_id = cfg["target"]
        e.target_box = nodes[cfg["target"]].box
        src = nodes[cfg["source"]]
        if src is lb:
            lb.out_edges[e.id] = e
        else:
            src.out_edge = e
        edges.append(e)

    tl = _injection_timelines(sim, lb, {e.id: e for e in edges})
    if tl is not None:                               # _start_events, :339-342
        env.process(tl[0]())
        env.process(tl[1]())
    env.process(gen.run())                           # _start_all_processes, :301-326
    env.process(client.run())
    for s in servers:
        env.process(s.dispatch())
    if lb is not None:
        env.process(lb.run())
    env.process(_collector(sim, edges, servers, p["sim_settings"]["sample_period_s"]))
    env.run(until=T)

    return {
        "generated": gen.count,
        "completed": len(client.clocks),
        "clocks": client.clocks,
        "edge_sent": {e.id: e.sent for e in edges},
        "edge_dropped": {e.id: e.dropped for e in edges},
        "server_series": {s.id: s.series for s in servers},
        "edge_series": {e.id: ({"edge_concurrent_connection": e.series}
                               if e.series is not None else {}) for e in edges},
        "heap_events": next(env._eid),
    }
