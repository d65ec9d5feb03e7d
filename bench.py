#!/usr/bin/env python
"""bench.py -- simulated request-completions/s of the replica engine (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c3|c2|c4|c5]
                    [--dump-outputs DIR]

Default workload (BASELINE.json configs[2], the one the north-star target is quoted on):
client -> LB -> {srv-1, srv-2} (README dashboard example), 100 000 replicas per GPU,
every edge's latency swept over RTT 1-50 ms (mean) x jitter 10-50 % (normal, sigma =
jitter * mean), fixed seed.  A *step* is one full pass of the hot path over that
batch: every replica simulated from t=0 to the horizon.  `--config` selects the other
BASELINE shapes (configs[1], [3], [4]); see WORKLOADS below.

* value  -- whole-job completions/s, sweep rows already resident in HBM, device-timed
            (CUDA events on the engine's stream; max over ranks).
* e2e    -- the same through SweepRunner's public calls: pinned-host sweep rows H2D, simulation,
            per-replica statistics / edge counters / sampled aggregates D2H.
* N > 1  -- every rank runs one Monte-Carlo repetition of the same parameter grid (its own replica
            ids, hence its own random numbers): equal work per rank by construction, no traffic during
            simulation, one NCCL all-gather of each rank's summary block (reduced latency histogram +
            totals) per step.

`--dump-outputs DIR` writes, after the timed steps, what the last one handed its caller as
DIR/<name>.npy (float64; see dump_outputs), so two builds can be compared output for output: with the
same arguments the inputs are the same in every run.

`--impl reference` times the reference's CPU path (oracle/des_port.py: the actor
generators on a simpy-4.1.1-compatible heap, restated because simpy is not installable
here; see DESIGN.md) on all the host cores this process may use, on a bounded sample of the
same workload.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from dataclasses import dataclass
from pathlib import Path
from typing import Callable

import numpy as np
import yaml

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SEED = 0xA5F10
METRIC = "simulated request-completions/sec"
UNIT = "completions/s"
SM_COUNT, SMSP_PER_SM = 148, 4


# --------------------------------------------------------------------------- workloads
def _scenario(name: str, horizon: int | None) -> dict:
    payload = yaml.safe_load((ROOT / "tests" / "scenarios" / name).read_text())
    if horizon is not None:
        payload["sim_settings"]["total_simulation_time"] = horizon
    return payload


def workload(n_replicas: int, horizon: int):
    """configs[2]: C3 with normal-jitter edges (kept under its round-1 name: tests import it)."""
    payload = _scenario("c3_lb_two_servers.yml", horizon)
    for e in payload["topology_graph"]["edges"]:          # "+ jitter": normal latency, sigma swept
        e["latency"] = {"mean": e["latency"]["mean"], "distribution": "normal",
                        "variance": 0.3 * e["latency"]["mean"]}
    return payload


def sweep_rows(replica_ids: np.ndarray, per_gpu: int):
    """configs[2]'s RTT x jitter grid, a pure function of the GLOBAL replica id: the grid has `per_gpu`
    points and repeats every `per_gpu` ids, so each rank's contiguous id range covers all of it."""
    i = np.asarray(replica_ids) % per_gpu
    n_j = 100
    n_r = max(per_gpu // n_j, 1)
    rtt = 0.001 + (0.050 - 0.001) * ((i // n_j) % n_r) / max(n_r - 1, 1)
    jit = 0.1 + 0.4 * (i % n_j) / (n_j - 1)
    return rtt, jit * rtt


@dataclass
class Workload:
    key: str
    title: str                       # BASELINE.json's wording
    payload: dict
    replicas: int                    # per GPU
    horizon: int
    horizon_note: str
    events_per_completion: float     # timed events per completion (SURVEY.md 8d): 1 + hops + CPU bursts + IO runs
    columns: Callable                # (flat, global replica ids, replicas per GPU) -> {selector: values}
    total: int = 0                   # replicas of the BASELINE configuration (all GPUs)

    @property
    def bytes_per_completion(self) -> float:     # SURVEY.md 8d: 96 B per timed event + 8 B histogram RMW
        return 96.0 * self.events_per_completion + 8.0


def _c3_cols(flat, ids, per_gpu):
    rtt, sig = sweep_rows(ids, per_gpu)
    cols = {}
    for e in flat.edge_ids:
        cols[("edge_mean", e)] = rtt
        cols[("edge_sigma", e)] = sig
    return cols


def _c2_cols(flat, ids, per_gpu):
    # avg_active_users 10..1000; consecutive ids are far apart in load (stride 61 is coprime with every
    # BASELINE size), so the saturated points are spread over the launch instead of bunched at its end
    i = (np.asarray(ids) % per_gpu) * 61 % per_gpu
    return {("users_mean",): 10.0 + 990.0 * i / max(per_gpu - 1, 1)}


def _c4_cols(flat, ids, per_gpu):
    # Monte-Carlo over the injected failure: spike amplitude 15-50 ms x client<->LB RTT 1-10 ms
    i = np.asarray(ids) % per_gpu
    n_a = 250
    amp = 0.015 + 0.035 * (i % n_a) / (n_a - 1)
    rtt = 0.001 + 0.009 * ((i // n_a) % max(per_gpu // n_a, 1)) / max(per_gpu // n_a - 1, 1)
    return {("spike_delta", "ev-spike"): amp, ("edge_mean", "client-lb"): rtt}


C5_CORES = (1, 2, 3, 4)
C5_RAM = (512, 1024, 1536, 2048, 3072)


def _c5_cols(flat, ids, per_gpu):
    # users x cpu_cores x ram_mb grid (100 x 4 x 5 = 2000 points, the rest of the ids are Monte-Carlo repeats);
    # cores and RAM are those of the ten back-end servers every request ends on
    i = np.asarray(ids) % per_gpu
    users = 600.0 + 1800.0 * (i % 100) / 99.0
    cores = np.asarray(C5_CORES, dtype=np.float64)[(i // 100) % len(C5_CORES)]
    ram = np.asarray(C5_RAM, dtype=np.float64)[(i // (100 * len(C5_CORES))) % len(C5_RAM)]
    cols = {("users_mean",): users}
    for s in flat.server_ids:
        if s.startswith("be-"):
            cols[("server_cpu_cores", s)] = cores
            cols[("server_ram_mb", s)] = ram
    return cols


def make_workload(key: str, horizon: int | None = None, replicas: int | None = None) -> Workload:
    if key == "c3":
        h = horizon or 60
        return Workload("c3", "configs[2]: client->LB->{srv-1,srv-2} (README dashboard example), 100 000 replicas "
                        "sweeping edge RTT 1-50 ms x jitter 10-50 % (normal), 1xB200", workload(0, h), replicas or 100_000, h,
                        "reference YAML horizon is 600 s; the metric is a rate, the horizon only scales step length",
                        7.0, _c3_cols, 100_000)
    if key == "c2":
        h = horizon or 60
        return Workload("c2", "configs[1]: README my_service.yml single-server topology, 10 000 replicas sweeping "
                        "avg_active_users 10-1000, 1xB200", _scenario("c1_my_service.yml", h), replicas or 10_000, h,
                        "BASELINE horizon (60 s)", 6.0, _c2_cols, 10_000)
    if key == "c4":
        h = horizon or 300
        return Workload("c4", "configs[3]: 8-server fan-out behind LB with event injection (60 s network spike + srv-3 "
                        "outage), 1 000 000 replicas over 8xB200", _scenario("c4_lb8_events.yml", h), replicas or 125_000, h,
                        "scenario horizon (300 s: spike 100-160 s, outage 180-240 s)", 7.0, _c4_cols, 1_000_000)
    if key == "c5":
        h = horizon or 30
        return Workload("c5", "configs[4]: 32-node multi-hop topology, mixed endpoint pipelines, 4 000 000-replica grid "
                        "over users x cpu_cores x ram_mb, 8xB200", _scenario("c5_multihop32.yml", h), replicas or 500_000, h,
                        "scenario YAML horizon is 120 s; the metric is a rate, the horizon only scales step length",
                        12.0, _c5_cols, 4_000_000)
    raise SystemExit(f"bench.py: unknown --config {key!r}")


# --------------------------------------------------------------------------- CPU path
def effective_cores() -> tuple[int, dict]:
    """Host cores this process can really use: the affinity mask capped by the cgroup CPU quota
    (os.cpu_count() reports the machine, not the lease -- VERDICT r1)."""
    info: dict = {"os_cpu_count": os.cpu_count()}
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = os.cpu_count() or 1
    info["affinity"] = aff
    quota = None
    for p in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = Path(p).read_text().split()
            if p.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            break
        except (OSError, ValueError, IndexError):
            continue
    info["cgroup_quota_cpus"] = quota
    n = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    return n, info


def _cpu_one(args):
    payload, seed, replica = args
    sys.path[:0] = [str(ROOT / "oracle"), str(ROOT / "oracle" / "simpy_shim")]
    import des_port
    t0 = time.perf_counter()
    r = des_port.simulate(payload, seed=seed, replica=replica)
    return r["completed"], r["heap_events"], time.perf_counter() - t0


_POOL = None


def _noop(_):
    return 0


def cpu_pool(cores: int):
    """A warm process pool (fork + imports are NOT part of what gets timed)."""
    global _POOL
    if _POOL is None and cores > 1:
        import multiprocessing as mp
        _POOL = mp.get_context("fork").Pool(cores)
        _POOL.map(_noop, range(cores * 4))
    return _POOL


def cpu_pool_close() -> None:
    global _POOL
    if _POOL is not None:
        _POOL.close()
        _POOL.join()
        _POOL = None


def cpu_jobs(w: Workload, replica_ids) -> list:
    """(payload of the sweep row, seed, replica id) for the reference's CPU path."""
    from asyncflow_b200 import SweepSpec, flatten
    flat = flatten(w.payload)
    ids = np.asarray(replica_ids, dtype=np.int64)
    spec = SweepSpec(flat, len(ids), w.columns(flat, ids, w.replicas))
    return [(spec.payload_for(w.payload, i), SEED, int(r)) for i, r in enumerate(ids)]


def cpu_path(w: Workload, replica_ids, cores: int):
    """Simulate `replica_ids` with the reference's CPU path on `cores` processes."""
    jobs = cpu_jobs(w, replica_ids)
    pool = cpu_pool(cores)
    t0 = time.perf_counter()
    out = pool.map(_cpu_one, jobs, chunksize=1) if pool is not None else [_cpu_one(j) for j in jobs]
    dt = time.perf_counter() - t0
    busy = sum(t for _, _, t in out)
    return sum(c for c, _, _ in out), sum(h for _, h, _ in out), dt, busy


def cpu_one_process(w: Workload, replica_ids):
    """The reference's real execution model: one process, one core."""
    out = [_cpu_one(j) for j in cpu_jobs(w, replica_ids)]
    dt = sum(t for _, _, t in out)
    return sum(c for c, _, _ in out) / dt, sum(h for _, h, _ in out) / dt, dt


def cpu_sample_size(cores: int, one_process_value: float, completions_per_replica: float, seconds: float) -> int:
    """Replicas that keep `cores` processes busy for about `seconds` (the contract's bounded CPU sample: 10-30 s)."""
    k = int(seconds * cores * one_process_value / max(completions_per_replica, 1.0))
    return max(3 * cores, min(k, 8192))


def spaced(total: int, k: int) -> np.ndarray:
    return np.unique(np.linspace(0, total - 1, k).astype(np.int64))


def cpu_block(w: Workload, cores: int, info: dict, n, h, dt, busy, k, one) -> dict:
    return {"value": n / dt, "unit": UNIT, "cores": cores,
            # measured, not declared: how many one-process equivalents the pool delivered (a lease's vCPUs can be
            # throttled below what the affinity mask and the cgroup quota admit)
            "cores_effective": round((n / dt) / one[0], 2), "cores_detail": info,
            "kind": "port",
            "one_process_value": one[0], "one_process_heap_events_per_s": one[1],
            "per_core_value": n / busy,       # completions per busy process-second inside the pool
            "sample": f"{k} replicas spaced over the sweep, horizon {w.horizon}s, {cores} processes "
                      f"(multiprocessing, one per usable core), oracle/des_port.py on oracle/simpy_shim ({dt:.1f} s); "
                      f"one_process_value: 1 process, {one[2]:.1f} s",
            "heap_events_per_s": h / dt}


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int) -> None:
        self.rows: list[list[str]] = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self) -> None:
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_median": float(np.median(pw)) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def latency_delta_vs_reference(device: int):
    """BASELINE.json's second half: p50/p95/p99 latency delta vs the SimPy reference.  The reference
    side is tests/golden/reference_numpy_stats.json (the unmodified reference on its own numpy RNG,
    96 replicas of C3 at the reference's parameters, 60 s horizon: oracle/make_reference_stats.py);
    the engine side is a 4096-replica run of the same scenario, outside the timed region."""
    from asyncflow_b200 import SweepRunner, flatten
    fx = ROOT / "tests" / "golden" / "reference_numpy_stats.json"
    if not fx.exists():
        return None
    ref = json.loads(fx.read_text())["c3_lb_two_servers.yml"]
    payload = _scenario("c3_lb_two_servers.yml", ref["horizon"])
    sw = SweepRunner(flatten(payload), 4096, seed=SEED + 1, device=device)
    st = sw.run().stats
    sw.close()
    mine = {"mean": float((st["lat_sum"] / st["completed"]).mean()), "median": float(st["p50"].mean()),
            "p95": float(st["p95"].mean()), "p99": float(st["p99"].mean())}
    return {"scenario": "c3_lb_two_servers.yml (reference parameters, horizon %d s)" % ref["horizon"],
            "reference": "unmodified AsyncFlow actors, numpy PCG64, %d replicas" % ref["replicas"],
            "engine_replicas": 4096,
            "delta_pct": {k: 100.0 * (mine[k] - ref["mean"][k]) / ref["mean"][k] for k in mine},
            "reference_s": {k: ref["mean"][k] for k in mine}, "engine_s": mine}


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except (KeyError, ValueError):
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def profiled(config_key: str) -> dict:
    """ncu-derived constants of the dominant kernel for this configuration (profiles/kernel_metrics.json, written
    from the committed ncu CSVs by tools/ncu_issue_summary.py): DRAM bytes per launch, warp-instructions per timed
    event, issue-active %.  Empty when the configuration has not been profiled."""
    p = ROOT / "profiles" / "kernel_metrics.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(config_key) or {}
        except ValueError:
            return {}
    return {}


# --------------------------------------------------------------------------- outputs
DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, res) -> None:
    """The last end-to-end step's results (SweepRunner.collect's per-replica arrays and the all-gathered
    summary) as float64 DIR/<name>.npy, at most DUMP_BYTES in all: past that, every per-replica array keeps
    the same fixed, seeded sample of rows, and replica_rows.npy names them (this rank's rows)."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    g = res.global_summary
    whole = {"summary_histogram": g.histogram,
             "summary_counts": np.array([g.completed, g.generated, g.events, g.replicas, g.overflowed]),
             "summary_latency": np.array([g.lat_sum, g.lat_min, g.lat_max])}
    per_replica = {f"stats_{f}": res.stats[f] for f in res.stats.dtype.names}
    per_replica.update(edge_sent=res.edge_sent, edge_dropped=res.edge_dropped,
                       sampled_sum=res.samp_sum, sampled_max=res.samp_max)
    if res.throughput is not None:
        per_replica["throughput"] = res.throughput
    n = len(res)
    row_bytes = 8 + sum(8 * int(np.prod(a.shape[1:])) for a in per_replica.values())        # + replica_rows
    budget = DUMP_BYTES - sum(8 * a.size for a in whole.values()) - 256 * (len(whole) + len(per_replica) + 1)
    rows = np.arange(n)
    if n * row_bytes > budget:
        rows = np.sort(np.random.default_rng(SEED).choice(n, budget // row_bytes, replace=False))
    out = {**whole, **{k: a[rows] for k, a in per_replica.items()}, "replica_rows": rows}
    for name, a in out.items():
        np.save(d / f"{name}.npy", np.asarray(a, dtype=np.float64))


# --------------------------------------------------------------------------- arms
def run_reference(a) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores, info = effective_cores()
    w = make_workload(a.config, a.horizon, a.replicas)
    total = w.replicas * a.gpus
    one = cpu_one_process(w, spaced(total, 2))
    cpr = one[0] * one[2] / 2.0                           # completions per replica of this workload
    per_step = cpu_sample_size(cores, one[0], cpr, seconds=10.0)      # ~10 s of all-core work per step
    ids = spaced(total, per_step * (a.steps + a.warmup))
    chunks = [ids[i::(a.steps + a.warmup)] for i in range(a.steps + a.warmup)]
    for c in chunks[: a.warmup]:
        cpu_path(w, c, cores)
    comp = ev = 0
    dt = busy = 0.0
    for c in chunks[a.warmup:]:
        n, h, t, b = cpu_path(w, c, cores)
        comp += n; ev += h; dt += t; busy += b
    value = comp / dt
    block = cpu_block(w, cores, info, comp, ev, dt, busy, len(chunks[0]), one)
    block["sample"] = f"{len(chunks[0])} replicas/step spaced over the sweep; " + block["sample"]
    emit({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(w, a.gpus),
        "cpu_baseline": block,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def config_dict(w: Workload, gpus: int) -> dict:
    return {"workload": w.title, "config_key": w.key,
            "replicas_per_gpu": w.replicas, "replicas_total": w.replicas * gpus, "horizon_s": w.horizon,
            "horizon_note": w.horizon_note,
            "seed": hex(SEED), "parallelism": f"replica-range x{gpus} (each rank: one Monte-Carlo repetition of the grid)",
            "l2": "per-replica latency histograms (16 KB each) exceed the 126 MB L2 from 8 000 replicas up; "
                  "a 256 MB buffer is also overwritten between timed steps"}


def run_ours(a) -> None:
    import torch
    import torch.distributed as dist

    from asyncflow_b200 import SweepRunner, flatten
    from asyncflow_b200._capi import STATS_DTYPE as res_dtype
    from asyncflow_b200.distributed import all_gather_summary, summary_block

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        sys.exit("bench.py: no CUDA device (asyncflow_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    w = make_workload(a.config, a.horizon, a.replicas)
    n = w.replicas
    total = n * world
    begin = rank * n
    flat = flatten(w.payload)
    ids = np.arange(begin, begin + n, dtype=np.int64)
    # one SweepRunner per rank holding this rank's rows; replica ids stay global
    sw = SweepRunner(flat, n, w.columns(flat, ids, n), seed=SEED, device=local, histogram=True, throughput=False)
    eng = sw.engine()
    if a.engine:
        eng.set_mode(a.engine)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def launch():
        eng.configure(request_capacity=sw.request_capacity, event_capacity=sw.event_capacity,
                      histogram=True, throughput=False, warps_per_block=a.wpb)
        eng.run(SEED, begin, begin + n)

    empty_stats = np.zeros(0, dtype=res_dtype)

    def summarise(res_stats=None):
        """This rank's summary block (device-reduced histogram + totals), all-gathered over
        NCCL when world > 1 -- the sweep's only collective."""
        ints, flts = summary_block(empty_stats if res_stats is None else res_stats, eng.reduced_histogram())
        return all_gather_summary(ints, flts, device="cuda" if world > 1 else None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def resident_step():
        launch()
        eng.sync()
        ms_total, ms_sim = eng.last_run_ms()
        summarise()
        return ms_total, ms_sim

    def e2e_step():
        eng.upload_sweep(sw.spec, begin, row_first=0, row_count=n)
        launch()
        res = sw.collect(begin)
        res.global_summary = summarise(res.stats)
        return res

    # sweep rows resident for the `value` steps
    eng.upload_sweep(sw.spec, begin, row_first=0, row_count=n)
    for _ in range(a.warmup):
        resident_step()
    sampler = ClockSampler(local) if rank == 0 else None

    # ---- value: K steps, inputs resident, device-timed ---------------------------
    launches0 = eng.launch_count
    dev_ms = sim_ms = 0.0
    barrier()
    w0 = time.perf_counter()
    for _ in range(a.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        mt, ms = resident_step()
        dev_ms += mt; sim_ms += ms
    barrier()
    wall_resident = time.perf_counter() - w0
    launches = eng.launch_count - launches0
    passes = eng.last_run_passes()

    # ---- e2e: K steps through the public API, host buffers ------------------------
    if a.e2e_warm:
        res = e2e_step()                                # untimed: allocates the pinned result buffers
    barrier()
    w0 = time.perf_counter()
    for _ in range(a.steps):
        res = e2e_step()
    barrier()
    wall_e2e = time.perf_counter() - w0
    clocks = sampler.stop() if sampler else None

    st = res.stats
    mine = np.array([float(st["completed"].sum()), float(st["n_events"].sum()), dev_ms, sim_ms, wall_e2e,
                     wall_resident, float(res.overflowed.sum()), float(passes["warp_replicas"] if passes["lane_pass"] else 0)])
    per_rank_ms = [dev_ms / a.steps]
    if world > 1:
        t = torch.tensor(mine, device="cuda", dtype=torch.float64)
        tot = t.clone(); dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        gathered = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(gathered, t)
        per_rank_ms = [g[2].item() / a.steps for g in gathered]
        completed, events, overflow, rerun = tot[0].item(), tot[1].item(), tot[6].item(), tot[7].item()
        dev_ms, sim_ms, wall_e2e, wall_resident = mx[2].item(), mx[3].item(), mx[4].item(), mx[5].item()
    else:
        completed, events, overflow, rerun = mine[0], mine[1], mine[6], mine[7]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    if a.dump_outputs:
        dump_outputs(a.dump_outputs, res)

    value = completed * a.steps / (dev_ms / 1e3)
    e2e_value = completed * a.steps / wall_e2e
    peak, peak_src = hbm_peak()
    per_launch_completions = float(st["completed"].sum())
    per_launch_events = float(st["n_events"].sum())
    sim_s = sim_ms / a.steps / 1e3
    achieved = per_launch_completions * w.bytes_per_completion / sim_s / 1e9
    kernel = "af_lane_kernel" if passes["lane_pass"] else "af_sim_kernel"
    prof = profiled(f"{w.key}:{kernel}")
    sm_hz = (clocks or {}).get("sm_mhz") or 1965.0
    slots = SM_COUNT * SMSP_PER_SM * sm_hz * 1e6                   # warp-instruction issue slots per second
    issue = {"events_per_s_one_gpu": per_launch_events / sim_s,
             "peak_slots_per_s": slots, "peak_source": "148 SMs x 4 SMSPs x the SM clock sampled during the run",
             "warp_inst_per_event": prof.get("warp_inst_per_event"), "issue_active_pct": prof.get("issue_active_pct"),
             "source": prof.get("source"), "profiled_build": prof.get("build")}
    if prof.get("warp_inst_per_event"):
        issue["achieved_slots_per_s"] = per_launch_events / sim_s * prof["warp_inst_per_event"]
        issue["frac"] = issue["achieved_slots_per_s"] / slots
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": dev_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config_dict(w, world),
        "events_per_s": events * a.steps / (dev_ms / 1e3),
        "per_rank_ms": per_rank_ms,
        "wall_ms_per_step_resident": wall_resident / a.steps * 1e3,
        "replicas_overflowed": overflow,
        "passes": {"kernel": kernel, "lane_warps_per_sm": passes["lane_warps_per_sm"], "lane_bytes_per_replica": passes["lane_bytes"],
                   "lane_events_in_smem": passes["lane_events_smem"], "lane_requests_in_smem": passes["lane_requests_smem"],
                   "replicas_rerun_per_warp": rerun},
        "latency_all_replicas": {"mean_s": res.global_summary.mean_latency, "p50_s": res.global_summary.percentile(50),
                                 "p95_s": res.global_summary.percentile(95), "p99_s": res.global_summary.percentile(99),
                                 "source": "merged (all-gathered) histogram"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(sw.spec.values.nbytes),
                "d2h_bytes_per_step": int(sw.d2h_bytes + (4096 * 8)), "ms_per_step": wall_e2e / a.steps * 1e3},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "peak_source": peak_src,
                     "algorithmic_bytes_per_completion": w.bytes_per_completion,
                     "traffic": prof.get("dram_bytes_per_launch"),
                     "issue": issue,
                     "note": "replica state lives in shared memory: the HBM fraction is the contract's figure, the "
                             "issue block is the limiter (DESIGN.md 'Roofline')"},
    }
    if w.key == "c3":
        out["latency_delta_vs_reference"] = latency_delta_vs_reference(local)
    if world == 1 and not a.no_cpu_baseline:
        cores, info = effective_cores()
        one = cpu_one_process(w, spaced(total, 2))         # also pages in the interpreter state; calibrates the sample
        k = cpu_sample_size(cores, one[0], per_launch_completions / n, seconds=15.0)
        cpu_path(w, spaced(total, cores), cores)         # untimed: warm the pool
        nn, h, dt, busy = cpu_path(w, spaced(total, k), cores)
        out["cpu_baseline"] = cpu_block(w, cores, info, nn, h, dt, busy, k, one)
    emit(out)
    if world > 1:
        dist.destroy_process_group()


_RESULT_FD = None


def claim_stdout() -> None:
    """Keep stdout for the ONE JSON line: native libraries write there too (NCCL prints its version
    banner with printf at communicator creation), so fd 1 is pointed at stderr for the run and the
    result goes to the saved descriptor."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(obj: dict) -> None:
    sys.stdout.flush()
    os.write(_RESULT_FD if _RESULT_FD is not None else 1, (json.dumps(obj) + "\n").encode())


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=["c2", "c3", "c4", "c5"],
                    help="BASELINE.json configs[1..4] (default c3 = configs[2], the one the metric is quoted on)")
    ap.add_argument("--replicas", type=int, default=None, help="replicas per GPU (default: the configuration's)")
    ap.add_argument("--horizon", type=int, default=None, help="simulated seconds (default: the configuration's)")
    ap.add_argument("--engine", default="", choices=["", "auto", "two_pass", "warp", "lane"], help="pin the pass structure (experiments)")
    ap.add_argument("--wpb", type=int, default=0, help="warps per SM of the thread-per-replica pass (experiments)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-warm", type=int, default=1, help="0: no untimed end-to-end step before the timed ones (the first timed "
                    "one then also allocates the pinned result buffers; for the multi-minute BASELINE-size runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's results to DIR/<name>.npy (float64, at most 64 MB)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the results of the engine (--impl ours)")
    a.warmup = max(a.warmup, 0)
    claim_stdout()
    try:
        if a.impl == "reference":
            run_reference(a)
        else:
            run_ours(a)
    finally:
        cpu_pool_close()


if __name__ == "__main__":
    main()
