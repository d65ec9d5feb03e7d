"""Run the UNMODIFIED reference actors on the oracle kernel with AF-RNG injected.

ORACLE / TEST INFRASTRUCTURE ONLY.  Needs a checkout of the reference, its ``src/``
directory named by ``ASYNCFLOW_REFERENCE_SRC``; its job is to generate the golden
data committed under ``tests/golden/`` (``oracle/make_golden.py``,
``oracle/make_reference_runs.py``), which pins ``oracle/des_port.py`` and the
engine to the real reference code.

What is "unmodified": every class under ``/root/reference/src/asyncflow`` is
imported and executed as shipped -- ``SimulationRunner.run()``
(``runtime/simulation_runner.py:349-376``) builds, wires and starts the actors
exactly as upstream.  Three seams are used, none edits reference source:

1. ``simpy`` resolves to ``oracle/simpy_shim/simpy`` (upstream 4.1.1 is absent).
2. ``runner.rng`` is replaced before ``run()`` by :class:`PhiloxDuckRng`, the
   seam the reference's own tests use
   (``tests/integration/single_server/test_int_single_server.py:36``); the
   actors accept any duck type (``tests/unit/runtime/actors/test_edge.py:31``).
   The duck looks at its *caller's frame* to learn which request/hop is asking,
   because AF-RNG keys draws by (request id, hop) -- see ``oracle/afrng.py``.
3. ``math.log`` inside the two sampler modules is pointed at ``af_log`` so the
   inter-arrival gaps are bit-identical to the device's (libm's log differs from
   ``af_log`` by <=1 ulp; ``tests/test_afrng.py`` quantifies it).
"""

from __future__ import annotations

import os
import sys
import types
from pathlib import Path

_HERE = Path(__file__).resolve().parent
REFERENCE_SRC = Path(os.environ.get("ASYNCFLOW_REFERENCE_SRC", "")).resolve()

if str(_HERE) not in sys.path:
    sys.path.insert(0, str(_HERE))

import afrng  # noqa: E402


def reference_available() -> bool:
    return bool(os.environ.get("ASYNCFLOW_REFERENCE_SRC")) and (REFERENCE_SRC / "asyncflow" / "__init__.py").is_file()


def _ensure_paths() -> None:
    shim = str(_HERE / "simpy_shim")
    if shim not in sys.path:
        sys.path.insert(0, shim)
    if str(REFERENCE_SRC) not in sys.path:
        sys.path.insert(0, str(REFERENCE_SRC))


class PhiloxDuckRng:
    """Duck-typed ``numpy.random.Generator`` backed by AF-RNG.

    Implements exactly the methods the reference calls
    (``samplers/common_helpers.py:13,20,31,40,47``, ``runtime/actors/edge.py:78``,
    ``runtime/actors/server.py:101``).
    """

    _EDGE_FN = "_deliver"
    _SERVER_FN = "_handle_request"
    _GEN_FNS = ("poisson_poisson_sampling", "gaussian_poisson_sampling")

    def __init__(self, seed: int, replica: int) -> None:
        self.seed = seed
        self.replica = replica
        self.gen = afrng.GenStream(seed, replica)
        self._cur_key = None
        self._cur_draw = None
        self.sent: dict[str, int] = {}
        self.dropped: dict[str, int] = {}

    # context ---------------------------------------------------------------
    def _source(self):
        f = sys._getframe(2)
        while f is not None:
            name = f.f_code.co_name
            if name in self._GEN_FNS:
                return self.gen, None
            if name == self._EDGE_FN or name == self._SERVER_FN:
                state = f.f_locals["state"]
                purpose = afrng.P_EDGE if name == self._EDGE_FN else afrng.P_SERVER
                key = (purpose, state.id, len(state.history))
                if key != self._cur_key:
                    self._cur_key = key
                    self._cur_draw = afrng.RequestDraw(
                        self.seed, self.replica, purpose, state.id, len(state.history))
                return self._cur_draw, f
            f = f.f_back
        msg = "PhiloxDuckRng called outside a known reference actor"
        raise RuntimeError(msg)

    # numpy.Generator surface ----------------------------------------------
    def random(self) -> float:
        src, _ = self._source()
        return src.next53()

    def uniform(self) -> float:
        src, frame = self._source()
        u = src.head53()
        cfg = frame.f_locals["self"].edge_config
        self.sent[cfg.id] = self.sent.get(cfg.id, 0) + 1
        if u < cfg.dropout_rate:
            self.dropped[cfg.id] = self.dropped.get(cfg.id, 0) + 1
        return u

    def exponential(self, scale: float) -> float:
        src, _ = self._source()
        return scale * afrng.std_exponential(src)

    def normal(self, loc: float, scale: float) -> float:
        src, _ = self._source()
        return loc + scale * afrng.std_normal(src)

    def lognormal(self, mean: float, sigma: float) -> float:
        src, _ = self._source()
        return afrng.af_exp(mean + sigma * afrng.std_normal(src))

    def poisson(self, lam: float) -> int:
        src, _ = self._source()
        return afrng.poisson(float(lam), src)

    def integers(self, low: int = 0, high: int | None = None) -> int:
        src, _ = self._source()
        assert low == 0 and high is not None
        return (src.block(0)[0] * high) >> 32


def run_reference(payload_dict: dict, *, seed: int, replica: int) -> dict:
    """One replica through the reference's ``SimulationRunner``; raw results."""
    _ensure_paths()
    import simpy  # the shim
    import asyncflow.samplers.gaussian_poisson as gp
    import asyncflow.samplers.poisson_poisson as pp
    from asyncflow.runtime.simulation_runner import SimulationRunner
    from asyncflow.schemas.payload import SimulationPayload

    payload = SimulationPayload.model_validate(payload_dict)
    env = simpy.Environment()
    runner = SimulationRunner(env=env, simulation_input=payload)
    rng = PhiloxDuckRng(seed, replica)
    runner.rng = rng

    det_math = types.SimpleNamespace(log=afrng.af_log)
    saved = (pp.math, gp.math)
    pp.math = gp.math = det_math
    try:
        analyzer = runner.run()
    finally:
        pp.math, gp.math = saved

    client = next(iter(runner._client_runtime.values()))
    gen = next(iter(runner._rqs_runtime.values()))
    clocks = [(c.start, c.finish) for c in client.rqs_clock]
    out = {
        "generated": gen.id_counter,
        "completed": len(clocks),
        "clocks": clocks,
        "edge_sent": {e.id: rng.sent.get(e.id, 0) for e in payload.topology_graph.edges},
        "edge_dropped": {e.id: rng.dropped.get(e.id, 0) for e in payload.topology_graph.edges},
        "server_series": {
            sid: {k.value: list(v) for k, v in srv.enabled_metrics.items()}
            for sid, srv in runner._servers_runtime.items()
        },
        "edge_series": {
            er.edge_config.id: {k.value: list(v) for k, v in er.enabled_metrics.items()}
            for er in runner._edges_runtime.values()
        },
        "analyzer": analyzer,
        "payload_dump": payload.model_dump(mode="json"),
    }
    return out
