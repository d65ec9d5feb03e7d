"""Shared fixtures.  `gpu` marks tests that need a real B200 (driver runs them with -m gpu)."""

from __future__ import annotations

import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "oracle", ROOT / "oracle" / "simpy_shim", ROOT / "tests"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

SEED = 0xA5F10


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


def pytest_collection_modifyitems(config, items):
    """A plain `pytest` on a box without a device skips the gpu tier instead of erroring in every fixture
    (the product has no CPU fallback: Engine(0) raises EngineUnavailable there)."""
    gpu_items = [it for it in items if it.get_closest_marker("gpu")]
    if not gpu_items:
        return
    have = any(Path(p).exists() for p in ("/dev/nvidiactl", "/dev/nvidia0", "/dev/dxg"))
    if not have:
        skip = pytest.mark.skip(reason="no CUDA device: the gpu tier needs a B200 (asyncflow_b200 has no CPU fallback)")
        for it in gpu_items:
            it.add_marker(skip)


@pytest.fixture(scope="session", autouse=True)
def _native_code_is_built():
    """A fresh checkout has no .so files (they are git-ignored): build them once per session."""
    lib = ROOT / "asyncflow_b200" / "_lib" / "libasyncflow_b200.so"
    if not lib.exists():
        import __graft_entry__
        __graft_entry__.build()


@pytest.fixture(scope="session")
def scenarios_dir() -> Path:
    return ROOT / "tests" / "scenarios"
