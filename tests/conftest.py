"""Test configuration.  `-m "not gpu"` runs here (no GPU): oracle vs reference build / golden vectors, host builders, the host
emulation of the device arithmetic, C-ABI symbol checks, gloo world-size-2 logic.  `-m gpu` is the parity suite proper
(CUDA through the C-ABI vs the oracle) and runs on a B200."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


def _has_gpu() -> bool:
    try:
        from opencl_render_b200 import _lib
        return _lib.load().oclr_device_count() > 0
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def port():
    import port as _port
    _port.load()
    return _port


@pytest.fixture(scope="session")
def hostemu():
    """tests/_build/libhostemu.so: the product's device arithmetic (rt_core.h) compiled for the host -- test-only."""
    import ctypes as C
    out = ROOT / "tests" / "_build"
    out.mkdir(exist_ok=True)
    lib = out / "libhostemu.so"
    srcs = [ROOT / "tests" / "hostemu" / "hostemu.cpp", ROOT / "opencl_render_b200" / "csrc" / "scene_pack.cpp"]
    deps = srcs + list((ROOT / "opencl_render_b200" / "csrc").glob("*.h"))
    if not lib.is_file() or lib.stat().st_mtime < max(p.stat().st_mtime for p in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-I/usr/local/cuda/include", "-pthread",
                        *map(str, srcs), "-o", str(lib)], check=True)
    return C.CDLL(str(lib))


from tests.helpers import *  # noqa: E402,F401,F403
