"""Ray queries without a GPU: the production walk's host form (tests/hostemu, rt_walk.h) against the reference's cell walk
(oracle/raytrace_port.c port_walk_grid) on caller rays -- the known-answer cases of SURVEY.md section 8c(iii) that whole renders never
produce -- plus the screening rules' claims about the reference, the no-GPU error and the Python argument checks."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

from opencl_render_b200 import _lib, api
from tests import helpers, port_rays, query_rays

ROOT = Path(__file__).resolve().parent.parent

# walk modes of the trace stage: 2 = wf_pipe_kernel's packed walk, 1001 = the brick-plane bursts of the tail hand-off (rt_tail.cuh)
WALK_MODES = ["2", "1001"]


@pytest.fixture(scope="module")
def hostemu_rays():
    """tests/_build/libhostemu_rays.so: the production walk (rt_walk.h, rt_core.h) compiled for the host -- test-only."""
    lib = ROOT / "tests" / "_build" / "libhostemu_rays.so"
    srcs = [ROOT / "tests" / "hostemu" / "hostemu_rays.cpp", ROOT / "opencl_render_b200" / "csrc" / "scene_pack.cpp"]
    deps = srcs + list((ROOT / "opencl_render_b200" / "csrc").glob("*.h"))
    if not lib.is_file() or lib.stat().st_mtime < max(p.stat().st_mtime for p in deps):
        lib.parent.mkdir(exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-I/usr/local/cuda/include", "-pthread",
                        *map(str, srcs), "-o", str(lib)], check=True)
    return C.CDLL(str(lib))


def hostemu_walk_rays(lib, sc, o4, d4, excl, threads=8):
    out = np.zeros((o4.shape[0], 4), np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
    d = sc.desc()
    lib.hostemu_walk_rays.restype = C.c_int
    assert lib.hostemu_walk_rays(C.byref(d), C.c_size_t(o4.shape[0]), p(o4), p(d4), p(excl), p(out), C.c_int(threads))
    return out


def _case(name):
    sc, cam, _, _ = helpers.make_case(name)
    return sc, cam


@pytest.mark.parametrize("mode", WALK_MODES)
@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_hostemu_walk_rays_equal_port(name, mode, hostemu_rays, monkeypatch):
    sc, cam = _case(name)
    o4, d4, excl = query_rays.all_families(sc, cam, n=384, seed=7)
    traced = ~query_rays.is_screened(o4, d4) & ~query_rays.is_empty(o4, d4)
    o4, d4, excl = o4[traced], d4[traced], excl[traced]
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", mode)
    got = hostemu_walk_rays(hostemu_rays, sc, o4, d4, excl)
    ref = port_rays.walk_rays(sc, o4, d4, excl)
    bad = np.nonzero((got.view(np.uint32) != ref.view(np.uint32)).any(1))[0]
    assert bad.size == 0, (bad.size, o4[bad[:3]], d4[bad[:3]], got[bad[:3]], ref[bad[:3]])
    hits = (ref[:, 0].view(np.uint32) != query_rays.NONE).sum()
    assert 0 < hits < len(ref)   # the families reach both outcomes


@pytest.mark.parametrize("name", ["soup_mirror_glass", "spheres", "terrain_textured", "coarse_grid"])
def test_empty_range_and_zero_direction_miss_in_the_reference(name):
    """The rays the library answers without a trace -- !(minD < maxD), zero direction -- are misses with t = maxD in the reference too,
    and their transmittance is (1, 1, 1)."""
    sc, cam = _case(name)
    o4, d4, excl = query_rays.family("empty_range", sc, cam, n=1024, seed=3)
    assert query_rays.is_empty(o4, d4).all()
    ref = port_rays.walk_rays(sc, o4, d4, excl)
    assert (ref[:, 0].view(np.uint32) == query_rays.NONE).all()
    assert np.array_equal(ref[:, 1].view(np.uint32), d4[:, 3].view(np.uint32))
    assert (ref[:, 2:] == 0).all()
    att = port_rays.transmit_rays(sc, o4, d4, excl)
    assert (att[:, :3] == 1).all() and (att[:, 3].view(np.uint32) == query_rays.NONE).all()


def test_port_transmit_follows_the_closest_hits():
    """port_transmit is the closest-hit loop: the first blocker it reports is the closest hit of the ray whenever the loop stops there."""
    sc, cam = _case("soup_mirror_glass")
    o4, d4, excl = query_rays.family("shadow", sc, cam, n=2048, seed=5)
    hit = port_rays.walk_rays(sc, o4, d4, excl)
    att = port_rays.transmit_rays(sc, o4, d4, excl)
    miss = hit[:, 0].view(np.uint32) == query_rays.NONE
    assert (att[miss, :3] == 1).all() and (att[miss, 3].view(np.uint32) == query_rays.NONE).all()
    assert (att[~miss, 3].view(np.uint32) != query_rays.NONE).all()
    stopped = ~miss & ~((att[:, :3] > 0).all(1))
    assert stopped.any() and (att[:, :3] < 1).any()


def test_query_entries_fail_without_scene():
    lib = _lib.load()
    out = np.zeros((1, 4), np.float32)
    o = np.zeros((1, 4), np.float32)
    for entry in ("oclr_scene_intersect", "oclr_scene_transmittance"):
        assert getattr(lib, entry)(None, 1, o.ctypes.data, o.ctypes.data, None, out.ctypes.data, 0, 0, None, None) == 0
        assert entry in _lib.last_error() and "null scene" in _lib.last_error()


def test_query_entries_fail_without_gpu():
    """Without a usable device no scene exists, so a query cannot run; a scene cannot be created either."""
    lib = _lib.load()
    if lib.oclr_device_count() > 0:
        pytest.skip("a CUDA device is present")
    sc, _ = _case("coarse_grid")
    with pytest.raises(api.OclrError):
        api.DeviceScene(sc)


class _FakeScene(api.DeviceScene):
    """A DeviceScene whose native calls must never happen: argument errors are raised before them."""

    def __init__(self):
        self.handle, self.device = None, 0

        class _NoLib:
            def __getattr__(self, name):
                raise AssertionError(f"native call {name} reached")
        self._lib = _NoLib()

    def close(self):
        pass


@pytest.mark.parametrize("call", ["intersect", "transmittance"])
def test_query_argument_validation(call):
    s = _FakeScene()
    f = getattr(s, call)
    o3, d3 = np.zeros((4, 3), np.float32), np.ones((4, 3), np.float32)
    o4, d4 = np.zeros((4, 4), np.float32), np.ones((4, 4), np.float32)
    bad = [
        lambda: f(np.zeros((4, 2), np.float32), d3),                    # wrong width
        lambda: f(np.zeros(4, np.float32), d3),                         # 1-D
        lambda: f(o3, np.ones((5, 3), np.float32)),                     # ray counts differ
        lambda: f(o3.astype(np.int32), d3),                             # not floating point
        lambda: f(o3, d3, t_min=np.zeros(3)),                           # range of the wrong length
        lambda: f(o3, d3, t_max="far"),                                 # range not a number
        lambda: f(o4, d4, t_min=0.5),                                   # [N,4] carries its range already
        lambda: f(o3, d4, t_max=2.0),
        lambda: f(o3, d3, exclude=np.zeros(4, np.float32)),             # excluded ids not integers
        lambda: f(o3, d3, exclude=np.zeros(5, np.uint32)),              # ... of the wrong length
    ]
    for k, b in enumerate(bad):
        with pytest.raises(ValueError):
            b()
