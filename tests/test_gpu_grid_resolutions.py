"""Grid resolutions on the GPU (tests/grid_scenes.py: 1, 2, 4, 8, 32, 128, 512 and 1024 cells per axis), bit for bit: frames of both
kernel variants against the port and the host emulation's flags, the counting build's counters, ray queries against their restatements,
the device grid builder and the device packers against the host ones, the off-by-default walks (super-brick level, tail hand-off, run-time
split) in processes of their own, and the two limits that are refusals: 2^17 entries in one cell's list (the packer) and 2^31
(triangle, cell) candidates (the device grid builder).  Which special case each resolution reaches is asserted on the host by
tests/test_grid_resolutions_host.py."""
import copy
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from opencl_render_b200 import api, scenes
from tests import grid_scenes, helpers, port_radiance, port_rays, query_rays
from tests.grid_scenes import CASES, FINE

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
NONE = query_rays.NONE
COUNTERS = ("segments", "primCandidates", "gridRays", "cells", "cellsNonEmpty", "gridCandidates", "shadedHits", "occluderLookups")


@pytest.fixture(scope="module", params=list(CASES))
def grid_case(request):
    """(name, (scene, camera, lists, samples), DeviceScene): every test of one case runs before the next case is built."""
    name = request.param
    c = grid_scenes.case(name)
    ds = api.DeviceScene(c[0], 0)
    yield name, c, ds
    ds.close()
    grid_scenes.release()


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _equal(img, want):
    return all(np.array_equal(img[k], want[k]) for k in range(3))


def test_frames_equal_port(grid_case, port, hostemu, monkeypatch):
    name, (sc, cam, lists, samples), ds = grid_case
    want = port.render(cam, lists, sc, 2, want_ids=True)
    monkeypatch.delenv("HOSTEMU_HIERARCHICAL", raising=False)
    flags = helpers.hostemu_render(hostemu, cam, lists, sc, 2, threads=8)[2]
    fr = api.DeviceFrame(ds, cam, lists)
    for variant in (api.KERNEL_PIPE, api.KERNEL_SIMPLE):
        fr.render(2, variant=variant)
        assert _equal(fr.read(), want) and np.array_equal(fr.primary_ids(), want[3]), (name, variant)
        assert np.array_equal(fr.undefined_flags(), flags), (name, variant)
    if CASES[name][1] in (2, FINE):
        try:
            for mode in (0, 1, 2):
                api.set_option("ahead", mode)
                fr.render(2)
                assert _equal(fr.read(), want) and np.array_equal(fr.primary_ids(), want[3]), (name, mode)
        finally:
            api.set_option("ahead", -1)
    fr.close()


def test_counters_equal_host_emulation(grid_case, hostemu, monkeypatch):
    name, (sc, cam, lists, _), ds = grid_case
    monkeypatch.delenv("HOSTEMU_HIERARCHICAL", raising=False)
    want = helpers.hostemu_render(hostemu, cam, lists, sc, 1, threads=8)[3]
    fr = api.DeviceFrame(ds, cam, lists)
    cnt = fr.render(1, variant=api.KERNEL_SIMPLE, count=True)[2]
    for k in COUNTERS:
        assert cnt[k] == want[k], (name, k, cnt[k], want[k])
    cnt = fr.render(1, variant=api.KERNEL_PIPE, count=True)[2]   # the counting instantiation of the logic kernel
    for k in ("segments", "shadedHits", "occluderLookups"):
        assert cnt[k] == want[k], (name, k, cnt[k], want[k])
    fr.close()


def test_queries_equal_restatements(grid_case):
    name, (sc, cam, _, _), ds = grid_case
    o4, d4, excl = grid_scenes.rays(name)
    ok = ~query_rays.is_screened(o4, d4)
    assert ok.all()
    ids, t, ab, ac = ds.intersect(o4, d4, exclude=excl)
    ref = port_rays.walk_rays(sc, o4, d4, excl)
    assert np.array_equal(ids, _bits(ref[:, 0])) and np.array_equal(_bits(t), _bits(ref[:, 1])), name
    assert np.array_equal(_bits(ab), _bits(ref[:, 2])) and np.array_equal(_bits(ac), _bits(ref[:, 3])), name
    assert 0 < (ids != NONE).sum() < len(ids)
    att, last = ds.transmittance(o4, d4, exclude=excl)
    ref = port_rays.transmit_rays(sc, o4, d4, excl)
    assert np.array_equal(_bits(att), _bits(ref[:, :3])) and np.array_equal(last, _bits(ref[:, 3])), name
    inf = d4[:, 3] == np.inf   # radiance rays have no far limit: the rays of the families that have one are left out
    o4, d4, excl = o4[inf], d4[inf], excl[inf]
    rgb, ids, flags = ds.radiance(o4, d4, exclude=excl, camera=cam, flags=True)
    ref, ref_flags, _ = port_radiance.shade_rays(sc, o4, d4, excl, camera=cam)
    nan = np.isnan(ref[:, :3])
    assert np.array_equal(np.isnan(rgb), nan) and np.array_equal(_bits(rgb)[~nan], _bits(ref[:, :3])[~nan]), name
    assert np.array_equal(ids, _bits(ref[:, 3])) and np.array_equal(flags, ref_flags), name
    assert (rgb[~nan] > 0).any()


def test_device_grid_builder_equals_host_builder(grid_case):
    name, (sc, _, _, _), _ = grid_case
    dev = copy.copy(sc)
    api.scene_triangle_list(dev, sc.axes_div, device=0)
    assert dev.axes_div == sc.axes_div
    assert np.array_equal(dev.box_min.view(np.uint32), sc.box_min.view(np.uint32)), name
    assert np.array_equal(dev.grid_start, sc.grid_start), name
    assert dev.grid_list.size == sc.grid_list.size and np.array_equal(dev.grid_list, sc.grid_list), name


def test_upload_without_grid_equals_upload_with_host_grid(grid_case):
    name, (sc, _, _, _), ds = grid_case
    bare = copy.copy(sc)
    bare.box_min = bare.grid_start = bare.grid_list = None
    b = api.DeviceScene(bare, 0, axes_div=sc.axes_div)
    for which in range(7):
        assert np.array_equal(ds.debug_read(which), b.debug_read(which)), (name, which)
    b.close()


def test_device_packers_equal_host_packer(grid_case, hostemu, monkeypatch):
    """pack_kernels.cuh (bricks of side n < 4, 2^24 bricks and 2^30 cells at 1024) against scene_pack.cpp, byte for byte."""
    monkeypatch.delenv("OCLR_SUPER", raising=False)
    name, (sc, _, _, _), ds = grid_case
    n, N = sc.axes_div, sc.triangle_count
    nb = max(n // 4, 1)
    nonempty = int((np.diff(sc.grid_start) > 0).sum())
    geo, shade = np.zeros(64 * N, np.uint8), np.zeros(128 * N, np.uint8)
    bricks, planes = np.zeros(16 * nb ** 3, np.uint8), np.zeros(12 * (n + 1), np.uint8)
    ranges, masks = np.zeros(8 * max(nonempty, 1), np.uint8), np.zeros(24 * max(nonempty, 1), np.uint8)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    hostemu.hostemu_pack.restype = C.c_long
    cnt = hostemu.hostemu_pack(C.byref(sc.desc()), p(geo), p(shade), p(bricks), p(ranges), C.c_size_t(ranges.size), p(planes), p(masks))
    assert cnt == nonempty
    assert np.array_equal(ds.debug_read(0), geo) and np.array_equal(ds.debug_read(1), shade), name
    assert np.array_equal(ds.debug_read(2), bricks) and np.array_equal(ds.debug_read(4), planes), name
    assert np.array_equal(ds.debug_read(3)[:8 * cnt], ranges[:8 * cnt]), name
    assert np.array_equal(ds.debug_read(5).view(np.uint32), sc.grid_list), name
    assert np.array_equal(ds.debug_read(6)[:24 * cnt], masks[:24 * cnt]), name


# ---- off-by-default walks, one process per setting (their knobs are read once per process) -----------------------------------------
_PROBE = r"""
import hashlib, json, os, sys
import numpy as np
sys.path.insert(0, os.getcwd())
from opencl_render_b200 import api
from tests import grid_scenes
out = {}
for name in sys.argv[1].split(","):
    sc, cam, lists, samples = grid_scenes.case(name)
    res = {}
    for policy in sys.argv[2].split(","):
        os.environ["OCLR_SUPER"] = policy
        ds = api.DeviceScene(sc, 0)
        fr = api.DeviceFrame(ds, cam, lists)
        _, _, cnt = fr.render(2, count=True)
        h = hashlib.sha256()
        for a in (*fr.read(), fr.primary_ids(), fr.undefined_flags()):
            h.update(np.ascontiguousarray(a).tobytes())
        res[policy] = dict(sha=h.hexdigest(), brick_bytes=len(ds.debug_read(2)),
                           **{k: cnt[k] for k in ("superSteps", "superEnters", "coarseSteps", "bricksLoaded", "splitsDone")})
        fr.close(); ds.close()
    out[name] = res
    grid_scenes.release()
print("GRID_PROBE " + json.dumps(out))
"""


def _want_sha(port, hostemu, name):
    sc, cam, lists, _ = grid_scenes.case(name)
    ref = port.render(cam, lists, sc, 2, want_ids=True)
    os.environ.pop("HOSTEMU_HIERARCHICAL", None)
    flags = helpers.hostemu_render(hostemu, cam, lists, sc, 2, threads=8)[2]
    h = hashlib.sha256()
    for a in (*ref[:3], ref[3], flags):
        h.update(np.ascontiguousarray(a).tobytes())
    grid_scenes.release()
    return h.hexdigest()


def _probe(names, policies, env):
    r = subprocess.run([sys.executable, "-c", _PROBE, ",".join(names), ",".join(policies)], cwd=ROOT, env=dict(os.environ, **env),
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("GRID_PROBE ")][-1][len("GRID_PROBE "):])


def test_super_brick_level_at_every_fine_resolution(port, hostemu):
    """The variant library whose trace kernel has the super-brick level (see test_gpu_progressive.py::
    test_super_brick_level_of_the_walk_is_invisible), at 32, 128 and 1024 cells per axis: packed without the flags (two-level walk) and
    with them, the same planes, ids and flags as the port and the host emulation; the soups take super-brick steps."""
    lib = ROOT / "opencl_render_b200" / "libopencl_render_b200_super.so"
    if not lib.is_file():
        pytest.skip("variant library with the super-brick level not built (python -m opencl_render_b200.build --variant super -DOCLR_SUPER_LEVEL=1)")
    names = [k for k, (_, n) in CASES.items() if n in (32, 128, FINE)]
    out = _probe(names, ["0", "1"], dict(OCLR_LIB=str(lib), OCLR_HIERARCHICAL="2"))
    for name in names:
        o, want = out[name], _want_sha(port, hostemu, name)
        assert o["0"]["sha"] == want and o["1"]["sha"] == want, (name, o)
        assert o["0"]["superSteps"] == 0 and o["0"]["superEnters"] == 0, (name, o)
        if CASES[name][0] in ("soup", "sparse"):
            assert o["1"]["superSteps"] > 0 and o["1"]["bricksLoaded"] < o["0"]["bricksLoaded"], (name, o)
            assert o["1"]["brick_bytes"] > o["0"]["brick_bytes"], (name, o)


@pytest.mark.parametrize("setting", ["handoff-0", "split"])
def test_tail_walks_at_2_and_1024_cells(setting, port, hostemu):
    """The tail hand-off forced at age 0 (every ray still walking when its warp sees the queue dry goes through the brick-plane burst
    walker) and the run-time split of long walks, on the 2-cell grids (no brick level) and the 1024-cell grids (full 10-bit fields)."""
    if setting == "split":
        env = dict(OCLR_SPLIT_MIN="8", OCLR_SPLIT_PART="4", OCLR_SPLIT_EARLY="2")
    else:
        env = dict(OCLR_HANDOFF_MAX_PATHS="4000000000", OCLR_HANDOFF_AFTER="0", OCLR_TAIL_BRICKS="1")
    names = [k for k, (_, n) in CASES.items() if n in (2, FINE)]
    out = _probe(names, ["0"], env)
    for name in names:
        assert out[name]["0"]["sha"] == _want_sha(port, hostemu, name), (setting, name, out[name])
    if setting == "split":
        assert sum(out[name]["0"]["splitsDone"] for name in names if CASES[name][1] == FINE) > 0, out


# ---- resolutions and limits that are refusals ------------------------------------------------------------------------------------
def _known_frame():
    sc, cam, lists, samples = helpers.make_case("coarse_grid")
    want = np.load(ROOT / "tests" / "golden" / "coarse_grid.npz")
    return sc, cam, lists, samples, (want["r"], want["g"], want["b"])


def _renders_known_frame():
    sc, cam, lists, samples, want = _known_frame()
    assert _equal(api.raytrace_all(1, cam, lists, samples, sc), want)


@pytest.mark.parametrize("n", [0, -4, 3, 48, 2048])
def test_device_scene_refuses_bad_resolutions(n):
    sc = scenes.soup(20, seed=1)
    with pytest.raises(api.OclrError, match="axesDivCount"):
        api.DeviceScene(sc, 0, axes_div=n)
    with pytest.raises(api.OclrError, match="axesDivCount"):
        api.scene_triangle_list(scenes.soup(20, seed=1), n, device=0)
    if n in (0, 3, 48):   # a caller-supplied grid with that axesDivCount
        sc = helpers.make_case("coarse_grid")[0]
        sc.axes_div = n
        with pytest.raises(api.OclrError, match="axesDivCount"):
            api.DeviceScene(sc, 0)
    _renders_known_frame()


def _one_cell_scene(tris):
    sc = scenes.soup(tris, seed=17)
    api.scene_triangle_list(sc, 1)
    assert sc.grid_start.tolist() == [0, tris]
    return sc


def test_one_cell_list_of_2_17_entries_is_refused():
    sc = _one_cell_scene(1 << 17)
    with pytest.raises(api.OclrError, match="131072 triangles or more"):
        api.DeviceScene(sc, 0)
    _renders_known_frame()


def test_one_cell_list_of_2_17_minus_1_entries_renders(port):
    sc = _one_cell_scene((1 << 17) - 1)
    m = sc.meta["camera"]
    cam = api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], 16, 12)
    lists = api.camera_triangle_list(cam, sc)
    want = port.render(cam, lists, sc, 1, want_ids=True)
    ds = api.DeviceScene(sc, 0)
    fr = api.DeviceFrame(ds, cam, lists)
    fr.render(1)
    assert _equal(fr.read(), want) and np.array_equal(fr.primary_ids(), want[3])
    assert (want[3] != NONE).any()
    fr.close()
    ds.close()
    _renders_known_frame()


def test_device_builder_refuses_more_than_2_31_candidates():
    """Three tilted triangles from corner to corner of a 1024^3 grid, among 1200 small ones (enough vertices for split planes of real
    width): each big triangle's candidate block is the whole grid, 2^30 cells, over 2^31 in all.  The device builder refuses; the host
    builder, which walks only the cells each triangle reaches, builds the grid."""
    big = np.array([[-3, -1, -3], [3, 3, 3], [3, -0.5, 0.2], [-3, -1, -3], [3, 3, 3], [-0.6, 2.8, -0.1],
                    [-3, -1, -3], [3, 3, 3], [0.3, 0.1, -2.9]], np.float32)
    vertex = np.concatenate([scenes.soup(1200, seed=17).vertex[:, :3], big])
    tri = np.arange(vertex.shape[0], dtype=np.int32).reshape(-1, 3)
    atlas = scenes.MaterialAtlas()
    atlas.add(color=(200, 200, 200))
    sc = scenes._scene("corner_to_corner", vertex, tri, np.zeros(len(tri), np.int32),
                       np.tile(np.array([[0, 0], [1, 0], [0, 1]], np.float32), (len(tri), 1, 1)), scenes._flat_normals(vertex, tri), atlas,
                       [helpers._SPOT])
    with pytest.raises(api.OclrError, match=r"more than 2\^31"):
        api.scene_triangle_list(copy.copy(sc), FINE, device=0)
    _renders_known_frame()
    api.scene_triangle_list(sc, FINE)
    blocks = grid_scenes.candidate_block_cells(sc)
    assert (blocks[-3:] == FINE ** 3).all() and blocks.sum() > 1 << 31
    assert sc.grid_start[-1] == sc.grid_list.size > 0
