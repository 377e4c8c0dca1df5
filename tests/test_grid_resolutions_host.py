"""Grid resolutions without a GPU (tests/grid_scenes.py): at 1, 2, 4, 8, 32, 128, 512 and 1024 cells per axis, every walk the trace
stage has (rt_walk.h, compiled for the host by tests/hostemu) equals the port bit for bit, on frames and on caller rays, and each case is
asserted to reach the special case of the code it exists for, so that a change to a scene cannot quietly make it ordinary.  Resolutions
outside the accepted range are refused with a message."""
import ctypes as C

import numpy as np
import pytest

from opencl_render_b200 import api, scenes
from tests import grid_scenes, helpers, port_rays, query_rays
from tests.grid_scenes import CASES, FINE
from tests.test_query_host import WALK_MODES, hostemu_rays, hostemu_walk_rays  # noqa: F401 (fixture)

BAD_RESOLUTIONS = [0, -4, 3, 48, 2048]
# cells / gridRays of the counting host emulation (the reference's cell walk) on the 256-cell cases of tests/helpers.py: 160 (soup) to 214
# (terrain_textured); measured on the 1024-cell cases: 758 (soup_1024) and 754 (sparse_1024)
WALK_CELLS_1024 = 600


@pytest.fixture(scope="module", params=list(CASES))
def grid_case(request):
    """Module scope and parameters: pytest runs every test of one case before it builds the next, so a 4 GiB grid is built once."""
    name = request.param
    yield name, grid_scenes.case(name)
    grid_scenes.release()


def _render(lib, monkeypatch, c, mode=None, super_level=None):
    sc, cam, lists, samples = c
    if mode is None:
        monkeypatch.delenv("HOSTEMU_HIERARCHICAL", raising=False)
    else:
        monkeypatch.setenv("HOSTEMU_HIERARCHICAL", mode)
    if super_level is None:
        monkeypatch.delenv("OCLR_SUPER", raising=False)
    else:
        monkeypatch.setenv("OCLR_SUPER", super_level)
    return helpers.hostemu_render(lib, cam, lists, sc, samples, threads=8)


def _same(a, b):
    return all(np.array_equal(a[0][c], b[0][c]) for c in range(3)) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])


def test_walks_equal_port(grid_case, hostemu, port, monkeypatch):
    """Every walk against the port's planes and ids and the reference cell walk's flags, with the counter relations of
    tests/test_hostemu_parity.py."""
    name, c = grid_case
    sc, cam, lists, samples = c
    ref = port.render(cam, lists, sc, samples, want_ids=True)
    flat = _render(hostemu, monkeypatch, c)
    assert all(np.array_equal(flat[0][k], ref[k]) for k in range(3)) and np.array_equal(flat[1], ref[3]), name
    assert (ref[3] != api.NO_TRIANGLE).any()
    if name.startswith("terrain_textured"):
        assert flat[2].any()   # bump maps: the undefined-result flags are exercised
    fc = flat[3]
    # the two-level walk: the reference's brick sequence, fewer cells
    hier = _render(hostemu, monkeypatch, c, "1")
    assert _same(flat, hier), name
    assert hier[3]["bricksLoaded"] == fc["bricksLoaded"] and hier[3]["gridCandidates"] == fc["gridCandidates"]
    assert hier[3]["cellsNonEmpty"] == fc["cellsNonEmpty"] and hier[3]["cells"] <= fc["cells"]
    # the packed walk (production), without and with the super-brick level
    two = _render(hostemu, monkeypatch, c, "2", "0")
    assert _same(flat, two), name
    assert two[3]["bricksLoaded"] == fc["bricksLoaded"] and two[3]["superSteps"] == 0
    assert two[3]["cellsNonEmpty"] == fc["cellsNonEmpty"] and two[3]["gridCandidates"] <= fc["gridCandidates"] and two[3]["cells"] <= fc["cells"]
    three = _render(hostemu, monkeypatch, c, "2", "1")
    assert _same(flat, three), name
    for k in ("cells", "cellsNonEmpty", "gridCandidates", "coarseEnters", "gridRays"):
        assert three[3][k] == two[3][k], (name, k)
    assert three[3]["superEnters"] >= three[3]["superRefines"]
    # split walks, the run-time split, cooperative bursts, brick-plane bursts
    for mode in ("3", "40", "2308"):
        split = _render(hostemu, monkeypatch, c, mode)
        assert _same(flat, split), (name, mode)
        assert split[3]["cellsNonEmpty"] == fc["cellsNonEmpty"], (name, mode)
    coop = _render(hostemu, monkeypatch, c, "1000")
    assert _same(flat, coop), name
    assert coop[3]["cellsNonEmpty"] == fc["cellsNonEmpty"]
    bricks = _render(hostemu, monkeypatch, c, "1001")
    assert _same(flat, bricks), name
    assert bricks[3]["cellsNonEmpty"] == fc["cellsNonEmpty"] and bricks[3]["gridRays"] == two[3]["gridRays"]
    # the case reaches its special case
    kind, n = CASES[name]
    if n >= 32 and kind in ("soup", "sparse") or name == "terrain_textured_128":
        assert three[3]["superSteps"] > 0, name
    elif kind == "flat" or n < 32:   # (a flat scene: every super-brick holds a piece of the plane in its zero-width y layers)
        assert three[3]["superSteps"] == 0, name
    if n < 32:
        assert three[3]["superSteps"] == 0 and three[3]["coarseSteps"] == two[3]["coarseSteps"], name
    if n < 4:   # no brick level (pwalk_setup: coarseOk = n >= 4)
        assert two[3]["coarseSteps"] == 0 and two[3]["coarseEnters"] == 0, name
    if n == FINE:
        assert fc["cells"] > WALK_CELLS_1024 * fc["gridRays"], (name, fc["cells"] / fc["gridRays"])


@pytest.mark.parametrize("mode", WALK_MODES)
def test_caller_rays_equal_port(grid_case, mode, hostemu_rays, monkeypatch):  # noqa: F811
    name, c = grid_case
    sc, cam = c[0], c[1]
    o4, d4, excl = grid_scenes.rays(name)
    traced = ~query_rays.is_screened(o4, d4) & ~query_rays.is_empty(o4, d4)
    o4, d4, excl = o4[traced], d4[traced], excl[traced]
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", mode)
    got = hostemu_walk_rays(hostemu_rays, sc, o4, d4, excl)
    ref = port_rays.walk_rays(sc, o4, d4, excl)
    bad = np.nonzero((got.view(np.uint32) != ref.view(np.uint32)).any(1))[0]
    assert bad.size == 0, (name, bad.size, o4[bad[:3]], d4[bad[:3]], got[bad[:3]], ref[bad[:3]])
    hits = (ref[:, 0].view(np.uint32) != query_rays.NONE).sum()
    assert 0 < hits < len(ref)


def _host_pack(lib, sc):
    """(bricks uint32 [nb^3, 4], cell ranges uint32 [cells, 2]) of the host packer (scene_pack.cpp pack_grid)."""
    n = sc.axes_div
    nb = max(n // 4, 1)
    nonempty = int((np.diff(sc.grid_start) > 0).sum())
    geo, shade = np.zeros(64 * sc.triangle_count, np.uint8), np.zeros(128 * sc.triangle_count, np.uint8)
    bricks, planes = np.zeros((nb ** 3, 4), np.uint32), np.zeros(3 * (n + 1), np.float32)
    ranges = np.zeros((max(nonempty, 1), 2), np.uint32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    lib.hostemu_pack.restype = C.c_long
    cnt = lib.hostemu_pack(C.byref(sc.desc()), p(geo), p(shade), p(bricks), p(ranges), C.c_size_t(ranges.nbytes), p(planes), None)
    assert cnt == nonempty
    return bricks, ranges[:cnt]


def test_case_reaches_its_special_case(grid_case, hostemu, monkeypatch):
    """What each resolution exists for, from the grid arrays and the host packer (the walks' counters are asserted in
    test_walks_equal_port)."""
    monkeypatch.delenv("OCLR_SUPER", raising=False)
    name, (sc, _, _, _) = grid_case
    kind, n = CASES[name]
    assert sc.axes_div == n and sc.grid_start.size == n ** 3 + 1
    lengths = np.diff(sc.grid_start)
    planes = sc.box_min[:, :3]
    if n <= 2:
        # one brick, partly filled: its mask has bits only for the n^3 cells (x | y << 2 | z << 4 with x, y, z < n)
        bricks, _ = _host_pack(hostemu, sc)
        inside = sum(1 << (x | y << 2 | z << 4) for x in range(n) for y in range(n) for z in range(n))
        mask = int(bricks[0, 0]) | int(bricks[0, 1]) << 32
        assert bricks.shape[0] == 1 and mask != 0 and mask & ~inside == 0, (name, hex(mask))
        assert bin(mask).count("1") == int((lengths > 0).sum())
    if n <= 4:
        assert lengths.max() > 32, (name, lengths.max())   # lists scanned past their 32-entry face masks
    if kind == "sparse":
        assert sc.vertex_count < n
        for a in range(3):   # repeated split planes strictly inside the scene's extent: zero-width cells in the middle of the grid
            p = planes[:, a]
            inner = (p[:-1] == p[1:]) & (p[:-1] > p[0]) & (p[1:] < p[-1])
            assert inner.sum() >= n // 8, (name, a, int(inner.sum()))
    if kind == "flat":
        assert (planes[:, 1] == planes[0, 1]).all()   # all n + 1 planes of the y axis coincide
    # the device builder's candidate blocks (grid_range_kernel): every listed cell lies in its triangle's block, and on fine grids most
    # blocks are filled by the one-CTA kernel (more than 512 cells).  Measured: 10 (sparse_128) to all; 126 of 127 (sparse_512)
    blocks = grid_scenes.candidate_block_cells(sc)
    assert (np.bincount(sc.grid_list, minlength=sc.triangle_count) <= blocks).all()
    large = int((blocks > grid_scenes.GRID_SMALL_BLOCK).sum())
    if n >= 512:
        assert 10 * large >= 9 * sc.triangle_count, (name, large)
    elif n >= 128:
        assert large >= 8, (name, large)


@pytest.mark.parametrize("n", BAD_RESOLUTIONS)
def test_host_builder_refuses_bad_resolutions(n):
    sc = scenes.soup(20, seed=1)
    with pytest.raises(api.OclrError, match="axesDivCount"):
        api.scene_triangle_list(sc, n)
    assert sc.box_min is None


@pytest.mark.parametrize("n", [0, 3, 48])
def test_caller_grid_with_bad_resolution_is_refused(n, hostemu, capfd):
    """validate_scene (scene_pack.cpp), which scene upload runs first, on a caller-supplied grid whose axesDivCount is not a power of two:
    the host emulation, which runs the same check, returns an error with the message instead of reading the grid."""
    sc, cam, lists, _ = helpers.make_case("coarse_grid")
    sc.axes_div = n
    h, w = cam.height, cam.width
    out = [np.zeros((h, w), np.uint16) for _ in range(3)]
    ids, flags, cnt = np.zeros((h, w), np.uint32), np.zeros((h, w), np.uint8), helpers._lib.Counters()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    hostemu.hostemu_render.restype = C.c_int
    ok = hostemu.hostemu_render(C.byref(sc.desc()), C.byref(cam.c()), p(lists.start), p(lists.end), p(lists.list), C.c_uint32(1),
                                C.c_uint32(0), C.c_uint32(h), p(out[0]), p(out[1]), p(out[2]), p(ids), p(flags), C.byref(cnt), C.c_int(1))
    assert ok == 0 and "axesDivCount must be a power of two" in capfd.readouterr().err


@pytest.mark.parametrize("n", BAD_RESOLUTIONS)
def test_device_scene_passes_the_resolution_through(n, monkeypatch):
    """DeviceScene(bare scene, axes_div=n) hands n to the library as it is (it used to turn 0 into the default 256), so the library's
    refusal is what the caller sees."""
    seen = []

    class _Lib:
        def oclr_scene_create(self, device, desc):
            seen.append(desc._obj.axesDivCount)
            return None

    monkeypatch.setattr(api._lib, "load", lambda: _Lib())
    monkeypatch.setattr(api._lib, "last_error", lambda: "oclr_scene_create: refused")
    with pytest.raises(api.OclrError):
        api.DeviceScene(scenes.soup(20, seed=1), 0, axes_div=n)
    assert seen == [n]
