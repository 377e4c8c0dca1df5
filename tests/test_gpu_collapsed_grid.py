"""The walk grid on the device (rt_types.h; runtime.cu grid_stage): the device collapse equals the host form (scene_pack.cpp
pack_walk_grid) byte for byte, config 2 walks a y axis of 56 cells, config 3 gets no second grid, and a geometry edit rebuilds it.  The
production path against the per-pixel kernel, which walks the reference grid, on the edited scene."""
import copy

import numpy as np
import pytest

from opencl_render_b200 import api, scenes
from tests import grid_scenes, helpers
from tests.test_collapsed_grid_host import malformed_spheres, walk_grid, walkgrid  # noqa: F401 (fixture)

pytestmark = pytest.mark.gpu


def _device_walk_grid(ds):
    return dict(extents=ds.debug_read(11).view(np.uint32), bricks=ds.debug_read(7).view(np.uint32), ranges=ds.debug_read(8).view(np.uint32),
                masks=ds.debug_read(9).view(np.uint32), planes=ds.debug_read(10).view(np.float32))


def _assert_equal_host(ds, sc, walkgrid):
    host = walk_grid(walkgrid, sc)
    dev = _device_walk_grid(ds)
    if host is None:
        assert (dev["extents"] == sc.axes_div).all() and dev["bricks"].size == 0
        return dev
    assert np.array_equal(dev["extents"], host["extents"].astype(np.uint32))
    assert np.array_equal(dev["bricks"], host["bricks"])
    assert np.array_equal(dev["planes"], host["planes"])
    cnt = host["ranges"].size // 2
    assert np.array_equal(dev["ranges"][:2 * cnt], host["ranges"]) and np.array_equal(dev["masks"][:6 * cnt], host["masks"])
    return dev


def _frames_equal(ds, cam, lists, samples):
    fr = api.DeviceFrame(ds, cam, lists)
    fr.render(samples, variant=api.KERNEL_SIMPLE)
    want = fr.read(), fr.primary_ids()
    fr.render(samples)
    got = fr.read(), fr.primary_ids()
    fr.close()
    assert all(np.array_equal(got[0][c], want[0][c]) for c in range(3)) and np.array_equal(got[1], want[1])


@pytest.mark.parametrize("name", ["spheres", "spheres_mirror", "terrain", "flat_32", "sparse_128"])
def test_device_collapse_equals_host(name, walkgrid):
    sc, cam, lists, samples = grid_scenes.case(name) if name in grid_scenes.CASES else helpers.make_case(name)
    ds = api.DeviceScene(sc)
    _assert_equal_host(ds, sc, walkgrid)
    _frames_equal(ds, cam, lists, samples)
    ds.close()


def _config_extents(k):
    sc = scenes.CONFIGS[k]["make"]()
    ds = api.DeviceScene(sc, 0, axes_div=256)   # grid built on the device, as RaytraceAll does
    ext = ds.debug_read(11).view(np.uint32).tolist()
    walk_bytes = ds.debug_read(7).size
    ds.close()
    return ext, walk_bytes


def test_config2_walk_grid():
    ext, walk_bytes = _config_extents(2)
    assert ext == [256, 56, 256] and walk_bytes == 16 * 64 ** 3


def test_config3_no_walk_grid():
    ext, walk_bytes = _config_extents(3)
    assert ext == [256, 256, 256] and walk_bytes == 0


def test_update_geometry_rebuilds(walkgrid):
    sc, cam, lists, samples = helpers.make_case("spheres")
    other = copy.copy(sc)
    api.scene_triangle_list(other, 128)   # the same geometry on a grid of 128 cells per axis
    ds = api.DeviceScene(sc)
    before = _assert_equal_host(ds, sc, walkgrid)
    ds.update_geometry(other.vertex, other.tri_idx, other.tri_mat, other.tri_uv, other.tri_normal,
                       grid=(other.box_min, other.grid_start, other.grid_list))
    after = _assert_equal_host(ds, other, walkgrid)
    assert not np.array_equal(before["extents"], after["extents"])
    _frames_equal(ds, cam, lists, samples)
    ds.update_geometry(sc.vertex, sc.tri_idx, sc.tri_mat, sc.tri_uv, sc.tri_normal, axes_div=sc.axes_div)   # built on the device
    _assert_equal_host(ds, sc, walkgrid)
    _frames_equal(ds, cam, lists, samples)
    ds.close()


def test_malformed_csr_in_a_run_is_refused():
    """A caller's grid whose CSR is not monotone inside a collapsible run: the scene is refused with the packers' message, and the run
    check reads no entry of the bad ranges (no device fault: a scene created afterwards renders)."""
    sc = malformed_spheres()[0]
    with pytest.raises(api.OclrError, match="monotone CSR"):
        api.DeviceScene(sc)
    sc, cam, lists, samples = helpers.make_case("spheres")
    ds = api.DeviceScene(sc)
    _frames_equal(ds, cam, lists, samples)
    ds.close()
