"""Argument checks of the scene and camera edits (DeviceScene.update / update_geometry, DeviceFrame.set_camera) that run before the
library is called, and the part bits of oclr_scene_update: no GPU needed."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

from opencl_render_b200 import _lib, api, scenes


def _scene_stub(device=0):
    """A DeviceScene whose native handle is never reached: every call below fails its argument checks first."""
    ds = api.DeviceScene.__new__(api.DeviceScene)
    ds._lib, ds.handle, ds.device = _lib.load(), None, device
    ds.host = scenes.soup(20, seed=3).normalise()
    return ds


def _geometry(n_tri=20):
    sc = scenes.soup(n_tri, seed=3).normalise()
    return dict(vertex=sc.vertex, tri_idx=sc.tri_idx, tri_mat=sc.tri_mat, tri_uv=sc.tri_uv, tri_normal=sc.tri_normal)


@pytest.mark.parametrize("name, bad", [
    ("vertex", np.zeros((10, 3), np.float32)),
    ("tri_idx", np.zeros((20, 3), np.int32)),
    ("tri_mat", np.zeros((20, 2), np.int32)),
    ("tri_uv", np.zeros((20, 3, 3), np.float32)),
    ("tri_normal", np.zeros((20, 3), np.float32)),
    ("tri_mat", np.zeros(19, np.int32)),          # a triangle count that disagrees with tri_idx
    ("tri_normal", np.zeros((21, 3, 4), np.float32)),
])
def test_update_geometry_refuses_wrong_shapes(name, bad):
    g = _geometry()
    g[name] = bad
    with pytest.raises(ValueError):
        _scene_stub().update_geometry(**g)


def test_update_geometry_checks_the_grid_and_axes_div():
    ds, g = _scene_stub(), _geometry()
    with pytest.raises(ValueError, match="axes_div"):
        ds.update_geometry(**g, axes_div=12)
    with pytest.raises(ValueError, match="grid_start"):
        ds.update_geometry(**g, grid=(np.zeros((5, 4), np.float32), np.zeros(10, np.uint32), np.zeros(0, np.uint32)))
    with pytest.raises(ValueError, match="grid must be"):
        ds.update_geometry(**g, grid=(np.zeros((5, 4), np.float32),))
    with pytest.raises(ValueError, match="axes_div is taken from the grid"):
        ds.update_geometry(**g, grid=(np.zeros((5, 4), np.float32), np.zeros(65, np.uint32), np.zeros(0, np.uint32)), axes_div=4)


def test_update_geometry_refuses_mixed_numpy_and_torch():
    torch = pytest.importorskip("torch")
    g = _geometry()
    g["vertex"] = torch.from_numpy(g["vertex"])
    with pytest.raises(ValueError, match="mix numpy arrays and torch tensors"):
        _scene_stub().update_geometry(**g)


def test_update_geometry_refuses_torch_tensors_off_the_scenes_device():
    torch = pytest.importorskip("torch")
    g = {k: torch.from_numpy(v) for k, v in _geometry().items()}   # host tensors: not on the scene's CUDA device
    with pytest.raises(ValueError, match="the scene is on cuda:0"):
        _scene_stub().update_geometry(**g)
    g = {k: torch.empty(v.shape, dtype=v.dtype, device="meta") for k, v in g.items()}
    with pytest.raises(ValueError, match="the scene is on cuda:0"):
        _scene_stub().update_geometry(**g)


def test_update_needs_a_part_and_a_host_scene():
    ds = _scene_stub()
    with pytest.raises(ValueError, match="at least one part"):
        ds.update(ds.host)
    with pytest.raises(ValueError, match="HostScene"):
        ds.update(_geometry(), geometry=True)


@pytest.mark.parametrize("parts", [0, 8, 1 | 16, 0xFFFFFFFF])
def test_scene_update_refuses_unknown_part_bits(parts):
    lib = _lib.load()
    d = scenes.soup(20, seed=3).normalise().desc(allow_missing_grid=True)
    assert lib.oclr_scene_update(None, C.byref(d), parts, api.QUERY_HOST_MEMORY) == 0
    assert "parts must be a non-empty combination" in _lib.last_error()


def test_scene_update_refuses_a_null_scene_and_unknown_memory():
    lib = _lib.load()
    d = scenes.soup(20, seed=3).normalise().desc(allow_missing_grid=True)
    assert lib.oclr_scene_update(None, C.byref(d), api.SCENE_LIGHTS, api.QUERY_HOST_MEMORY) == 0
    assert "null scene" in _lib.last_error()
    for memory in (2, -1):
        assert lib.oclr_scene_update(None, C.byref(d), api.SCENE_LIGHTS, memory) == 0
        assert f"unknown memory kind {memory}" in _lib.last_error()
    assert lib.oclr_frame_set_camera(None, None) == 0
    assert lib.oclr_frame_set_camera_lists(None, None, None, None, None, 0) == 0


def _frame_stub(w=32, h=24):
    fr = api.DeviceFrame.__new__(api.DeviceFrame)
    fr._lib, fr.handle = _lib.load(), None
    fr.camera = api.set_camera((0, 0, -5), (0, 0, 0), (0, 1, 0), 0.8, w, h)
    return fr


def test_set_camera_refuses_another_image_size_and_bad_lists():
    fr = _frame_stub()
    with pytest.raises(ValueError, match="keeps its image size"):
        fr.set_camera(api.set_camera((0, 0, -5), (0, 0, 0), (0, 1, 0), 0.8, 32, 25))
    with pytest.raises(ValueError, match="CameraSetup"):
        fr.set_camera(fr.camera.c())
    lists = api.CameraLists(np.zeros(32 * 24 - 1, np.uint32), np.zeros(32 * 24, np.uint32), np.zeros(0, np.uint32))
    with pytest.raises(ValueError, match="width \\* height"):
        fr.set_camera(fr.camera, lists)


def test_path_state_reallocates_when_the_ring_depth_changes(tmp_path):
    """The decision PathState::reserve and the frame's launch take before a render (runtime.h path_state_regrow), compiled for the host:
    a materials edit that changes the scene's ring depth (2 <-> 12 slots) reallocates a frame's path state in both directions, at no
    smaller capacity, before the next render writes to the ring."""
    src = tmp_path / "regrow.cpp"
    src.write_text('#include "runtime.h"\nextern "C" unsigned regrow(unsigned c, int r, unsigned q, int s) { return oclr::path_state_regrow(c, r, q, s); }\n')
    lib = tmp_path / "libregrow.so"
    csrc = Path(__file__).resolve().parent.parent / "opencl_render_b200" / "csrc"
    subprocess.run(["g++", "-std=c++17", "-fPIC", "-shared", f"-I{csrc}", "-I/usr/local/cuda/include", str(src), "-o", str(lib)], check=True)
    regrow = C.CDLL(str(lib)).regrow
    regrow.restype = C.c_uint
    regrow.argtypes = [C.c_uint, C.c_int, C.c_uint, C.c_int]
    assert regrow(0, 0, 1000, 2) == 1000          # first render
    assert regrow(1000, 2, 1000, 2) == 0          # same domain, same ring: the buffers serve it
    assert regrow(1000, 2, 500, 2) == 0           # a smaller domain fits
    assert regrow(1000, 2, 1000, 12) == 1000      # materials edit 2 -> 12 slots: reallocate before the ring is written
    assert regrow(1000, 2, 500, 12) == 1000       # ... at no smaller capacity
    assert regrow(1000, 12, 1000, 2) == 1000      # and back, 12 -> 2
    assert regrow(1000, 12, 2000, 12) == 2000     # growth as before
