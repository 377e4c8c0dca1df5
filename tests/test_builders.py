"""Host builders (product code: opencl_render_b200/csrc/builders.cpp) against the reference's own
CameraTriangleList::New / SceneTriangleList::New / SetCamera (source/util/trianglelist.cpp, render.cpp:461-491), through
what the reference build returned, stored under tests/golden (digests of the lists, the camera vectors themselves)."""
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

from opencl_render_b200 import api, scenes

GOLDEN = Path(__file__).resolve().parent / "golden" / "builders.json"


def _digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


CASES = {
    "soup": (lambda: scenes.soup(400, seed=11), 192, 160),
    "spheres": (lambda: scenes.sphere_grid(3, 12, 24), 320, 180),
    "terrain": (lambda: scenes.terrain(48), 240, 135),
    "terrain_big_tris": (lambda: scenes.terrain(6), 160, 90),
}


def _build(name):
    make, w, h = CASES[name]
    sc = make()
    m = sc.meta["camera"]
    cam = api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], w, h)
    lists = api.camera_triangle_list(cam, sc)
    api.scene_triangle_list(sc, 256)
    return sc, cam, lists


@pytest.mark.parametrize("name", list(CASES))
def test_builders_equal_reference(name):
    # builders.json: digests of the reference's CameraTriangleList::New / SceneTriangleList::New output (make_golden.py)
    gold = json.loads(GOLDEN.read_text())[name]
    sc, cam, lists = _build(name)
    assert _digest(lists.start, lists.end, lists.list) == gold["camera_lists"]
    assert _digest(sc.box_min, sc.grid_start, sc.grid_list) == gold["scene_grid"]


@pytest.mark.parametrize("name", list(CASES))
def test_builders_equal_golden(name):
    if not GOLDEN.is_file():
        pytest.skip("golden digests not generated")
    gold = json.loads(GOLDEN.read_text())[name]
    sc, cam, lists = _build(name)
    assert _digest(cam.eye, cam.eye_to_top_left, cam.left_to_right, cam.top_to_bottom, np.float32(cam.pixel_size_inv)) == gold["camera"]
    assert _digest(lists.start, lists.end, lists.list) == gold["camera_lists"]
    assert _digest(sc.box_min, sc.grid_start, sc.grid_list) == gold["scene_grid"]


def test_lists_are_sorted_and_complete():
    sc, cam, lists = _build("soup")
    # per-pixel candidate lists ascending (trianglelist.cpp:565-573 sorts pixel*N+tri keys)
    for p in range(0, cam.width * cam.height, 97):
        seg = lists.list[lists.start[p]:lists.end[p]]
        assert (np.diff(seg.astype(np.int64)) > 0).all()
    # grid CSR monotone, per-cell ascending
    assert (np.diff(sc.grid_start.astype(np.int64)) >= 0).all()
    assert sc.grid_start[-1] == sc.grid_list.size
    nz = np.nonzero(np.diff(sc.grid_start))[0][::211]
    for c in nz:
        seg = sc.grid_list[sc.grid_start[c]:sc.grid_start[c + 1]]
        assert (np.diff(seg.astype(np.int64)) > 0).all()


def test_grid_other_divisions_consistent():
    # the kernel accepts any power-of-two axesDivCount (raytrace_opencl.c:174-193); the builder generalises AXES_DIVISION
    sc = scenes.soup(100, seed=2)
    for n in (1, 2, 16, 64):
        api.scene_triangle_list(sc, n)
        assert sc.box_min.shape == (n + 1, 4) and sc.grid_start.size == n ** 3 + 1
        assert set(np.unique(sc.grid_list)) == set(range(100))      # every triangle lands in at least one cell
    with pytest.raises(api.OclrError):
        api.scene_triangle_list(sc, 48)


def test_empty_scene_builders():
    sc = scenes.soup(0, seed=1)
    cam = api.set_camera((0, 4.4, -8), (0, 0, 0), (0, 1, 0), 0.9, 32, 24)
    lists = api.camera_triangle_list(cam, sc)
    assert lists.list.size == 0 and (lists.start == 0).all() and (lists.end == 0).all()
    api.scene_triangle_list(sc, 16)
    assert sc.grid_list.size == 0 and (sc.grid_start == 0).all()


def test_sub_band_sets_partition_a_ranks_band_set():
    """launch_wavefront cuts the band set of rank r in world N into slices = the band sets of ranks r + N*k in world N*K
    (b % (N*K) == r + N*k implies b % N == r): together they are exactly the rows rank r owns, without overlap."""
    from opencl_render_b200 import api
    for height, band, world, slices in ((1080, 16, 8, 4), (2160, 128, 2, 3), (75, 8, 3, 2), (600, 128, 2, 5)):
        for rank in range(world):
            own = {y for a, b in api.band_partition(height, rank, world, band_rows=band) for y in range(a, b)}
            parts = [{y for a, b in api.band_partition(height, rank + world * k, world * slices, band_rows=band) for y in range(a, b)}
                     for k in range(slices)]
            assert set().union(*parts) == own and sum(len(p) for p in parts) == len(own)


def test_set_camera_equals_reference():
    """oclr_set_camera against the reference's own SetCamera (render.cpp:461-491, cut out of render.cpp by oracle/build_ref.py): bit
    for bit on 1 000 random cameras, including the image shapes of the five configs.  golden/set_camera.npy holds the reference's
    (eye_to_top_left, left_to_right, top_to_bottom, pixel_size_inv) per camera, recorded from oclr_set_camera, which matched it
    bit for bit."""
    stored = np.load(GOLDEN.parent / "set_camera.npy")
    rng = np.random.default_rng(20261018)
    shapes = [(512, 512), (1920, 1080), (3840, 2160), (7680, 4320), (1024, 768), (1, 1), (333, 7)]
    for k in range(1000):
        eye = rng.uniform(-50, 50, 3).astype(np.float32)
        look = (eye + rng.uniform(-20, 20, 3)).astype(np.float32)
        up = rng.uniform(-1, 1, 3).astype(np.float32)
        if k % 4 == 0:
            up = np.array([0, 1, 0], np.float32)
        fov = float(np.float32(rng.uniform(0.05, 3.0)))
        w, h = shapes[k % len(shapes)]
        cam = api.set_camera(eye, look, up, fov, w, h)
        got = np.concatenate([np.asarray(cam.eye_to_top_left, np.float32)[:3], np.asarray(cam.left_to_right, np.float32)[:3],
                              np.asarray(cam.top_to_bottom, np.float32)[:3], [np.float32(cam.pixel_size_inv)]]).astype(np.float32)
        want = stored[k]
        assert got.tobytes() == want.tobytes(), (k, got, want)       # NaNs included: byte comparison
