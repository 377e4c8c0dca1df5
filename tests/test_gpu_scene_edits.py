"""Edits of a resident scene (DeviceScene.update / update_geometry) and of a frame's camera (DeviceFrame.set_camera): after an edit the
scene is byte for byte, and renders and answers queries bit for bit, what a scene created from the merged arrays is and does."""
import dataclasses

import numpy as np
import pytest

from opencl_render_b200 import api, scenes
from tests import helpers
from tests.test_gpu_parity import GOLDEN

pytestmark = pytest.mark.gpu


def _copy(sc, **kw):
    return dataclasses.replace(sc, **{k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in kw.items()})


def _packed(ds):
    return [ds.debug_read(i) for i in range(7)] + [ds.device_bytes]


def _assert_packed_equal(a, b):
    for i, (x, y) in enumerate(zip(a, b)):
        assert np.array_equal(x, y), f"packed array {i} differs" if i < 7 else f"device bytes {x} != {y}"


def _scene(sc):
    return api.DeviceScene(sc, 0, axes_div=sc.axes_div)


def _render(fr, samples):
    fr.render(samples)
    return fr.read(), fr.primary_ids(), fr.undefined_flags()


def _assert_render_equal(a, b):
    for x, y, what in zip(a[0], b[0], "rgb"):
        assert np.array_equal(x, y), f"plane {what} differs"
    assert np.array_equal(a[1], b[1]), "primary ids differ"
    assert np.array_equal(a[2], b[2]), "flags differ"


def _fresh(sc, cam, samples, lists=None):
    ds = api.DeviceScene(sc, 0)
    fr = api.DeviceFrame(ds, cam, lists)
    out = _render(fr, samples), _packed(ds)
    fr.close()
    ds.close()
    return out


def _assert_golden(name, img, flags):
    gold = np.load(GOLDEN / f"{name}.npz")
    res = helpers.compare_rgb(img, (gold["r"], gold["g"], gold["b"]), mask=(flags == 0))
    assert res["diff_pixels"] == 0, res
    assert helpers.compare_rgb(img, (gold["r"], gold["g"], gold["b"]))["diff_pixels"] <= int(flags.sum())


def _other_lights(sc):
    lt, pos, dr, col, rad, half = scenes._lights([helpers._SUN, helpers._OMNI] if sc.light_count != 2 else [helpers._AREA])
    return _copy(sc, light_type=lt, light_pos=pos, light_dir=dr, light_colour=col, light_radius=rad, light_half=half).normalise()


def _other_materials(sc):
    return _copy(sc, textures=(255 - sc.textures).astype(np.uint8))


def _other_geometry(sc, axes):
    """The case's topology on shrunken, shifted vertices, with a device-built grid at another resolution."""
    v = sc.vertex.copy()
    v[:, :3] = v[:, :3] * 0.6 + np.float32(0.25)
    out = _copy(sc, vertex=v, axes_div=axes)
    out.box_min = out.grid_start = out.grid_list = None
    return out


def _start_scene(sc, part):
    other_axes = 32 if sc.axes_div != 32 else 16
    if part == "lights":
        return _other_lights(sc)
    if part == "materials":
        return _other_materials(sc)
    if part in ("geometry_grid", "geometry_device_grid"):
        return _other_geometry(sc, other_axes)
    return _other_materials(_other_lights(_other_geometry(sc, other_axes)))


@pytest.mark.parametrize("part", ["lights", "materials", "geometry_grid", "geometry_device_grid", "all"])
@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_edit_equals_a_fresh_scene_and_the_golden_planes(name, part):
    sc, cam, lists, samples = helpers.make_case(name)
    start = _start_scene(sc, part)
    ds = _scene(start)
    fr = api.DeviceFrame(ds, cam)   # device-built lists: entry for entry the host builder's
    _render(fr, samples)
    if part == "lights":
        ds.update(sc, lights=True)
    elif part == "materials":
        ds.update(sc, materials=True)
    elif part == "geometry_grid":
        ds.update(sc, geometry=True)
    elif part == "geometry_device_grid":
        ds.update_geometry(sc.vertex, sc.tri_idx, sc.tri_mat, sc.tri_uv, sc.tri_normal, axes_div=sc.axes_div)
    else:
        ds.update(sc, lights=True, materials=True, geometry=True)
    edited = _render(fr, samples)
    fresh, packed = _fresh(sc, cam, samples)
    _assert_packed_equal(_packed(ds), packed)
    _assert_render_equal(edited, fresh)
    _assert_golden(name, edited[0], edited[2])
    assert ds.host.axes_div == sc.axes_div and np.array_equal(ds.host.textures, sc.textures)
    if part.startswith("geometry") or part == "all":
        assert np.array_equal(fr.camera_lists().list, lists.list)
    fr.close()
    ds.close()


def test_light_counts_4_1_0_and_all_types():
    sc, cam, _, samples = helpers.make_case("soup_all_light_types")
    steps = [[helpers._OMNI, helpers._SPOT, helpers._AREA, helpers._SUN], [helpers._SPOT], [], helpers._ALL_TYPES]
    first = helpers._with_lights(_copy(sc), steps[0])
    ds = _scene(first)
    fr = api.DeviceFrame(ds, cam)
    _render(fr, samples)
    for entries in steps[1:]:
        target = helpers._with_lights(_copy(sc), entries)
        ds.update(target, lights=True)
        edited = _render(fr, samples)
        fresh, packed = _fresh(target, cam, samples)
        _assert_packed_equal(_packed(ds), packed)
        _assert_render_equal(edited, fresh)
    _assert_golden("soup_all_light_types", edited[0], edited[2])
    fr.close()
    ds.close()


def _black_mirrors(sc):
    """Every reflection and transparency channel replaced by one black texel appended to the atlas: a 2-slot ring."""
    tex = np.concatenate([sc.textures, np.zeros((1, 4), np.uint8)])
    size, start = sc.mat_size.copy(), sc.mat_start.copy()
    for m in range(sc.material_count):
        for ch in (api.CH_REFLECTION, api.CH_TRANSPARENCY):
            size[5 * m + ch] = (1, 1)
            start[5 * m + ch] = sc.textures.shape[0]
    return _copy(sc, textures=tex, mat_size=size, mat_start=start)


def test_ring_depth_follows_a_materials_edit():
    sc, cam, _, samples = helpers.make_case("spheres_mirror")
    paths = cam.width * ((cam.height + 7) // 8 * 8)
    ds = _scene(_black_mirrors(sc))
    fr = api.DeviceFrame(ds, cam)
    _render(fr, samples)
    assert fr.state_bytes / paths < 520
    ds.update(sc, materials=True)
    edited = _render(fr, samples)
    assert fr.state_bytes / paths > 980
    _assert_golden("spheres_mirror", edited[0], edited[2])
    _assert_render_equal(edited, _fresh(sc, cam, samples)[0])
    ds.update(_black_mirrors(sc), materials=True)
    back = _render(fr, samples)
    assert fr.state_bytes / paths < 520
    _assert_render_equal(back, _fresh(_black_mirrors(sc), cam, samples)[0])
    fr.close()
    ds.close()


def test_geometry_from_torch_equals_geometry_from_numpy():
    torch = pytest.importorskip("torch")
    sc, cam, _, samples = helpers.make_case("soup_mirror_glass")
    dev = torch.device("cuda", 0)
    results = []
    for kind in ("numpy", "torch", "torch_grid"):
        ds = _scene(_other_geometry(sc, 16))
        fr = api.DeviceFrame(ds, cam)
        _render(fr, samples)
        arrays = [sc.vertex, sc.tri_idx, sc.tri_mat, sc.tri_uv, sc.tri_normal]
        grid = None
        if kind != "numpy":
            arrays = [torch.from_numpy(a).to(dev) for a in arrays]
        if kind == "torch_grid":
            grid = tuple(torch.from_numpy(a).to(dev) for a in (sc.box_min, sc.grid_start, sc.grid_list))
        ds.update_geometry(*arrays, grid=grid, axes_div=None if grid else sc.axes_div)
        results.append((_packed(ds), _render(fr, samples)))
        fr.close()
        ds.close()
    for packed, img in results[1:]:
        _assert_packed_equal(packed, results[0][0])
        _assert_render_equal(img, results[0][1])
    _assert_golden("soup_mirror_glass", results[0][1][0], results[0][1][2])


def test_camera_moves_through_the_sweep():
    sc, cam0, lists0, samples = helpers.make_case("terrain")
    ds = api.DeviceScene(sc, 0)
    moved_dev = api.DeviceFrame(ds, cam0)
    moved_host = api.DeviceFrame(ds, cam0, lists0)
    for m in scenes.sweep_cameras(sc, 4):
        cam = api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], cam0.width, cam0.height)
        lists = api.camera_triangle_list(cam, sc)
        moved_dev.set_camera(cam)
        moved_host.set_camera(cam, lists)
        fresh = api.DeviceFrame(ds, cam)
        want = _render(fresh, samples)
        fresh.close()
        _assert_render_equal(_render(moved_dev, samples), want)
        _assert_render_equal(_render(moved_host, samples), want)
        got = moved_dev.camera_lists()
        assert np.array_equal(got.start, lists.start) and np.array_equal(got.end, lists.end) and np.array_equal(got.list, lists.list)
    # the device-built lists follow a geometry edit
    other = _other_geometry(sc, 64)
    ds.update(other, geometry=True)
    got, want = moved_dev.camera_lists(), api.camera_triangle_list(moved_dev.camera, other)
    assert np.array_equal(got.start, want.start) and np.array_equal(got.end, want.end) and np.array_equal(got.list, want.list)
    with pytest.raises(ValueError):
        moved_dev.set_camera(api.set_camera((0, 5, -9), (0, 0, 0), (0, 1, 0), 0.8, cam0.width + 8, cam0.height))
    moved_dev.close()
    moved_host.close()
    ds.close()


def test_caller_lists_are_refused_after_a_geometry_edit():
    sc, cam, lists, samples = helpers.make_case("soup")
    small = scenes.soup(60, seed=8).normalise()   # fewer triangles: the old lists name triangles that no longer exist
    small.tri_mat = np.minimum(small.tri_mat, sc.material_count - 1).astype(np.int32)
    ds = api.DeviceScene(sc, 0)
    fr = api.DeviceFrame(ds, cam, lists)
    _render(fr, samples)
    ds.update(small, geometry=True)
    with pytest.raises(api.OclrError, match="geometry changed"):
        fr.render(samples)
    with pytest.raises(api.OclrError, match="geometry changed"):
        fr.camera_lists()
    merged = _copy(sc, vertex=small.vertex, tri_idx=small.tri_idx, tri_mat=small.tri_mat, tri_uv=small.tri_uv, tri_normal=small.tri_normal,
                   axes_div=sc.axes_div)
    merged.box_min = merged.grid_start = merged.grid_list = None
    new_lists = api.camera_triangle_list(cam, merged)
    fr.set_camera(cam, new_lists)
    _assert_render_equal(_render(fr, samples), _fresh(merged, cam, samples, new_lists)[0])
    fr.close()
    ds.close()


def _rays(sc, cam, n=4096, seed=5):
    rng = np.random.default_rng(seed)
    o = np.tile(cam.eye[:3], (n, 1)).astype(np.float32)
    d = (np.asarray(sc.meta["camera"]["look_at"], np.float32) - cam.eye[:3] + rng.normal(0, 2.0, (n, 3))).astype(np.float32)
    return o, d


def _multi_material_case():
    for name in helpers.CASE_NAMES:
        sc, cam, lists, samples = helpers.make_case(name)
        if sc.material_count >= 2 and int(sc.tri_mat.max()) == sc.material_count - 1:
            return name, sc, cam, lists, samples
    pytest.fail("no case uses its last material")


def test_failed_updates_leave_the_scene_untouched():
    torch = pytest.importorskip("torch")
    name, sc, cam, lists, samples = _multi_material_case()
    ds = api.DeviceScene(sc, 0)
    fr = api.DeviceFrame(ds, cam, lists)
    before, packed = _render(fr, samples), _packed(ds)
    bad_idx = sc.tri_idx.copy()
    bad_idx[len(bad_idx) // 2, 1] = sc.vertex_count + 7
    M = sc.material_count - 1
    attempts = [
        ("VertexIndex out of range", lambda: ds.update(_copy(sc, tri_idx=bad_idx), geometry=True)),
        ("VertexIndex out of range", lambda: ds.update_geometry(sc.vertex, bad_idx, sc.tri_mat, sc.tri_uv, sc.tri_normal, axes_div=16)),
        ("VertexIndex out of range", lambda: ds.update_geometry(*[torch.from_numpy(a).cuda() for a in
                                                           (sc.vertex, bad_idx, sc.tri_mat, sc.tri_uv, sc.tri_normal)], axes_div=16)),
        ("VertexIndex out of range", lambda: ds.update_geometry(*[torch.from_numpy(a).cuda() for a in
                                                           (sc.vertex, bad_idx, sc.tri_mat, sc.tri_uv, sc.tri_normal)],
                                                          grid=tuple(torch.from_numpy(a).cuda() for a in (sc.box_min, sc.grid_start, sc.grid_list)))),
        ("triangleMaterialId out of range", lambda: ds.update(_copy(sc, mat_size=sc.mat_size[:5 * M], mat_start=sc.mat_start[:5 * M + 1]),
                                                              materials=True)),
        ("outside the texture atlas", lambda: ds.update(_copy(sc, mat_start=np.where(sc.mat_size[:, 0] > 0, sc.textures.shape[0],
                                                                                       sc.mat_start[:-1]).tolist() + [sc.mat_start[-1]]),
                                                        materials=True)),
        ("light arrays missing", lambda: ds.update(_copy(sc, light_radius=np.zeros(0, np.float32)), lights=True)),
    ]
    for msg, attempt in attempts:
        with pytest.raises(api.OclrError, match=msg):
            attempt()
        _assert_packed_equal(_packed(ds), packed)
        _assert_render_equal(_render(fr, samples), before)
    fr.close()
    ds.close()


def test_queries_on_an_edited_scene_equal_a_fresh_scene():
    sc, cam, _, _ = helpers.make_case("soup_mirror_glass")
    start = _other_materials(_other_lights(_other_geometry(sc, 16)))
    ds = _scene(start)
    o, d = _rays(sc, cam)
    ds.intersect(o, d)
    ds.update(sc, lights=True, materials=True, geometry=True)
    fresh = api.DeviceScene(_copy(sc), 0)
    for a, b in ((ds.intersect(o, d), fresh.intersect(o, d)), (ds.transmittance(o, d), fresh.transmittance(o, d)),
                 (ds.radiance(o, d, samples=2, camera=cam), fresh.radiance(o, d, samples=2, camera=cam))):
        for x, y in zip(a, b):
            assert np.array_equal(np.ascontiguousarray(x).view(np.uint8), np.ascontiguousarray(y).view(np.uint8))
    # a BUMP channel added by an edit needs a camera; removing it again lifts that
    bump_size = sc.mat_size.copy()
    bump_size[api.CH_BUMP] = sc.mat_size[api.CH_COLOR]
    bump_start = sc.mat_start.copy()
    bump_start[api.CH_BUMP] = sc.mat_start[api.CH_COLOR]
    if bump_size[api.CH_BUMP, 0] == 0:
        bump_size[api.CH_BUMP] = (1, 1)
        bump_start[api.CH_BUMP] = 0
    ds.update(_copy(sc, mat_size=bump_size, mat_start=bump_start), materials=True)
    with pytest.raises((ValueError, api.OclrError)):
        ds.radiance(o, d)
    ds.update(sc, materials=True)
    a, b = ds.radiance(o, d), fresh.radiance(o, d)
    assert all(np.array_equal(np.ascontiguousarray(x).view(np.uint8), np.ascontiguousarray(y).view(np.uint8)) for x, y in zip(a, b))
    fresh.close()
    ds.close()
