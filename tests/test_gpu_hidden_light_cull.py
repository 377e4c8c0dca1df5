"""The hidden-side light cull of the logic kernel (rt_wavefront.cuh, GO_LIGHTS; oclr_set_option("cull_hidden_lights"), on by default).
A light on the side of a surface its segment does not see adds only to the face the colour step never reads, so its shadow ray (and the
re-traces through transparent occluders) is skipped.  The planes, ids and flags must be bit for bit those of a run that traces every shadow
ray, on every golden and deep case and on every path that runs the logic kernel; a scene whose every shadow ray is culled shows that the
cull really fires."""
import numpy as np
import pytest

from opencl_render_b200 import api, scenes
from tests import deep_scenes, helpers, query_rays

pytestmark = pytest.mark.gpu
MULTI_LIGHT = ["soup_lights_sun_last", "soup_lights_omni_last", "soup_all_light_types", "many_lights3", "panes8"]


@pytest.fixture
def cull():
    yield lambda on: api.set_option("cull_hidden_lights", on)
    api.set_option("cull_hidden_lights", 1)


def _case(name):
    return deep_scenes.case(name) if name in deep_scenes.CASES else helpers.make_case(name)


def _open(name):
    sc, cam, lists, samples = _case(name)
    ds = api.DeviceScene(sc, 0)
    return ds, api.DeviceFrame(ds, cam, lists), samples


def _outputs(fr):
    return (*fr.read(), fr.primary_ids(), fr.undefined_flags())


def _equal(a, b):
    return len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _off_on(cull, run):
    out = []
    for on in (0, 1):
        cull(on)
        out.append(run())
    return out


@pytest.mark.parametrize("name", helpers.CASE_NAMES + list(deep_scenes.CASES))
def test_frames_equal_without_cull(name, cull):
    """Every golden and deep case, at its own sample count and at S = 1 or S = 2."""
    ds, fr, samples = _open(name)
    for s in sorted({samples, 1 if samples > 1 else 2}):
        def run():
            fr.render(s)
            return _outputs(fr)
        off, on = _off_on(cull, run)
        assert _equal(off, on), (name, s)
    fr.close()
    ds.close()


@pytest.mark.parametrize("slices", [1, 2])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_slices_ahead_modes_and_bands(mode, slices, cull):
    """Several lights per hit: with the last light culled, a path finishes its segment and queues the next closest hit in the same round,
    so the cull never needs more rounds than tracing every shadow ray (the second render enqueues exactly the rounds the first needed)."""
    try:
        api.set_option("ahead", mode)
        api.set_option("slices", slices)
        for name in MULTI_LIGHT:
            ds, fr, samples = _open(name)
            cam = fr.camera

            def run():
                fr.render(samples)
                whole = _outputs(fr)
                out = tuple(np.zeros((cam.height, cam.width), np.uint16) for _ in range(3))
                for rank in range(2):
                    fr.render_bands(samples, 16, rank, 2)
                    for rows in api.band_partition(cam.height, rank, 2, band_rows=16):
                        fr.read(rows=rows, out=out)
                fr.render(1)
                fr.render(1)   # one sample: enqueues exactly the rounds the first call needed, three launches each
                return whole, out, fr.last_launches

            (off, off_bands, off_launches), (on, on_bands, on_launches) = _off_on(cull, run)
            assert _equal(off, on) and _equal(off_bands, on_bands) and _equal(on_bands, on[:3]), name
            assert on_launches <= off_launches, (name, off_launches, on_launches)
            fr.close()
            ds.close()
    finally:
        api.set_option("ahead", -1)
        api.set_option("slices", 0)


@pytest.mark.parametrize("name", ["soup_lights_sun_last", "soup_mirror_glass", "spheres_mirror", "panes8", "many_lights3"])
def test_float_accumulation_and_progressive(name, cull):
    ds, fr, samples = _open(name)
    s = max(samples, 2)

    def run():
        fr.set_accumulation(api.ACCUMULATE_FLOAT)
        fr.render(s)
        acc = fr.read_accum()
        planes = _outputs(fr)
        fr.set_accumulation(api.ACCUMULATE_REFERENCE_16BIT)
        for k in range(s):   # one call per sample
            fr.render(s, samples=(k, k + 1))
        return (_bits(acc), *planes, *_outputs(fr))

    off, on = _off_on(cull, run)
    assert _equal(off, on), name
    fr.close()
    ds.close()


@pytest.mark.parametrize("name", MULTI_LIGHT[:3] + ["spheres_mirror", "terrain_textured"])
def test_radiance_equals_without_cull(name, cull):
    sc, cam, _, _ = _case(name)
    ds = api.DeviceScene(sc, 0)
    o4, d4, ex = query_rays.all_families(sc, cam, 256, seed=7)
    d4[:, 3] = np.inf

    def run():
        rgb, ids, flags = ds.radiance(o4, d4, exclude=ex, samples=2, index_base=11, camera=cam, flags=True)
        return _bits(rgb), ids, flags

    off, on = _off_on(cull, run)
    assert _equal(off, on)
    ds.close()


def test_radiance_from_inside_the_closed_box(cull):
    ds = api.DeviceScene(deep_scenes.closed_box(), 0)
    o4, d4 = deep_scenes.box_rays(2048, 4)

    def run():
        rgb, ids, flags = ds.radiance(o4, d4, samples=3, index_base=5, flags=True)
        return _bits(rgb), ids, flags

    off, on = _off_on(cull, run)
    assert _equal(off, on)
    ds.close()


def test_cull_fires_on_a_quad_seen_from_below(cull):
    """One quad with a black COLOR channel, seen from below, lit from above: every shadow ray would leave on the unseen side, and with a
    black colour and no REFLECTION / TRANSPARENCY channel no segment is spawned.  With the cull no ray is traced at all."""
    atlas = scenes.MaterialAtlas()
    mat = atlas.add(color=(0, 0, 0))
    corners, tris = deep_scenes._quad((0.0, 0.0, 0.0), (6.0, 0.0, 0.0), (0.0, 0.0, 6.0))
    vertex = np.array(corners, np.float32)
    tri_idx = np.array(tris, np.int32)
    sc = scenes._scene("quad_from_below", vertex, tri_idx, np.full(2, mat, np.int32), np.tile(deep_scenes._UV, (2, 1, 1)),
                       scenes._flat_normals(vertex, tri_idx), atlas, [dict(type=api.LIGHT_SPOT, pos=(0.5, 5.0, 0.3), colour=(1, 1, 1))])
    api.scene_triangle_list(sc, 16)
    cam = api.set_camera((0.2, -3.0, 0.1), (0.0, 0.0, 0.0), (0.0, 0.0, 1.0), 0.8, 512, 512)
    ds = api.DeviceScene(sc, 0)
    fr = api.DeviceFrame(ds, cam, api.camera_triangle_list(cam, sc))
    outs, traced = [], []
    for on in (0, 1):
        cull(on)
        fr.render(1)
        outs.append(_outputs(fr))
        traced.append(fr.last_trace_launches)
    assert (outs[0][3] != api.NO_TRIANGLE).all()   # the quad fills the view
    assert _equal(outs[0], outs[1])
    assert traced == [1, 0], traced
    fr.close()
    ds.close()
