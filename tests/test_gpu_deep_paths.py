"""Deep paths on the GPU (tests/deep_scenes.py), bit for bit against the port (frames) and the restatements of the radiance and
transmittance queries: full rings with skipped spawns, samples of hundreds to thousands of trace rounds (far beyond the 64-entry round log
the round driver reads), launch-domain slices that finish hundreds of rounds apart, shadow loops that suspend and resume a hundred times in
one path, and scenes with more than 65 536 lights (the light index a suspended path resumes from does not fit 16 bits).  How deep each case
goes is asserted on the host by tests/test_deep_paths_host.py."""
import numpy as np
import pytest

from opencl_render_b200 import api
from tests import deep_scenes, helpers, port_radiance, port_rays
from tests.deep_scenes import case, stack_rays

pytestmark = pytest.mark.gpu
VARIANTS = [api.KERNEL_PIPE, api.KERNEL_SIMPLE]
FRAMES = ["panes8", "panes24", "panes100"]
ROUND_LOG = 64
_ref = {}


def _port(port, name, samples):
    if (name, samples) not in _ref:
        sc, cam, lists, _ = case(name)
        _ref[name, samples] = port.render(cam, lists, sc, samples, want_ids=True)
    return _ref[name, samples]


def _equal(img, want):
    return all(np.array_equal(img[c], want[c]) for c in range(3))


def _frame(name):
    sc, cam, lists, _ = case(name)
    ds = api.DeviceScene(sc, 0)
    return ds, api.DeviceFrame(ds, cam, lists)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("name", FRAMES + ["many_lights", "many_lights3"])
def test_frame_equals_port(name, variant, port):
    """S = 2: sample 1's first chunk of rounds is as long as sample 0 needed, far beyond the round log; rendered twice, so that the second
    call's first sample starts from the first call's round count."""
    ds, fr = _frame(name)
    want = _port(port, name, 2)
    for _ in range(2):
        _, launches, _ = fr.render(2, variant=variant)
        assert _equal(fr.read(), want) and np.array_equal(fr.primary_ids(), want[3]) and not fr.undefined_flags().any()
        if variant == api.KERNEL_PIPE and name in FRAMES:
            assert launches > 3 * ROUND_LOG   # every round is a logic, a setup and a trace launch
    fr.close()
    ds.close()


@pytest.mark.parametrize("name", FRAMES + ["many_lights3"])
def test_ahead_modes(name, port):
    ds, fr = _frame(name)
    want = _port(port, name, 2)
    try:
        for mode in (0, 1, 2):
            api.set_option("ahead", mode)
            fr.render(2)
            assert _equal(fr.read(), want) and np.array_equal(fr.primary_ids(), want[3]), mode
    finally:
        api.set_option("ahead", -1)
    fr.close()
    ds.close()


@pytest.mark.parametrize("slices", [1, 2, 4])
def test_slices(slices, port):
    """The stack covers only the middle rows: slices over the top or bottom rows finish in a few rounds, those over the stack hundreds
    of rounds later."""
    try:
        api.set_option("slices", slices)
        for name in ("panes8", "panes100"):
            ds, fr = _frame(name)
            want = _port(port, name, 2)
            _, launches, cnt = fr.render(2, count=True)
            assert _equal(fr.read(), want) and np.array_equal(fr.primary_ids(), want[3]), name
            assert launches > 3 * ROUND_LOG and cnt["segments"] > 0
            fr.close()
            ds.close()
    finally:
        api.set_option("slices", 0)


@pytest.mark.parametrize("variant", VARIANTS)
def test_sample_ranges_equal_the_whole_job(variant, port):
    for name in ("panes8", "panes100"):
        ds, fr = _frame(name)
        fr.render(2, variant=variant, samples=(0, 1))
        fr.render(2, variant=variant, samples=(1, 2))
        assert _equal(fr.read(), _port(port, name, 2)), name
        fr.close()
        ds.close()


def test_float_accumulation_one_sample(port):
    for name in FRAMES:
        ds, fr = _frame(name)
        fr.set_accumulation(api.ACCUMULATE_FLOAT)
        fr.render(1)
        assert _equal(fr.read(), _port(port, name, 1)), name
        assert (fr.read_accum()[..., 3] == 1.0).all()
        fr.close()
        ds.close()


@pytest.mark.parametrize("name", ["panes8", "panes100", "many_lights"])
def test_counters_equal_host_emulation(name, hostemu):
    sc, cam, lists, samples = case(name)
    _, _, _, want = helpers.hostemu_render(hostemu, cam, lists, sc, 1, threads=8)
    ds, fr = _frame(name)
    _, _, cnt = fr.render(1, variant=api.KERNEL_SIMPLE, count=True)
    for k in ("segments", "primCandidates", "gridRays", "cells", "cellsNonEmpty", "gridCandidates", "shadedHits", "occluderLookups"):
        assert cnt[k] == want[k], (k, cnt[k], want[k])
    _, _, cnt = fr.render(1, variant=api.KERNEL_PIPE, count=True)   # the counting instantiation of the logic kernel
    for k in ("segments", "shadedHits", "occluderLookups"):
        assert cnt[k] == want[k], (k, cnt[k], want[k])
    fr.close()
    ds.close()


@pytest.mark.parametrize("samples", [1, 3])
def test_radiance_from_inside_the_closed_box(samples):
    sc = deep_scenes.closed_box()
    ds = api.DeviceScene(sc, 0)
    o4, d4 = deep_scenes.box_rays(512, 1)
    base = 70_001
    rgb, ids, flags, cnt = ds.radiance(o4, d4, samples=samples, index_base=base, flags=True, count=True)
    ref, ref_flags, ref_cnt = port_radiance.shade_rays(sc, o4, d4, samples=samples, index_base=base)
    assert np.array_equal(_bits(rgb), _bits(ref[:, :3])) and np.array_equal(ids, _bits(ref[:, 3])) and np.array_equal(flags, ref_flags)
    for k in ("segments", "shadedHits", "gridRays"):
        assert cnt[k] == ref_cnt[k], (k, cnt[k], ref_cnt[k])
    ds.close()


@pytest.mark.parametrize("name", ["many_lights", "many_lights3"])
def test_radiance_with_many_lights(name):
    """Eye rays through the pixel centres of the deep scenes' camera, S = 2."""
    sc, cam, _, _ = case(name)
    ds = api.DeviceScene(sc, 0)
    ys, xs = np.mgrid[0:cam.height, 0:cam.width].astype(np.float32) + np.float32(0.5)
    d = cam.eye_to_top_left[:3] + xs.reshape(-1, 1) * cam.left_to_right[:3] + ys.reshape(-1, 1) * cam.top_to_bottom[:3]
    o4 = np.zeros((d.shape[0], 4), np.float32)
    o4[:, :3] = cam.eye[:3]
    d4 = np.full((d.shape[0], 4), np.inf, np.float32)
    d4[:, :3] = d
    rgb, ids, flags = ds.radiance(o4, d4, samples=2, index_base=9, flags=True)
    ref, ref_flags, _ = port_radiance.shade_rays(sc, o4, d4, samples=2, index_base=9)
    assert np.array_equal(_bits(rgb), _bits(ref[:, :3])) and np.array_equal(ids, _bits(ref[:, 3])) and np.array_equal(flags, ref_flags)
    assert (rgb > 0).any()
    ds.close()


@pytest.mark.parametrize("stop", [None, 57])
def test_transmittance_through_the_hundred_pane_stack(stop):
    sc = deep_scenes.panes(100, 60, 240, stop=stop)
    ds = api.DeviceScene(sc, 0)
    o4, d4 = stack_rays()
    att, last = ds.transmittance(o4, d4)
    ref = port_rays.transmit_rays(sc, o4, d4)
    assert np.array_equal(_bits(att), _bits(ref[:, :3])) and np.array_equal(last, _bits(ref[:, 3]))
    assert (last != api.NO_TRIANGLE).all()
    ds.close()
