"""Deep paths without a GPU (tests/deep_scenes.py): the restatement of the ring loop that the GPU tests compare against
(tests/port_radiance.c) and the host emulation of the device arithmetic (tests/hostemu, rt_core.h) equal the port on scenes whose paths
fill the ring, need hundreds to thousands of sequential traces and walk shadow loops over a hundred blockers, and on scenes with more
than 65 536 lights.  Each case's depth is measured on the port's control flow (tests/port_depth.c) and asserted, so that a change to a
scene cannot make it shallow without a test failing."""
import numpy as np
import pytest

import port
from opencl_render_b200 import api
from tests import deep_scenes, helpers, port_depth, port_radiance, port_rays
from tests.deep_scenes import CASES, case, stack_rays


@pytest.mark.parametrize("name", list(CASES))
def test_restatement_entered_from_the_camera_equals_the_port(name):
    sc, cam, lists, samples = case(name)
    ref = port.render(cam, lists, sc, samples, want_ids=True)
    assert ref[0].any()
    got, ids = port_radiance.shade_frame(cam, lists, sc, samples)
    for c in range(3):
        assert np.array_equal(got[c], ref[c]), (name, c, int((got[c] != ref[c]).sum()))
    assert np.array_equal(ids, ref[3])
    # the depth counts come from the same control flow: its planes and ids equal the port's too
    got, ids, cnt = port_depth.depth_frame(cam, lists, sc, samples)
    for c in range(3):
        assert np.array_equal(got[c], ref[c]), (name, c, int((got[c] != ref[c]).sum()))
    assert np.array_equal(ids, ref[3])
    ring_full, traces, segments = CASES[name][4:]
    assert cnt["ringFull"] >= ring_full, cnt                # panes: the ring fills and spawns are skipped
    assert cnt["longestWalks"] >= traces, cnt               # panes: far more sequential traces than the 64-entry round log holds
    assert cnt["longestSegments"] >= segments, cnt          # panes: branching chains, not one mirror chain of the maximum depth


@pytest.mark.parametrize("name", list(CASES))
def test_host_emulation_equals_the_port(name, hostemu):
    sc, cam, lists, samples = case(name)
    ref = port.render(cam, lists, sc, samples, want_ids=True)
    img, ids, flags, _ = helpers.hostemu_render(hostemu, cam, lists, sc, samples, threads=8)
    for c in range(3):
        assert np.array_equal(img[c], ref[c]), (name, c, int((img[c] != ref[c]).sum()))
    assert np.array_equal(ids, ref[3]) and not flags.any()


def test_many_light_scenes_have_lights_past_16_bits():
    sc = case("many_lights")[0]
    assert sc.light_count == 65537 and sc.light_type[65536] != deep_scenes._QUIET and (sc.light_type[:65536] == deep_scenes._QUIET).all()
    sc = case("many_lights3")[0]
    assert sc.light_count == 65538 and (sc.light_type[65535:] != deep_scenes._QUIET).all()
    assert (sc.light_type[:65535] == deep_scenes._QUIET).all()


@pytest.mark.parametrize("samples", [1, 3])
def test_rays_inside_the_closed_box_stay_inside(samples):
    """Every ray from inside meets a wall, and the longest ray-sample needs more sequential traces than the round log holds."""
    sc = deep_scenes.closed_box()
    o4, d4 = deep_scenes.box_rays(512, 1)
    out, flags, _ = port_radiance.shade_rays(sc, o4, d4, samples=samples, index_base=40_000)
    assert (out[:, 3].view(np.uint32) != api.NO_TRIANGLE).all()
    assert not flags.any() and (out[:, :3] > 0).all()
    got, cnt = port_depth.depth_rays(sc, o4, d4, samples=samples, index_base=40_000)
    assert np.array_equal(got.view(np.uint32), out.view(np.uint32))
    assert cnt["longestWalks"] > 150 and cnt["longestSegments"] > 40, cnt


def test_transmittance_through_the_hundred_pane_stack():
    """Shadow rays through all 100 panes: the attenuation is the product of 100 texels and the last blocker is a triangle of the last
    pane; with a pane whose texel has a zero green channel the loop stops there, with the attenuation at that pane."""
    o4, d4 = stack_rays()
    t = np.float32(240) / np.float32(255)
    sc = deep_scenes.panes(100, 60, 240)
    ref = port_rays.transmit_rays(sc, o4, d4)
    assert np.allclose(ref[:, :3], float(t) ** 100, rtol=1e-4)
    assert np.isin(ref[:, 3].view(np.uint32), [198, 199]).all()   # pane k is triangles 2k and 2k + 1
    sc = deep_scenes.panes(100, 60, 240, stop=57)
    ref = port_rays.transmit_rays(sc, o4, d4)
    assert (ref[:, 1] == 0).all() and np.allclose(ref[:, [0, 2]], float(t) ** 58, rtol=1e-4)
    assert np.isin(ref[:, 3].view(np.uint32), [114, 115]).all()
