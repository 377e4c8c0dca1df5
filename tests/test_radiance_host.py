"""Radiance queries without a GPU: the restatement of the reference's ring loop that the GPU tests compare against (tests/port_radiance.c)
is pinned to the port (oracle/raytrace_port.c, itself pinned to the reference), and DeviceScene.radiance rejects bad arguments before the
library is called."""
import numpy as np
import pytest

import port
from opencl_render_b200 import _lib, api
from tests import helpers, port_radiance, query_rays


@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_restatement_entered_from_the_camera_equals_the_port(name):
    """Whole frames at the case's own sample count: the restatement's planes and primary ids equal port_render_rows' bit for bit."""
    sc, cam, lists, samples = helpers.make_case(name)
    ref = port.render(cam, lists, sc, samples, want_ids=True)
    got, ids = port_radiance.shade_frame(cam, lists, sc, samples)
    for c in range(3):
        assert np.array_equal(got[c], ref[c]), (name, c, int((got[c] != ref[c]).sum()))
    assert np.array_equal(ids, ref[3])
    assert ref[0].any()


def test_restatement_of_caller_rays():
    """Eye rays through pixel centres: the first hit is the closest hit of the ray (the grid walk), untraced rays get the library's
    answers, and the seed rule makes a split job equal the whole one."""
    from tests import port_rays
    sc, cam, _, _ = helpers.make_case("soup_mirror_glass")
    o4, d4, excl = query_rays.all_families(sc, cam, n=128, seed=3, names=["eye", "bounce", "outside", "glass"])
    d4[:, 3] = np.inf
    out, flags, cnt = port_radiance.shade_rays(sc, o4, d4, excl, samples=3, index_base=7)
    hits = port_rays.walk_rays(sc, o4, d4, excl)
    assert np.array_equal(out[:, 3].view(np.uint32), hits[:, 0].view(np.uint32))
    assert (out[:, :3] >= 0).all() and (out[:, :3] <= 1).all() and out[:, :3].any()
    assert cnt["segments"] >= len(o4) and cnt["gridRays"] >= cnt["segments"]
    half = len(o4) // 2
    a, _, _ = port_radiance.shade_rays(sc, o4[:half], d4[:half], excl[:half], samples=3, index_base=7)
    b, _, _ = port_radiance.shade_rays(sc, o4[half:], d4[half:], excl[half:], samples=3, index_base=7 + half)
    assert np.array_equal(np.concatenate([a, b]).view(np.uint32), out.view(np.uint32))
    scr_o, scr_d, _ = query_rays.family("screened", sc, cam, n=12, seed=1)
    scr_d[:, 3] = np.where(np.arange(12) % 6 == 2, np.float32(5.0), scr_d[:, 3])   # NaN maxD -> finite maxD: refused as well
    res, _, c0 = port_radiance.shade_rays(sc, scr_o, scr_d)
    assert np.isnan(res[:, :3]).all() and (res[:, 3].view(np.uint32) == api.NO_TRIANGLE).all() and c0["segments"] == 0


class _FakeScene(api.DeviceScene):
    """A DeviceScene whose native calls must never happen: argument errors are raised before them."""

    def __init__(self, host=None):
        self.handle, self.device, self.host = None, 0, host

        class _NoLib:
            def __getattr__(self, name):
                raise AssertionError(f"native call {name} reached")
        self._lib = _NoLib()

    def close(self):
        pass


def test_radiance_argument_validation():
    s = _FakeScene()
    o3, d3 = np.zeros((4, 3), np.float32), np.ones((4, 3), np.float32)
    o4, d4 = np.zeros((4, 4), np.float32), np.ones((4, 4), np.float32)
    bad = [
        lambda: s.radiance(np.zeros((4, 2), np.float32), d3),             # wrong width
        lambda: s.radiance(np.zeros(4, np.float32), d3),                  # 1-D
        lambda: s.radiance(o3, np.ones((5, 3), np.float32)),              # ray counts differ
        lambda: s.radiance(o3.astype(np.int32), d3),                      # not floating point
        lambda: s.radiance(o3, d3, t_min=np.zeros(3)),                    # range of the wrong length
        lambda: s.radiance(o4, d4, t_min=0.5),                            # [N,4] carries its range already
        lambda: s.radiance(o3, d3, exclude=np.zeros(4, np.float32)),      # excluded ids not integers
        lambda: s.radiance(o3, d3, exclude=np.zeros(5, np.uint32)),       # ... of the wrong length
        lambda: s.radiance(o3, d3, samples=0),                            # at least one sample
        lambda: s.radiance(o3, d3, samples=1.5),
        lambda: s.radiance(o3, d3, index_base=-1),                        # seeds are unsigned 64-bit
        lambda: s.radiance(o3, d3, index_base=1 << 64),
        lambda: s.radiance(o3, d3, camera="pinhole"),                     # not a CameraSetup
    ]
    for b in bad:
        with pytest.raises(ValueError):
            b()


def test_radiance_needs_a_camera_on_a_bump_scene():
    sc, cam, _, _ = helpers.make_case("terrain_textured")
    assert (sc.mat_size[api.CH_BUMP::api.MATERIAL_CHANNEL_COUNT, 0] > 0).any()
    with pytest.raises(ValueError, match="camera"):
        _FakeScene(sc).radiance(np.zeros((2, 3), np.float32), np.ones((2, 3), np.float32))


def test_radiance_mixed_numpy_and_torch_inputs_are_refused():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("mixed inputs are told apart only for CUDA tensors")
    s = _FakeScene()
    with pytest.raises(ValueError):
        s.radiance(np.zeros((2, 3), np.float32), torch.ones((2, 3), device="cuda"))


def test_radiance_entry_fails_without_scene():
    lib = _lib.load()
    o = np.zeros((1, 4), np.float32)
    out = np.zeros((1, 4), np.float32)
    assert lib.oclr_scene_radiance(None, None, 1, o.ctypes.data, o.ctypes.data, None, 0, 1, out.ctypes.data, None, 0, 0, None, None) == 0
    assert "oclr_scene_radiance" in _lib.last_error() and "null scene" in _lib.last_error()


@pytest.mark.parametrize("eye, look_at, up", [((0, 9.0, -16.0), (0, 0.5, 0), (0, 1, 0)),      # config 2: looking down
                                               ((0, 4.4, -8), (0, 0, 0), (0, 1, 0)),
                                               ((3, -2, 5), (0, 1, 0), (0.2, 1, -0.3))])      # a tilted pole
def test_equirect_directions_are_a_level_panorama(eye, look_at, up):
    """render.py --projection equirect: the basis is orthonormal with --up as the pole, every direction is a unit vector, row y lies at
    latitude theta(y) and column x at longitude phi(x) (0 towards the look-at point)."""
    from opencl_render_b200 import render
    right, pole, forward = (v.astype(np.float64) for v in render.equirect_basis(eye, look_at, up))
    basis = np.stack([right, pole, forward])
    assert np.allclose(basis @ basis.T, np.eye(3), atol=1e-6)
    assert np.allclose(pole, np.asarray(up, np.float64) / np.linalg.norm(up), atol=1e-6)
    view = np.asarray(look_at, np.float64) - np.asarray(eye, np.float64)
    assert np.dot(view, forward) > 0 and abs(np.dot(view, right)) < 1e-5 * np.linalg.norm(view)
    cam = api.set_camera(eye, look_at, up, 0.9, 64, 32)   # right is the pinhole camera's left-to-right direction
    assert np.dot(right, cam.left_to_right[:3]) > 0
    w, h = 64, 32
    d = render.equirect_directions(render.equirect_basis(eye, look_at, up), w, h).astype(np.float64).reshape(h, w, 3)
    assert np.allclose(np.linalg.norm(d, axis=2), 1, atol=1e-6)
    theta = np.pi / 2 - np.pi * (np.arange(h) + 0.5) / h
    phi = 2 * np.pi * (np.arange(w) + 0.5) / w - np.pi
    assert np.allclose(np.arcsin(np.clip(d @ pole, -1, 1)), theta[:, None], atol=1e-5)
    assert np.allclose(np.arctan2(d @ right, d @ forward), phi[None, :], atol=1e-5)
    part = render.equirect_directions(render.equirect_basis(eye, look_at, up), w, h, (5, 9))   # a chunk of rows equals those rows
    assert np.array_equal(part.view(np.uint32), d.astype(np.float32).reshape(-1, 3)[5 * w:9 * w].view(np.uint32))


def test_equirect_basis_needs_a_horizontal_view():
    from opencl_render_b200 import render
    with pytest.raises(ValueError):
        render.equirect_basis((0, 5, 0), (0, 0, 0), (0, 1, 0))


@pytest.mark.parametrize("flag", [["--checkpoint", "job.npz"], ["--float-accum"], ["--pass-samples", "2"], ["--preview"]])
def test_equirect_refuses_the_pinhole_pass_options(flag, capsys):
    from opencl_render_b200 import render
    with pytest.raises(SystemExit):
        render.main(["config2", "--projection", "equirect", *flag])
    assert "not supported with --projection equirect" in capsys.readouterr().err
