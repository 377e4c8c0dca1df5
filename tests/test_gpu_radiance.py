"""Radiance queries on a resident scene (DeviceScene.radiance, oclr_scene_radiance) against the restatement of the reference's ring loop
(tests/port_radiance.c, pinned to the port by tests/test_radiance_host.py), bit for bit: colours, first hits, flags and counters."""
import ctypes as C

import numpy as np
import pytest

from opencl_render_b200 import _lib, api, render
from tests import helpers, port_radiance, query_rays

pytestmark = pytest.mark.gpu
NONE = query_rays.NONE
FAMILIES = [f for f in query_rays.TRACED_FAMILIES] + query_rays.SCREENED_FAMILIES + ["finite_max", "infinite_min"]

_scenes = {}


def _scene(name):
    if name not in _scenes:
        sc, cam, lists, samples = helpers.make_case(name)
        _scenes[name] = (sc, cam, api.DeviceScene(sc))
    return _scenes[name]


def _rays(sc, cam, n=256, seed=21):
    """The query families with maxD = +inf (ring segments have no far limit), plus rays with a finite maxD, which are refused, and rays with
    minD = +inf, which meet nothing."""
    parts = []
    for f in FAMILIES:
        o4, d4, ex = query_rays.family("eye" if f in ("finite_max", "infinite_min") else f, sc, cam, n, seed)
        if f == "finite_max":
            d4[:, 3] = np.float32(1.0) + np.arange(n, dtype=np.float32)
        elif f == "infinite_min":
            o4[:, 3] = np.inf
            d4[:, 3] = np.inf
        elif f not in query_rays.SCREENED_FAMILIES:
            d4[:, 3] = np.inf
        parts.append((o4, d4, ex))
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(3))


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _check(o4, d4, rgb, ids, ref, flags=None, ref_flags=None):
    assert np.array_equal(ids, _bits(ref[:, 3]))
    nan = np.isnan(ref[:, :3])
    assert np.array_equal(np.isnan(rgb), nan)
    assert np.array_equal(_bits(rgb)[~nan], _bits(ref[:, :3])[~nan])
    scr = query_rays.is_screened(o4, d4) | (d4[:, 3] != np.inf)
    assert nan[scr].all() and not nan[~scr].any()
    empty = ~scr & ((o4[:, 3] == np.inf) | (d4[:, :3] == 0).all(1))   # meets nothing: black, no hit
    assert (rgb[empty] == 0).all() and (ids[empty] == NONE).all()
    if flags is not None:
        assert np.array_equal(flags, ref_flags)


@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_radiance_equals_restatement(name):
    sc, cam, ds = _scene(name)
    o4, d4, excl = _rays(sc, cam)
    rgb, ids, flags = ds.radiance(o4, d4, exclude=excl, camera=cam, flags=True)
    ref, ref_flags, _ = port_radiance.shade_rays(sc, o4, d4, excl, camera=cam)
    _check(o4, d4, rgb, ids, ref, flags, ref_flags)
    assert (ids != NONE).any() and (rgb[~np.isnan(rgb)] > 0).any()


@pytest.mark.parametrize("samples", [1, 3])
def test_samples_and_index_base(samples):
    sc, cam, ds = _scene("soup_mirror_glass")
    o4, d4, excl = _rays(sc, cam, n=128, seed=22)
    base = 1_000_003
    rgb, ids = ds.radiance(o4, d4, exclude=excl, samples=samples, index_base=base, camera=cam)
    ref, _, _ = port_radiance.shade_rays(sc, o4, d4, excl, samples=samples, index_base=base, camera=cam)
    _check(o4, d4, rgb, ids, ref)
    half = len(o4) // 2   # a job split across calls gives the same bits
    a = ds.radiance(o4[half:], d4[half:], exclude=excl[half:], samples=samples, index_base=base + half, camera=cam)
    assert np.array_equal(_bits(a[0]), _bits(rgb[half:])) and np.array_equal(a[1], ids[half:])


def test_bump_scene_camera_and_flags():
    sc, cam, ds = _scene("terrain_textured")
    o4, d4, excl = _rays(sc, cam, n=256, seed=23)
    short = query_rays.family("bounce", sc, cam, 512, 24)   # directions shorter than a pixel step: the helper ray may miss the plane
    so4, sd4, sex = short
    sd4[:, :3] *= np.float32(1e-3)
    sd4[:, 3] = np.inf
    o4, d4, excl = np.concatenate([o4, so4]), np.concatenate([d4, sd4]), np.concatenate([excl, sex])
    rgb, ids, flags = ds.radiance(o4, d4, exclude=excl, camera=cam, flags=True)
    ref, ref_flags, _ = port_radiance.shade_rays(sc, o4, d4, excl, camera=cam)
    _check(o4, d4, rgb, ids, ref, flags, ref_flags)
    assert ref_flags.any()
    lib = _lib.load()
    out = np.zeros((len(o4), 4), np.float32)
    assert lib.oclr_scene_radiance(ds.handle, None, len(o4), o4.ctypes.data, d4.ctypes.data, None, 0, 1, out.ctypes.data, None,
                                   api.QUERY_HOST_MEMORY, 0, None, None) == 0
    assert "oclr_scene_radiance" in _lib.last_error() and "camera" in _lib.last_error()
    # no bump channel: the camera is not needed and not read
    sc2, cam2, ds2 = _scene("soup")
    o2, d2, e2 = _rays(sc2, cam2, n=64, seed=25)
    with_cam = ds2.radiance(o2, d2, exclude=e2, camera=cam2)
    without = ds2.radiance(o2, d2, exclude=e2)
    assert np.array_equal(_bits(with_cam[0]), _bits(without[0])) and np.array_equal(with_cam[1], without[1])


def test_ahead_modes_agree():
    sc, cam, ds = _scene("spheres_mirror")
    o4, d4, excl = _rays(sc, cam, n=128, seed=26)
    res = []
    try:
        for m in (0, 1, 2):
            api.set_option("ahead", m)
            res.append(ds.radiance(o4, d4, exclude=excl, samples=2, camera=cam))
    finally:
        api.set_option("ahead", -1)
    for r in res[1:]:
        assert np.array_equal(_bits(r[0]), _bits(res[0][0])) and np.array_equal(r[1], res[0][1])
    ref, _, _ = port_radiance.shade_rays(sc, o4, d4, excl, samples=2, camera=cam)
    _check(o4, d4, res[0][0], res[0][1], ref)


def test_host_and_device_memory_agree():
    torch = pytest.importorskip("torch")
    sc, cam, ds = _scene("soup_mirror_glass")
    o4, d4, excl = _rays(sc, cam, n=128, seed=27)
    dev = torch.device("cuda", ds.device)
    s = torch.cuda.Stream(device=dev)
    to, td, te = (torch.from_numpy(a).to(dev) for a in (o4, d4, excl.view(np.int32)))
    torch.cuda.synchronize(dev)
    h = ds.radiance(o4, d4, exclude=excl, samples=2, camera=cam, flags=True)
    g = ds.radiance(to, td, exclude=te, samples=2, camera=cam, flags=True, stream=s)
    s.synchronize()
    assert isinstance(g[0], torch.Tensor)
    assert np.array_equal(_bits(h[0]), _bits(g[0].cpu().numpy()))
    assert np.array_equal(h[1], g[1].cpu().numpy()) and np.array_equal(h[2], g[2].cpu().numpy())
    traced = d4[:, 3] == np.inf   # [N,3] inputs (maxD = +inf) give the same as the [N,4] layout
    h3 = ds.radiance(o4[traced, :3], d4[traced, :3], t_min=o4[traced, 3], exclude=excl[traced], samples=2, camera=cam)
    assert np.array_equal(_bits(h3[0]), _bits(h[0][traced])) and np.array_equal(h3[1], h[1][traced])
    g3 = ds.radiance(to[:, :3], td[:, :3], t_min=to[:, 3], exclude=te, samples=2, camera=cam)
    torch.cuda.synchronize(dev)
    same = traced & ~query_rays.is_screened(o4, d4)
    assert np.array_equal(_bits(g3[0].cpu().numpy()[same]), _bits(h[0][same]))


@pytest.mark.parametrize("count", [0, 1, 31, 33, api.RADIANCE_BATCH + 1])
def test_counts(count):
    sc, cam, ds = _scene("soup")
    rng = np.random.default_rng(count)
    base_o, base_d, base_e = _rays(sc, cam, n=128, seed=28)
    pick = rng.integers(0, len(base_o), count)
    o4, d4, excl = base_o[pick], base_d[pick], base_e[pick]
    rgb, ids = ds.radiance(o4, d4, exclude=excl, index_base=5, camera=cam)
    assert rgb.shape == (count, 3) and ids.shape == (count,)
    if count == 0:
        return
    sub = np.unique(np.concatenate([rng.integers(0, count, 2000), [0, count - 1],
                                    np.arange(max(0, api.RADIANCE_BATCH - 4), min(count, api.RADIANCE_BATCH + 1))]))
    ref = np.concatenate([port_radiance.shade_rays(sc, o4[k:k + 1], d4[k:k + 1], excl[k:k + 1], index_base=5 + int(k), camera=cam, threads=1)[0]
                          for k in sub])
    _check(o4[sub], d4[sub], rgb[sub], ids[sub], ref)


def test_counters():
    sc, cam, ds = _scene("soup_mirror_glass")
    o4, d4, excl = _rays(sc, cam, n=128, seed=29)
    *_, cnt = ds.radiance(o4, d4, exclude=excl, samples=2, camera=cam, count=True)
    _, _, ref = port_radiance.shade_rays(sc, o4, d4, excl, samples=2, camera=cam)
    for k in ("segments", "shadedHits", "gridRays"):
        assert cnt[k] == ref[k], (k, cnt[k], ref[k])
    assert cnt["occluderLookups"] > 0


def _raw(ds, cam, n, o, d, out, flags=None, memory=api.QUERY_DEVICE_MEMORY):
    lib = _lib.load()
    c = cam.c()
    return lib.oclr_scene_radiance(ds.handle, C.byref(c), n, C.c_void_p(o), C.c_void_p(d), None, 0, 1, C.c_void_p(out),
                                   C.c_void_p(flags) if flags else None, memory, 0, None, None)


def test_bad_arguments_fail_cleanly():
    torch = pytest.importorskip("torch")
    sc, cam, ds = _scene("soup")
    o4, d4, excl = query_rays.family("eye", sc, cam, n=64, seed=30)
    d4[:, 3] = np.inf
    dev = torch.device("cuda", ds.device)
    to, td = torch.from_numpy(o4).to(dev), torch.from_numpy(d4).to(dev)
    out = torch.empty((65, 4), dtype=torch.float32, device=dev)
    big = torch.cat([to, to[:1]]).contiguous()
    cases = [
        (0, td.data_ptr(), out.data_ptr()),                           # null origin, count > 0
        (to.data_ptr(), td.data_ptr(), 0),                            # null output
        (big.data_ptr() + 4, td.data_ptr(), out.data_ptr()),          # misaligned origin
        (to.data_ptr(), td.data_ptr(), out.data_ptr() + 8),           # misaligned output
        (o4.ctypes.data, td.data_ptr(), out.data_ptr()),              # host memory passed as device memory
    ]
    for o, d, r in cases:
        assert _raw(ds, cam, 64, o, d, r) == 0, (o, d, r)
        assert "oclr_scene_radiance" in _lib.last_error()
    host_flags = np.zeros(64, np.uint8)
    assert _raw(ds, cam, 64, to.data_ptr(), td.data_ptr(), out.data_ptr(), flags=host_flags.ctypes.data) == 0   # host flags as device
    assert "flags" in _lib.last_error()
    lib = _lib.load()
    assert lib.oclr_scene_radiance(ds.handle, None, 64, o4.ctypes.data, d4.ctypes.data, None, 0, 0, out.data_ptr(), None,
                                   api.QUERY_HOST_MEMORY, 0, None, None) == 0   # zero samples
    assert "sampleCount" in _lib.last_error()
    # the device is still usable
    rgb, ids = ds.radiance(to, td, camera=cam)
    torch.cuda.synchronize(dev)
    ref, _, _ = port_radiance.shade_rays(sc, o4, d4, camera=cam)
    _check(o4, d4, rgb.cpu().numpy(), ids.cpu().numpy(), ref)


def _equirect_restated(basis, width, height):
    """The panorama's directions restated from render.py's docstring: float32 angle tables over the whole image, then the basis sum."""
    right, up, forward = (np.asarray(v, np.float32) for v in basis)
    phi = np.float32(2 * np.pi) * (np.arange(width, dtype=np.float32) + np.float32(0.5)) / np.float32(width) - np.float32(np.pi)
    theta = np.float32(np.pi / 2) - np.float32(np.pi) * (np.arange(height, dtype=np.float32) + np.float32(0.5)) / np.float32(height)
    ct, st = np.cos(theta)[:, None, None], np.sin(theta)[:, None, None]
    d = ct * np.sin(phi)[None, :, None] * right + st * up + ct * np.cos(phi)[None, :, None] * forward
    return np.ascontiguousarray(d.reshape(-1, 3), np.float32)


def test_equirect_render_equals_restatement(tmp_path):
    """render.py --projection equirect: the harness's planes equal (int)(mean * 65535) of the restatement over the restated directions."""
    name = "soup_mirror_glass"
    sc, cam, ds = _scene(name)
    m = sc.meta["camera"]
    w, h, samples = 96, 48, 2
    basis = render.equirect_basis(m["eye"], m["look_at"], m["up"])
    planes = render.render_equirect(ds, cam, basis, w, h, samples)
    d = _equirect_restated(basis, w, h)
    o4 = np.zeros((len(d), 4), np.float32)
    o4[:, :3] = np.asarray(cam.eye[:3], np.float32)
    d4 = np.zeros((len(d), 4), np.float32)
    d4[:, :3] = d
    d4[:, 3] = np.inf
    ref, _, _ = port_radiance.shade_rays(sc, o4, d4, samples=samples, camera=cam)
    v = np.clip(np.trunc(np.nan_to_num(ref[:, :3] * np.float32(65535))), 0, 65535).astype(np.uint16)
    for c in range(3):
        assert np.array_equal(planes[c], v[:, c].reshape(h, w)), c
    assert planes[0].any()
    out = tmp_path / "pano.png"
    api.write_image(out, planes)
    assert out.stat().st_size > 0


def _read_ppm16(path):
    data = path.read_bytes()
    magic, size, maxval, rest = data.split(b"\n", 3)
    w, h = (int(v) for v in size.split())
    assert magic == b"P6" and maxval == b"65535"
    px = np.frombuffer(rest, ">u2").reshape(h, w, 3)
    return tuple(px[:, :, c].astype(np.uint16) for c in range(3))


def test_equirect_command_line(tmp_path):
    """The harness end to end: the basis taken from the config's camera, the chunked render, the image written."""
    from opencl_render_b200 import scenes
    out = tmp_path / "pano.ppm"
    assert render.main(["config2", "--projection", "equirect", "--size", "128x64", "--samples", "2", "--out", str(out), "--quiet"]) == 0
    got = _read_ppm16(out)
    sc = scenes.CONFIGS[2]["make"]()
    m = sc.meta["camera"]
    cam = api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], 128, 64)
    ds = api.DeviceScene(sc)
    want = render.render_equirect(ds, cam, render.equirect_basis(m["eye"], m["look_at"], m["up"]), 128, 64, 2)
    ds.close()
    for c in range(3):
        assert np.array_equal(got[c], want[c]), c
    assert got[0].any()
