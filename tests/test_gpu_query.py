"""Ray queries on a resident scene (DeviceScene.intersect / transmittance, oclr_scene_intersect / oclr_scene_transmittance) against
the reference's closest-hit walk and shadow loop (oracle/raytrace_port.c port_walk_grid, and the shadow loop of tests/port_rays.c), bit for bit."""
import ctypes as C

import numpy as np
import pytest

from opencl_render_b200 import _lib, api
from tests import helpers, port_rays, query_rays

pytestmark = pytest.mark.gpu
NONE = query_rays.NONE

_scenes = {}


def _scene(name):
    if name not in _scenes:
        sc, cam, _, _ = helpers.make_case(name)
        _scenes[name] = (sc, cam, api.DeviceScene(sc))
    return _scenes[name]


def _rays(sc, cam, n=384, seed=11):
    fam = query_rays.all_families(sc, cam, n=n, seed=seed, names=query_rays.TRACED_FAMILIES + query_rays.SCREENED_FAMILIES)
    return fam


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _check_hits(o4, d4, ids, t, ab, ac, ref):
    scr = query_rays.is_screened(o4, d4)
    ok = ~scr
    assert np.array_equal(ids[ok], _bits(ref[ok, 0]))
    assert np.array_equal(_bits(t[ok]), _bits(ref[ok, 1]))
    assert np.array_equal(_bits(ab[ok]), _bits(ref[ok, 2])) and np.array_equal(_bits(ac[ok]), _bits(ref[ok, 3]))
    assert (ids[scr] == NONE).all() and np.isnan(t[scr]).all() and (ab[scr] == 0).all() and (ac[scr] == 0).all()
    empty = ok & query_rays.is_empty(o4, d4)   # answered without a trace: the ordinary miss
    assert (ids[empty] == NONE).all() and np.array_equal(_bits(t[empty]), _bits(d4[empty, 3]))


def _check_att(o4, d4, att, last, ref):
    scr = query_rays.is_screened(o4, d4)
    ok = ~scr
    assert np.array_equal(_bits(att[ok]), _bits(ref[ok, :3]))
    assert np.array_equal(last[ok], _bits(ref[ok, 3]))
    assert np.isnan(att[scr]).all() and (last[scr] == NONE).all()


@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_intersect_equals_port(name):
    sc, cam, ds = _scene(name)
    o4, d4, excl = _rays(sc, cam)
    ids, t, ab, ac = ds.intersect(o4, d4, exclude=excl)
    _check_hits(o4, d4, ids, t, ab, ac, port_rays.walk_rays(sc, o4, d4, excl))


@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_transmittance_equals_port(name):
    sc, cam, ds = _scene(name)
    o4, d4, excl = _rays(sc, cam, seed=12)
    att, last = ds.transmittance(o4, d4, exclude=excl)
    ref = port_rays.transmit_rays(sc, o4, d4, excl)
    _check_att(o4, d4, att, last, ref)
    if name == "soup_mirror_glass":   # partly transparent materials: attenuation between 0 and 1 is exercised
        ok = ~query_rays.is_screened(o4, d4)
        assert ((att[ok] > 0) & (att[ok] < 1)).any()


def test_host_and_device_memory_agree():
    torch = pytest.importorskip("torch")
    sc, cam, ds = _scene("soup_mirror_glass")
    o4, d4, excl = _rays(sc, cam, seed=13)
    dev = torch.device("cuda", ds.device)
    s = torch.cuda.Stream(device=dev)
    to, td, te = (torch.from_numpy(a).to(dev) for a in (o4, d4, excl.view(np.int32)))
    torch.cuda.synchronize(dev)
    h = ds.intersect(o4, d4, exclude=excl)
    g = ds.intersect(to, td, exclude=te, stream=s)
    s.synchronize()
    assert isinstance(g[0], torch.Tensor)
    for a, b in zip(h, g):
        assert np.array_equal(a.view(np.uint32), b.cpu().numpy().view(np.uint32))
    ha, hl = ds.transmittance(o4, d4, exclude=excl)
    ga, gl = ds.transmittance(to, td, exclude=te, stream=s)
    s.synchronize()
    assert np.array_equal(_bits(ha), _bits(ga.cpu().numpy())) and np.array_equal(hl, gl.cpu().numpy())
    # [N,3] inputs with scalar / per-ray ranges give the same as the [N,4] layout
    h3 = ds.intersect(o4[:, :3], d4[:, :3], t_min=o4[:, 3], t_max=d4[:, 3], exclude=excl)
    for a, b in zip(h, h3):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    g3 = ds.intersect(to[:, :3], td[:, :3], t_min=0.0, exclude=te)
    r3 = ds.intersect(o4[:, :3], d4[:, :3], exclude=excl)
    assert np.array_equal(g3[0].cpu().numpy(), r3[0])


@pytest.mark.parametrize("count", [0, 1, 31, 33, api.QUERY_BATCH + 1])
def test_counts(count):
    sc, cam, ds = _scene("soup")
    rng = np.random.default_rng(count)
    base_o, base_d, base_e = query_rays.all_families(sc, cam, n=256, seed=14)
    pick = rng.integers(0, len(base_o), count)
    o4, d4, excl = base_o[pick], base_d[pick], base_e[pick]
    ids, t, ab, ac = ds.intersect(o4, d4, exclude=excl)
    att, last = ds.transmittance(o4, d4, exclude=excl)
    assert ids.shape == (count,) and att.shape == (count, 3)
    if count == 0:
        return
    sub = np.unique(np.concatenate([rng.integers(0, count, 2000), [0, count - 1], np.arange(max(0, api.QUERY_BATCH - 4), min(count, api.QUERY_BATCH + 1))]))
    _check_hits(o4[sub], d4[sub], ids[sub], t[sub], ab[sub], ac[sub], port_rays.walk_rays(sc, o4[sub], d4[sub], excl[sub]))
    _check_att(o4[sub], d4[sub], att[sub], last[sub], port_rays.transmit_rays(sc, o4[sub], d4[sub], excl[sub]))


def test_scene_with_device_built_grid():
    sc, cam, _, _ = helpers.make_case("terrain_textured")
    bare = api.HostScene(**{k: getattr(sc, k) for k in ("vertex", "tri_idx", "tri_mat", "tri_uv", "tri_normal", "mat_size", "mat_start",
                                                        "textures", "light_type", "light_pos", "light_dir", "light_colour", "light_radius",
                                                        "light_half")})
    ds = api.DeviceScene(bare, axes_div=sc.axes_div)
    o4, d4, excl = _rays(sc, cam, seed=15)
    _check_hits(o4, d4, *ds.intersect(o4, d4, exclude=excl), port_rays.walk_rays(sc, o4, d4, excl))
    _check_att(o4, d4, *ds.transmittance(o4, d4, exclude=excl), port_rays.transmit_rays(sc, o4, d4, excl))
    ds.close()


def test_counters():
    sc, cam, ds = _scene("soup_mirror_glass")
    o4, d4, excl = _rays(sc, cam, seed=16)
    traced = ~query_rays.is_screened(o4, d4) & ~query_rays.is_empty(o4, d4)
    *_, cnt = ds.intersect(o4, d4, exclude=excl, count=True)
    assert cnt["gridRays"] == traced.sum()
    att, last, cnt = ds.transmittance(o4, d4, exclude=excl, count=True)
    # closest-hit traces of the shadow loop, replayed with the port: a ray stops at a miss or at the blocker that zeroes a component
    # (a triangle is met at most once: minD grows strictly)
    zeroed = ~(att > 0).all(1)
    o, d, e, fin, z = o4[traced].copy(), d4[traced], excl[traced], last[traced], zeroed[traced]
    active = np.ones(len(o), bool)
    traces = 0
    while active.any():
        traces += int(active.sum())
        h = port_rays.walk_rays(sc, o[active], d[active], e[active])
        tri = h[:, 0].view(np.uint32)
        idx = np.nonzero(active)[0]
        stop = (tri == NONE) | ((tri == fin[idx]) & z[idx])
        o[idx[~stop], 3] = h[~stop, 1]
        active[idx[stop]] = False
    assert cnt["gridRays"] == traces


def _raw(ds, entry, n, o, d, e, out, memory=api.QUERY_DEVICE_MEMORY):
    lib = _lib.load()
    return getattr(lib, entry)(ds.handle, n, C.c_void_p(o), C.c_void_p(d), C.c_void_p(e) if e else None, C.c_void_p(out), memory, 0,
                               None, None)


def test_bad_arguments_fail_cleanly():
    torch = pytest.importorskip("torch")
    sc, cam, ds = _scene("soup")
    o4, d4, excl = query_rays.family("eye", sc, cam, n=64, seed=17)
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
    if torch.cuda.device_count() > 1:
        other = torch.from_numpy(o4).to(torch.device("cuda", (ds.device + 1) % torch.cuda.device_count()))
        cases.append((other.data_ptr(), td.data_ptr(), out.data_ptr()))   # another device's memory
    for entry in ("oclr_scene_intersect", "oclr_scene_transmittance"):
        for o, d, r in cases:
            assert _raw(ds, entry, 64, o, d, 0, r) == 0, (entry, o, d, r)
            assert entry in _lib.last_error()
    # through the Python layer: a contiguous [N,4] float32 tensor is used in place, so a misaligned one reaches the library
    flat = torch.empty(64 * 4 + 1, dtype=torch.float32, device=dev)
    shifted = flat[1:].view(64, 4)
    shifted.copy_(to)
    with pytest.raises(api.OclrError, match="aligned"):
        ds.intersect(shifted, td)
    # the device is still usable
    ids, t, ab, ac = ds.intersect(to, td)
    torch.cuda.synchronize(dev)
    ref = port_rays.walk_rays(sc, o4, d4)
    assert np.array_equal(ids.cpu().numpy(), _bits(ref[:, 0])) and np.array_equal(_bits(t.cpu().numpy()), _bits(ref[:, 1]))

