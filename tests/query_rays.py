"""Seeded ray families for the ray-query tests (tests/test_query_host.py, tests/test_gpu_query.py): rays in the reference's layout,
origin4 = (o.xyz, minD), direction4 = (d.xyz, maxD), plus the excluded triangle of each ray."""
import numpy as np

from opencl_render_b200 import api

NONE = api.NO_TRIANGLE

# families the trace stage runs; SCREENED_FAMILIES break its preconditions (minD < 0, NaN range, non-finite components)
TRACED_FAMILIES = ["eye", "bounce", "shadow", "axis", "split_planes", "outside", "glass", "empty_range", "magnitudes"]
SCREENED_FAMILIES = ["screened"]


def _unit(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def _tri_points(sc, rng, n):
    """Points on random triangles (barycentric, in float32) and those triangles' ids."""
    tri = rng.integers(0, sc.triangle_count, n)
    idx = sc.tri_idx[tri, :3]
    a, b, c = (sc.vertex[idx[:, k], :3].astype(np.float64) for k in range(3))
    u, v = rng.random(n), rng.random(n)
    flip = u + v > 1
    u[flip], v[flip] = 1 - u[flip], 1 - v[flip]
    return (a + u[:, None] * (b - a) + v[:, None] * (c - a)), tri.astype(np.uint32)


def _pack(o, d, lo, hi):
    n = len(o)
    o4, d4 = np.zeros((n, 4), np.float32), np.zeros((n, 4), np.float32)
    o4[:, :3], d4[:, :3] = o, d
    o4[:, 3], d4[:, 3] = lo, hi
    return o4, d4


def family(name, sc, cam, n=512, seed=0):
    """(origin4 [n,4], direction4 [n,4], excluded uint32 [n]) of one family on scene `sc` seen by camera `cam`."""
    rng = np.random.default_rng([seed, TRACED_FAMILIES.index(name) if name in TRACED_FAMILIES else 99])
    inf = np.float32(np.inf)
    excl = np.full(n, NONE, np.uint32)
    lo_box, hi_box = sc.box_min[0, :3], sc.box_min[-1, :3]
    centre = (lo_box.astype(np.float64) + hi_box) / 2
    eye = np.broadcast_to(cam.eye[:3], (n, 3))
    px, py = rng.random(n) * cam.width, rng.random(n) * cam.height
    eye_dir = cam.eye_to_top_left[:3] + px[:, None] * cam.left_to_right[:3] + py[:, None] * cam.top_to_bottom[:3]
    if name == "eye":
        o4, d4 = _pack(eye, eye_dir, 0.0, inf)
    elif name == "bounce":
        p, tri = _tri_points(sc, rng, n)
        o4, d4 = _pack(p, _unit(rng, n), 0.0, inf)
        excl = tri
    elif name == "shadow":
        p, tri = _tri_points(sc, rng, n)
        lights = sc.light_pos[:, :3] if sc.light_count else np.array([[0.0, 10.0, 0.0]], np.float32)
        to = lights[rng.integers(0, len(lights), n)].astype(np.float64) - p
        dist = np.linalg.norm(to, axis=1)
        o4, d4 = _pack(p, to / dist[:, None], 0.0, dist)
        excl = tri
    elif name == "axis":   # one or two zero direction components, +0.0 and -0.0
        p, tri = _tri_points(sc, rng, n)
        d = _unit(rng, n)
        zeros = rng.integers(1, 3, n)
        for i in range(n):
            for ax in rng.choice(3, zeros[i], replace=False):
                d[i, ax] = -0.0 if rng.random() < 0.5 else 0.0
        o4, d4 = _pack(p, d, 0.0, np.where(rng.random(n) < 0.5, inf, np.float32(rng.random(n) * 20)))
        excl = tri
        o4[1::3, :3] = eye[1::3]
        excl[1::3] = NONE
    elif name == "split_planes":   # origin coordinates exactly on split planes (sceneBoxMin values) and on the grid's faces
        planes = sc.box_min[:, :3]
        k = rng.integers(0, planes.shape[0], (n, 3))
        o = np.stack([planes[k[:, a], a] for a in range(3)], axis=1)
        o[::4] = np.where(rng.random((len(o[::4]), 3)) < 0.5, lo_box, hi_box)
        o4, d4 = _pack(o, _unit(rng, n), 0.0, inf)
        o4[:, :3] = o.astype(np.float32)   # (exact plane values, no float64 round trip)
    elif name == "outside":   # starts outside the grid, towards it and away from it
        half = (hi_box.astype(np.float64) - lo_box) / 2
        o = centre + _unit(rng, n) * (np.linalg.norm(half) * (1.2 + 2 * rng.random(n)))[:, None]
        to = centre + (rng.random((n, 3)) - 0.5) * half - o
        d = np.where(rng.random(n)[:, None] < 0.7, to, -to)
        o4, d4 = _pack(o, d, 0.0, np.where(rng.random(n) < 0.7, inf, np.float32(1 + rng.random(n))))
    elif name == "glass":   # minD > 0: the glass segment continues the same ray behind the surface
        o4, d4 = _pack(eye, eye_dir, np.float32(rng.random(n) * 3), inf)
    elif name == "empty_range":   # !(minD < maxD) and zero directions: misses without a trace
        o4, d4 = _pack(eye, eye_dir, np.float32(rng.random(n) * 5), 0.0)
        d4[:, 3] = np.where(rng.random(n) < 0.5, o4[:, 3], o4[:, 3] * np.float32(0.5))
        d4[::5, 3] = -inf
        z = slice(2, None, 4)
        o4[z, 3], d4[z, 3] = 0.0, inf
        d4[z, :3] = np.where(rng.random((len(d4[z]), 3)) < 0.5, -0.0, 0.0)
    elif name == "magnitudes":   # very small and very large direction lengths (t scales inversely) and far origins
        scale = 10.0 ** rng.uniform(-15, 15, n)
        o = np.where(rng.random(n)[:, None] < 0.3, centre + _unit(rng, n) * 1e5, eye)
        d = np.where(o == eye, eye_dir, centre - o) * scale[:, None]
        o4, d4 = _pack(o, d, 0.0, inf)
    elif name == "screened":
        o4, d4 = _pack(eye, eye_dir, 0.0, inf)
        kinds = np.arange(n) % 6
        o4[kinds == 0, 3] = -np.float32(rng.random((kinds == 0).sum()) + 1e-3)   # minD < 0
        o4[kinds == 1, 3] = np.nan
        d4[kinds == 2, 3] = np.nan
        o4[kinds == 3, rng.integers(0, 3)] = np.inf
        d4[kinds == 4, rng.integers(0, 3)] = -np.inf
        d4[kinds == 5, rng.integers(0, 3)] = np.nan
    else:
        raise KeyError(name)
    return np.ascontiguousarray(o4, np.float32), np.ascontiguousarray(d4, np.float32), excl


def all_families(sc, cam, n=512, seed=0, names=None):
    """All traced families concatenated: (origin4, direction4, excluded)."""
    parts = [family(f, sc, cam, n, seed) for f in (names or TRACED_FAMILIES)]
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(3))


def is_screened(o4, d4):
    """Rays the library does not trace because they break the trace stage's preconditions."""
    with np.errstate(invalid="ignore"):
        return ~((o4[:, 3] >= 0) & ~np.isnan(d4[:, 3]) & np.isfinite(o4[:, :3]).all(1) & np.isfinite(d4[:, :3]).all(1))


def is_empty(o4, d4):
    """Rays that meet nothing by definition: !(minD < maxD) or a zero direction."""
    with np.errstate(invalid="ignore"):
        return ~(o4[:, 3] < d4[:, 3]) | (d4[:, :3] == 0).all(1)
