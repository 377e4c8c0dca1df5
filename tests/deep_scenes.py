"""Scenes whose paths go deep: materials with both a REFLECTION and a TRANSPARENCY channel, so that every hit spawns a mirror AND a glass
segment.  The config generators never make such a material, and without one a hit spawns at most two segments, one of them a diffuse leaf:
the ring never holds more than two live segments, a pixel-sample needs a dozen traces at most and a shadow loop walks a few blockers.  These
scenes reach what exists for long paths -- the full ring and its skipped spawns, the depth-12 cutoff, more than 64 trace rounds per sample,
shadow loops over a hundred blockers -- and scenes with more than 65 536 lights.

All geometry lies in front of the camera (scenes.py: triangles behind the eye break the camera lists).  tests/port_depth.py measures
how deep each case goes; tests/test_deep_paths_host.py asserts it, so that a change here cannot make a case shallow again."""
import math

import numpy as np

from opencl_render_b200 import api, scenes

EYE, LOOK_AT, UP, FOV = (0.3, 0.2, -6.0), (0.0, 0.0, 10.0), (0.0, 1.0, 0.0), 0.9
AXES = 64
_UV = np.array([[0, 0], [1, 0], [0, 1]], np.float32)
_SPOT = dict(type=api.LIGHT_SPOT, pos=(0.5, 1.0, 60.0), colour=(1.0, 0.95, 0.9), radius=0.3)
_QUIET = 11   # a light type outside the reference's switch (raytrace_opencl.c:566-607): casts no ray, adds nothing


def _quad(c, ex, ey):
    """Two triangles of the parallelogram c +- ex +- ey."""
    c, ex, ey = (np.asarray(v, np.float64) for v in (c, ex, ey))
    return [c - ex - ey, c + ex - ey, c + ex + ey, c - ex + ey], [(0, 1, 2), (0, 2, 3)]


def _mesh(name, quads, atlas, lights):
    """quads: list of (corners, triangles, material)."""
    vs, ts, ms = [], [], []
    for corners, tris, mat in quads:
        base = sum(len(v) for v in vs)
        vs.append(np.array(corners, np.float64))
        ts.append(np.array(tris, np.int32) + base)
        ms += [mat] * len(tris)
    vertex = np.concatenate(vs).astype(np.float32)
    tri_idx = np.concatenate(ts).astype(np.int32)
    uv = np.tile(_UV, (tri_idx.shape[0], 1, 1))
    return scenes._scene(name, vertex, tri_idx, np.array(ms, np.int32), uv, scenes._flat_normals(vertex, tri_idx), atlas, lights,
                         meta=dict(camera=dict(eye=EYE, look_at=LOOK_AT, up=UP, fov=FOV)))


def _pane_quads(k_count, mat, stop=None, stop_mat=None):
    """k_count panes 0.25 apart along +z, each tilted a little about x and y (differently per pane, so mirror chains wander)."""
    out = []
    for k in range(k_count):
        ay, ax = 0.08 + 0.013 * (k % 7), 0.05 - 0.011 * (k % 5)
        ex = (1.6 * math.cos(ay), 0.0, 1.6 * math.sin(ay))
        ey = (0.0, 1.2 * math.cos(ax), 1.2 * math.sin(ax))
        corners, tris = _quad((0.0, 0.0, 0.25 * k), ex, ey)
        out.append((corners, tris, stop_mat if k == stop else mat))
    return out


def _floor(mat):
    corners, tris = _quad((0.0, -1.5, 33.0), (8.0, 0.0, 0.0), (0.0, 0.0, 37.0))   # z from -4 to 70: in front of the eye at z = -6
    return corners, tris, mat


def panes(k_count, refl, transp, stop=None, lights=None):
    """k_count panes of one white material with REFLECTION (refl,)*3 and TRANSPARENCY (transp,)*3, a diffuse floor and a spot light behind
    the stack.  `stop`: pane index whose TRANSPARENCY texel has a zero green channel (a shadow loop ends at it).  `lights`: replaces the
    spot light."""
    atlas = scenes.MaterialAtlas()
    m_pane = atlas.add(color=(255, 255, 255), reflection=(refl,) * 3, transparency=(transp,) * 3, luminance=(0, 0, 0))
    m_floor = atlas.add(color=(180, 180, 170), reflection=(0, 0, 0), transparency=(0, 0, 0), luminance=(0, 0, 0))
    m_stop = atlas.add(color=(255, 255, 255), reflection=(refl,) * 3, transparency=(transp, 0, transp), luminance=(0, 0, 0))
    quads = _pane_quads(k_count, m_pane, stop, m_stop) + [_floor(m_floor)]
    sc = _mesh(f"panes{k_count}_{refl}_{transp}", quads, atlas, lights if lights is not None else [_SPOT])
    return api.scene_triangle_list(sc, AXES)


def closed_box():
    """A closed box around [-2, 2]^3 (its corners moved a little, so that no wall is axis-aligned): mirror walls at -+x, mirror-and-glass
    walls at -+y and -+z, a tilted glass pane inside, a spot light inside and a distant light outside (its shadow rays cross the glass walls
    and stop at a mirror wall, which has no TRANSPARENCY channel).  For radiance rays that start inside: no camera lists are needed.
    axesDivCount 32: with 64 or more cells per axis the grid builder (the reference's SceneTriangleList::New, which the host builder
    reproduces) lists these walls, which cross the whole grid, in too few cells, and a third of the rays from inside walk through them."""
    atlas = scenes.MaterialAtlas()
    m_mirror = atlas.add(color=(235, 235, 240), reflection=(200, 200, 200), luminance=(0, 0, 0))
    m_both = atlas.add(color=(250, 245, 240), reflection=(140, 140, 140), transparency=(150, 160, 140), luminance=(6, 4, 2))
    m_glass = atlas.add(color=(220, 240, 230), reflection=(60, 60, 60), transparency=(190, 180, 200), luminance=(0, 0, 0))
    corner = np.array([[2.0 * (1 - 2 * ((i >> a) & 1)) for a in range(3)] for i in range(8)])   # corner i: bit a set = -2 along axis a
    corner += np.random.default_rng(5).uniform(-0.15, 0.15, corner.shape)
    quads = []
    for axis, mat in ((0, m_mirror), (1, m_both), (2, m_both)):
        a1, a2 = (axis + 1) % 3, (axis + 2) % 3
        for side in (0, 1):
            ring = [i for i in ((0, 1 << a1, (1 << a1) | (1 << a2), 1 << a2))]
            quads.append((corner[[i | (side << axis) for i in ring]], [(0, 1, 2), (0, 2, 3)], mat))
    corners, tris = _quad((0.2, -0.1, 0.3), (1.1, 0.2, 0.3), (-0.1, 0.9, 0.4))
    quads.append((corners, tris, m_glass))
    lights = [dict(type=api.LIGHT_SPOT, pos=(0.6, 1.1, -0.7), colour=(0.9, 0.85, 0.8), radius=0.2),
              dict(type=api.LIGHT_DISTANT, dir=(-0.3, -0.8, 0.5), colour=(0.4, 0.45, 0.5), radius=0.5)]
    sc = _mesh("closed_box", quads, atlas, lights)
    return api.scene_triangle_list(sc, 32)


def box_rays(n, seed):
    """Rays from points inside the closed box in all directions: o4 = (o, 0), d4 = (d, +inf)."""
    rng = np.random.default_rng(seed)
    o4 = np.zeros((n, 4), np.float32)
    d4 = np.zeros((n, 4), np.float32)
    o4[:, :3] = rng.uniform(-1.7, 1.7, (n, 3))
    d = rng.normal(size=(n, 3))
    d4[:, :3] = d / np.linalg.norm(d, axis=1, keepdims=True)
    d4[:, 3] = np.inf
    return o4, d4


def many_lights(casting=(65536,)):
    """One pane and the floor, then lights of the quiet type at every index but `casting`, where a spot light sits; the light count is
    max(casting) + 1.  A path that suspends on light 65 536 or later needs a light index wider than 16 bits.  The paths are kept short:
    every hit loops over all the lights, and what these scenes test is the light index, not the depth."""
    n = max(casting) + 1
    lights = [dict(type=_QUIET, pos=(0.0, 5.0, 0.0), colour=(1, 1, 1), radius=0.3)] * n
    for i, j in enumerate(sorted(casting)):
        lights[j] = dict(_SPOT, pos=(0.5 + 0.7 * i, 1.0 - 0.4 * i, 60.0 - 5.0 * i))
    sc = panes(1, 60, 90, lights=lights)
    sc.name = f"many_lights{n}"
    return sc


def camera(width, height):
    return api.set_camera(EYE, LOOK_AT, UP, FOV, width, height)


def frame_case(sc, width, height):
    """(camera, camera lists) of the deep scenes' camera at width x height."""
    cam = camera(width, height)
    return cam, api.camera_triangle_list(cam, sc)


def stack_rays(n=256, seed=3):
    """Rays from in front of the pane stack to a point beyond its last pane, all inside the panes' outline: o4 = (o, 0), d4 = (d, 1)."""
    rng = np.random.default_rng(seed)
    o = np.stack([rng.uniform(-0.5, 0.5, n), rng.uniform(-0.4, 0.4, n), np.full(n, -1.0)], 1)
    to = np.stack([rng.uniform(-0.5, 0.5, n), rng.uniform(-0.4, 0.4, n), np.full(n, 26.0)], 1)
    o4 = np.zeros((n, 4), np.float32)
    d4 = np.ones((n, 4), np.float32)
    o4[:, :3] = o
    d4[:, :3] = to - o
    return o4, d4


# name: (make, width, height, samples, least ring-full spawns, least sequential traces and least segments of the longest pixel-sample)
CASES = {
    "panes8": (lambda: panes(8, 128, 128), 48, 32, 1, 1000, 300, 50),
    "panes24": (lambda: panes(24, 140, 140), 48, 32, 1, 1000, 1000, 60),
    "panes100": (lambda: panes(100, 60, 240), 48, 32, 1, 1000, 5000, 60),
    "many_lights": (lambda: many_lights(), 24, 16, 1, 0, 5, 4),
    "many_lights3": (lambda: many_lights((65535, 65536, 65537)), 24, 16, 1, 0, 15, 4),
}
_made = {}


def case(name):
    """(scene, camera, camera lists, samples) of a deep case, built once per process."""
    if name not in _made:
        make, w, h, samples = CASES[name][:4]
        sc = make()
        cam, lists = frame_case(sc, w, h)
        _made[name] = (sc, cam, lists, samples)
    return _made[name]
