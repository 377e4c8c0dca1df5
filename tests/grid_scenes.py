"""Scenes at every grid resolution the library accepts that the other tests do not use (axesDivCount 16, 64 and 256 are covered by
tests/helpers.py make_case and tests/deep_scenes.py).  Each resolution exists for a special case of the code:

- n = 1, 2: the grid is smaller than one 4x4x4 brick (pack_grid / brick_mask: one brick, side n, a partly filled mask) and the walk has no
  brick level (pwalk_setup: coarseOk needs n >= 4); every list is long, so lists are scanned past their 32-entry face masks;
- n = 4: exactly one brick, full mask;
- n = 8: two bricks per axis, no super-brick level;
- n = 32, 128, 512: the super-brick level of the three-level walk starts at 32 (super_bricks_per_axis);
- n = 1024: the packed walk's 10-bit coordinate fields are full (rt_walk.h kPkBits), 2^24 brick records, grid_start of 2^30 + 1
  entries (4 GiB), 3 x 1025 split planes in the trace kernels' shared memory.

Scenes per resolution: a soup with mirror and glass materials and four lights; a sparse soup with fewer vertices than cells per axis
(n >= 32: the quantile rule repeats split planes, so the grid has zero-width cells); the textured terrain with bump maps (n <= 128); a flat
terrain (all n + 1 planes of the y axis coincide), up to 128.  At 1024 only the two soups, at 100 x 75 pixels: grid_start alone is 4 GiB.
tests/test_grid_resolutions_host.py asserts that each case reaches its special case."""
import copy

import numpy as np

from opencl_render_b200 import api, scenes
from tests import helpers, query_rays

RESOLUTIONS = [1, 2, 4, 8, 32, 128, 512, 1024]
_LIGHTS = [helpers._OMNI, helpers._SPOT, helpers._AREA, helpers._SUN]


def _two_clusters(sc):
    """Every second triangle moved by (5, 4, 5): two clusters on a diagonal, so that the median split planes leave six of the eight
    octants empty and a grid of 32 cells or more has empty super-bricks (16^3 cells) for the three-level walk to cross."""
    v = sc.vertex.reshape(-1, 3, 4)   # (the soups' vertices are per triangle: tri_idx = arange)
    v[1::2, :, :3] += np.float32([5.0, 4.0, 5.0])
    return sc


def _soup(n):
    """800 triangles on grids of at most one brick (so that cells list more than 32 triangles), 180 on finer ones, in two clusters from
    32 cells per axis on."""
    sc = helpers._with_lights(scenes.soup(800 if n <= 4 else 180, seed=100 + n, reflective=True, transparent=True), _LIGHTS)
    return _two_clusters(sc) if n >= 32 else sc


def _sparse(n):
    """Fewer vertices than cells per axis: n // 4 - 1 triangles (3 vertices each), from 7 to 255, in two clusters."""
    tris = max(7, min(n // 4 - 1, 255))
    return _two_clusters(helpers._with_lights(scenes.soup(tris, seed=200 + n, reflective=True, transparent=True), _LIGHTS))


_terrain = {}


def _terrain_textured(n):
    """One scene (its textures take seconds to make), a copy per resolution."""
    if "t" not in _terrain:
        _terrain["t"] = scenes.terrain(12, textured=True, tile_quads=4, mirror_spheres=1)
    return copy.copy(_terrain["t"])


def _flat(n):
    """A flat terrain fills every cell of its footprint in all n zero-width layers of the y axis: n^3 non-empty cells.  At 512 that is
    1.3e8 cells, minutes for the host builder and the host packer, so the flat case stops at 128."""
    return scenes.terrain(16, seed=3, height=0.0)


# kind: (make, width, height, samples, resolutions); at 1024 cells per axis every frame is 100 x 75
KINDS = {
    "soup": (_soup, 96, 72, 2, RESOLUTIONS),
    "sparse": (_sparse, 96, 72, 2, [32, 128, 512, 1024]),
    "terrain_textured": (_terrain_textured, 120, 68, 1, [1, 2, 4, 8, 32, 128]),
    "flat": (_flat, 96, 54, 1, [1, 2, 4, 8, 32, 128]),
}
FINE = 1024
CASES = {f"{kind}_{n}": (kind, n) for kind, (_, _, _, _, ns) in KINDS.items() for n in ns}
_made = {}


def case(name):
    """(scene, camera, camera lists, samples) of a resolution case, grid built by the host builder.  Built once per process; a 1024-cell
    case (a 4 GiB grid) is kept only until another case is asked for."""
    if name not in _made:
        if any(CASES[k][1] == FINE for k in _made) or CASES[name][1] == FINE:
            _made.clear()
        kind, n = CASES[name]
        make, w, h, samples = KINDS[kind][:4]
        if n == FINE:
            w, h = 100, 75
        sc = make(n)
        m = sc.meta["camera"]
        cam = api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], w, h)
        lists = api.camera_triangle_list(cam, sc)
        api.scene_triangle_list(sc, n)
        _made[name] = (sc, cam, lists, samples)
    return _made[name]


def release():
    _made.clear()


def rays(name, n=192, seed=7):
    """The traced query families (tests/query_rays.py) on a case: origins on split planes and grid faces included."""
    sc, cam, _, _ = case(name)
    return query_rays.all_families(sc, cam, n=n, seed=seed)


def _first_cell_reaching(p, v):
    """grid_builder.cuh first_cell_reaching, vectorised: lowest c in [0, n-1] with p[c + 1] >= v (n - 1 when none)."""
    n = len(p) - 1
    return np.minimum(np.searchsorted(p[1:], v, side="left"), n - 1)


def _last_cell_reached(p, v):
    """grid_builder.cuh last_cell_reached: highest c in [0, n-1] with p[c] <= v (0 when none)."""
    n = len(p) - 1
    return np.clip(np.searchsorted(p[:n], v, side="right") - 1, 0, n - 1)


def _box_address(p, v):
    """rt_core.h box_address along one axis: the binary search of raytrace_opencl.c:174-193."""
    n = len(p) - 1
    c = np.zeros(v.shape, np.int64)
    while n > 1:
        n //= 2
        c += np.where(p[c + n] < v, n, 0)
    return c


def candidate_block_cells(sc):
    """Cells in each triangle's candidate block, by the rule of grid_builder.cuh grid_range_kernel: the cells whose closed boxes overlap
    the triangle's bounding box, widened to the cell of vertex a.  The device builder fills blocks of more than kGridSmallBlock (512)
    cells with grid_fill_large_kernel."""
    n = sc.axes_div
    v = sc.vertex[:, :3][sc.tri_idx[:, :3]]   # [N, 3 vertices, 3 axes], float32
    size = np.ones(sc.triangle_count, np.int64)
    for a in range(3):
        p = np.ascontiguousarray(sc.box_min[:, a])   # float32, non-decreasing
        lo = _first_cell_reaching(p, v[:, :, a].min(1))
        hi = _last_cell_reached(p, v[:, :, a].max(1))
        s = _box_address(p, v[:, 0, a])
        size *= np.maximum(hi, s) - np.minimum(lo, s) + 1
    return size


GRID_SMALL_BLOCK = 512
