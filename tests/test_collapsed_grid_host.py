"""The walk grid without a GPU (rt_types.h: each run of coincident split planes whose zero-width cells hold the same lists in every column
is one cell of the grid the production trace stage walks).  Its host form (scene_pack.cpp pack_walk_grid) against a numpy statement of the
rule; a hand-edited grid whose run must stay; and the trace kernels' packed walk over it (rt_walk.h, compiled for the host) against the
reference's cell walk on frames and against the port on caller rays -- planes, ids and flags bit for bit, with fewer cells walked wherever
a run collapsed."""
import ctypes as C
import subprocess
import types
from pathlib import Path

import numpy as np
import pytest

from opencl_render_b200 import _lib
from tests import grid_scenes, helpers, port_rays, query_rays
from tests.grid_scenes import CASES

ROOT = Path(__file__).resolve().parent.parent
# the grid-resolution cases of 32 cells or more whose split planes repeat: the flat terrain (all n + 1 planes of y coincide) and the
# sparse soups, whose runs hold different lists in some column (they stay: the grid is the reference grid)
REPEATED = [k for k, (kind, n) in CASES.items() if n >= 32 and kind in ("sparse", "flat")]


@pytest.fixture(scope="module")
def walkgrid():
    """tests/_build/libhostemu_walkgrid.so -- test-only."""
    lib = ROOT / "tests" / "_build" / "libhostemu_walkgrid.so"
    srcs = [ROOT / "tests" / "hostemu" / "hostemu_walkgrid.cpp", ROOT / "opencl_render_b200" / "csrc" / "scene_pack.cpp"]
    deps = srcs + list((ROOT / "opencl_render_b200" / "csrc").glob("*.h"))
    if not lib.is_file() or lib.stat().st_mtime < max(p.stat().st_mtime for p in deps):
        lib.parent.mkdir(exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-I/usr/local/cuda/include", "-pthread",
                        *map(str, srcs), "-o", str(lib)], check=True)
    return C.CDLL(str(lib))


def walk_grid(lib, sc):
    """The host form: None when no run collapses, else dict(extents, map, planes, bricks, ranges, masks)."""
    n = sc.axes_div
    nb = max(n // 4, 1)
    cap = int((np.diff(sc.grid_start.astype(np.int64)) > 0).sum()) + 1
    ext, cmap = np.zeros(3, np.int32), np.zeros(3 * n, np.int32)
    planes = np.zeros(3 * (n + 1), np.float32)
    bricks, ranges, masks = np.zeros(4 * nb ** 3, np.uint32), np.zeros(2 * cap, np.uint32), np.zeros(6 * cap, np.uint32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    lib.hostemu_walk_grid.restype = C.c_long
    cnt = lib.hostemu_walk_grid(C.byref(sc.desc()), p(ext), p(cmap), p(planes), p(bricks), p(ranges), C.c_size_t(ranges.nbytes), p(masks))
    assert cnt >= 0, cnt
    if cnt == 0:
        return None
    return dict(extents=ext, map=cmap.reshape(3, n), planes=planes, bricks=bricks, ranges=ranges[:2 * cnt], masks=masks[:6 * cnt])


def expected_map(sc):
    """The rule of rt_types.h in numpy: (map [3, n] with -1 past each extent, extents), or None when no run collapses."""
    n = sc.axes_div
    start = sc.grid_start.astype(np.int64)
    lst = sc.grid_list
    stride = np.array([1, n, n * n])
    keep = np.ones((3, n), bool)
    runs = []
    for a in range(3):
        p = sc.box_min[:, a]
        zero = p[:-1] == p[1:]
        c = 0
        while c < n:
            e = c
            while e < n and zero[e]:
                e += 1
            if e - c >= 2 and n >= 4:
                runs.append((a, c, e - c))
            c = max(e, c + 1)
    collapsed = []
    for a, first, count in runs:
        u, v = [b for b in range(3) if b != a]
        jj, ii = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
        base = (first * stride[a] + ii * stride[u] + jj * stride[v]).ravel()
        ok = True
        for k in range(1, count):
            ids = base + k * stride[a]
            ln0, ln = start[base + 1] - start[base], start[ids + 1] - start[ids]
            if not np.array_equal(ln0, ln):
                ok = False
                break
            rep = np.repeat(np.arange(len(base)), ln)
            off = np.arange(rep.size) - np.repeat(np.cumsum(ln) - ln, ln)
            if not np.array_equal(lst[start[base][rep] + off], lst[start[ids][rep] + off]):
                ok = False
                break
        collapsed.append(ok)
        if ok:
            keep[a, first + 1:first + count] = False
    if not any(collapsed):
        return None
    for (a, first, count), ok in zip(runs, collapsed):   # pad to a multiple of 4: cells of collapsed runs kept again, in run order
        for k in range(1, count):
            if ok and (n - keep[a].sum()) % 4:
                keep[a, first + k] = True
    if (keep.sum(1) == n).all():   # the padding kept every cell again: no walk grid
        return None
    cmap = np.full((3, n), -1, np.int32)
    for a in range(3):
        kept = np.nonzero(keep[a])[0]
        cmap[a, :kept.size] = kept
    return cmap, keep.sum(1)


def _check_form(sc, got):
    want = expected_map(sc)
    assert (got is None) == (want is None)
    if got is None:
        return
    cmap, ext = want
    assert np.array_equal(got["map"], cmap) and np.array_equal(got["extents"], ext)
    n = sc.axes_div
    assert (ext % 4 == 0).all() and (ext <= n).all() and (ext < n).any()
    for a in range(3):
        p = sc.box_min[:, a]
        kept = cmap[a, :ext[a]]
        assert np.array_equal(got["planes"][a * (n + 1):a * (n + 1) + ext[a]], p[kept])
        assert (got["planes"][a * (n + 1) + ext[a]:(a + 1) * (n + 1)] == p[n]).all()   # padded with the last plane
        assert set(np.nonzero(p[:-1] != p[1:])[0]) <= set(kept)   # every positive-width cell is kept
    # every walk cell's range is the list of the reference cell it stands for (the non-empty cells in brick-major order)
    nb = max(n // 4, 1)
    start = sc.grid_start.astype(np.int64)
    want_ranges = []
    by, bx, lz, ly, lx = np.indices((nb, nb, 4, 4, 4)).reshape(5, -1)
    for bz in range(nb):   # brick-major order, one layer of bricks at a time
        c = [bx * 4 + lx, by * 4 + ly, bz * 4 + lz]
        inside = (c[0] < ext[0]) & (c[1] < ext[1]) & (c[2] < ext[2])
        rid = np.zeros(inside.sum(), np.int64)
        for a in range(3):
            rid += cmap[a, c[a][inside]].astype(np.int64) * n ** a
        full = start[rid] < start[rid + 1]
        want_ranges.append(np.stack([start[rid][full], start[rid + 1][full]], 1).ravel())
    want_ranges = np.concatenate(want_ranges)
    assert np.array_equal(got["ranges"], np.array(want_ranges, np.uint32))


def test_spheres_collapse(walkgrid):
    sc = helpers.make_case("spheres")[0]
    got = walk_grid(walkgrid, sc)
    _check_form(sc, got)
    assert got is not None and got["extents"][1] < sc.axes_div // 2   # UV spheres: the y axis repeats its ring heights


@pytest.mark.parametrize("name", [k for k in REPEATED if CASES[k][1] <= 128])
def test_repeated_planes_collapse(name, walkgrid):
    sc = grid_scenes.case(name)[0]
    got = walk_grid(walkgrid, sc)
    _check_form(sc, got)
    if name.startswith("flat"):
        assert got is not None and got["extents"][1] == 4, name   # all n + 1 planes of y coincide: one cell and three duplicates
    else:
        assert got is None, name


def _edited_spheres():
    """The spheres case with one cell inside a collapsible y run given another list (same length, one entry changed)."""
    sc, cam, lists, samples = helpers.make_case("spheres")
    n = sc.axes_div
    start = sc.grid_start.astype(np.int64)
    p = sc.box_min[:, 1]
    zero = np.nonzero(p[:-1] == p[1:])[0]
    for y in zero:
        if y + 1 not in zero or y - 1 in zero:   # y: first cell of a run of >= 2 zero-width cells
            continue
        ids = np.arange(n * n) % n + n * (y + 1) + n * n * (np.arange(n * n) // n)
        full = ids[start[ids + 1] > start[ids]]
        if full.size:
            cid = int(full[0])
            lst = sc.grid_list.copy()
            e = int(start[cid + 1]) - 1
            lst[e] = (lst[e] + 1) % sc.triangle_count
            sc.grid_list = lst
            return sc, cam, lists, samples, int(y)
    raise AssertionError("no run to edit")


def test_edited_run_stays(walkgrid, hostemu):
    sc, cam, lists, samples, y = _edited_spheres()
    got = walk_grid(walkgrid, sc)
    _check_form(sc, got)
    assert got is not None
    kept = set(got["map"][1, :got["extents"][1]].tolist())
    assert {y, y + 1} <= kept   # the edited run keeps its cells
    ref = helpers.hostemu_render(hostemu, cam, lists, sc, samples, threads=8)
    wg = _render(walkgrid, cam, lists, sc, samples)
    assert _same(ref, wg)


def malformed_spheres():
    """The spheres case with a non-monotone CSR inside a collapsible y run: two cells of one column claim the range [0, 2^31)."""
    sc, cam, lists, samples = helpers.make_case("spheres")
    n = sc.axes_div
    p = sc.box_min[:, 1]
    y = int(np.nonzero((p[:-2] == p[1:-1]) & (p[1:-1] == p[2:]))[0][0])   # first cell of a run of >= 2 zero-width cells
    start = sc.grid_start.copy()
    for cid in (n // 2 + n * y + n * n * (n // 2), n // 2 + n * (y + 1) + n * n * (n // 2)):
        start[cid], start[cid + 1] = 0, 1 << 31
    sc.grid_start = start
    return sc, cam, lists, samples


def test_malformed_csr_is_refused(walkgrid):
    """The host packer refuses the grid before the walk grid reads any list (scene_pack.cpp pack_grid, walk_run_collapses)."""
    sc = malformed_spheres()[0]
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    z = np.zeros(16, np.uint32)
    lib = walkgrid
    lib.hostemu_walk_grid.restype = C.c_long
    assert lib.hostemu_walk_grid(C.byref(sc.desc()), p(z), p(z), p(z), p(z), p(z), C.c_size_t(z.nbytes), p(z)) == -1


def _render(lib, cam, lists, sc, samples):
    return helpers.hostemu_render(types.SimpleNamespace(hostemu_render=lib.hostemu_walkgrid_render), cam, lists, sc, samples, threads=8)


def _same(a, b):
    return all(np.array_equal(a[0][c], b[0][c]) for c in range(3)) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])


def _frames_equal_reference(walkgrid, hostemu, monkeypatch, name, sc, cam, lists, samples):
    monkeypatch.delenv("HOSTEMU_HIERARCHICAL", raising=False)
    monkeypatch.delenv("OCLR_SUPER", raising=False)
    ref = helpers.hostemu_render(hostemu, cam, lists, sc, samples, threads=8)   # the reference's cell walk
    wg = _render(walkgrid, cam, lists, sc, samples)
    assert _same(ref, wg), name
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", "2")   # the same packed walk on the reference grid
    packed = helpers.hostemu_render(hostemu, cam, lists, sc, samples, threads=8)[3]
    c = wg[3]
    for k in ("segments", "gridRays", "shadedHits", "occluderLookups", "gridCandidates"):   # (face masks: every repeated list is skipped whole)
        assert c[k] == packed[k], (name, k)
    if expected_map(sc) is None:
        assert c == packed, name
    else:
        # fewer occupied cells opened.  (Not always fewer cells: a walk grid packs more cells into each brick, so a scene whose runs are
        # short and many -- the 48-quad terrain at 256 cells -- crosses fewer empty bricks whole; the UV spheres walk half the cells.)
        assert c["cellsNonEmpty"] < packed["cellsNonEmpty"], (name, c, packed)
        if name.startswith("spheres"):
            assert c["cells"] < packed["cells"] and c["coarseSteps"] < packed["coarseSteps"], (name, c, packed)


@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_frames_equal_reference(name, walkgrid, hostemu, monkeypatch):
    _frames_equal_reference(walkgrid, hostemu, monkeypatch, name, *helpers.make_case(name))


@pytest.mark.parametrize("name", list(CASES))
def test_grid_resolution_frames_equal_reference(name, walkgrid, hostemu, monkeypatch):
    try:
        _frames_equal_reference(walkgrid, hostemu, monkeypatch, name, *grid_scenes.case(name))
    finally:
        grid_scenes.release()


def _walk_rays(lib, sc, o4, d4, excl):
    out = np.zeros((o4.shape[0], 4), np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
    lib.hostemu_walkgrid_rays.restype = C.c_int
    assert lib.hostemu_walkgrid_rays(C.byref(sc.desc()), C.c_size_t(o4.shape[0]), p(o4), p(d4), p(excl), p(out), C.c_int(8))
    return out


def _plane_rays(sc, rng, count):
    """Origins exactly on collapsed y planes (the run's value), half of them with r.y == 0: lying in the plane."""
    p = sc.box_min[:, 1]
    values = np.unique(p[:-1][p[:-1] == p[1:]])
    lo, hi = sc.box_min[0, :3], sc.box_min[-1, :3]
    o = rng.uniform(lo, hi, (count, 3)).astype(np.float32)
    o[:, 1] = rng.choice(values, count)
    d = rng.normal(size=(count, 3)).astype(np.float32)
    d[::2, 1] = 0.0
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o4, d4 = np.zeros((count, 4), np.float32), np.zeros((count, 4), np.float32)
    o4[:, :3], d4[:, :3] = o, d
    o4[:, 3] = np.where(np.arange(count) % 3 == 0, 0.0, 1e-3)
    d4[:, 3] = np.where(np.arange(count) % 4 == 0, np.float32(np.inf), rng.uniform(0.5, 20.0, count).astype(np.float32))
    return o4, d4, np.full(count, query_rays.NONE, np.uint32)


@pytest.mark.parametrize("name", ["spheres", "spheres_mirror"])
def test_caller_rays_equal_port(name, walkgrid):
    sc, cam, _, _ = helpers.make_case(name)
    assert expected_map(sc) is not None
    o4, d4, excl = query_rays.all_families(sc, cam, n=384, seed=7)
    traced = ~query_rays.is_screened(o4, d4) & ~query_rays.is_empty(o4, d4)
    po, pd, pe = _plane_rays(sc, np.random.default_rng(5), 3000)
    o4, d4, excl = np.concatenate([o4[traced], po]), np.concatenate([d4[traced], pd]), np.concatenate([excl[traced], pe])
    got = _walk_rays(walkgrid, sc, o4, d4, excl)
    ref = port_rays.walk_rays(sc, o4, d4, excl)
    bad = np.nonzero((got.view(np.uint32) != ref.view(np.uint32)).any(1))[0]
    assert bad.size == 0, (bad.size, o4[bad[:3]], d4[bad[:3]], got[bad[:3]], ref[bad[:3]])
    hits = (ref[-len(po):, 0].view(np.uint32) != query_rays.NONE).sum()
    assert 0 < hits < len(po)
