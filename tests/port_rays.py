"""TEST INFRASTRUCTURE ONLY: the reference of the batched ray queries -- tests/port_rays.c, the plain-C port of the reference's
raytrace path (oracle/raytrace_port.c) plus batch doors over its closest-hit walk and the shadow loop -- built into tests/_build/."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

import port

HERE = Path(__file__).resolve().parent
SRC = HERE / "port_rays.c"
LIB = HERE / "_build" / "libport_rays.so"
_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        deps = [SRC, Path(port.SRC)]
        if not LIB.is_file() or LIB.stat().st_mtime < max(p.stat().st_mtime for p in deps):
            LIB.parent.mkdir(exist_ok=True)
            subprocess.run(["gcc", "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wno-unused-function", str(SRC),
                            "-o", str(LIB), "-lm", "-lpthread"], check=True)
        lib = C.CDLL(str(LIB))
        lib.port_job_size.restype = C.c_size_t
        assert lib.port_job_size() == C.sizeof(port.Job), "port_job layout mismatch"
        for name in ("port_walk_rays", "port_transmit_rays"):
            getattr(lib, name).restype = None
            getattr(lib, name).argtypes = [C.POINTER(port.Job), C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        _lib = lib
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


def _rays(entry, scene, o4, d4, excl, threads):
    lib = load()
    o4 = np.ascontiguousarray(o4, np.float32)
    d4 = np.ascontiguousarray(d4, np.float32)
    assert o4.ndim == 2 and o4.shape[1] == 4 and d4.shape == o4.shape
    ex = None if excl is None else np.ascontiguousarray(excl, np.uint32)
    out = np.zeros((o4.shape[0], 4), np.float32)
    j = port.Job()
    j.vertex, j.tri_index, j.tri_material = _p(scene.vertex), _p(scene.tri_idx), _p(scene.tri_mat)
    j.tri_uv, j.tri_normal = _p(scene.tri_uv), _p(scene.tri_normal)
    j.divisions = scene.axes_div
    j.planes, j.cell_start, j.cell_list = _p(scene.box_min), _p(scene.grid_start), _p(scene.grid_list)
    j.mat_size, j.mat_start, j.texels = _p(scene.mat_size), _p(scene.mat_start), _p(scene.textures)
    getattr(lib, entry)(C.byref(j), o4.shape[0], _p(o4), _p(d4), _p(ex), _p(out), threads or (os.cpu_count() or 1))
    return out


def walk_rays(scene, o4, d4, excl=None, threads: int | None = None):
    """RayIntersectsTriangles (port_walk_grid) per ray: o4 = (o.xyz, minD), d4 = (d.xyz, maxD) [N,4].  Returns float32 [N,4]
    (as_float(triangle), t, abL, acL)."""
    return _rays("port_walk_rays", scene, o4, d4, excl, threads)


def transmit_rays(scene, o4, d4, excl=None, threads: int | None = None):
    """The shadow loop (port_transmit) per ray.  Returns float32 [N,4] (att.rgb, as_float(last blocker))."""
    return _rays("port_transmit_rays", scene, o4, d4, excl, threads)
