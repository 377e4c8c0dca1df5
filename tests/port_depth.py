"""TEST INFRASTRUCTURE ONLY: how deep the paths of a scene go (tests/port_depth.c: the ring loop of the plain-C port with depth counts), built
into tests/_build/."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

import port
from tests import port_radiance

HERE = Path(__file__).resolve().parent
SRC = HERE / "port_depth.c"
LIB = HERE / "_build" / "libport_depth.so"
_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        deps = [SRC, port_radiance.SRC, Path(port.SRC)]
        if not LIB.is_file() or LIB.stat().st_mtime < max(p.stat().st_mtime for p in deps):
            LIB.parent.mkdir(exist_ok=True)
            subprocess.run(["gcc", "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wno-unused-function", str(SRC),
                            "-o", str(LIB), "-lm", "-lpthread"], check=True)
        lib = C.CDLL(str(LIB))
        lib.port_job_size.restype = C.c_size_t
        assert lib.port_job_size() == C.sizeof(port.Job), "port_job layout mismatch"
        lib.port_depth_frame.restype = None
        lib.port_depth_frame.argtypes = [C.POINTER(port.Job), C.c_void_p, C.c_int]
        lib.port_depth_rays.restype = None
        lib.port_depth_rays.argtypes = [C.POINTER(port.Job), C.c_size_t, C.c_void_p, C.c_void_p, C.c_ulonglong, C.c_uint32, C.c_void_p,
                                        C.c_void_p, C.c_int]
        _lib = lib
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _counts(c):
    """segments and gridRays as the library counts them; ringFull = spawns after which the ring held 11 live segments (the hit's remaining
    spawns are skipped); longestSegments / longestWalks = the largest segment count and number of sequential grid walks (non-camera
    closest hits plus shadow-loop steps) of one pixel-sample or ray-sample."""
    return dict(segments=int(c[0]), gridRays=int(c[1]), ringFull=int(c[2]), longestSegments=int(c[3]), longestWalks=int(c[4]))


def depth_frame(camera, lists, scene, samples=1, threads=None):
    """Every pixel-sample of a frame from the camera: planes (r, g, b) uint16 [H,W] and primary ids uint32 [H,W] as the port renders them,
    and the counts dict (_counts)."""
    lib = load()
    h, w = camera.height, camera.width
    out = [np.zeros((h, w), np.uint16) for _ in range(3)]
    ids = np.full((h, w), 0xFFFFFFFF, np.uint32)
    start, end = np.ascontiguousarray(lists.start, np.uint32), np.ascontiguousarray(lists.end, np.uint32)
    lst = np.ascontiguousarray(lists.list, np.uint32) if lists.list.size else np.zeros(1, np.uint32)
    j = port_radiance._job(scene, camera, samples)
    j.cam_start, j.cam_end, j.cam_list = _p(start), _p(end), _p(lst)
    j.out_r, j.out_g, j.out_b = _p(out[0]), _p(out[1]), _p(out[2])
    j.primary_id = _p(ids)
    counts = np.zeros(5, np.uint64)
    lib.port_depth_frame(C.byref(j), _p(counts), threads or (os.cpu_count() or 1))
    return tuple(out), ids, _counts(counts)


def depth_rays(scene, o4, d4, samples=1, index_base=0, threads=None):
    """Traced caller rays (0 <= minD < inf, maxD = +inf, finite non-zero directions) as ring slot 0: out float32 [N,4] as
    port_radiance.shade_rays returns it, and the counts dict (_counts)."""
    lib = load()
    o4 = np.ascontiguousarray(o4, np.float32)
    d4 = np.ascontiguousarray(d4, np.float32)
    assert o4.ndim == 2 and o4.shape[1] == 4 and d4.shape == o4.shape
    assert (o4[:, 3] >= 0).all() and np.isfinite(o4).all() and (d4[:, 3] == np.inf).all() and np.isfinite(d4[:, :3]).all()
    assert (d4[:, :3] != 0).any(axis=1).all()
    out = np.zeros((o4.shape[0], 4), np.float32)
    counts = np.zeros(5, np.uint64)
    j = port_radiance._job(scene, None, samples)
    lib.port_depth_rays(C.byref(j), o4.shape[0], _p(o4), _p(d4), index_base, samples, _p(out), _p(counts), threads or (os.cpu_count() or 1))
    return out, _counts(counts)
