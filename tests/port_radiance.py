"""TEST INFRASTRUCTURE ONLY: the reference of the radiance queries (oclr_scene_radiance) -- tests/port_radiance.c, a restatement of the
ring loop of the plain-C port (oracle/raytrace_port.c port_pixel_sample) entered from a caller ray or from the camera -- built into
tests/_build/."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

import port

HERE = Path(__file__).resolve().parent
SRC = HERE / "port_radiance.c"
LIB = HERE / "_build" / "libport_radiance.so"
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
        lib.port_shade_rays.restype = None
        lib.port_shade_rays.argtypes = [C.POINTER(port.Job), C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_ulonglong, C.c_uint32,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        lib.port_shade_frame.restype = None
        lib.port_shade_frame.argtypes = [C.POINTER(port.Job), C.c_int]
        _lib = lib
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


def _job(scene, camera=None, samples=1):
    j = port.Job()
    if camera is not None:
        j.width, j.height = camera.width, camera.height
        for name, v in (("eye", camera.eye), ("top_left", camera.eye_to_top_left), ("step_right", camera.left_to_right),
                        ("step_down", camera.top_to_bottom)):
            setattr(j, name, port.V3(float(v[0]), float(v[1]), float(v[2])))
        j.pixel_size_inv = float(camera.pixel_size_inv)
    j.samples = samples
    j.vertex, j.tri_index, j.tri_material = _p(scene.vertex), _p(scene.tri_idx), _p(scene.tri_mat)
    j.tri_uv, j.tri_normal = _p(scene.tri_uv), _p(scene.tri_normal)
    j.divisions = scene.axes_div
    j.planes, j.cell_start, j.cell_list = _p(scene.box_min), _p(scene.grid_start), _p(scene.grid_list)
    j.mat_size, j.mat_start, j.texels = _p(scene.mat_size), _p(scene.mat_start), _p(scene.textures)
    j.light_count = scene.light_count
    j.light_type, j.light_pos, j.light_dir = _p(scene.light_type), _p(scene.light_pos), _p(scene.light_dir)
    j.light_colour, j.light_radius, j.light_half = _p(scene.light_colour), _p(scene.light_radius), _p(scene.light_half)
    return j


def shade_rays(scene, o4, d4, excl=None, samples=1, index_base=0, camera=None, threads=None):
    """The restatement entered with each caller ray as ring slot 0.  o4 = (o.xyz, minD), d4 = (d.xyz, maxD) [N,4]; `camera` gives the pixel
    step vectors bump normals read.  Returns (out float32 [N,4] = (mean rgb, as_float(first hit of sample 0)), flags uint8 [N],
    counts dict(segments, shadedHits, gridRays))."""
    lib = load()
    o4 = np.ascontiguousarray(o4, np.float32)
    d4 = np.ascontiguousarray(d4, np.float32)
    assert o4.ndim == 2 and o4.shape[1] == 4 and d4.shape == o4.shape
    ex = None if excl is None else np.ascontiguousarray(excl, np.uint32)
    out = np.zeros((o4.shape[0], 4), np.float32)
    flags = np.zeros(o4.shape[0], np.uint8)
    counts = np.zeros(3, np.uint64)
    j = _job(scene, camera, samples)
    lib.port_shade_rays(C.byref(j), o4.shape[0], _p(o4), _p(d4), _p(ex), index_base, samples, _p(out), _p(flags), _p(counts),
                        threads or (os.cpu_count() or 1))
    return out, flags, dict(segments=int(counts[0]), shadedHits=int(counts[1]), gridRays=int(counts[2]))


def shade_frame(camera, lists, scene, samples=1, threads=None):
    """The restatement entered with the camera segment, every pixel-sample of a frame: planes (r, g, b) uint16 [H,W] with the port's
    per-sample conversion, and primary ids uint32 [H,W]."""
    lib = load()
    h, w = camera.height, camera.width
    out = [np.zeros((h, w), np.uint16) for _ in range(3)]
    ids = np.full((h, w), 0xFFFFFFFF, np.uint32)
    start = np.ascontiguousarray(lists.start, np.uint32)
    end = np.ascontiguousarray(lists.end, np.uint32)
    lst = np.ascontiguousarray(lists.list, np.uint32)
    j = _job(scene, camera, samples)
    j.cam_start, j.cam_end, j.cam_list = _p(start), _p(end), _p(lst)
    j.out_r, j.out_g, j.out_b = _p(out[0]), _p(out[1]), _p(out[2])
    j.primary_id = _p(ids)
    lib.port_shade_frame(C.byref(j), threads or (os.cpu_count() or 1))
    return tuple(out), ids

