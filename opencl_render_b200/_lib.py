"""ctypes binding of libopencl_render_b200.so (include/oclr_abi.h).  Loading fails loudly: there is no Python or
CPU fallback for any compute entry point."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libopencl_render_b200.so"

c_uint_p = C.POINTER(C.c_uint32)
c_int_p = C.POINTER(C.c_int32)
c_float_p = C.POINTER(C.c_float)
c_ushort_p = C.POINTER(C.c_uint16)


class SceneDesc(C.Structure):
    """oclr_scene_desc"""
    _fields_ = [
        ("vertexCount", C.c_uint32), ("vertex", C.c_void_p),
        ("triangleCount", C.c_uint32), ("triangleVertexIndex", C.c_void_p), ("triangleMaterialId", C.c_void_p),
        ("triangleUv", C.c_void_p), ("triangleNormal", C.c_void_p),
        ("axesDivCount", C.c_int32), ("sceneBoxMin", C.c_void_p), ("scenePixelTriangleListStart", C.c_void_p),
        ("scenePixelTriangleList", C.c_void_p),
        ("materialCount", C.c_uint32), ("materialImageSize", C.c_void_p), ("materialImageStart", C.c_void_p),
        ("texturesSize", C.c_uint32), ("textures", C.c_void_p),
        ("lightCount", C.c_uint32), ("lightType", C.c_void_p), ("lightPosition", C.c_void_p), ("lightDirection", C.c_void_p),
        ("lightColour", C.c_void_p), ("lightRadius", C.c_void_p), ("lightHalfAttenuationDistance", C.c_void_p),
    ]


class Camera(C.Structure):
    """oclr_camera"""
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("eye", C.c_float * 4), ("eyeToTopLeft", C.c_float * 4),
                ("leftToRight", C.c_float * 4), ("topToBottom", C.c_float * 4), ("pixelSizeInv", C.c_float)]


class Counters(C.Structure):
    """oclr_counters"""
    _fields_ = [(n, C.c_ulonglong) for n in ("segments", "primCandidates", "gridRays", "cells", "cellsNonEmpty",
                                              "gridCandidates", "shadedHits", "occluderLookups", "bricksLoaded", "emptyBrickCells", "walkWarpIters", "walkLaneIters", "testWarpIters",
                                              "testLaneIters", "mailboxSkips", "coarseSteps", "coarseEnters", "switchWarpIters", "switchLaneIters", "walkIdleLanes", "walkParkedLanes", "walkFinishedLanes", "walkLowIters", "walkExhaustedIters",
                                              "splitAttempts", "splitsDone", "splitParts", "splitCancelled", "superSteps", "superEnters", "superRefines") +
                                             tuple("exitHist%02d" % i for i in range(16)) + tuple("exhaustHist%02d" % i for i in range(16)) +
                                             ("warpOuterItersMax", "warpOuterItersSum", "warpsRun")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class RenderStats(C.Structure):
    """oclr_render_stats"""
    _fields_ = [("deviceMs", C.c_float), ("launches", C.c_uint32), ("traceMs", C.c_float), ("traceLaunches", C.c_uint32),
                ("counters", Counters)]


class CameraLists(C.Structure):
    """oclr_camera_lists"""
    _fields_ = [("start", c_uint_p), ("end", c_uint_p), ("list", c_uint_p), ("listSize", C.c_size_t), ("pixelCount", C.c_uint32)]


class SceneGrid(C.Structure):
    """oclr_scene_grid"""
    _fields_ = [("axesDivCount", C.c_int32), ("boxMin", C.c_void_p), ("start", c_uint_p), ("list", c_uint_p), ("listSize", C.c_size_t)]


EXPORTS = [
    # Part 1: source/opencl/raytrace.h:37-106
    "dot", "cross", "normalize", "vector", "bindf", "GetPointToLineSqLen", "RayIntersectsTriangle", "GetBoxAddress",
    "InitOpenCL", "ResetComputationType", "GetIsComputationTypeUpdated", "GetComputationTypeCount", "GetComputationTypeName",
    "GetProgress", "SetProgress", "GetStartTime", "GetEndTime", "ResetTime", "RaytraceAll",
    # Part 2: extension
    "oclr_last_error", "oclr_device_count", "oclr_version", "oclr_scene_create", "oclr_scene_destroy", "oclr_scene_device_bytes", "oclr_scene_debug_read",
    "oclr_set_camera", "oclr_frame_create", "oclr_frame_create_device_lists", "oclr_frame_camera_list_size",
    "oclr_frame_read_camera_lists", "oclr_frame_destroy", "oclr_frame_state_bytes", "oclr_frame_render", "oclr_frame_render_bands", "oclr_frame_read",
    "oclr_frame_read_primary_ids", "oclr_frame_read_flags", "oclr_frame_last_launches", "oclr_frame_device_planes", "oclr_band_partition", "oclr_raytrace_all_p",
    "oclr_build_camera_lists", "oclr_build_scene_grid", "oclr_build_scene_grid_device", "oclr_free_camera_lists", "oclr_free_scene_grid",
    # progressive rendering, progress, image output (SURVEY.md section 8f-3, 8f-4)
    "oclr_frame_render_samples", "oclr_frame_render_bands_samples", "oclr_frame_write", "oclr_frame_set_accumulation", "oclr_frame_read_accum",
    "oclr_frame_write_accum", "oclr_frame_progress", "oclr_estimated_seconds_left", "oclr_write_bmp", "oclr_write_ppm16", "oclr_write_png16",
    "oclr_set_option", "oclr_frame_push_rows",
    # batched ray queries on a resident scene
    "oclr_scene_intersect", "oclr_scene_transmittance", "oclr_scene_radiance",
    # edits of a resident scene and of a frame's camera
    "oclr_scene_update", "oclr_frame_set_camera", "oclr_frame_set_camera_lists",
]

_lib = None


def load() -> C.CDLL:
    """Load the native library (building it first when nvcc is present and sources changed)."""
    global _lib
    if _lib is not None:
        return _lib
    if os.environ.get("OCLR_NO_BUILD") != "1":
        try:
            from . import build as _build
            _build.build()
        except Exception as e:  # a prebuilt .so may still be usable (GPU box without a changed tree)
            if not LIB_PATH.is_file():
                raise RuntimeError(f"libopencl_render_b200.so is missing and could not be built: {e}") from e
    if not LIB_PATH.is_file():
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -m opencl_render_b200.build` "
                           "(there is no Python/CPU fallback)")
    lib = C.CDLL(os.environ.get("OCLR_LIB") or str(LIB_PATH))     # OCLR_LIB: developer knob for A/B builds of the same library
    lib.oclr_last_error.restype = C.c_char_p
    lib.oclr_version.restype = C.c_char_p
    lib.oclr_device_count.restype = C.c_int
    lib.oclr_scene_create.restype = C.c_void_p
    lib.oclr_scene_create.argtypes = [C.c_int, C.POINTER(SceneDesc)]
    lib.oclr_scene_destroy.argtypes = [C.c_void_p]
    lib.oclr_scene_destroy.restype = None
    lib.oclr_scene_device_bytes.restype = C.c_size_t
    lib.oclr_scene_device_bytes.argtypes = [C.c_void_p]
    lib.oclr_scene_debug_read.restype = C.c_size_t
    lib.oclr_scene_debug_read.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    lib.oclr_set_camera.restype = None
    lib.oclr_set_camera.argtypes = [C.POINTER(Camera), c_float_p, c_float_p, c_float_p, C.c_float, C.c_uint32, C.c_uint32]
    lib.oclr_frame_create.restype = C.c_void_p
    lib.oclr_frame_create.argtypes = [C.c_void_p, C.POINTER(Camera), C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    lib.oclr_frame_create_device_lists.restype = C.c_void_p
    lib.oclr_frame_create_device_lists.argtypes = [C.c_void_p, C.POINTER(Camera)]
    lib.oclr_frame_camera_list_size.restype = C.c_size_t
    lib.oclr_frame_camera_list_size.argtypes = [C.c_void_p]
    lib.oclr_frame_read_camera_lists.restype = C.c_int
    lib.oclr_frame_read_camera_lists.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.oclr_frame_destroy.argtypes = [C.c_void_p]
    lib.oclr_frame_state_bytes.argtypes = [C.c_void_p]
    lib.oclr_frame_state_bytes.restype = C.c_size_t
    lib.oclr_frame_destroy.restype = None
    lib.oclr_frame_render.restype = C.c_int
    lib.oclr_frame_render.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_void_p,
                                      C.POINTER(RenderStats)]
    lib.oclr_frame_render_bands.restype = C.c_int
    lib.oclr_frame_render_bands.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                            C.POINTER(RenderStats)]
    lib.oclr_frame_read.restype = C.c_int
    lib.oclr_frame_read.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.oclr_frame_read_primary_ids.restype = C.c_int
    lib.oclr_frame_read_primary_ids.argtypes = [C.c_void_p, C.c_void_p]
    lib.oclr_frame_read_flags.restype = C.c_int
    lib.oclr_frame_read_flags.argtypes = [C.c_void_p, C.c_void_p]
    lib.oclr_frame_last_launches.restype = C.c_uint32
    lib.oclr_frame_last_launches.argtypes = [C.c_void_p]
    lib.oclr_frame_device_planes.restype = None
    lib.oclr_frame_device_planes.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
    lib.oclr_band_partition.restype = C.c_int
    lib.oclr_band_partition.argtypes = [C.c_uint32, C.c_uint32, C.c_int, C.c_int, c_uint_p, C.c_int]
    lib.oclr_raytrace_all_p.restype = C.c_uint32
    lib.oclr_raytrace_all_p.argtypes = [C.c_uint32, c_uint_p, c_float_p, c_float_p, c_float_p, c_float_p, C.c_float,
                                        C.POINTER(SceneDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_uint32,
                                        C.c_void_p, C.c_void_p, C.c_void_p]
    lib.oclr_build_camera_lists.restype = C.c_int
    lib.oclr_build_camera_lists.argtypes = [C.POINTER(Camera), C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(CameraLists)]
    lib.oclr_build_scene_grid.restype = C.c_int
    lib.oclr_build_scene_grid.argtypes = [C.c_int32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(SceneGrid)]
    lib.oclr_build_scene_grid_device.restype = C.c_int
    lib.oclr_build_scene_grid_device.argtypes = [C.c_int, C.c_int32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(SceneGrid)]
    lib.oclr_free_camera_lists.argtypes = [C.POINTER(CameraLists)]
    lib.oclr_free_camera_lists.restype = None
    lib.oclr_free_scene_grid.argtypes = [C.POINTER(SceneGrid)]
    lib.oclr_free_scene_grid.restype = None
    lib.oclr_frame_render_samples.restype = C.c_int
    lib.oclr_frame_render_samples.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_int,
                                              C.c_void_p, C.POINTER(RenderStats)]
    lib.oclr_frame_render_bands_samples.restype = C.c_int
    lib.oclr_frame_render_bands_samples.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int,
                                                    C.c_int, C.c_void_p, C.POINTER(RenderStats)]
    lib.oclr_frame_write.restype = C.c_int
    lib.oclr_frame_write.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.oclr_frame_set_accumulation.restype = C.c_int
    lib.oclr_frame_set_accumulation.argtypes = [C.c_void_p, C.c_int]
    lib.oclr_frame_read_accum.restype = C.c_int
    lib.oclr_frame_read_accum.argtypes = [C.c_void_p, C.c_void_p]
    lib.oclr_frame_write_accum.restype = C.c_int
    lib.oclr_frame_write_accum.argtypes = [C.c_void_p, C.c_void_p]
    lib.oclr_frame_progress.restype = C.c_int
    lib.oclr_frame_progress.argtypes = [C.c_void_p, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]
    lib.oclr_estimated_seconds_left.restype = C.c_double
    for name in ("oclr_write_ppm16", "oclr_write_png16"):
        getattr(lib, name).restype = C.c_int
        getattr(lib, name).argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.oclr_write_bmp.restype = C.c_int
    lib.oclr_write_bmp.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    lib.oclr_frame_push_rows.restype = C.c_int
    lib.oclr_frame_push_rows.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.c_void_p]
    for name in ("oclr_scene_intersect", "oclr_scene_transmittance"):
        getattr(lib, name).restype = C.c_int
        getattr(lib, name).argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                       C.POINTER(RenderStats)]
    lib.oclr_scene_radiance.restype = C.c_int
    lib.oclr_scene_radiance.argtypes = [C.c_void_p, C.POINTER(Camera), C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_ulonglong, C.c_uint32,
                                        C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(RenderStats)]
    lib.oclr_scene_update.restype = C.c_int
    lib.oclr_scene_update.argtypes = [C.c_void_p, C.POINTER(SceneDesc), C.c_uint, C.c_int]
    lib.oclr_frame_set_camera.restype = C.c_int
    lib.oclr_frame_set_camera.argtypes = [C.c_void_p, C.POINTER(Camera)]
    lib.oclr_frame_set_camera_lists.restype = C.c_int
    lib.oclr_frame_set_camera_lists.argtypes = [C.c_void_p, C.POINTER(Camera), C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    lib.oclr_set_option.restype = C.c_int
    lib.oclr_set_option.argtypes = [C.c_char_p, C.c_int]
    lib.InitOpenCL.restype = None
    lib.ResetComputationType.restype = None
    lib.GetIsComputationTypeUpdated.restype = C.c_uint32
    lib.GetComputationTypeCount.restype = C.c_size_t
    lib.GetComputationTypeName.restype = C.c_uint32
    lib.GetComputationTypeName.argtypes = [C.c_size_t, C.c_size_t, C.c_char_p]
    lib.GetProgress.restype = C.c_float
    lib.SetProgress.argtypes = [C.c_float]
    lib.SetProgress.restype = None
    lib.GetStartTime.restype = C.c_long
    lib.GetEndTime.restype = C.c_long
    lib.ResetTime.restype = None
    _lib = lib
    return lib


def last_error() -> str:
    return load().oclr_last_error().decode("utf-8", "replace")
