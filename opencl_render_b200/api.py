"""Host-side mirror of the reference's render interface (source/opencl/raytrace.h:46-106, called from
source/render.cpp:1311-1352), on top of the C-ABI of libopencl_render_b200.so.

Names and argument meaning follow the reference: `raytrace_all` is `RaytraceAll`, `set_camera` is `SetCamera`
(render.cpp:461-491), `camera_triangle_list` / `scene_triangle_list` are `CameraTriangleList::New` /
`SceneTriangleList::New` (source/util/trianglelist.cpp:520-626, 655-737).  Arrays use the reference's element layouts
(cl_float3 = 4 floats, cl_int3 = 4 ints, cl_uchar3 = 4 bytes).  Every compute call goes to the CUDA library; there is
no Python implementation behind any of them.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from dataclasses import dataclass, field

import numpy as np

from . import _lib

AXES_DIVISION = 256          # SceneTriangleList::AXES_DIVISION, trianglelist.h:44
MATERIAL_CHANNEL_COUNT = 5   # raytrace_opencl.h:14-22
CH_COLOR, CH_REFLECTION, CH_TRANSPARENCY, CH_BUMP, CH_LUMINANCE = range(5)
LIGHT_OMNI, LIGHT_SPOT, LIGHT_SPOTRECT, LIGHT_DISTANT, LIGHT_PARALLEL, LIGHT_PARSPOT, LIGHT_PARSPOTRECT, LIGHT_TUBE, \
    LIGHT_AREA, LIGHT_PHOTOMETRIC = range(10)
KERNEL_SIMPLE, KERNEL_PIPE, KERNEL_DEFAULT = 0, 2, -1
ACCUMULATE_REFERENCE_16BIT, ACCUMULATE_FLOAT = 0, 1
NO_TRIANGLE = 0xFFFFFFFF
QUERY_HOST_MEMORY, QUERY_DEVICE_MEMORY = 0, 1
SCENE_LIGHTS, SCENE_MATERIALS, SCENE_GEOMETRY = 1, 2, 4   # parts of oclr_scene_update
QUERY_BATCH = 1 << 21        # rays per internal batch of a query (runtime.h kQueryBatch)
RADIANCE_BATCH = 1 << 20     # rays per internal batch of a radiance query (runtime.h kRadianceBatch)


class OclrError(RuntimeError):
    pass


def _c(a, dtype, shape_tail=None):
    a = np.ascontiguousarray(a, dtype=dtype)
    if shape_tail is not None and tuple(a.shape[1:]) != tuple(shape_tail):
        raise ValueError(f"expected trailing shape {shape_tail}, got {a.shape}")
    return a


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


@dataclass
class HostScene:
    """The scene arrays the plugin hands to RaytraceAll (everything except camera, camera lists and outputs)."""
    vertex: np.ndarray               # float32 [V,4]
    tri_idx: np.ndarray              # int32   [N,4]
    tri_mat: np.ndarray              # int32   [N]
    tri_uv: np.ndarray               # float32 [N,3,2]
    tri_normal: np.ndarray           # float32 [N,3,4]
    mat_size: np.ndarray             # uint32  [5*M,2]
    mat_start: np.ndarray            # int32   [5*M+1]
    textures: np.ndarray             # uint8   [T,4]
    light_type: np.ndarray           # int32   [L]
    light_pos: np.ndarray            # float32 [L,4]
    light_dir: np.ndarray            # float32 [L,4]
    light_colour: np.ndarray         # float32 [L,4]
    light_radius: np.ndarray         # float32 [L]
    light_half: np.ndarray           # float32 [L]
    axes_div: int = AXES_DIVISION
    box_min: np.ndarray | None = None     # float32 [axes_div+1,4]
    grid_start: np.ndarray | None = None  # uint32 [axes_div^3+1]
    grid_list: np.ndarray | None = None   # uint32
    name: str = ""
    meta: dict = field(default_factory=dict)

    def normalise(self) -> "HostScene":
        self.vertex = _c(self.vertex, np.float32, (4,))
        self.tri_idx = _c(self.tri_idx, np.int32, (4,))
        self.tri_mat = _c(self.tri_mat, np.int32)
        self.tri_uv = _c(self.tri_uv, np.float32, (3, 2))
        self.tri_normal = _c(self.tri_normal, np.float32, (3, 4))
        self.mat_size = _c(self.mat_size, np.uint32, (2,))
        self.mat_start = _c(self.mat_start, np.int32)
        self.textures = _c(self.textures, np.uint8, (4,))
        self.light_type = _c(self.light_type, np.int32)
        self.light_pos = _c(self.light_pos, np.float32, (4,))
        self.light_dir = _c(self.light_dir, np.float32, (4,))
        self.light_colour = _c(self.light_colour, np.float32, (4,))
        self.light_radius = _c(self.light_radius, np.float32)
        self.light_half = _c(self.light_half, np.float32)
        if self.box_min is not None:
            self.box_min = _c(self.box_min, np.float32, (4,))
            self.grid_start = _c(self.grid_start, np.uint32)
            self.grid_list = _c(self.grid_list, np.uint32)
        return self

    @property
    def triangle_count(self) -> int:
        return int(self.tri_idx.shape[0])

    @property
    def vertex_count(self) -> int:
        return int(self.vertex.shape[0])

    @property
    def material_count(self) -> int:
        return int(self.mat_size.shape[0] // MATERIAL_CHANNEL_COUNT)

    @property
    def light_count(self) -> int:
        return int(self.light_type.shape[0])

    def desc(self, allow_missing_grid: bool = False) -> _lib.SceneDesc:
        if self.box_min is None and not allow_missing_grid:
            raise OclrError("scene has no grid: call scene_triangle_list(scene) first")
        d = _lib.SceneDesc()
        d.vertexCount = self.vertex_count
        d.vertex = _ptr(self.vertex)
        d.triangleCount = self.triangle_count
        d.triangleVertexIndex = _ptr(self.tri_idx)
        d.triangleMaterialId = _ptr(self.tri_mat)
        d.triangleUv = _ptr(self.tri_uv)
        d.triangleNormal = _ptr(self.tri_normal)
        d.axesDivCount = self.axes_div
        if self.box_min is not None:
            d.sceneBoxMin = _ptr(self.box_min)
            d.scenePixelTriangleListStart = _ptr(self.grid_start)
            d.scenePixelTriangleList = _ptr(self.grid_list)
        d.materialCount = self.material_count
        d.materialImageSize = _ptr(self.mat_size)
        d.materialImageStart = _ptr(self.mat_start)
        d.texturesSize = int(self.textures.shape[0])
        d.textures = _ptr(self.textures)
        d.lightCount = self.light_count
        d.lightType = _ptr(self.light_type)
        d.lightPosition = _ptr(self.light_pos)
        d.lightDirection = _ptr(self.light_dir)
        d.lightColour = _ptr(self.light_colour)
        d.lightRadius = _ptr(self.light_radius)
        d.lightHalfAttenuationDistance = _ptr(self.light_half)
        return d


@dataclass
class CameraSetup:
    """Output of SetCamera (render.cpp:461-491) + the image size."""
    width: int
    height: int
    eye: np.ndarray
    eye_to_top_left: np.ndarray
    left_to_right: np.ndarray
    top_to_bottom: np.ndarray
    pixel_size_inv: float

    def c(self) -> _lib.Camera:
        k = _lib.Camera()
        k.width, k.height = self.width, self.height
        for i in range(3):
            k.eye[i] = float(self.eye[i])
            k.eyeToTopLeft[i] = float(self.eye_to_top_left[i])
            k.leftToRight[i] = float(self.left_to_right[i])
            k.topToBottom[i] = float(self.top_to_bottom[i])
        k.pixelSizeInv = float(self.pixel_size_inv)
        return k


@dataclass
class CameraLists:
    """CameraTriangleList: per-pixel candidate triangles (Start/End have W*H entries, no +1)."""
    start: np.ndarray
    end: np.ndarray
    list: np.ndarray


def set_camera(position, look_at, up, fov: float, width: int, height: int) -> CameraSetup:
    """SetCamera (render.cpp:461-491): fov is the horizontal field of view in radians."""
    lib = _lib.load()
    out = _lib.Camera()
    f3 = lambda v: (C.c_float * 3)(*[float(x) for x in v[:3]])
    lib.oclr_set_camera(C.byref(out), f3(position), f3(look_at), f3(up), C.c_float(fov), width, height)
    g = lambda a: np.array([a[0], a[1], a[2], 0.0], dtype=np.float32)
    return CameraSetup(width, height, g(out.eye), g(out.eyeToTopLeft), g(out.leftToRight), g(out.topToBottom),
                       float(np.float32(out.pixelSizeInv)))


def camera_triangle_list(camera: CameraSetup, scene: HostScene) -> CameraLists:
    """CameraTriangleList::New (trianglelist.cpp:520-626)."""
    lib = _lib.load()
    scene.normalise()
    out = _lib.CameraLists()
    cam = camera.c()
    if not lib.oclr_build_camera_lists(C.byref(cam), scene.vertex_count, _ptr(scene.vertex), scene.triangle_count,
                                       _ptr(scene.tri_idx), C.byref(out)):
        raise OclrError(_lib.last_error())
    try:
        p = int(out.pixelCount)
        start = np.ctypeslib.as_array(out.start, shape=(p,)).copy()
        end = np.ctypeslib.as_array(out.end, shape=(p,)).copy()
        lst = np.ctypeslib.as_array(out.list, shape=(max(int(out.listSize), 1),))[:int(out.listSize)].copy()
    finally:
        lib.oclr_free_camera_lists(C.byref(out))
    return CameraLists(start, end, lst)


def scene_triangle_list(scene: HostScene, axes_div: int = AXES_DIVISION, device: int | None = None) -> HostScene:
    """SceneTriangleList::New (trianglelist.cpp:655-737): fills scene.box_min / grid_start / grid_list.  `device` = a CUDA device
    index: the builder runs on the GPU (same output, entry for entry); None: the host builder."""
    lib = _lib.load()
    scene.normalise()
    out = _lib.SceneGrid()
    if device is None:
        ok = lib.oclr_build_scene_grid(axes_div, scene.vertex_count, _ptr(scene.vertex), scene.triangle_count, _ptr(scene.tri_idx), C.byref(out))
    else:
        ok = lib.oclr_build_scene_grid_device(device, axes_div, scene.vertex_count, _ptr(scene.vertex), scene.triangle_count,
                                              _ptr(scene.tri_idx), C.byref(out))
    if not ok:
        raise OclrError(_lib.last_error())
    try:
        n = int(out.axesDivCount)
        scene.axes_div = n
        scene.box_min = np.ctypeslib.as_array(C.cast(out.boxMin, C.POINTER(C.c_float)), shape=(n + 1, 4)).copy()
        scene.grid_start = np.ctypeslib.as_array(out.start, shape=(n ** 3 + 1,)).copy()
        scene.grid_list = np.ctypeslib.as_array(out.list, shape=(max(int(out.listSize), 1),))[:int(out.listSize)].copy()
    finally:
        lib.oclr_free_scene_grid(C.byref(out))
    return scene


def computation_types() -> list[str]:
    """InitOpenCL + GetComputationTypeCount/Name (raytrace.c:78-153): index 0 is a label only."""
    lib = _lib.load()
    lib.InitOpenCL()
    names = []
    for i in range(lib.GetComputationTypeCount()):
        buf = C.create_string_buffer(256)
        names.append(buf.value.decode() if lib.GetComputationTypeName(i, 255, buf) else "")
    return names


def raytrace_all(computation_type: int, camera: CameraSetup, lists: CameraLists, sample_count: int, scene: HostScene,
                 out=None):
    """RaytraceAll (raytrace.h:58-106) with HOST arrays in and out: upload, repack, trace, read back.
    Returns (red, green, blue) uint16 [H,W].  Raises OclrError where the reference returns CL_FALSE."""
    lib = _lib.load()
    scene.normalise()
    w, h = camera.width, camera.height
    if out is None:
        out = tuple(np.empty((h, w), dtype=np.uint16) for _ in range(3))
    r, g, b = out
    dim = (C.c_uint32 * 2)(w, h)
    f = lambda v: np.ascontiguousarray(v, dtype=np.float32).ctypes.data_as(_lib.c_float_p)
    start = _c(lists.start, np.uint32)
    end = _c(lists.end, np.uint32)
    lst = _c(lists.list, np.uint32)
    d = scene.desc()
    ok = lib.oclr_raytrace_all_p(computation_type, dim, f(camera.eye), f(camera.eye_to_top_left), f(camera.left_to_right),
                                 f(camera.top_to_bottom), C.c_float(camera.pixel_size_inv), C.byref(d), _ptr(start), _ptr(end),
                                 _ptr(lst), int(lst.size), sample_count, _ptr(r), _ptr(g), _ptr(b))
    if not ok:
        raise OclrError(_lib.last_error())
    return r, g, b


class DeviceScene:
    """Resident scene (extension): uploaded and repacked once, rendered many times."""

    def __init__(self, scene: HostScene, device: int = 0, axes_div: int | None = None):
        """A scene without a grid (scene_triangle_list not called) is accepted: SceneTriangleList::New then runs on the device
        during the upload and the grid never exists on the host (`axes_div` = its axesDivCount, default 256)."""
        self._lib = _lib.load()
        scene.normalise()
        if scene.box_min is None:
            scene.axes_div = AXES_DIVISION if axes_div is None else axes_div
        d = scene.desc(allow_missing_grid=True)
        self.handle = self._lib.oclr_scene_create(device, C.byref(d))
        if not self.handle:
            raise OclrError(_lib.last_error())
        self.device = device
        self.host = scene

    @property
    def device_bytes(self) -> int:
        return int(self._lib.oclr_scene_device_bytes(self.handle))

    def update(self, scene: HostScene, lights: bool = False, materials: bool = False, geometry: bool = False):
        """Replaces the parts named with those of `scene` (numpy arrays) in place (oclr_scene_update): afterwards the scene is byte for
        byte what DeviceScene would make from the new parts plus the ones it holds.  geometry=True takes scene's grid when it has one,
        else builds it on the device at scene.axes_div.  A failed update raises OclrError and leaves the scene as it was."""
        parts = (SCENE_LIGHTS if lights else 0) | (SCENE_MATERIALS if materials else 0) | (SCENE_GEOMETRY if geometry else 0)
        if not parts:
            raise ValueError("update: name at least one part (lights, materials, geometry)")
        if not isinstance(scene, HostScene):
            raise ValueError("update: scene must be a HostScene (update_geometry takes bare arrays)")
        scene.normalise()
        d = scene.desc(allow_missing_grid=True)
        if not self._lib.oclr_scene_update(self.handle, C.byref(d), parts, QUERY_HOST_MEMORY):
            raise OclrError(_lib.last_error())
        keep = {}
        if lights:
            keep.update({k: getattr(scene, k) for k in ("light_type", "light_pos", "light_dir", "light_colour", "light_radius", "light_half")})
        if materials:
            keep.update(mat_size=scene.mat_size, mat_start=scene.mat_start, textures=scene.textures)
        if geometry:
            keep.update({k: getattr(scene, k) for k in ("vertex", "tri_idx", "tri_mat", "tri_uv", "tri_normal", "axes_div", "box_min",
                                                         "grid_start", "grid_list")})
        self.host = dataclasses.replace(self.host, **keep)

    def update_geometry(self, vertex, tri_idx, tri_mat, tri_uv, tri_normal, grid=None, axes_div: int | None = None):
        """Replaces the geometry in place (oclr_scene_update with OCLR_SCENE_GEOMETRY).  Arrays in HostScene's shapes: vertex [V,4]
        float32, tri_idx [N,4] int32, tri_mat [N] int32, tri_uv [N,3,2] float32, tri_normal [N,3,4] float32 -- all numpy, or all CUDA
        torch tensors on the scene's device (read in place, e.g. a simulation's output).  grid = (box_min [n+1,4] float32,
        grid_start [n^3+1] uint32, grid_list [K] uint32) in the same kind of memory, or None: built on the device at `axes_div` cells
        per axis (default: the current one).  `host` then holds the arrays given (torch tensors stay tensors)."""
        arrays = {"vertex": vertex, "tri_idx": tri_idx, "tri_mat": tri_mat, "tri_uv": tri_uv, "tri_normal": tri_normal}
        if grid is not None:
            if len(grid) != 3:
                raise ValueError("grid must be (box_min, grid_start, grid_list)")
            if axes_div is not None:
                raise ValueError("axes_div is taken from the grid given (box_min has axes_div + 1 rows)")
            arrays.update(box_min=grid[0], grid_start=grid[1], grid_list=grid[2])
        torch = _torch_if_any(arrays.values())
        if torch is None:
            a = _geometry_arrays_numpy(arrays, self.host.axes_div if axes_div is None else axes_div)
            memory, ptr = QUERY_HOST_MEMORY, _ptr
        else:
            a = _geometry_arrays_torch(torch, torch.device("cuda", self.device), arrays,
                                       self.host.axes_div if axes_div is None else axes_div)
            memory, ptr = QUERY_DEVICE_MEMORY, lambda t: C.c_void_p(t.data_ptr()) if t is not None and t.numel() else None
        d = _lib.SceneDesc()
        d.vertexCount, d.vertex = a["vertex"].shape[0], ptr(a["vertex"])
        d.triangleCount = a["tri_idx"].shape[0]
        d.triangleVertexIndex, d.triangleMaterialId = ptr(a["tri_idx"]), ptr(a["tri_mat"])
        d.triangleUv, d.triangleNormal = ptr(a["tri_uv"]), ptr(a["tri_normal"])
        d.axesDivCount = a["axes_div"]
        if grid is not None:
            d.sceneBoxMin, d.scenePixelTriangleListStart, d.scenePixelTriangleList = ptr(a["box_min"]), ptr(a["grid_start"]), ptr(a["grid_list"])
        if torch is not None:
            torch.cuda.current_stream(torch.device("cuda", self.device)).synchronize()   # the arrays are complete before the library reads them
        if not self._lib.oclr_scene_update(self.handle, C.byref(d), SCENE_GEOMETRY, memory):
            raise OclrError(_lib.last_error())
        self.host = dataclasses.replace(self.host, vertex=a["vertex"], tri_idx=a["tri_idx"], tri_mat=a["tri_mat"], tri_uv=a["tri_uv"],
                                        tri_normal=a["tri_normal"], axes_div=a["axes_div"], box_min=a.get("box_min"),
                                        grid_start=a.get("grid_start"), grid_list=a.get("grid_list"))

    def debug_read(self, which: int) -> np.ndarray:
        """Packed device array as bytes (0 triGeo, 1 triShade, 2 bricks, 3 cellRange, 4 planes, 5 cellList)."""
        n = int(self._lib.oclr_scene_debug_read(self.handle, which, None, 0))
        out = np.zeros(max(n, 1), np.uint8)
        self._lib.oclr_scene_debug_read(self.handle, which, _ptr(out), n)
        return out[:n]

    def intersect(self, origins, directions, t_min=None, t_max=None, exclude=None, stream=None, count: bool = False):
        """Closest hit of every ray, RayIntersectsTriangles exactly (raytrace_opencl.c:324-401; semantics and preconditions in
        include/oclr_abi.h).  origins / directions: [N,3], or [N,4] with minD / maxD in column 3; t_min / t_max (scalars or [N]) give the
        range of [N,3] rays (default 0 and +inf) and may not be combined with [N,4] inputs; exclude: [N] triangle ids or None.
        numpy inputs run through host memory and return numpy; CUDA torch tensors on the scene's device run in place (contiguous [N,4]
        float32 inputs are not copied) on `stream` (torch stream or cudaStream_t handle; default: torch's current stream) and return
        tensors.  Returns (ids uint32[N], t float32[N], abL float32[N], acL float32[N]) -- a miss is (NO_TRIANGLE, maxD, 0, 0), a ray
        that breaks the preconditions (minD < 0, NaN range, non-finite component) (NO_TRIANGLE, NaN, 0, 0) -- plus the counters dict
        when count=True."""
        out, _, cnt = self._query(self._entry("oclr_scene_intersect"), origins, directions, t_min, t_max, exclude, stream, count)
        res = (self._ids(out[:, 0]), out[:, 1], out[:, 2], out[:, 3])
        return res + (cnt,) if count else res

    def transmittance(self, origins, directions, t_min=None, t_max=None, exclude=None, stream=None, count: bool = False):
        """Transmittance along every ray: the shadow loop of raytrace_opencl.c:608-627 (att starts at (1,1,1) and is multiplied by the
        TRANSPARENCY texel of each blocker, 0 without that channel, until a component reaches 0 or the ray is clear).  Arguments as in
        intersect().  Returns (att float32[N,3], last blocker uint32[N] or NO_TRIANGLE) (+ counters dict when count=True)."""
        out, _, cnt = self._query(self._entry("oclr_scene_transmittance"), origins, directions, t_min, t_max, exclude, stream, count)
        res = (out[:, :3], self._ids(out[:, 3]))
        return res + (cnt,) if count else res

    def radiance(self, origins, directions, t_min=None, exclude=None, samples: int = 1, index_base: int = 0, camera: CameraSetup | None = None,
                 stream=None, flags: bool = False, count: bool = False):
        """Colour arriving along every ray: the reference's pixel-sample loop (raytrace_opencl.c:452-725) with the camera segment replaced by
        the ray (semantics in include/oclr_abi.h, oclr_scene_radiance).  origins / directions as in intersect(), but a ray has no far
        limit: [N,4] directions carry +inf in column 3 (a finite one is refused per ray, with a NaN result).  Sample s of ray i is seeded
        (index_base + i) * samples + s + 1, so a job split over calls gives the same colours.  `camera` (CameraSetup): its pixel step
        vectors are what bump-mapped normals read; required when a material has a BUMP channel.  Returns (rgb float32[N,3] = mean over
        the samples, first-hit ids uint32[N] = the ray's own hit in sample 0), plus flags uint8[N] (bit 0: the reference's result is
        undefined for the ray) when flags=True and the counters dict when count=True."""
        if isinstance(samples, bool) or not isinstance(samples, (int, np.integer)) or samples < 1:
            raise ValueError(f"samples must be an integer >= 1, got {samples!r}")
        if isinstance(index_base, bool) or not isinstance(index_base, (int, np.integer)) or not 0 <= index_base < 1 << 64:
            raise ValueError(f"index_base must be an integer in [0, 2^64), got {index_base!r}")
        if camera is not None and not isinstance(camera, CameraSetup):
            raise ValueError("camera must be a CameraSetup (set_camera) or None")
        host = getattr(self, "host", None)
        if camera is None and host is not None and host.material_count and (host.mat_size[CH_BUMP::MATERIAL_CHANNEL_COUNT, 0] > 0).any():
            raise ValueError("the scene has bump-mapped materials, whose normals read the camera's pixel step vectors: pass camera=")
        cam = C.byref(camera.c()) if camera is not None else None

        def native(n, o, d, ex, out, fl, memory, cnt, st, stats):
            return self._lib.oclr_scene_radiance(self.handle, cam, n, o, d, ex, int(index_base), int(samples), out, fl, memory, cnt, st, stats)
        out, fl, cnt = self._query(native, origins, directions, t_min, None, exclude, stream, count, flags)
        res = (out[:, :3], self._ids(out[:, 3]))
        if flags:
            res += (fl,)
        return res + (cnt,) if count else res

    @staticmethod
    def _ids(col):
        if isinstance(col, np.ndarray):
            return np.ascontiguousarray(col).view(np.uint32)
        import torch
        return col.contiguous().view(torch.uint32)

    def _entry(self, name):
        """The native call of oclr_scene_intersect / oclr_scene_transmittance in _query's argument order."""
        def native(n, o, d, ex, out, fl, memory, cnt, st, stats):
            return getattr(self._lib, name)(self.handle, n, o, d, ex, out, memory, cnt, st, stats)
        return native

    def _query(self, native, origins, directions, t_min, t_max, exclude, stream, count, flags=False):
        """Runs native(n, origin4, direction4, excluded, out4, flags, memory, countEvents, stream, stats) on validated rays: numpy inputs
        through host memory, CUDA torch tensors in place on `stream`.  Returns (out [N,4], flags uint8 [N] or None, counters dict or None)."""
        torch = _torch_if_tensor(origins)
        if torch is None:
            if _torch_if_tensor(directions) is not None:
                raise ValueError("directions is a torch tensor, origins a numpy array: a query takes numpy or torch inputs, not both")
            o, d, ex = _query_rays_numpy(origins, directions, t_min, t_max, exclude)
            out = np.empty((o.shape[0], 4), np.float32)
            fl = np.zeros(o.shape[0], np.uint8) if flags else None
            stats = _lib.RenderStats()
            if not native(o.shape[0], _ptr(o), _ptr(d), _ptr(ex), _ptr(out), _ptr(fl), QUERY_HOST_MEMORY, 1 if count else 0, None,
                          C.byref(stats) if count else None):
                raise OclrError(_lib.last_error())
            return out, fl, (stats.counters.as_dict() if count else None)
        dev = torch.device("cuda", self.device)
        for name, a in (("origins", origins), ("directions", directions), ("exclude", exclude), ("t_min", t_min), ("t_max", t_max)):
            if isinstance(a, torch.Tensor) and a.device != dev:
                raise ValueError(f"{name} is on {a.device}, the scene is on {dev}")
            if isinstance(a, np.ndarray) and a.ndim > 0:
                raise ValueError(f"{name} is a numpy array: a query takes numpy or torch inputs, not both")
        if isinstance(stream, torch.cuda.Stream):
            ts = stream
        elif stream:
            ts = torch.cuda.ExternalStream(int(stream), device=dev)
        else:
            ts = torch.cuda.current_stream(dev)
        with torch.cuda.device(dev), torch.cuda.stream(ts):
            o, d, ex = _query_rays_torch(torch, dev, origins, directions, t_min, t_max, exclude)
            out = torch.empty((o.shape[0], 4), dtype=torch.float32, device=dev)
            fl = torch.zeros(o.shape[0], dtype=torch.uint8, device=dev) if flags else None
            stats = _lib.RenderStats()
            if not native(o.shape[0], C.c_void_p(o.data_ptr()), C.c_void_p(d.data_ptr()), C.c_void_p(ex.data_ptr()) if ex is not None else None,
                          C.c_void_p(out.data_ptr()), C.c_void_p(fl.data_ptr()) if fl is not None else None, QUERY_DEVICE_MEMORY,
                          1 if count else 0, C.c_void_p(ts.cuda_stream), C.byref(stats) if count else None):
                raise OclrError(_lib.last_error())
        cur = torch.cuda.current_stream(dev)
        if cur != ts:   # results are used on the caller's current stream
            cur.wait_stream(ts)
            out.record_stream(cur)
            if fl is not None:
                fl.record_stream(cur)
        return out, fl, (stats.counters.as_dict() if count else None)

    def close(self):
        if getattr(self, "handle", None):
            self._lib.oclr_scene_destroy(self.handle)
            self.handle = None

    def __del__(self):
        self.close()


_GEOMETRY_SHAPES = {"vertex": ("float32", (4,)), "tri_idx": ("int32", (4,)), "tri_mat": ("int32", ()), "tri_uv": ("float32", (3, 2)),
                    "tri_normal": ("float32", (3, 4)), "box_min": ("float32", (4,)), "grid_start": ("uint32", ()), "grid_list": ("uint32", ())}


def _torch_if_any(arrays):
    """The torch module when any of `arrays` is a torch tensor (torch is imported only then), else None; numpy and torch do not mix."""
    kinds = {type(a).__module__.startswith("torch") for a in arrays if a is not None}
    if kinds == {True, False}:
        raise ValueError("the geometry arrays mix numpy arrays and torch tensors: give all of them in one kind of memory")
    if kinds == {True}:
        import torch
        return torch
    return None


def _check_geometry_shapes(a: dict, shape_of, axes_div: int | None):
    """Shapes of the geometry arrays (HostScene's) and their agreement: one triangle count, a grid of axes_div cells per axis."""
    for name, (_, tail) in _GEOMETRY_SHAPES.items():
        if name in a and (len(shape_of(a[name])) != 1 + len(tail) or tuple(shape_of(a[name])[1:]) != tail):
            raise ValueError(f"{name} must be [K{''.join(f',{t}' for t in tail)}], got {tuple(shape_of(a[name]))}")
    n = shape_of(a["tri_idx"])[0]
    for name in ("tri_mat", "tri_uv", "tri_normal"):
        if shape_of(a[name])[0] != n:
            raise ValueError(f"tri_idx has {n} triangles, {name} {shape_of(a[name])[0]}")
    if "box_min" in a:
        axes_div = shape_of(a["box_min"])[0] - 1
        if shape_of(a["grid_start"])[0] != axes_div ** 3 + 1:
            raise ValueError(f"box_min has {axes_div + 1} rows (axes_div {axes_div}): grid_start must have {axes_div ** 3 + 1} entries, "
                             f"got {shape_of(a['grid_start'])[0]}")
    if isinstance(axes_div, bool) or not isinstance(axes_div, (int, np.integer)) or axes_div < 1 or axes_div & (axes_div - 1) or axes_div > 1024:
        raise ValueError(f"axes_div must be a power of two <= 1024, got {axes_div!r}")
    a["axes_div"] = int(axes_div)
    return a


def _geometry_arrays_numpy(arrays: dict, axes_div):
    a = {k: np.asarray(v) for k, v in arrays.items()}
    _check_geometry_shapes(a, lambda x: x.shape, axes_div)
    for name, (dt, _) in _GEOMETRY_SHAPES.items():
        if name in a:
            a[name] = np.ascontiguousarray(a[name], dtype=dt)
    return a


def _geometry_arrays_torch(torch, dev, arrays: dict, axes_div):
    for name, v in arrays.items():
        if not isinstance(v, torch.Tensor) or v.device != dev:
            raise ValueError(f"{name} is on {getattr(v, 'device', 'the host')}, the scene is on {dev}: torch geometry is read in place")
    a = dict(arrays)
    _check_geometry_shapes(a, lambda x: tuple(x.shape), axes_div)
    for name, (dt, _) in _GEOMETRY_SHAPES.items():
        if name in a:
            want = getattr(torch, dt)
            if a[name].dtype != want:
                raise ValueError(f"{name} must be {dt}, got {a[name].dtype}")
            a[name] = a[name].contiguous()
    return a


def _torch_if_tensor(a):
    """The torch module when `a` is a torch tensor (torch is imported only then), else None."""
    mod = type(a).__module__
    if mod.startswith("torch"):
        import torch
        if isinstance(a, torch.Tensor):
            if not a.is_cuda:
                raise ValueError("torch inputs of a query must be CUDA tensors (numpy arrays take the host path)")
            return torch
    return None


def _ray_shape(name, shape):
    if len(shape) != 2 or shape[1] not in (3, 4):
        raise ValueError(f"{name} must be [N,3] or [N,4], got {tuple(shape)}")


def _query_range(name, v, n):
    a = np.asarray(v)
    if a.dtype.kind not in "fiu" or (a.ndim != 0 and a.shape != (n,)):
        raise ValueError(f"{name} must be a real scalar or [N={n}] array, got {a.dtype} {a.shape}")
    return a


def _query_rays_numpy(origins, directions, t_min, t_max, exclude):
    """Validated contiguous (origin4, direction4, excluded | None) host arrays."""
    o, d = np.asarray(origins), np.asarray(directions)
    for name, a in (("origins", o), ("directions", d)):
        _ray_shape(name, a.shape)
        if a.dtype.kind != "f":
            raise ValueError(f"{name} must be floating point, got {a.dtype}")
    n = o.shape[0]
    if d.shape[0] != n:
        raise ValueError(f"origins has {n} rays, directions {d.shape[0]}")
    rays = []
    for name, a, rng, dflt in (("origins", o, t_min, 0.0), ("directions", d, t_max, np.inf)):
        if a.shape[1] == 4:
            if rng is not None:
                raise ValueError(f"{name} is [N,4] (range in column 3): {'t_min' if dflt == 0.0 else 't_max'} cannot be given too")
            rays.append(np.ascontiguousarray(a, np.float32))
        else:
            r = _query_range("t_min" if dflt == 0.0 else "t_max", dflt if rng is None else rng, n)
            a4 = np.empty((n, 4), np.float32)
            a4[:, :3] = a
            a4[:, 3] = r
            rays.append(a4)
    ex = None
    if exclude is not None:
        e = np.asarray(exclude)
        if e.dtype.kind not in "iu" or e.shape != (n,):
            raise ValueError(f"exclude must be an integer [N={n}] array, got {e.dtype} {e.shape}")
        ex = np.ascontiguousarray(e.astype(np.int64) & 0xFFFFFFFF, np.uint32) if e.dtype != np.uint32 else np.ascontiguousarray(e)
    return rays[0], rays[1], ex


def _query_rays_torch(torch, dev, origins, directions, t_min, t_max, exclude):
    """Validated contiguous (origin4, direction4, excluded | None) CUDA tensors; contiguous [N,4] float32 inputs are used as they are."""
    if not isinstance(directions, torch.Tensor):
        raise ValueError("directions must be a torch tensor like origins")
    for name, a in (("origins", origins), ("directions", directions)):
        _ray_shape(name, a.shape)
        if not a.dtype.is_floating_point:
            raise ValueError(f"{name} must be floating point, got {a.dtype}")
    n = origins.shape[0]
    if directions.shape[0] != n:
        raise ValueError(f"origins has {n} rays, directions {directions.shape[0]}")
    rays = []
    for name, a, rng, dflt in (("origins", origins, t_min, 0.0), ("directions", directions, t_max, float("inf"))):
        rname = "t_min" if dflt == 0.0 else "t_max"
        if a.shape[1] == 4:
            if rng is not None:
                raise ValueError(f"{name} is [N,4] (range in column 3): {rname} cannot be given too")
            rays.append(a.to(torch.float32).contiguous())
        else:
            rng = dflt if rng is None else rng
            if isinstance(rng, torch.Tensor):
                if rng.ndim != 0 and tuple(rng.shape) != (n,):
                    raise ValueError(f"{rname} must be a scalar or [N={n}] tensor, got {tuple(rng.shape)}")
            else:
                rng = _query_range(rname, rng, n)
                rng = float(rng) if rng.ndim == 0 else torch.as_tensor(rng, device=dev)
            a4 = torch.empty((n, 4), dtype=torch.float32, device=dev)
            a4[:, :3] = a
            a4[:, 3] = rng
            rays.append(a4)
    ex = None
    if exclude is not None:
        if not isinstance(exclude, torch.Tensor) or exclude.dtype not in (torch.int32, torch.uint32, torch.int64) or tuple(exclude.shape) != (n,):
            raise ValueError(f"exclude must be an int32 / uint32 / int64 [N={n}] CUDA tensor")
        ex = exclude.contiguous() if exclude.dtype != torch.int64 else (exclude & 0xFFFFFFFF).to(torch.int32).contiguous()
    return rays[0], rays[1], ex


class DeviceFrame:
    """One camera on a resident scene: camera lists + three 16-bit planes in HBM."""

    def __init__(self, scene: DeviceScene, camera: CameraSetup, lists: CameraLists | None = None):
        """`lists` = CameraTriangleList::New output built on the host, or None: the lists are built on the device from the
        resident scene (entry-for-entry the same; see camera_lists())."""
        self._lib = _lib.load()
        self.scene = scene
        self.camera = camera
        cam = camera.c()
        if lists is None:
            self.handle = self._lib.oclr_frame_create_device_lists(scene.handle, C.byref(cam))
        else:
            start = _c(lists.start, np.uint32)
            end = _c(lists.end, np.uint32)
            lst = _c(lists.list, np.uint32)
            self.handle = self._lib.oclr_frame_create(scene.handle, C.byref(cam), _ptr(start), _ptr(end), _ptr(lst), int(lst.size))
        if not self.handle:
            raise OclrError(_lib.last_error())

    def set_camera(self, camera: CameraSetup, lists: CameraLists | None = None):
        """Moves the frame's camera (same width and height): `lists` = CameraTriangleList::New output for the new camera and the
        scene's current geometry, or None: built on the device.  Planes, path state, accumulation mode and progress stay.  A call that
        fails in the library (OclrError) leaves the frame with the new camera and no lists: `camera` follows, and the frame refuses to
        render until a camera is set successfully."""
        if not isinstance(camera, CameraSetup):
            raise ValueError("camera must be a CameraSetup (set_camera)")
        if (camera.width, camera.height) != (self.camera.width, self.camera.height):
            raise ValueError(f"the camera is {camera.width}x{camera.height}, the frame {self.camera.width}x{self.camera.height}: "
                             "a frame keeps its image size (make a new DeviceFrame)")
        cam = camera.c()
        if lists is None:
            ok = self._lib.oclr_frame_set_camera(self.handle, C.byref(cam))
        else:
            P = camera.width * camera.height
            start, end, lst = _c(lists.start, np.uint32), _c(lists.end, np.uint32), _c(lists.list, np.uint32)
            if start.shape != (P,) or end.shape != (P,) or lst.ndim != 1:
                raise ValueError(f"lists: start and end must be [{P}] (width * height), list 1-D; got {start.shape}, {end.shape}, {lst.shape}")
            ok = self._lib.oclr_frame_set_camera_lists(self.handle, C.byref(cam), _ptr(start), _ptr(end), _ptr(lst), int(lst.size))
        self.camera = camera
        if not ok:
            raise OclrError(_lib.last_error())

    @property
    def state_bytes(self) -> int:
        """Wavefront path state held in HBM (0 before the first render)."""
        return int(self._lib.oclr_frame_state_bytes(self.handle))

    def camera_lists(self) -> "CameraLists":
        """Copies the frame's camera lists (uploaded or device-built) back to the host."""
        P = self.camera.width * self.camera.height
        n = int(self._lib.oclr_frame_camera_list_size(self.handle))
        start, end, lst = np.empty(P, np.uint32), np.empty(P, np.uint32), np.empty(max(n, 1), np.uint32)
        if not self._lib.oclr_frame_read_camera_lists(self.handle, _ptr(start), _ptr(end), _ptr(lst)):
            raise OclrError(_lib.last_error())
        return CameraLists(start, end, lst[:n])

    def render(self, sample_count: int = 1, rows=None, variant: int = KERNEL_DEFAULT, count: bool = False, stream: int = 0,
               sync: bool = True, samples=None):
        """Trace rows [rows[0], rows[1]) (default: all).  `samples` = (begin, end): only that range of the sample_count-sample
        job (progressive rendering: sample 0 overwrites the planes, later samples add).  Returns (device_ms, launches,
        counters dict | None)."""
        r0, r1 = rows if rows is not None else (0, self.camera.height)
        s0, s1 = samples if samples is not None else (0, sample_count)
        stats = _lib.RenderStats()
        ok = self._lib.oclr_frame_render_samples(self.handle, sample_count, s0, s1, r0, r1, variant, 1 if count else 0,
                                                 C.c_void_p(stream), C.byref(stats) if (sync or count) else None)
        if not ok:
            raise OclrError(_lib.last_error())
        self.last_trace_ms, self.last_trace_launches = float(stats.traceMs), int(stats.traceLaunches)
        return float(stats.deviceMs), int(stats.launches), (stats.counters.as_dict() if count else None)

    def render_bands(self, sample_count: int, band_rows: int, rank: int, world: int, variant: int = KERNEL_DEFAULT,
                     count: bool = False, stream: int = 0, sync: bool = True, samples=None):
        """Trace the rows y with (y // band_rows) % world == rank in one launch."""
        s0, s1 = samples if samples is not None else (0, sample_count)
        stats = _lib.RenderStats()
        ok = self._lib.oclr_frame_render_bands_samples(self.handle, sample_count, s0, s1, band_rows, rank, world, variant,
                                                       1 if count else 0, C.c_void_p(stream),
                                                       C.byref(stats) if (sync or count) else None)
        if not ok:
            raise OclrError(_lib.last_error())
        self.last_trace_ms, self.last_trace_launches = float(stats.traceMs), int(stats.traceLaunches)
        return float(stats.deviceMs), int(stats.launches), (stats.counters.as_dict() if count else None)

    def read(self, rows=None, out=None, stream: int = 0):
        h, w = self.camera.height, self.camera.width
        r0, r1 = rows if rows is not None else (0, h)
        if out is None:
            out = tuple(np.zeros((h, w), dtype=np.uint16) for _ in range(3))
        if not self._lib.oclr_frame_read(self.handle, r0, r1, _ptr(out[0]), _ptr(out[1]), _ptr(out[2]), C.c_void_p(stream)):
            raise OclrError(_lib.last_error())
        return out

    def write(self, planes, rows=None, stream: int = 0):
        """Uploads full-frame uint16 planes (rows [rows[0], rows[1]) of them): restores a checkpoint taken with read()."""
        r0, r1 = rows if rows is not None else (0, self.camera.height)
        p = [_c(a, np.uint16) for a in planes]
        if not self._lib.oclr_frame_write(self.handle, r0, r1, _ptr(p[0]), _ptr(p[1]), _ptr(p[2]), C.c_void_p(stream)):
            raise OclrError(_lib.last_error())

    def set_accumulation(self, mode: int):
        """ACCUMULATE_REFERENCE_16BIT (default, raytrace_opencl.c:726-741) or ACCUMULATE_FLOAT (fp32 sums, no per-sample truncation)."""
        if not self._lib.oclr_frame_set_accumulation(self.handle, mode):
            raise OclrError(_lib.last_error())

    def read_accum(self) -> np.ndarray:
        """float32 [H,W,4]: (sum r, sum g, sum b, samples) of the float accumulator."""
        out = np.empty((self.camera.height, self.camera.width, 4), np.float32)
        if not self._lib.oclr_frame_read_accum(self.handle, _ptr(out)):
            raise OclrError(_lib.last_error())
        return out

    def write_accum(self, acc: np.ndarray):
        a = _c(acc, np.float32)
        if not self._lib.oclr_frame_write_accum(self.handle, _ptr(a)):
            raise OclrError(_lib.last_error())

    def progress(self):
        """(done, total) pixel-samples of the render call in flight (thread-safe)."""
        d, t = C.c_ulonglong(), C.c_ulonglong()
        if not self._lib.oclr_frame_progress(self.handle, C.byref(d), C.byref(t)):
            raise OclrError(_lib.last_error())
        return int(d.value), int(t.value)

    def primary_ids(self) -> np.ndarray:
        ids = np.empty((self.camera.height, self.camera.width), dtype=np.uint32)
        if not self._lib.oclr_frame_read_primary_ids(self.handle, _ptr(ids)):
            raise OclrError(_lib.last_error())
        return ids

    def undefined_flags(self) -> np.ndarray:
        """uint8 [H,W]: 1 where the reference's own result is undefined (uninitialised read, see oclr_abi.h)."""
        flags = np.empty((self.camera.height, self.camera.width), dtype=np.uint8)
        if not self._lib.oclr_frame_read_flags(self.handle, _ptr(flags)):
            raise OclrError(_lib.last_error())
        return flags

    @property
    def last_launches(self) -> int:
        return int(self._lib.oclr_frame_last_launches(self.handle))

    def push_rows(self, band_rows: int, rank: int, world: int, peer_planes, stream: int = 0):
        """Stores this rank's rows into the full-frame planes of every GPU in `peer_planes` (device addresses, one per rank)."""
        arr = (C.c_void_p * world)(*[int(p) for p in peer_planes])
        if not self._lib.oclr_frame_push_rows(self.handle, band_rows, rank, world, arr, C.c_void_p(stream)):
            raise OclrError(_lib.last_error())

    def device_planes(self):
        r, g, b = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._lib.oclr_frame_device_planes(self.handle, C.byref(r), C.byref(g), C.byref(b))
        return r.value, g.value, b.value

    def close(self):
        if getattr(self, "handle", None):
            self._lib.oclr_frame_destroy(self.handle)
            self.handle = None

    def __del__(self):
        self.close()


def write_image(path: str, planes, fmt: str | None = None, bmp_reference_cast: bool = False):
    """Writes uint16 [H,W] planes (r, g, b): .bmp (24 bit, value/256 -- or the reference's low-byte cast, writebmp.cpp:136-141),
    .ppm (16 bit) or .png (16 bit)."""
    lib = _lib.load()
    r, g, b = (_c(a, np.uint16) for a in planes)
    h, w = r.shape
    fmt = (fmt or str(path).rsplit(".", 1)[-1]).lower()
    p = str(path).encode()
    if fmt == "bmp":
        ok = lib.oclr_write_bmp(p, w, h, _ptr(r), _ptr(g), _ptr(b), 1 if bmp_reference_cast else 0)
    elif fmt == "ppm":
        ok = lib.oclr_write_ppm16(p, w, h, _ptr(r), _ptr(g), _ptr(b))
    elif fmt == "png":
        ok = lib.oclr_write_png16(p, w, h, _ptr(r), _ptr(g), _ptr(b))
    else:
        raise ValueError(f"unknown image format {fmt!r}")
    if not ok:
        raise OclrError(f"could not write {path}")


def set_option(name: str, value: int):
    if not _lib.load().oclr_set_option(name.encode(), int(value)):
        raise OclrError(_lib.last_error())


def band_partition(height: int, rank: int, world: int, band_rows: int = 128) -> list[tuple[int, int]]:
    """Rows owned by `rank`: bands of 128 rows (the reference's tile height, raytrace.c:507) dealt round-robin."""
    lib = _lib.load()
    n = lib.oclr_band_partition(height, band_rows, rank, world, None, 0)
    rows = (C.c_uint32 * (2 * max(n, 1)))()
    lib.oclr_band_partition(height, band_rows, rank, world, rows, n)
    return [(int(rows[2 * i]), int(rows[2 * i + 1])) for i in range(n)]
