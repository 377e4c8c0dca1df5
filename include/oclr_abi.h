/* oclr_abi.h -- C-ABI of libopencl_render_b200.so: the B200-native drop-in for the raytracer core loop of
 * ChrisHekmanOtoy/opencl_render (the OpenCL `Raytrace` kernel + the host code that launches it).
 *
 * Part 1 re-declares, with identical names, argument order, types and calling convention, every symbol the
 * reference declares in source/opencl/raytrace.h:37-106 -- that header is the reference's whole boundary between
 * the Cinema4D plugin (source/render.cpp) and the compute path.  A plugin built against the reference header links
 * against this library unchanged.
 * Part 2 is an extension the reference does not have: resident scenes and per-camera frames, so a scene is uploaded
 * once and rendered many times (the reference re-creates context, program and all 35 buffers on every call,
 * raytrace.c:283-491), rows can be split across GPUs, and foreign-function callers (ctypes) that cannot pass the
 * OpenCL vector unions by value get pointer-only doors.
 *
 * There is NO CPU implementation in this library: every compute entry point fails (returns 0 / NULL and sets
 * oclr_last_error()) when no sm_100 CUDA device is usable.
 */
#ifndef OCLR_ABI_H
#define OCLR_ABI_H

#include <stddef.h>
#include <stdint.h>
#include <time.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---------------------------------------------------------------------------------------------------------------
 * OpenCL host types.  If the real <CL/cl.h> was included first, use it; otherwise define layout- AND
 * calling-convention-compatible equivalents of source/3rdparty/opencl-1.2/include/CL/cl_platform.h:
 *   cl_float4/cl_float3  :995-1025  16 B, 16-aligned, carries a 128-bit vector member under __SSE__  (=> passed in ONE
 *                                   XMM register on x86-64 SysV, not two)
 *   cl_int4/cl_int3      :719-760   16 B, vector member under __SSE2__
 *   cl_uint2             :770-781   8 B, 64-bit vector member under __MMX__
 *   cl_float2            :995-1006  8 B;   cl_uchar4/cl_uchar3 :495-512  4 B;   cl_bool == cl_uint (CL/cl.h:49)
 * ------------------------------------------------------------------------------------------------------------- */
#if !defined(__CL_PLATFORM_H) && !defined(__OPENCL_CL_H)
typedef int8_t cl_char;
typedef uint8_t cl_uchar;
typedef uint16_t cl_ushort;
typedef int32_t cl_int;
typedef uint32_t cl_uint;
typedef uint64_t cl_ulong;
typedef float cl_float;
typedef double cl_double;
typedef cl_uint cl_bool;
#define CL_FALSE 0
#define CL_TRUE 1

#if defined(__GNUC__)
#define OCLR_ALIGNED(n) __attribute__((aligned(n)))
#else
#define OCLR_ALIGNED(n)
#endif
#if defined(__GNUC__) && defined(__MMX__)
#define OCLR_HAVE_V8 1
typedef cl_float oclr_v2f __attribute__((vector_size(8)));
typedef cl_int oclr_v2i __attribute__((vector_size(8)));
typedef cl_uint oclr_v2u __attribute__((vector_size(8)));
#endif
#if defined(__GNUC__) && defined(__SSE2__)
#define OCLR_HAVE_V16 1
typedef cl_float oclr_v4f __attribute__((vector_size(16)));
typedef cl_int oclr_v4i __attribute__((vector_size(16)));
#endif

typedef union {
    cl_float OCLR_ALIGNED(8) s[2];
#ifdef OCLR_HAVE_V8
    oclr_v2f v2;
#endif
} cl_float2;

typedef union {
    cl_float OCLR_ALIGNED(16) s[4];
#ifdef OCLR_HAVE_V8
    oclr_v2f v2[2];
#endif
#ifdef OCLR_HAVE_V16
    oclr_v4f v4;
#endif
} cl_float4;
typedef cl_float4 cl_float3;

typedef union {
    cl_int OCLR_ALIGNED(8) s[2];
#ifdef OCLR_HAVE_V8
    oclr_v2i v2;
#endif
} cl_int2;

typedef union {
    cl_int OCLR_ALIGNED(16) s[4];
#ifdef OCLR_HAVE_V8
    oclr_v2i v2[2];
#endif
#ifdef OCLR_HAVE_V16
    oclr_v4i v4;
#endif
} cl_int4;
typedef cl_int4 cl_int3;

typedef union {
    cl_uint OCLR_ALIGNED(8) s[2];
#ifdef OCLR_HAVE_V8
    oclr_v2u v2;
#endif
} cl_uint2;

typedef union {
    cl_uchar OCLR_ALIGNED(4) s[4];
} cl_uchar4;
typedef cl_uchar4 cl_uchar3;
#endif /* CL types */

/* Light types and material channels: source/opencl/raytrace_opencl.h:1-22 */
enum {
    OCLR_LIGHT_TYPE_OMNI = 0, OCLR_LIGHT_TYPE_SPOT = 1, OCLR_LIGHT_TYPE_SPOTRECT = 2, OCLR_LIGHT_TYPE_DISTANT = 3,
    OCLR_LIGHT_TYPE_PARALLEL = 4, OCLR_LIGHT_TYPE_PARSPOT = 5, OCLR_LIGHT_TYPE_PARSPOTRECT = 6, OCLR_LIGHT_TYPE_TUBE = 7,
    OCLR_LIGHT_TYPE_AREA = 8, OCLR_LIGHT_TYPE_PHOTOMETRIC = 9
};
enum {
    OCLR_MATERIAL_CHANNEL_COLOR = 0, OCLR_MATERIAL_CHANNEL_REFLECTION = 1, OCLR_MATERIAL_CHANNEL_TRANSPARENCY = 2,
    OCLR_MATERIAL_CHANNEL_BUMP = 3, OCLR_MATERIAL_CHANNEL_LUMINANCE = 4, OCLR_MATERIAL_CHANNEL_COUNT = 5
};

/* ===============================================================================================================
 * Part 1 -- the reference boundary, source/opencl/raytrace.h
 * ============================================================================================================= */

/* raytrace.h:37-44 -- small host helpers the reference's callers use (render.cpp:422,758-760,1197;
 * trianglelist.cpp:54-58,122-124,278,455).  Host-side fp32, reference operation order. */
cl_float dot(cl_float3 a, cl_float3 b);
cl_float3 cross(cl_float3 a, cl_float3 b);
cl_float3 normalize(cl_float3 v);
cl_float3 vector(cl_float3 a, cl_float3 b);
cl_float bindf(cl_float value, cl_float a, cl_float b);
cl_float GetPointToLineSqLen(cl_float3 origin, cl_float3 destination, cl_float3 point);
cl_bool RayIntersectsTriangle(cl_float3 origin, cl_float3 ray, cl_float minDistance, cl_float maxDistance, cl_float3 a,
                              cl_float3 b, cl_float3 c, cl_float* outRayMult, cl_float* outABL, cl_float* outACL);
cl_int3 GetBoxAddress(cl_int axesDivCount, cl_float3* boxMin, cl_float3 position);

/* raytrace.h:46-50 -- device list ("computation types").  Replaces the OpenCL platform/device enumeration of
 * raytrace.c:78-153 with CUDA device enumeration.  Index 0 keeps the reference's label "Local CPU single thread"
 * AS A NAME ONLY (there is no CPU path; RaytraceAll(0, ...) returns CL_FALSE); index k >= 1 is CUDA device k-1;
 * index deviceCount+1 (when deviceCount > 1) is "all CUDA devices of this box" (rows split across GPUs). */
void InitOpenCL(void);
void ResetComputationType(void);
cl_bool GetIsComputationTypeUpdated(void);
size_t GetComputationTypeCount(void);
cl_bool GetComputationTypeName(size_t id, size_t strLen, cl_char* str);

/* raytrace.h:52-56 -- progress / timing cells polled by the UI thread (raytrace.c:156-173).  Atomic here. */
cl_float GetProgress(void);
void SetProgress(cl_float p);
clock_t GetStartTime(void);
clock_t GetEndTime(void);
void ResetTime(void);

/* raytrace.h:58-106 -- render one frame.  Array length conventions as in raytrace.c:345-487:
 *   cameraPixelTriangleListStart/End: W*H entries each; cameraPixelTriangleList: cameraPixelTriangleListSize entries;
 *   scenePixelTriangleListStart: axesDivCount^3 + 1; scenePixelTriangleList: Start[axesDivCount^3] entries;
 *   sceneBoxMin: axesDivCount + 1 (axesDivCount a power of two); materialImageSize: 5*materialCount;
 *   materialImageStart: 5*materialCount + 1; triangleUv / triangleNormal: 3*triangleCount.
 * The caller owns every array; nothing is retained past return.  Output planes are overwritten (accumulated from
 * zero, as the OpenCL branch does, raytrace.c:476-486).  Returns CL_TRUE on success (raytrace.c:656). */
cl_bool RaytraceAll(cl_uint computationType,
                    cl_uint2 cameraImageDimension, cl_float3 cameraEye, cl_float3 cameraEyeToTopLeftVector,
                    cl_float3 cameraLeftToRightPixelSizeVector, cl_float3 cameraTopToBottomPixelSizeVector,
                    cl_float cameraPixelSizeInv,
                    cl_uint* cameraPixelTriangleListStart, cl_uint* cameraPixelTriangleListEnd,
                    cl_uint* cameraPixelTriangleList, ptrdiff_t cameraPixelTriangleListSize,
                    cl_uint sampleCount,
                    cl_uint vertexCount, cl_float3* vertex,
                    cl_uint triangleCount, cl_int3* triangleVertexIndex, cl_int* triangleMaterialId,
                    cl_float2* triangleUv, cl_float3* triangleNormal,
                    cl_int axesDivCount, cl_float3* sceneBoxMin, cl_uint* scenePixelTriangleListStart,
                    cl_uint* scenePixelTriangleList,
                    cl_uint materialCount, cl_uint2* materialImageSize, cl_int* materialImageStart,
                    cl_uint texturesSize, cl_uchar3* textures,
                    cl_uint lightCount, cl_int* lightType, cl_float3* lightPosition, cl_float3* lightDirection,
                    cl_float3* lightColour, cl_float* lightRadius, cl_float* lightHalfAttenuationDistance,
                    cl_ushort* outputRed, cl_ushort* outputGreen, cl_ushort* outputBlue);

/* ===============================================================================================================
 * Part 2 -- extension: resident scenes, frames, bands, pointer-only doors
 * ============================================================================================================= */

const char* oclr_last_error(void);          /* thread-local message of the last failing call on this thread */
int oclr_device_count(void);                /* CUDA devices visible (0 => every compute call fails) */
const char* oclr_version(void);

/* Scene arrays, exactly the reference's (same element types and length conventions as RaytraceAll). */
typedef struct oclr_scene_desc {
    cl_uint vertexCount;       const cl_float3* vertex;
    cl_uint triangleCount;     const cl_int3* triangleVertexIndex; const cl_int* triangleMaterialId;
    const cl_float2* triangleUv; const cl_float3* triangleNormal;
    cl_int axesDivCount;       const cl_float3* sceneBoxMin; const cl_uint* scenePixelTriangleListStart;
    const cl_uint* scenePixelTriangleList;
    cl_uint materialCount;     const cl_uint2* materialImageSize; const cl_int* materialImageStart;
    cl_uint texturesSize;      const cl_uchar3* textures;
    cl_uint lightCount;        const cl_int* lightType; const cl_float3* lightPosition; const cl_float3* lightDirection;
    const cl_float3* lightColour; const cl_float* lightRadius; const cl_float* lightHalfAttenuationDistance;
} oclr_scene_desc;

typedef struct oclr_camera {
    cl_uint width, height;
    cl_float eye[4];               /* cameraEye */
    cl_float eyeToTopLeft[4];      /* cameraEyeToTopLeftVector */
    cl_float leftToRight[4];       /* cameraLeftToRightPixelSizeVector */
    cl_float topToBottom[4];       /* cameraTopToBottomPixelSizeVector */
    cl_float pixelSizeInv;         /* cameraPixelSizeInv */
} oclr_camera;

typedef struct oclr_scene oclr_scene;
typedef struct oclr_frame oclr_frame;

/* Per-launch event counts behind the algorithmic-bytes figure (SURVEY.md section 8d). */
typedef struct oclr_counters {
    unsigned long long segments, primCandidates, gridRays, cells, cellsNonEmpty, gridCandidates, shadedHits,
        occluderLookups, bricksLoaded, emptyBrickCells, walkWarpIters, walkLaneIters, testWarpIters, testLaneIters,
        mailboxSkips, coarseSteps, coarseEnters, switchWarpIters, switchLaneIters,
        walkIdleLanes, walkParkedLanes, walkFinishedLanes, walkLowIters, walkExhaustedIters,
        splitAttempts, splitsDone, splitParts, splitCancelled,
        superSteps, superEnters, superRefines,   /* three-level walk: steps / level switches at super-brick granularity */
        /* per-warp timing of the trace kernel, counting build: when warps leave / see the queue dry, 32-us buckets since their start */
        exitHist00, exitHist01, exitHist02, exitHist03, exitHist04, exitHist05, exitHist06, exitHist07, exitHist08, exitHist09, exitHist10, exitHist11, exitHist12, exitHist13, exitHist14, exitHist15, exhaustHist00, exhaustHist01, exhaustHist02, exhaustHist03, exhaustHist04, exhaustHist05, exhaustHist06, exhaustHist07, exhaustHist08, exhaustHist09, exhaustHist10, exhaustHist11, exhaustHist12, exhaustHist13, exhaustHist14, exhaustHist15, warpOuterItersMax, warpOuterItersSum, warpsRun;   /* run-time split of long walks (experimental kernel instantiation) */
} oclr_counters;

typedef struct oclr_render_stats {
    float deviceMs;        /* CUDA-event time of the trace kernels on the launch stream */
    cl_uint launches;      /* kernels launched by this call */
    float traceMs;         /* CUDA-event time of the trace-stage launches alone (dominant kernel) */
    cl_uint traceLaunches; /* trace-stage rounds that had rays (rounds enqueued ahead that found none are not counted) */
    oclr_counters counters;
} oclr_render_stats;

/* 0: one thread per pixel (baseline, also the counting kernel of the reference accounting); 2: wavefront pipeline (production) */
enum { OCLR_KERNEL_SIMPLE = 0, OCLR_KERNEL_PIPE = 2, OCLR_KERNEL_DEFAULT = -1 };

/* Upload + repack a scene into the HBM of CUDA device `device`.  NULL on failure.  With sceneBoxMin ==
 * scenePixelTriangleListStart == NULL the grid (SceneTriangleList::New, axesDivCount cells per axis) is built on the device during
 * the upload and never exists on the host. */
oclr_scene* oclr_scene_create(int device, const oclr_scene_desc* desc);
void oclr_scene_destroy(oclr_scene* scene);
size_t oclr_scene_device_bytes(const oclr_scene* scene);

/* Test door: copies one packed device array back to `dst` (0 triGeo, 1 triShade, 2 bricks, 3 cellRange, 4 planes, 5 cellList,
 * 6 faceMask);
 * returns its size in bytes (nothing is copied when it exceeds `capacity`). */
size_t oclr_scene_debug_read(oclr_scene* scene, int which, void* dst, size_t capacity);

/* Camera (SetCamera, source/render.cpp:461-491): position / look-at / up / horizontal fov (radians) / size. */
void oclr_set_camera(oclr_camera* out, const cl_float position[3], const cl_float object[3], const cl_float up[3],
                     cl_float fov, cl_uint width, cl_uint height);

/* Per-camera triangle lists (CameraTriangleList::New output, source/util/trianglelist.cpp:520-626) uploaded to the
 * scene's device together with three zeroed 16-bit planes.  NULL on failure. */
oclr_frame* oclr_frame_create(oclr_scene* scene, const oclr_camera* camera, const cl_uint* cameraPixelTriangleListStart,
                              const cl_uint* cameraPixelTriangleListEnd, const cl_uint* cameraPixelTriangleList,
                              size_t cameraPixelTriangleListSize);
void oclr_frame_destroy(oclr_frame* frame);
/* Bytes of wavefront path state the frame holds in HBM (0 before its first render): about 510 B per path of the largest launch domain
 * so far for a scene without mirror / glass materials (ring of 2 slots), about 990 B otherwise (ring of 12, raytrace_opencl.c:461-468). */
size_t oclr_frame_state_bytes(const oclr_frame* frame);
/* Same frame, but CameraTriangleList::New (source/util/trianglelist.cpp:520-626) runs on the device from the resident scene:
 * no host lists are needed (they are per-frame inputs; the host builder costs 0.15-0.45 s per frame).  The lists are
 * entry-for-entry those of oclr_build_camera_lists(); oclr_frame_read_camera_lists() copies them back (`list` must hold
 * oclr_frame_camera_list_size() entries, `start`/`end` width*height entries each). */
oclr_frame* oclr_frame_create_device_lists(oclr_scene* scene, const oclr_camera* camera);
size_t oclr_frame_camera_list_size(const oclr_frame* frame);
int oclr_frame_read_camera_lists(oclr_frame* frame, cl_uint* start, cl_uint* end, cl_uint* list);

/* ---- edits of a resident scene and of a frame's camera ----
 * oclr_scene_update replaces the parts named in `parts` with the arrays of `desc` (same layout as oclr_scene_create; the fields of
 * other parts are ignored).  Afterwards the scene is byte for byte what oclr_scene_create would make from the new parts plus the
 * arrays it was created or last updated with: packed arrays, oclr_scene_device_bytes, path ring depth and every render and query result.
 *   OCLR_SCENE_LIGHTS     lightCount (0 included) and the six light arrays.
 *   OCLR_SCENE_MATERIALS  materialCount, materialImageSize, materialImageStart, texturesSize and textures, all together.  Without a
 *                         geometry edit in the same call the resident triangles' material ids are checked against the new count.
 *   OCLR_SCENE_GEOMETRY   vertices, triangle indices, material ids, UVs and normals at any counts; the grid from desc when given,
 *                         else built on the device at desc->axesDivCount cells per axis.
 * memory: OCLR_QUERY_HOST_MEMORY, or OCLR_QUERY_DEVICE_MEMORY -- the geometry arrays (the grid arrays included) are device memory of
 * the scene's device, read in place (vertex, indices, normals, sceneBoxMin 16-byte aligned, UVs 8, the rest 4).  Lights and
 * materials are always host arrays.
 * The call waits for all work already enqueued on the scene's device, builds the new parts into new buffers (a geometry edit can
 * briefly need twice the geometry's device bytes) and swaps them in only on success: a failed update returns 0 with oclr_last_error()
 * set and leaves the scene exactly as it was.  It returns with the edit in place; frames and queries see it from their next call.
 * Planes and float accumulators are not cleared: a progressive job continued across an edit mixes the two scenes.  After a geometry
 * edit a frame with device-built lists rebuilds them at its next use; a frame with caller lists refuses to render until
 * oclr_frame_set_camera_lists or oclr_frame_set_camera gives it lists for the new geometry.  Returns 1 on success. */
enum { OCLR_SCENE_LIGHTS = 1, OCLR_SCENE_MATERIALS = 2, OCLR_SCENE_GEOMETRY = 4 };
int oclr_scene_update(oclr_scene* scene, const oclr_scene_desc* desc, unsigned parts, int memory);
/* New camera of the same width x height; lists built on the device from the resident scene.  The frame keeps its planes, path state,
 * accumulation mode and progress counters; a different image size is refused (make a new frame).  The call waits for all work
 * enqueued on the frame's device.  A call that fails after the image-size check leaves the frame with the new camera and no lists: it
 * refuses to render until a camera is set successfully.  Returns 1 on success. */
int oclr_frame_set_camera(oclr_frame* frame, const oclr_camera* camera);
/* Same, with the caller's CameraTriangleList::New output (range-checked on the device as in oclr_frame_create). */
int oclr_frame_set_camera_lists(oclr_frame* frame, const oclr_camera* camera, const cl_uint* start, const cl_uint* end,
                                const cl_uint* list, size_t listSize);

/* Trace rows [rowBegin,rowEnd) with sampleCount samples per pixel on `cudaStream` (a cudaStream_t, NULL = default
 * stream).  `stats` may be NULL (then the call does not synchronise).  `countEvents` != 0 runs the counting build.
 * Returns 1 on success. */
int oclr_frame_render(oclr_frame* frame, cl_uint sampleCount, cl_uint rowBegin, cl_uint rowEnd, int kernelVariant,
                      int countEvents, void* cudaStream, oclr_render_stats* stats);
/* Same for the interleaved band set of one rank: the rows y with (y / bandRows) % worldSize == rank, in ONE launch. */
int oclr_frame_render_bands(oclr_frame* frame, cl_uint sampleCount, cl_uint bandRows, int rank, int worldSize, int kernelVariant,
                            int countEvents, void* cudaStream, oclr_render_stats* stats);
/* Progressive rendering (source/opencl/raytrace_opencl.c:726-741: every sample is truncated to an integer and ADDED to the 16-bit
 * planes -- the planes are the job's only partial state).  Samples [sampleBegin,sampleEnd) of a sampleCount-sample job: sample 0
 * overwrites the planes, later samples add, so a job of up to 16 384 samples (render.cpp:182) can be rendered over several calls,
 * looked at in between (oclr_frame_read), checkpointed and resumed on another frame or process (oclr_frame_write + sampleBegin). */
int oclr_frame_render_samples(oclr_frame* frame, cl_uint sampleCount, cl_uint sampleBegin, cl_uint sampleEnd, cl_uint rowBegin,
                              cl_uint rowEnd, int kernelVariant, int countEvents, void* cudaStream, oclr_render_stats* stats);
int oclr_frame_render_bands_samples(oclr_frame* frame, cl_uint sampleCount, cl_uint sampleBegin, cl_uint sampleEnd, cl_uint bandRows,
                                    int rank, int worldSize, int kernelVariant, int countEvents, void* cudaStream,
                                    oclr_render_stats* stats);
/* Host -> device copy of rows [rowBegin,rowEnd) of full-frame planes (restores a checkpoint). */
int oclr_frame_write(oclr_frame* frame, cl_uint rowBegin, cl_uint rowEnd, const cl_ushort* red, const cl_ushort* green,
                     const cl_ushort* blue, void* cudaStream);
/* Accumulation mode of a frame.  0 (default): the reference's rule above.  1: fp32 sums per pixel without per-sample truncation
 * (the reference loses up to one 16-bit step per sample: at 16 384 samples a quarter of the range); after every render call the
 * planes hold (int)(sum * 65535 / samples so far), i.e. the running mean converted by the reference's own rule.  With one sample
 * both modes give identical planes.  The accumulator is W*H x (sum r, sum g, sum b, samples) floats. */
enum { OCLR_ACCUMULATE_REFERENCE_16BIT = 0, OCLR_ACCUMULATE_FLOAT = 1 };
int oclr_frame_set_accumulation(oclr_frame* frame, int mode);
int oclr_frame_read_accum(oclr_frame* frame, cl_float* rgbn);
int oclr_frame_write_accum(oclr_frame* frame, const cl_float* rgbn);
/* Pixel-samples finished / requested by the render call in flight on this frame (callable from another thread). */
int oclr_frame_progress(oclr_frame* frame, unsigned long long* done, unsigned long long* total);
/* The "Estimated Time Left" of the plugin dialog (render.cpp:334-343) for the RaytraceAll in flight, on the wall clock; -1 while
 * unknown.  GetProgress() itself is live during RaytraceAll: it reads the device counter of every GPU taking part. */
double oclr_estimated_seconds_left(void);

/* Image output of finished planes (source/render.cpp:1372-1386, source/util/writebmp.cpp:124-177).  BMP mode 0: byte = value/256
 * (what the plugin displays); mode 1: the low byte, exactly what the reference's writebmp3s writes.  Return 1 on success. */
int oclr_write_bmp(const char* path, cl_uint width, cl_uint height, const cl_ushort* red, const cl_ushort* green, const cl_ushort* blue,
                   int mode);
int oclr_write_ppm16(const char* path, cl_uint width, cl_uint height, const cl_ushort* red, const cl_ushort* green, const cl_ushort* blue);
int oclr_write_png16(const char* path, cl_uint width, cl_uint height, const cl_ushort* red, const cl_ushort* green, const cl_ushort* blue);

/* Run-time options.  "slices": how many slices a launch domain is cut into (0 = automatic).  "ahead": tracing one round ahead
 * (0 never, 1 all segments but the camera's, 2 all, -1 automatic).  "cull_hidden_lights": 1 (default) skips the shadow rays of lights
 * on the side of a surface its segment does not see, whose contribution the shading never reads; 0 traces them all.  The planes are
 * the same either way.  "devices": the "all devices" computation type
 * (RaytraceAll(deviceCount + 1, ...), the analogue of the reference's multi-device tile loop raytrace.c:507-556) renders on the first
 * `value` GPUs of the box (0 = all of them).  Returns 1 if the option is known. */
int oclr_set_option(const char* name, int value);

/* Copy rows [rowBegin,rowEnd) of the planes to full-frame host arrays. */
int oclr_frame_read(oclr_frame* frame, cl_uint rowBegin, cl_uint rowEnd, cl_ushort* outputRed, cl_ushort* outputGreen,
                    cl_ushort* outputBlue, void* cudaStream);
/* Primary-hit triangle id per pixel of sample 0 (0xFFFFFFFF = miss); W*H entries. */
int oclr_frame_read_primary_ids(oclr_frame* frame, cl_uint* ids);
/* Per-pixel flags, W*H bytes: bit 0 = the reference's own result is undefined at this pixel (it reads uninitialised
 * barycentrics when a bump-mapped surface is hit by a non-camera ray whose first helper ray, raytrace_opencl.c:244, does
 * not meet the triangle plane); parity checks exclude exactly these pixels. */
int oclr_frame_read_flags(oclr_frame* frame, cl_uchar* flags);
/* Number of CUDA kernels the last render call on this frame launched. */
cl_uint oclr_frame_last_launches(const oclr_frame* frame);
/* Device addresses of the three planes (W*H cl_ushort each) -- for NCCL gathers issued by the host layer. */
void oclr_frame_device_planes(oclr_frame* frame, void** red, void** green, void** blue);

/* Frame assembly over NVLink peer memory: stores the rows `rank` owns (bands of bandRows rows dealt round-robin over worldSize)
 * from the frame's planes into the full-frame planes ([3][H][W] cl_ushort: red, green, blue) of EVERY GPU listed in peerPlanes --
 * worldSize device pointers valid in this process (the rank's own buffer and its peers', e.g. from CUDA IPC / symmetric memory).
 * One kernel on cudaStream; the caller orders a cross-GPU barrier behind it.  The reference has no counterpart (one device). */
int oclr_frame_push_rows(oclr_frame* frame, cl_uint bandRows, int rank, int worldSize, void* const* peerPlanes, void* cudaStream);

/* Batched ray queries on a resident scene, with the reference's own semantics.  The reference has no such door: its only caller of
 * RayIntersectsTriangles is the Raytrace kernel.  A query runs on the scene's device.
 *
 * Rays: origin4[i] = (ox, oy, oz, minD), direction4[i] = (dx, dy, dz, maxD) -- the reference's cl_float3 layout with the range in the
 * unused 4th component.  The direction is not normalised: t is in its units.  `excluded` = cl_uint[count] (the triangle the ray
 * starts on, RayIntersectsTriangles' `excludeTriangle`), or NULL = 0xFFFFFFFF for every ray.  The caller's input arrays are never
 * written.  count == 0 is accepted.
 *
 * oclr_scene_intersect: RayIntersectsTriangles (raytrace_opencl.c:324-401) exactly.  The first grid cell along the ray that holds any
 * hit with minD < t < maxD wins; inside it the smallest t, and on equal t the earliest entry of the cell's list.
 *   hit4[i] = (as_float(triangle), t, abL, acL); a miss is (as_float(0xFFFFFFFF), maxD, 0, 0).
 * oclr_scene_transmittance: the shadow loop of raytrace_opencl.c:608-627.  att = (1,1,1); closest hit with the same excluded triangle;
 * at each blocker att *= its TRANSPARENCY texel at (abL, acL) (0 without that channel) and the query continues from minD = t while all
 * three components are > 0 -- the loop stops as soon as ANY component reaches 0 and the others are returned as they are.
 *   att4[i] = (r, g, b, as_float(last triangle met, or 0xFFFFFFFF)).
 *
 * Preconditions.  The trace kernel orders the hits of a ray by the bit pattern of t, which requires t > 0 and so minD >= 0 (-0.0 is
 * allowed).  A ray with minD < 0, a NaN minD or maxD, or a non-finite origin or direction component is NOT traced: its result is
 * (0xFFFFFFFF, NaN, 0, 0), transmittance (NaN, NaN, NaN, 0xFFFFFFFF).  A real miss never has a NaN t.  A ray with !(minD < maxD) or a
 * zero direction is not traced either; no t can pass minD < t < maxD, so it gets the ordinary miss (0xFFFFFFFF, maxD, 0, 0) and att
 * (1, 1, 1).
 *
 * memory: OCLR_QUERY_HOST_MEMORY -- host arrays, staged through the library (the call synchronises).  OCLR_QUERY_DEVICE_MEMORY --
 * device memory of the scene's device; origin4 / direction4 / hit4 / att4 16-byte aligned, excluded 4-byte aligned; any other pointer
 * fails the call with a message.  Inputs are read in place.
 * Rays are processed in internal batches of 2^21 (2 097 152); scratch is allocated per call, stream-ordered on cudaStream (up to about
 * 190 MB for closest hit, 270 MB for transmittance, plus 110 MB of staging for host memory), so queries on one scene from different
 * streams share no state.
 * `stats` as in oclr_frame_render: NULL = no synchronisation for a device-memory closest-hit query; host-memory queries and transmittance
 * always synchronise (the loop reads its ray count back once per chunk of rounds).  stats->deviceMs is the whole call;
 * stats->traceLaunches the trace rounds enqueued; with countEvents, counters.gridRays counts every closest-hit trace (transmittance: of
 * every round).  Returns 1 on success. */
enum { OCLR_QUERY_HOST_MEMORY = 0, OCLR_QUERY_DEVICE_MEMORY = 1 };
int oclr_scene_intersect(oclr_scene* scene, size_t count, const cl_float* origin4, const cl_float* direction4, const cl_uint* excluded,
                         cl_float* hit4, int memory, int countEvents, void* cudaStream, oclr_render_stats* stats);
int oclr_scene_transmittance(oclr_scene* scene, size_t count, const cl_float* origin4, const cl_float* direction4, const cl_uint* excluded,
                             cl_float* att4, int memory, int countEvents, void* cudaStream, oclr_render_stats* stats);

/* Radiance along caller rays: the colour the reference computes for a pixel-sample (raytrace_opencl.c:452-725 -- shading, lights and
 * their shadow loops, the ring of diffuse / mirror / glass segments, the RNG draw order), with the camera segment replaced by the
 * caller's ray.  For light baking, light probes and projections the pinhole camera cannot express (panoramas, stereo, orthographic).
 *
 * Rays as for the queries above, with maxD = direction4[i].w = +inf (ring segments have no far limit).  Ring slot 0 is {o, d, minD,
 * excluded, weight (1,1,1), 12 bounces}, an ordinary grid segment: its closest hit is RayIntersectsTriangles, never a camera-list scan,
 * and so is that of its glass continuation.  There are no jitter draws: sample s of ray i starts from rng = (indexBase + i) *
 * sampleCount + s + 1 (64-bit), the frame's pixel * S + s + 1 rule with the ray's global index for the pixel, so a job split across
 * calls (indexBase = index of the call's first ray) gives the same results.  sampleCount >= 1; a call renders all samples.
 *   rgb4[i] = (R, G, B, as_float(tri0)): R = (colour_0 + colour_1 + ... ) / (float)sampleCount, an fp32 sum in sample order and one
 *   IEEE division, where colour_s is the value the reference converts at :726-741 (before its * 65535 / S truncation); tri0 = the
 *   triangle the ray itself hits in sample 0, or 0xFFFFFFFF.
 * A ray with minD < 0, a NaN minD, a maxD other than +inf, or a non-finite origin or direction component is not traced: (NaN, NaN,
 * NaN, 0xFFFFFFFF), which no real result has.  A zero direction or minD = +inf meets nothing: (0, 0, 0, 0xFFFFFFFF) without a trace.
 * flags: NULL or cl_uchar[count]; bit 0 = the reference's own result is undefined for this ray, as in oclr_frame_read_flags (every
 * caller ray is a non-camera segment, so this can happen on its very first hit).
 * camera: bump-mapped normals read its leftToRight, topToBottom and pixelSizeInv (raytrace_opencl.c:195-263), nothing else of it.
 * It may be NULL only if no material has a BUMP channel; otherwise the call fails.
 * memory, alignment (rgb4 16 bytes, flags 1), pointer checks, countEvents and cudaStream as for the queries above.  Rays go in
 * internal batches of 2^20 (1 048 576) with about 1 KB of path state per ray of a batch (about 1.1 GB stream-ordered scratch; host
 * memory adds about 55 MB of staging).  The call always synchronises (it reads each sample's round count back).  With countEvents,
 * counters.segments / shadedHits / gridRays / occluderLookups count ring segments, shaded hits, grid walks (closest hits and every
 * walk of the shadow loops) and transparency lookups of blockers.  Returns 1 on success. */
int oclr_scene_radiance(oclr_scene* scene, const oclr_camera* camera, size_t count, const cl_float* origin4, const cl_float* direction4,
                        const cl_uint* excluded, unsigned long long indexBase, cl_uint sampleCount, cl_float* rgb4, cl_uchar* flags,
                        int memory, int countEvents, void* cudaStream, oclr_render_stats* stats);

/* Rows of a W x H image owned by `rank` of `worldSize` when the image is cut into bands of `bandRows` rows dealt
 * round-robin (SURVEY.md section 8e; band height 128 = the reference's tile height, raytrace.c:507).  Writes up to
 * `maxBands` [begin,end) pairs to `rows` and returns the number of bands owned. */
int oclr_band_partition(cl_uint height, cl_uint bandRows, int rank, int worldSize, cl_uint* rows, int maxBands);

/* Pointer-only door onto RaytraceAll for foreign-function callers: the five by-value vectors become pointers
 * (dimension: 2 x cl_uint; the others: >= 3 x cl_float). */
cl_bool oclr_raytrace_all_p(cl_uint computationType, const cl_uint* cameraImageDimension, const cl_float* cameraEye,
                            const cl_float* cameraEyeToTopLeftVector, const cl_float* cameraLeftToRightPixelSizeVector,
                            const cl_float* cameraTopToBottomPixelSizeVector, cl_float cameraPixelSizeInv,
                            const oclr_scene_desc* scene, const cl_uint* cameraPixelTriangleListStart,
                            const cl_uint* cameraPixelTriangleListEnd, const cl_uint* cameraPixelTriangleList,
                            ptrdiff_t cameraPixelTriangleListSize, cl_uint sampleCount, cl_ushort* outputRed,
                            cl_ushort* outputGreen, cl_ushort* outputBlue);

/* Acceleration-list builders (host restatements of CameraTriangleList::New / SceneTriangleList::New,
 * source/util/trianglelist.cpp:520-626, 655-737): the inputs the kernel cannot run without.  Results are
 * malloc'ed; free with oclr_free(). */
typedef struct oclr_camera_lists {
    cl_uint* start; cl_uint* end; cl_uint* list; size_t listSize; cl_uint pixelCount;
} oclr_camera_lists;
typedef struct oclr_scene_grid {
    cl_int axesDivCount; cl_float3* boxMin; cl_uint* start; cl_uint* list; size_t listSize;
} oclr_scene_grid;
int oclr_build_camera_lists(const oclr_camera* camera, cl_uint vertexCount, const cl_float3* vertex, cl_uint triangleCount,
                            const cl_int3* triangleVertexIndex, oclr_camera_lists* out);
int oclr_build_scene_grid(cl_int axesDivCount, cl_uint vertexCount, const cl_float3* vertex, cl_uint triangleCount,
                          const cl_int3* triangleVertexIndex, oclr_scene_grid* out);
/* SceneTriangleList::New (source/util/trianglelist.cpp:655-737) on CUDA device `device`: same output as oclr_build_scene_grid,
 * entry for entry (the reference needs 10 s at 101 k triangles, the host builder 0.3 s, this tens of milliseconds). */
int oclr_build_scene_grid_device(int device, cl_int axesDivCount, cl_uint vertexCount, const cl_float3* vertex, cl_uint triangleCount,
                                 const cl_int3* triangleVertexIndex, oclr_scene_grid* out);
void oclr_free_camera_lists(oclr_camera_lists* lists);
void oclr_free_scene_grid(oclr_scene_grid* grid);

#ifdef __cplusplus
}
#endif
#endif /* OCLR_ABI_H */
