// abi.cpp -- the exported C-ABI (include/oclr_abi.h).  Part 1 mirrors source/opencl/raytrace.h:46-106 symbol for
// symbol; Part 2 is the resident scene/frame extension.  Compiled by g++ (the by-value OpenCL vector unions carry
// GCC vector members, see the header), calls into the CUDA runtime layer through runtime.h.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <atomic>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/oclr_abi.h"
#include "runtime.h"

namespace oclr {
void set_camera(oclr_camera* out, const float position[3], const float object[3], const float up3[3], float fov, uint32_t w,
                uint32_t h);
bool build_camera_lists(const oclr_camera* cam, uint32_t vertexCount, const float4* vertex, uint32_t triangleCount,
                        const int32_t* triIdx, oclr_camera_lists* out);
bool build_scene_grid(int32_t n, uint32_t vertexCount, const float4* vertex, uint32_t triangleCount, const int32_t* triIdx,
                      oclr_scene_grid* out);
}  // namespace oclr

using namespace oclr;

static_assert(sizeof(cl_float3) == 16 && sizeof(cl_int3) == 16 && sizeof(cl_uint2) == 8 && sizeof(cl_float2) == 8 &&
                  sizeof(cl_uchar3) == 4,
              "OpenCL host type layout (cl_platform.h)");
static_assert(sizeof(oclr_counters) == sizeof(Counters), "counter layout");
static_assert(sizeof(oclr_camera) == sizeof(Camera), "camera layout");

static thread_local std::string g_err;
static void fail(const std::string& m) {
    g_err = m;
    fprintf(stderr, "[opencl_render_b200] %s\n", m.c_str());
}

struct oclr_scene {
    Scene* impl;
};
struct oclr_frame {
    Frame* impl;
    oclr_scene* scene;
};

// ---- device list: raytrace.c:73-153 ------------------------------------------------------------------------------------
static std::mutex g_devMutex;
static std::atomic<cl_uint> g_devUpdated(CL_FALSE);
static int g_devCount = 0;
static char g_devName[256][256];

void InitOpenCL(void) {
    std::lock_guard<std::mutex> lock(g_devMutex);
    int n = device_count();
    if (n > 254) n = 254;
    for (int i = 0; i < n; ++i)
        if (!device_name(i, g_devName[i], sizeof(g_devName[i]))) snprintf(g_devName[i], sizeof(g_devName[i]), "CUDA device #%d", i);
    g_devCount = n;
    if (n > 1) snprintf(g_devName[n], sizeof(g_devName[n]), "CUDA all %d devices (row bands, shared upload over NVLink)", n);
    g_devUpdated = CL_TRUE;
}
void ResetComputationType(void) {
    std::lock_guard<std::mutex> lock(g_devMutex);
    if (g_devUpdated) {
        g_devUpdated = CL_FALSE;
        g_devCount = 0;
    }
}
cl_bool GetIsComputationTypeUpdated(void) { return g_devUpdated; }
size_t GetComputationTypeCount(void) {
    std::lock_guard<std::mutex> lock(g_devMutex);
    return 1 + (size_t)g_devCount + (g_devCount > 1 ? 1 : 0);
}
cl_bool GetComputationTypeName(size_t id, size_t strLen, cl_char* str) {
    std::lock_guard<std::mutex> lock(g_devMutex);
    const char* name = nullptr;
    if (id == 0)
        name = "Local CPU single thread";  // label kept for list-index compatibility; RaytraceAll(0) is refused
    else if (id - 1 < (size_t)g_devCount + (g_devCount > 1 ? 1 : 0))
        name = g_devName[id - 1];
    if (!name || !str) return CL_FALSE;
    // The reference accepts strlen(name) <= strLen and then strcpy's strlen + 1 bytes (raytrace.c:139-141: one past the caller's
    // buffer when the lengths are equal).  Here the name is returned only when it fits WITH its terminator.
    if (strlen(name) < strLen) {
        memcpy(str, name, strlen(name) + 1);
        return CL_TRUE;
    }
    return CL_FALSE;
}

// ---- progress / timing cells: raytrace.c:155-173 --------------------------------------------------------------------------
static std::atomic<float> g_progress(0.f);
static std::atomic<clock_t> g_startTime(0), g_endTime(0);
// Frames RaytraceAll is rendering right now: while there are any, GetProgress() is live -- pixel-samples finished (a device
// counter the logic kernel bumps, read through the frame's own stream) over pixel-samples requested -- instead of the
// reference's once-per-second event poll (raytrace.c:566-587).  Capped at 0.999 like the reference (:580); 1.0 is the caller's
// (render.cpp:1397).
static std::mutex g_liveMutex;
static std::vector<Frame*> g_liveFrames;
static std::atomic<double> g_wallStart(0.0), g_wallLastChange(0.0);
static double wall_now() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}
cl_float GetProgress(void) {
    std::lock_guard<std::mutex> lock(g_liveMutex);
    if (!g_liveFrames.empty()) {
        unsigned long long done = 0, total = 0;
        for (Frame* f : g_liveFrames) {
            unsigned long long d = 0, t = 0;
            if (frame_progress(f, &d, &t)) {
                done += d;
                total += t;
            }
        }
        if (total) {
            const float p = 0.999f * (float)((double)done / (double)total);
            if (p > g_progress.load()) {
                g_progress.store(p);
                g_wallLastChange.store(wall_now());
            }
        }
    }
    return g_progress.load();
}
void SetProgress(cl_float p) {
    g_progress.store(p);
    g_wallLastChange.store(wall_now());
}
// Estimated seconds left, the dialog's rule (render.cpp:334-343): (start - now) + (last progress change - start) / progress,
// on the wall clock; negative values are clamped to 0 and "unknown" (no progress yet) is reported as -1.
double oclr_estimated_seconds_left(void) {
    const float p = GetProgress();
    const double start = g_wallStart.load(), last = g_wallLastChange.load(), now = wall_now();
    if (!(p > 0.f) || start == 0.0) return -1.0;
    const double t = (start - now) + (last - start) / (double)p;
    return t < 0.0 ? 0.0 : t;
}
int oclr_frame_progress(oclr_frame* frame, unsigned long long* done, unsigned long long* total);
clock_t GetStartTime(void) { return g_startTime.load(); }
clock_t GetEndTime(void) { return g_endTime.load(); }
void ResetTime(void) {
    g_startTime = 0;
    g_endTime = 0;
}

// ---- extension -----------------------------------------------------------------------------------------------------------
const char* oclr_last_error(void) { return g_err.c_str(); }
int oclr_device_count(void) { return device_count(); }
const char* oclr_version(void) { return "opencl_render_b200 0.1 (sm_100a)"; }
// Devices the "all devices" computation type renders on: all of them, or the first k (oclr_set_option("devices", k)).
static std::atomic<int> g_allDevicesLimit(0);

int oclr_set_option(const char* name, int value) {
    if (name && strcmp(name, "slices") == 0) {
        set_slice_count(value);
        return 1;
    }
    if (name && strcmp(name, "ahead") == 0) {
        set_ahead_mode(value);
        return 1;
    }
    if (name && strcmp(name, "cull_hidden_lights") == 0) {
        set_cull_hidden_lights(value);
        return 1;
    }
    if (name && strcmp(name, "devices") == 0) {   // the "all devices" computation type uses the first `value` GPUs (0 = all)
        g_allDevicesLimit.store(value < 0 ? 0 : value);
        return 1;
    }
    fail(std::string("oclr_set_option: unknown option ") + (name ? name : "(null)"));
    return 0;
}

static HostScene to_host(const oclr_scene_desc* d) {
    HostScene h;
    h.vertexCount = d->vertexCount;
    h.vertex = (const float4*)d->vertex;
    h.triangleCount = d->triangleCount;
    h.triIdx = (const int32_t*)d->triangleVertexIndex;
    h.triMat = d->triangleMaterialId;
    h.triUv = (const float*)d->triangleUv;
    h.triNormal = (const float4*)d->triangleNormal;
    h.axesDivCount = d->axesDivCount;
    h.boxMin = (const float4*)d->sceneBoxMin;
    h.gridStart = d->scenePixelTriangleListStart;
    h.gridList = d->scenePixelTriangleList;
    h.materialCount = d->materialCount;
    h.matSize = (const uint2*)d->materialImageSize;
    h.matStart = d->materialImageStart;
    h.texturesSize = d->texturesSize;
    h.textures = (const uchar4*)d->textures;
    h.lightCount = d->lightCount;
    h.lightType = d->lightType;
    h.lightPos = (const float4*)d->lightPosition;
    h.lightDir = (const float4*)d->lightDirection;
    h.lightColour = (const float4*)d->lightColour;
    h.lightRadius = d->lightRadius;
    h.lightHalf = d->lightHalfAttenuationDistance;
    return h;
}

oclr_scene* oclr_scene_create(int device, const oclr_scene_desc* desc) {
    if (!desc) {
        fail("oclr_scene_create: null description");
        return nullptr;
    }
    std::string err;
    Scene* s = scene_create(device, to_host(desc), err);
    if (!s) {
        fail("oclr_scene_create: " + err);
        return nullptr;
    }
    oclr_scene* h = new oclr_scene();
    h->impl = s;
    return h;
}
void oclr_scene_destroy(oclr_scene* scene) {
    if (!scene) return;
    scene_destroy(scene->impl);
    delete scene;
}
size_t oclr_scene_debug_read(oclr_scene* scene, int which, void* dst, size_t capacity) {
    return scene ? scene_debug_read(scene->impl, which, dst, capacity) : 0;
}
size_t oclr_scene_device_bytes(const oclr_scene* scene) { return scene ? scene_device_bytes(scene->impl) : 0; }
static_assert(OCLR_SCENE_LIGHTS == kSceneLights && OCLR_SCENE_MATERIALS == kSceneMaterials && OCLR_SCENE_GEOMETRY == kSceneGeometry, "part bits");
int oclr_scene_update(oclr_scene* scene, const oclr_scene_desc* desc, unsigned parts, int memory) {
    if (parts == 0 || (parts & ~(unsigned)(OCLR_SCENE_LIGHTS | OCLR_SCENE_MATERIALS | OCLR_SCENE_GEOMETRY))) {
        fail("oclr_scene_update: parts must be a non-empty combination of OCLR_SCENE_LIGHTS, OCLR_SCENE_MATERIALS and OCLR_SCENE_GEOMETRY, "
             "got " + std::to_string(parts));
        return 0;
    }
    if (memory != OCLR_QUERY_HOST_MEMORY && memory != OCLR_QUERY_DEVICE_MEMORY) {
        fail("oclr_scene_update: unknown memory kind " + std::to_string(memory));
        return 0;
    }
    if (!scene || !desc) {
        fail("oclr_scene_update: null scene or description");
        return 0;
    }
    std::string err;
    if (!scene_update(scene->impl, to_host(desc), parts, memory == OCLR_QUERY_DEVICE_MEMORY, err)) {
        fail("oclr_scene_update: " + err);
        return 0;
    }
    return 1;
}

void oclr_set_camera(oclr_camera* out, const cl_float position[3], const cl_float object[3], const cl_float up[3], cl_float fov,
                     cl_uint width, cl_uint height) {
    set_camera(out, position, object, up, fov, width, height);
}

static Camera to_camera(const oclr_camera* c) {
    Camera k;
    memcpy(&k, c, sizeof(Camera));
    return k;
}

oclr_frame* oclr_frame_create(oclr_scene* scene, const oclr_camera* camera, const cl_uint* start, const cl_uint* end,
                              const cl_uint* list, size_t listSize) {
    if (!scene || !camera) {
        fail("oclr_frame_create: null scene or camera");
        return nullptr;
    }
    if (!start || !end) {
        fail("oclr_frame_create: camera triangle lists missing (oclr_frame_create_device_lists builds them on the device)");
        return nullptr;
    }
    std::string err;
    Frame* f = frame_create(scene->impl, to_camera(camera), start, end, list, listSize, err);
    if (!f) {
        fail("oclr_frame_create: " + err);
        return nullptr;
    }
    oclr_frame* h = new oclr_frame();
    h->impl = f;
    h->scene = scene;
    return h;
}
oclr_frame* oclr_frame_create_device_lists(oclr_scene* scene, const oclr_camera* camera) {
    if (!scene || !camera) {
        fail("oclr_frame_create_device_lists: null scene or camera");
        return nullptr;
    }
    std::string err;
    Frame* f = frame_create(scene->impl, to_camera(camera), nullptr, nullptr, nullptr, 0, err);
    if (!f) {
        fail("oclr_frame_create_device_lists: " + err);
        return nullptr;
    }
    oclr_frame* h = new oclr_frame();
    h->impl = f;
    h->scene = scene;
    return h;
}
int oclr_frame_set_camera(oclr_frame* frame, const oclr_camera* camera) {
    std::string err;
    if (!frame || !camera || !frame_set_camera(frame->impl, to_camera(camera), nullptr, nullptr, nullptr, 0, err)) {
        fail("oclr_frame_set_camera: " + (err.empty() ? std::string("null frame or camera") : err));
        return 0;
    }
    return 1;
}
int oclr_frame_set_camera_lists(oclr_frame* frame, const oclr_camera* camera, const cl_uint* start, const cl_uint* end, const cl_uint* list,
                                size_t listSize) {
    std::string err;
    if (!frame || !camera || !start || !end) {
        fail("oclr_frame_set_camera_lists: null frame, camera or camera triangle lists");
        return 0;
    }
    if (!frame_set_camera(frame->impl, to_camera(camera), start, end, list, listSize, err)) {
        fail("oclr_frame_set_camera_lists: " + err);
        return 0;
    }
    return 1;
}
size_t oclr_frame_camera_list_size(const oclr_frame* frame) { return frame ? frame_camera_list_size(frame->impl) : 0; }
int oclr_frame_read_camera_lists(oclr_frame* frame, cl_uint* start, cl_uint* end, cl_uint* list) {
    std::string err;
    if (!frame || !frame_read_camera_lists(frame->impl, start, end, list, err)) {
        fail("oclr_frame_read_camera_lists: " + (frame ? err : std::string("null frame")));
        return 0;
    }
    return 1;
}
size_t oclr_frame_state_bytes(const oclr_frame* frame) { return frame ? frame_state_bytes(frame->impl) : 0; }
void oclr_frame_destroy(oclr_frame* frame) {
    if (!frame) return;
    frame_destroy(frame->impl);
    delete frame;
}

static int default_variant() {
    static const int v = [] {
        const char* e = getenv("OCLR_KERNEL_VARIANT");   // experiment knob
        return e ? atoi(e) : (int)kKernelPipe;
    }();
    return v;
}
static int pick_variant(int v) { return v == OCLR_KERNEL_DEFAULT ? default_variant() : v; }

static void copy_stats(oclr_render_stats* stats, const RenderStats& rs) {
    stats->deviceMs = rs.deviceMs;
    stats->launches = rs.launches;
    stats->traceMs = rs.traceMs;
    stats->traceLaunches = rs.traceLaunches;
    memcpy(&stats->counters, &rs.counters, sizeof(Counters));
}

int oclr_frame_render_samples(oclr_frame* frame, cl_uint sampleCount, cl_uint sampleBegin, cl_uint sampleEnd, cl_uint rowBegin, cl_uint rowEnd,
                              int kernelVariant, int countEvents, void* cudaStream, oclr_render_stats* stats) {
    if (!frame) {
        fail("oclr_frame_render: null frame");
        return 0;
    }
    std::string err;
    RenderStats rs;
    if (!frame_render(frame->impl, sampleCount, sampleBegin, sampleEnd, rowBegin, rowEnd, pick_variant(kernelVariant), countEvents != 0,
                      cudaStream, stats ? &rs : nullptr, err)) {
        fail("oclr_frame_render: " + err);
        return 0;
    }
    if (stats) copy_stats(stats, rs);
    return 1;
}
int oclr_frame_render(oclr_frame* frame, cl_uint sampleCount, cl_uint rowBegin, cl_uint rowEnd, int kernelVariant, int countEvents,
                      void* cudaStream, oclr_render_stats* stats) {
    return oclr_frame_render_samples(frame, sampleCount, 0, sampleCount, rowBegin, rowEnd, kernelVariant, countEvents, cudaStream, stats);
}

// What every query entry checks before the runtime does: a scene and a known memory kind.
static bool query_entry_ok(const char* name, oclr_scene* scene, int memory) {
    if (!scene) {
        fail(std::string(name) + ": null scene");
        return false;
    }
    if (memory != OCLR_QUERY_HOST_MEMORY && memory != OCLR_QUERY_DEVICE_MEMORY) {
        fail(std::string(name) + ": unknown memory kind " + std::to_string(memory));
        return false;
    }
    return true;
}
static int scene_query_entry(const char* name, bool transmit, oclr_scene* scene, size_t count, const cl_float* origin4, const cl_float* direction4,
                             const cl_uint* excluded, cl_float* out4, int memory, int countEvents, void* cudaStream, oclr_render_stats* stats) {
    if (!query_entry_ok(name, scene, memory)) return 0;
    std::string err;
    RenderStats rs;
    const bool dev = memory == OCLR_QUERY_DEVICE_MEMORY;
    const bool ok = transmit ? scene_transmittance(scene->impl, count, origin4, direction4, excluded, out4, dev, countEvents != 0, cudaStream,
                                                   stats ? &rs : nullptr, err)
                             : scene_intersect(scene->impl, count, origin4, direction4, excluded, out4, dev, countEvents != 0, cudaStream,
                                               stats ? &rs : nullptr, err);
    if (!ok) {
        fail(std::string(name) + ": " + err);
        return 0;
    }
    if (stats) copy_stats(stats, rs);
    return 1;
}
int oclr_scene_intersect(oclr_scene* scene, size_t count, const cl_float* origin4, const cl_float* direction4, const cl_uint* excluded,
                         cl_float* hit4, int memory, int countEvents, void* cudaStream, oclr_render_stats* stats) {
    return scene_query_entry("oclr_scene_intersect", false, scene, count, origin4, direction4, excluded, hit4, memory, countEvents, cudaStream, stats);
}
int oclr_scene_transmittance(oclr_scene* scene, size_t count, const cl_float* origin4, const cl_float* direction4, const cl_uint* excluded,
                             cl_float* att4, int memory, int countEvents, void* cudaStream, oclr_render_stats* stats) {
    return scene_query_entry("oclr_scene_transmittance", true, scene, count, origin4, direction4, excluded, att4, memory, countEvents, cudaStream,
                             stats);
}
int oclr_scene_radiance(oclr_scene* scene, const oclr_camera* camera, size_t count, const cl_float* origin4, const cl_float* direction4,
                        const cl_uint* excluded, unsigned long long indexBase, cl_uint sampleCount, cl_float* rgb4, cl_uchar* flags, int memory,
                        int countEvents, void* cudaStream, oclr_render_stats* stats) {
    if (!query_entry_ok("oclr_scene_radiance", scene, memory)) return 0;
    std::string err;
    RenderStats rs;
    Camera cam;
    if (camera) cam = to_camera(camera);
    if (!scene_radiance(scene->impl, camera ? &cam : nullptr, count, origin4, direction4, excluded, indexBase, sampleCount, rgb4, flags,
                        memory == OCLR_QUERY_DEVICE_MEMORY, countEvents != 0, cudaStream, stats ? &rs : nullptr, err)) {
        fail("oclr_scene_radiance: " + err);
        return 0;
    }
    if (stats) copy_stats(stats, rs);
    return 1;
}

int oclr_frame_render_bands_samples(oclr_frame* frame, cl_uint sampleCount, cl_uint sampleBegin, cl_uint sampleEnd, cl_uint bandRows, int rank,
                                    int worldSize, int kernelVariant, int countEvents, void* cudaStream, oclr_render_stats* stats) {
    if (!frame || rank < 0 || worldSize < 1) {
        fail("oclr_frame_render_bands: bad argument");
        return 0;
    }
    std::string err;
    RenderStats rs;
    if (!frame_render_bands(frame->impl, sampleCount, sampleBegin, sampleEnd, bandRows, (uint32_t)rank, (uint32_t)worldSize,
                            pick_variant(kernelVariant), countEvents != 0, cudaStream, stats ? &rs : nullptr, err)) {
        fail("oclr_frame_render_bands: " + err);
        return 0;
    }
    if (stats) copy_stats(stats, rs);
    return 1;
}
int oclr_frame_render_bands(oclr_frame* frame, cl_uint sampleCount, cl_uint bandRows, int rank, int worldSize, int kernelVariant,
                            int countEvents, void* cudaStream, oclr_render_stats* stats) {
    return oclr_frame_render_bands_samples(frame, sampleCount, 0, sampleCount, bandRows, rank, worldSize, kernelVariant, countEvents, cudaStream,
                                           stats);
}

int oclr_frame_write(oclr_frame* frame, cl_uint rowBegin, cl_uint rowEnd, const cl_ushort* r, const cl_ushort* g, const cl_ushort* b,
                     void* cudaStream) {
    std::string err;
    if (!frame || !r || !g || !b || !frame_write(frame->impl, rowBegin, rowEnd, r, g, b, cudaStream, err)) {
        fail("oclr_frame_write: " + (err.empty() ? std::string("null argument") : err));
        return 0;
    }
    return 1;
}
int oclr_frame_set_accumulation(oclr_frame* frame, int mode) {
    std::string err;
    if (!frame || !frame_set_accumulation(frame->impl, mode, err)) {
        fail("oclr_frame_set_accumulation: " + (err.empty() ? std::string("null frame") : err));
        return 0;
    }
    return 1;
}
int oclr_frame_read_accum(oclr_frame* frame, cl_float* rgbn) {
    std::string err;
    if (!frame || !frame_accum_copy(frame->impl, rgbn, true, err)) {
        fail("oclr_frame_read_accum: " + (err.empty() ? std::string("null frame") : err));
        return 0;
    }
    return 1;
}
int oclr_frame_write_accum(oclr_frame* frame, const cl_float* rgbn) {
    std::string err;
    if (!frame || !frame_accum_copy(frame->impl, const_cast<cl_float*>(rgbn), false, err)) {
        fail("oclr_frame_write_accum: " + (err.empty() ? std::string("null frame") : err));
        return 0;
    }
    return 1;
}
int oclr_frame_progress(oclr_frame* frame, unsigned long long* done, unsigned long long* total) {
    unsigned long long d = 0, t = 0;
    if (!frame || !frame_progress(frame->impl, &d, &t)) {
        fail("oclr_frame_progress: query failed");
        return 0;
    }
    if (done) *done = d;
    if (total) *total = t;
    return 1;
}

int oclr_frame_read(oclr_frame* frame, cl_uint rowBegin, cl_uint rowEnd, cl_ushort* r, cl_ushort* g, cl_ushort* b, void* cudaStream) {
    if (!frame || !r || !g || !b) {
        fail("oclr_frame_read: null argument");
        return 0;
    }
    std::string err;
    if (!frame_read(frame->impl, rowBegin, rowEnd, r, g, b, cudaStream, err)) {
        fail("oclr_frame_read: " + err);
        return 0;
    }
    return 1;
}

int oclr_frame_read_primary_ids(oclr_frame* frame, cl_uint* ids) {
    if (!frame || !ids) {
        fail("oclr_frame_read_primary_ids: null argument");
        return 0;
    }
    std::string err;
    if (!frame_read_ids(frame->impl, ids, err)) {
        fail("oclr_frame_read_primary_ids: " + err);
        return 0;
    }
    return 1;
}

int oclr_frame_read_flags(oclr_frame* frame, cl_uchar* flags) {
    if (!frame || !flags) {
        fail("oclr_frame_read_flags: null argument");
        return 0;
    }
    std::string err;
    if (!frame_read_flags(frame->impl, flags, err)) {
        fail("oclr_frame_read_flags: " + err);
        return 0;
    }
    return 1;
}

cl_uint oclr_frame_last_launches(const oclr_frame* frame) { return frame ? frame_last_launches(frame->impl) : 0; }

int oclr_frame_push_rows(oclr_frame* frame, cl_uint bandRows, int rank, int worldSize, void* const* peerPlanes, void* cudaStream) {
    std::string err;
    if (!frame || rank < 0 || worldSize < 1 ||
        !frame_push_rows(frame->impl, bandRows, (uint32_t)rank, (uint32_t)worldSize, peerPlanes, cudaStream, err)) {
        fail("oclr_frame_push_rows: " + (err.empty() ? std::string("bad argument") : err));
        return 0;
    }
    return 1;
}

void oclr_frame_device_planes(oclr_frame* frame, void** red, void** green, void** blue) {
    if (frame) frame_device_planes(frame->impl, red, green, blue);
}

int oclr_band_partition(cl_uint height, cl_uint bandRows, int rank, int worldSize, cl_uint* rows, int maxBands) {
    if (bandRows == 0 || worldSize < 1 || rank < 0 || rank >= worldSize) return 0;
    int owned = 0;
    const cl_uint bands = (height + bandRows - 1) / bandRows;
    for (cl_uint b = (cl_uint)rank; b < bands; b += (cl_uint)worldSize) {
        if (rows && owned < maxBands) {
            rows[2 * owned] = b * bandRows;
            rows[2 * owned + 1] = (b + 1) * bandRows < height ? (b + 1) * bandRows : height;
        }
        ++owned;
    }
    return owned;
}

static double now_ms() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}

// ---- one frame on one device: upload, trace, read back ---------------------------------------------------------------------
// world > 1: this is one of `world` threads (one per GPU) rendering the rows y with (y / bandRows) % world == rank; `shareCtx` (when
// peer access is available) makes the N uploads ONE upload: every GPU pulls 1/N of each large array and fans it out over NVLink.
static bool render_rows_on_device(int device, const HostScene& h, const Camera& cam, const cl_uint* camStart, const cl_uint* camEnd,
                                  const cl_uint* camList, size_t camListSize, cl_uint sampleCount, int rank, int world, cl_uint bandRows,
                                  ShardCtx* shareCtx, cl_ushort* r, cl_ushort* g, cl_ushort* b, std::string& err) {
    const bool trace = getenv("OCLR_TRACE") != nullptr;
    static const bool overlap = [] { const char* v = getenv("OCLR_OVERLAP_UPLOAD"); return !v || atoi(v) != 0; }();
    static const bool cacheBlocks = [] { const char* v = getenv("OCLR_BLOCK_CACHE"); return !v || atoi(v) != 0; }();
    struct Scope {   // device blocks of this call are recycled by the next one (runtime.cu, BlockCache)
        void* s;
        ~Scope() {
            if (s) allocation_cache_leave(s);
        }
    } scope = {cacheBlocks ? allocation_cache_enter(device) : nullptr};
    const double t0 = now_ms();
    const uint32_t bandWorld = (uint32_t)(world > 1 ? world : 1);
    // The camera lists go up and the primary-ray round starts as soon as the triangles are on the device, under the upload of the
    // grid (scene_create's `early` hook + frame_prelaunch); the render call below continues from that round.
    Frame* f = nullptr;
    std::string frameErr;
    double tFrame = 0;
    UploadShare share;
    share.ctx = shareCtx;
    share.rank = rank;
    share.camStart = camStart;
    share.camEnd = camEnd;
    share.camList = camList;
    share.camListSize = camListSize;
    share.pixels = (size_t)cam.width * cam.height;
    const std::function<void(Scene*)> early = [&](Scene* partial) {
        const double a = now_ms();
        f = frame_create(partial, cam, camStart, camEnd, camList, camListSize, frameErr, false, shareCtx ? &share.staged : nullptr);
        std::string ignored;
        if (f && default_variant() == (int)kKernelPipe) frame_prelaunch(f, sampleCount, bandRows, (uint32_t)rank, bandWorld, ignored);
        tFrame = now_ms() - a;
    };
    Scene* s = scene_create(device, h, err, overlap && camStart && camEnd ? &early : nullptr, shareCtx ? &share : nullptr);
    if (!s) {
        if (f) frame_destroy(f);
        staged_release(share.staged);
        return false;
    }
    const double t1 = now_ms() - tFrame;
    if (!f) {
        if (!frameErr.empty()) {   // the hook ran and the frame could not be created
            err = frameErr;
            staged_release(share.staged);
            scene_destroy(s);
            return false;
        }
        const double a = now_ms();
        f = frame_create(s, cam, camStart, camEnd, camList, camListSize, err, true, shareCtx ? &share.staged : nullptr);
        tFrame = now_ms() - a;
    }
    staged_release(share.staged);   // (no-op once a frame has adopted the lists)
    const double t2 = t1 + tFrame;
    double tRender = 0, tRead = 0;
    bool ok = f != nullptr;
    if (ok) {
        {
            std::lock_guard<std::mutex> lock(g_liveMutex);
            g_liveFrames.push_back(f);
        }
        RenderStats rs;
        const double a = now_ms();
        // all bands of this device in one launch sequence
        // (render statistics -- an event pair around every trace launch and a synchronisation of their own -- only when somebody reads them)
        ok = frame_render_bands(f, sampleCount, 0, sampleCount, bandRows, (uint32_t)rank, bandWorld, default_variant(), false, nullptr,
                                trace ? &rs : nullptr, err);
        const double c = now_ms();
        ok = ok && frame_read_bands(f, bandRows, (uint32_t)rank, bandWorld, r, g, b, err);
        tRender += c - a;
        tRead += now_ms() - c;
        GetProgress();   // latch the last value of the device counter before the frame goes away
        std::lock_guard<std::mutex> lock(g_liveMutex);
        for (size_t i = 0; i < g_liveFrames.size(); ++i)
            if (g_liveFrames[i] == f) {
                g_liveFrames.erase(g_liveFrames.begin() + (long)i);
                break;
            }
    }
    const double t3 = now_ms();
    if (f) frame_destroy(f);
    scene_destroy(s);
    if (trace)
        fprintf(stderr, "[opencl_render_b200] RaytraceAll dev %d: scene upload+repack %.2f ms, camera lists %.2f ms, trace %.2f ms, read back %.2f ms, "
                        "release %.2f ms\n", device, t1 - t0, t2 - t1, tRender, tRead, now_ms() - t3);
    return ok;
}

static int all_devices_world(int devices) {
    const int k = g_allDevicesLimit.load();
    return k > 0 && k < devices ? k : devices;
}
// Band height of the all-devices mode: about eight bands per GPU (sky and geometry rows cost very different amounts), multiple of 8
// rows (the logic kernel's tile height), at most 128 = the reference's tile height (raytrace.c:507).
static cl_uint all_devices_band_rows(cl_uint height, int world) {
    static const int forced = [] { const char* v = getenv("OCLR_BAND_ROWS"); return v ? atoi(v) : 0; }();
    if (forced > 0) return (cl_uint)forced;
    cl_uint rows = height / (cl_uint)(world * 8);
    rows = rows / 8 * 8;
    return rows < 8 ? 8 : (rows > 128 ? 128 : rows);
}

static cl_bool raytrace_all_impl(cl_uint computationType, const Camera& cam, const HostScene& h, const cl_uint* camStart,
                                 const cl_uint* camEnd, const cl_uint* camList, ptrdiff_t camListSize, cl_uint sampleCount,
                                 cl_ushort* r, cl_ushort* g, cl_ushort* b) {
    if (computationType == 0) {
        fail("RaytraceAll: computation type 0 (\"Local CPU single thread\") is not implemented by this library -- "
             "it is a CUDA sm_100a drop-in with no CPU fallback; pick a CUDA device (type >= 1)");
        return CL_FALSE;
    }
    const int devices = device_count();
    if (devices <= 0) {
        fail("RaytraceAll: no CUDA device available (no CPU fallback)");
        return CL_FALSE;
    }
    if (!r || !g || !b || camListSize < 0 || sampleCount == 0) {
        fail("RaytraceAll: bad arguments");
        return CL_FALSE;
    }
    const int type = (int)computationType - 1;
    const bool allDevices = devices > 1 && type == devices;
    if (!allDevices && type >= devices) {
        fail("RaytraceAll: computation type out of range");
        return CL_FALSE;
    }
    g_progress.store(0.f);
    g_wallStart.store(wall_now());
    g_wallLastChange.store(g_wallStart.load());
    g_startTime = clock();
    g_endTime = g_startTime.load();
    bool ok = true;
    std::string err;
    const int world = allDevices ? all_devices_world(devices) : 1;
    if (world <= 1) {
        ok = render_rows_on_device(allDevices ? 0 : type, h, cam, camStart, camEnd, camList, (size_t)camListSize, sampleCount, 0, 1, 128, nullptr, r, g,
                                   b, err);
    } else {
        // Rows dealt in bands over the GPUs, ONE upload shared by all of them (each pulls 1/N over PCIe, NVLink fan-out), every GPU
        // copies its own rows back to the caller's planes (disjoint), so no gather step is needed inside one process.
        static const bool shareUpload = [] { const char* v = getenv("OCLR_SHARE_UPLOAD"); return !v || atoi(v) != 0; }();
        const cl_uint bandRows = all_devices_band_rows(cam.height, world);
        std::vector<std::string> errs(world);
        std::vector<char> oks(world, 1);
        ok = run_on_devices(world, shareUpload, [&](int d, ShardCtx* share) {
            oks[d] = render_rows_on_device(d, h, cam, camStart, camEnd, camList, (size_t)camListSize, sampleCount, d, world, bandRows, share, r, g, b,
                                           errs[d]);
        }, err);
        for (int d = 0; ok && d < world; ++d)
            if (!oks[d]) {
                ok = false;
                err = errs[d];
                break;
            }
    }
    g_endTime = clock();
    if (!ok) {
        fail("RaytraceAll: " + err);
        return CL_FALSE;
    }
    return CL_TRUE;
}

cl_bool oclr_raytrace_all_p(cl_uint computationType, const cl_uint* dim, const cl_float* eye, const cl_float* eyeToTopLeft,
                            const cl_float* leftToRight, const cl_float* topToBottom, cl_float pixelSizeInv,
                            const oclr_scene_desc* scene, const cl_uint* camStart, const cl_uint* camEnd, const cl_uint* camList,
                            ptrdiff_t camListSize, cl_uint sampleCount, cl_ushort* r, cl_ushort* g, cl_ushort* b) {
    if (!dim || !eye || !eyeToTopLeft || !leftToRight || !topToBottom || !scene) {
        fail("oclr_raytrace_all_p: null argument");
        return CL_FALSE;
    }
    Camera cam;
    memset(&cam, 0, sizeof(cam));
    cam.width = dim[0];
    cam.height = dim[1];
    for (int i = 0; i < 3; ++i) {
        cam.eye[i] = eye[i];
        cam.eyeToTopLeft[i] = eyeToTopLeft[i];
        cam.leftToRight[i] = leftToRight[i];
        cam.topToBottom[i] = topToBottom[i];
    }
    cam.pixelSizeInv = pixelSizeInv;
    return raytrace_all_impl(computationType, cam, to_host(scene), camStart, camEnd, camList, camListSize, sampleCount, r, g, b);
}

cl_bool RaytraceAll(cl_uint computationType, cl_uint2 dim, cl_float3 eye, cl_float3 eyeToTopLeft, cl_float3 leftToRight,
                    cl_float3 topToBottom, cl_float pixelSizeInv, cl_uint* camStart, cl_uint* camEnd, cl_uint* camList,
                    ptrdiff_t camListSize, cl_uint sampleCount, cl_uint vertexCount, cl_float3* vertex, cl_uint triangleCount,
                    cl_int3* triIdx, cl_int* triMat, cl_float2* triUv, cl_float3* triNormal, cl_int axesDivCount,
                    cl_float3* sceneBoxMin, cl_uint* gridStart, cl_uint* gridList, cl_uint materialCount, cl_uint2* matSize,
                    cl_int* matStart, cl_uint texturesSize, cl_uchar3* textures, cl_uint lightCount, cl_int* lightType,
                    cl_float3* lightPos, cl_float3* lightDir, cl_float3* lightColour, cl_float* lightRadius, cl_float* lightHalf,
                    cl_ushort* outR, cl_ushort* outG, cl_ushort* outB) {
    oclr_scene_desc d;
    memset(&d, 0, sizeof(d));
    d.vertexCount = vertexCount;
    d.vertex = vertex;
    d.triangleCount = triangleCount;
    d.triangleVertexIndex = triIdx;
    d.triangleMaterialId = triMat;
    d.triangleUv = triUv;
    d.triangleNormal = triNormal;
    d.axesDivCount = axesDivCount;
    d.sceneBoxMin = sceneBoxMin;
    d.scenePixelTriangleListStart = gridStart;
    d.scenePixelTriangleList = gridList;
    d.materialCount = materialCount;
    d.materialImageSize = matSize;
    d.materialImageStart = matStart;
    d.texturesSize = texturesSize;
    d.textures = textures;
    d.lightCount = lightCount;
    d.lightType = lightType;
    d.lightPosition = lightPos;
    d.lightDirection = lightDir;
    d.lightColour = lightColour;
    d.lightRadius = lightRadius;
    d.lightHalfAttenuationDistance = lightHalf;
    return oclr_raytrace_all_p(computationType, dim.s, eye.s, eyeToTopLeft.s, leftToRight.s, topToBottom.s, pixelSizeInv, &d, camStart,
                               camEnd, camList, camListSize, sampleCount, outR, outG, outB);
}

// ---- builders --------------------------------------------------------------------------------------------------------------
int oclr_build_camera_lists(const oclr_camera* camera, cl_uint vertexCount, const cl_float3* vertex, cl_uint triangleCount,
                            const cl_int3* triIdx, oclr_camera_lists* out) {
    if (!camera || !out || (triangleCount && (!vertex || !triIdx))) {
        fail("oclr_build_camera_lists: null argument");
        return 0;
    }
    memset(out, 0, sizeof(*out));
    if (!build_camera_lists(camera, vertexCount, (const float4*)vertex, triangleCount, (const int32_t*)triIdx, out)) {
        fail("oclr_build_camera_lists: out of memory");
        return 0;
    }
    return 1;
}
int oclr_build_scene_grid(cl_int axesDivCount, cl_uint vertexCount, const cl_float3* vertex, cl_uint triangleCount,
                          const cl_int3* triIdx, oclr_scene_grid* out) {
    if (!out || (triangleCount && (!vertex || !triIdx))) {
        fail("oclr_build_scene_grid: null argument");
        return 0;
    }
    memset(out, 0, sizeof(*out));
    if (!build_scene_grid(axesDivCount, vertexCount, (const float4*)vertex, triangleCount, (const int32_t*)triIdx, out)) {
        fail("oclr_build_scene_grid: bad axesDivCount (power of two <= 1024) or out of memory");
        return 0;
    }
    return 1;
}
int oclr_build_scene_grid_device(int device, cl_int axesDivCount, cl_uint vertexCount, const cl_float3* vertex, cl_uint triangleCount,
                                 const cl_int3* triIdx, oclr_scene_grid* out) {
    if (!out || (triangleCount && (!vertex || !triIdx))) {
        fail("oclr_build_scene_grid_device: null argument");
        return 0;
    }
    memset(out, 0, sizeof(*out));
    std::string err;
    float4* box = nullptr;
    uint32_t *start = nullptr, *list = nullptr;
    size_t listSize = 0;
    if (!build_scene_grid_device(device, axesDivCount, vertexCount, (const float4*)vertex, triangleCount, (const int32_t*)triIdx, &box, &start, &list,
                                 &listSize, err)) {
        fail("oclr_build_scene_grid_device: " + err);
        return 0;
    }
    out->axesDivCount = axesDivCount;
    out->boxMin = (cl_float3*)box;
    out->start = start;
    out->list = list;
    out->listSize = listSize;
    return 1;
}
void oclr_free_camera_lists(oclr_camera_lists* l) {
    if (!l) return;
    free(l->start);
    free(l->end);
    free(l->list);
    memset(l, 0, sizeof(*l));
}
void oclr_free_scene_grid(oclr_scene_grid* g) {
    if (!g) return;
    free(g->boxMin);
    free(g->start);
    free(g->list);
    memset(g, 0, sizeof(*g));
}
