// runtime.h -- internal C++ interface between the C-ABI (abi.cpp), the host-side packers/builders (g++) and the CUDA
// runtime + kernels (nvcc).  Replaces the OpenCL host setup of source/opencl/raytrace.c:283-603 (context, program
// build, 35 buffers, tile loop) with: one resident Scene per upload, one Frame per camera, kernels launched on a
// caller-chosen stream.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <functional>
#include <string>
#include <vector>

#include "rt_types.h"

namespace oclr {

// Host arrays exactly as the reference passes them to RaytraceAll (source/opencl/raytrace.h:58-106).
struct HostScene {
    uint32_t vertexCount = 0;
    const float4* vertex = nullptr;          // cl_float3 == 16 B
    uint32_t triangleCount = 0;
    const int32_t* triIdx = nullptr;         // cl_int3 == 16 B: 4 ints per triangle
    const int32_t* triMat = nullptr;
    const float* triUv = nullptr;            // cl_float2 x 3 per triangle
    const float4* triNormal = nullptr;       // cl_float3 x 3 per triangle
    int32_t axesDivCount = 0;
    const float4* boxMin = nullptr;          // axesDivCount + 1
    const uint32_t* gridStart = nullptr;     // axesDivCount^3 + 1
    const uint32_t* gridList = nullptr;
    uint32_t materialCount = 0;
    const uint2* matSize = nullptr;          // 5 * materialCount
    const int32_t* matStart = nullptr;       // 5 * materialCount + 1
    uint32_t texturesSize = 0;
    const uchar4* textures = nullptr;
    uint32_t lightCount = 0;
    const int32_t* lightType = nullptr;
    const float4* lightPos = nullptr;
    const float4* lightDir = nullptr;
    const float4* lightColour = nullptr;
    const float* lightRadius = nullptr;
    const float* lightHalf = nullptr;
};

// ---- host packers (scene_pack.cpp, g++ -ffp-contract=off) -------------------------------------------------------
struct PackedGrid {
    std::vector<uint4> bricks;
    std::vector<uint2> cellRange;
    std::vector<uint32_t> cellList;
    std::vector<uint32_t> faceMask;
    std::vector<float> planes;
    int32_t n = 0, nb = 0;
    // a walk grid (rt_types.h) only: walk cell j of axis a stands for reference cell cellMap[a * n + j] (-1 past the extent);
    // cells each axis has fewer than n (SceneView::walkTrim).  cellList stays empty: the ranges point into the reference's list.
    std::vector<int32_t> cellMap;
    uint32_t walkTrim = 0;
};
void pack_triangles(const HostScene& h, float4* triGeo /*4N*/, float4* triShade /*8N*/, int threads);
bool pack_grid(const HostScene& h, PackedGrid& out, std::string& err);
// Walk grid (rt_types.h) of a scene and its packed reference grid `ref`; walk.n == 0 when no run collapses or the padding to a multiple of
// 4 keeps every cell again (the walk runs on `ref`).
// The device builds it from the same pieces: walk_runs and walk_cell_map on the host, the run check and the packing on the device.
struct WalkRun {
    int axis, first, count;   // zero-width cells first .. first + count - 1 of `axis` (count >= 2): count + 1 equal planes
};
std::vector<WalkRun> walk_runs(const float* planes /* 3 x (n+1) */, int n);
// every cell of the run has, in every column across the other two axes, the list of the run's first cell (same length, same entries)
bool walk_run_collapses(const uint32_t* gridStart, const uint32_t* gridList, int n, const WalkRun& r);
// kept cells per axis -> map (3 x n, -1 past each extent); returns the cells removed per axis, packed (SceneView::walkTrim)
uint32_t walk_cell_map(int n, const std::vector<WalkRun>& runs, const std::vector<uint8_t>& collapses, std::vector<int32_t>& map);
void walk_planes(const float* planes, int n, const int32_t* map, float* out /* 3 x (n+1) */);
bool pack_walk_grid(const HostScene& h, const PackedGrid& ref, PackedGrid& walk, std::string& err);
// super-brick level of the three-level walk (rt_walk.h): records appended to the brick array, flags in the empty bricks' .w
int super_bricks_per_axis(int n);   // n / 16 for power-of-two grids of >= 32 cells per axis, else 0 (no super-brick level)
size_t super_brick_records(int n);  // records behind the nb^3 brick records (super-brick records sit at the brick strides)
int super_policy(int dflt);         // OCLR_SUPER (else dflt): 0 = no super-brick records / flags at all, 1 = flag every empty super-brick
void append_super_bricks(std::vector<uint4>& bricks, int n, int nb, int policy);
void pack_lights(const HostScene& h, std::vector<Light>& out);
// gridMayBeMissing: sceneBoxMin == scenePixelTriangleListStart == NULL is accepted (the device runtime then builds the grid itself)
bool validate_scene(const HostScene& h, std::string& err, bool gridMayBeMissing = false);

// ---- device runtime (runtime.cu) -----------------------------------------------------------------------------------
// Path state of a launch domain (runtime.cu PathState): the capacity to reallocate at before a domain of Q paths with a ring of `slots`
// slots runs on buffers sized for `capacity` paths and `ringSlots` slots, or 0 when they serve it as they are.  A new ring depth (a
// materials edit changed the scene's) reallocates in both directions, at no smaller capacity.
inline uint32_t path_state_regrow(uint32_t capacity, int ringSlots, uint32_t Q, int slots) {
    if (Q <= capacity && slots == ringSlots) return 0;
    return Q > capacity ? Q : capacity;
}

struct Scene;
struct Frame;

int device_count();
bool device_name(int dev, char* buf, size_t len);

// RaytraceAll(all devices): the N per-GPU scene_create calls of one frame share the upload -- each GPU pulls 1/N of every large array over
// PCIe and stores it into its peers over NVLink (runtime.cu, ShardCtx).  run_on_devices() runs fn(rank, share) on a persistent worker
// thread per GPU; `share` is null when peer access is unavailable (every GPU then uploads everything itself).
struct ShardCtx;
struct StagedCamLists {   // camera lists that went up with the scene; frame_create adopts them
    void* start = nullptr;
    void* end = nullptr;
    void* list = nullptr;
    size_t listSize = 0;
    bool adopted = false;
    bool borrowed = false;   // the lists live in the shared-upload landing arena: nobody frees them
};
struct UploadShare {
    ShardCtx* ctx = nullptr;
    int rank = 0;
    const uint32_t* camStart = nullptr;
    const uint32_t* camEnd = nullptr;
    const uint32_t* camList = nullptr;
    size_t camListSize = 0, pixels = 0;
    StagedCamLists staged;
};
// Inside RaytraceAll device blocks come from / go back to a per-device free list instead of the driver (runtime.cu, BlockCache): the
// calling thread brackets its work on `device` with these two.
void* allocation_cache_enter(int device);
void allocation_cache_leave(void* scope);
bool run_on_devices(int world, bool shareUpload, const std::function<void(int rank, ShardCtx* share)>& fn, std::string& err);
void staged_release(StagedCamLists& st);

// `early` (optional) is called once the triangles, materials and lights are on their way to the device and BEFORE the grid is
// uploaded, with the partly built scene: RaytraceAll uses it to start the primary-ray round under the grid upload (frame_prelaunch).
Scene* scene_create(int device, const HostScene& h, std::string& err, const std::function<void(Scene*)>* early = nullptr,
                    UploadShare* share = nullptr);
void scene_destroy(Scene* s);
size_t scene_device_bytes(const Scene* s);
size_t frame_state_bytes(Frame* f);
int scene_device(const Scene* s);
size_t scene_debug_read(Scene* s, int which, void* dst, size_t cap);

// Camera lists are per-frame inputs (CameraTriangleList::New output, trianglelist.cpp:520-626).  `camStart`/`camEnd`
// hold width*height entries; only rows [rowBegin,rowEnd) need to be valid (band-partitioned multi-GPU rendering).
Frame* frame_create(Scene* s, const Camera& cam, const uint32_t* camStart, const uint32_t* camEnd, const uint32_t* camList,
                    size_t camListSize, std::string& err, bool sync = true,   // sync = false: the host arrays outlive the copies
                    StagedCamLists* staged = nullptr);
void frame_destroy(Frame* f);
// Edits of a resident scene (semantics in include/oclr_abi.h, oclr_scene_update): the parts named are rebuilt from `h` by the stages
// scene_create runs, into new buffers swapped in on success.  deviceMemory: the geometry arrays are device memory of the scene's device.
enum { kSceneLights = 1, kSceneMaterials = 2, kSceneGeometry = 4 };
bool scene_update(Scene* s, const HostScene& h, unsigned parts, bool deviceMemory, std::string& err);
// A new camera of the same image size for a frame: caller lists (camStart != nullptr) or lists built on the device.
bool frame_set_camera(Frame* f, const Camera& cam, const uint32_t* camStart, const uint32_t* camEnd, const uint32_t* camList, size_t listSize,
                      std::string& err);
// camStart == nullptr: CameraTriangleList::New runs on the device from the resident scene (cam_builder.cuh).  The lists a frame
// holds (uploaded or device-built) can be copied back: `list` needs frame_camera_list_size() entries.
size_t frame_camera_list_size(Frame* f);
bool frame_read_camera_lists(Frame* f, uint32_t* start, uint32_t* end, uint32_t* list, std::string& err);

enum KernelVariant { kKernelSimple = 0, kKernelPipe = 2 };   // (1 was the lane-owned wavefront kernel, retired)

struct RenderStats {
    float deviceMs = 0.f;        // CUDA-event time of the trace kernel(s) on the launch stream
    uint32_t launches = 0;       // kernels launched
    float traceMs = 0.f;         // device time during which a trace-stage launch (wf_setup_kernel + wf_pipe_kernel, the dominant kernel) was in flight
    uint32_t traceLaunches = 0;
    Counters counters = {};      // filled when `count` was requested
};

// Renders rows [rowBegin,rowEnd) with `sampleCount` samples into the frame's device planes (zeroed first, like the
// OpenCL branch raytrace.c:476-486).  `stream` is a cudaStream_t (0 = default stream).  Synchronous w.r.t. the host
// only when `stats` is non-null (it needs the event time).
// Samples [sampleBegin,sampleEnd) of a sampleCount-sample job: sample 0 overwrites the planes, later samples add to them
// (raytrace_opencl.c:726-741), so a job can be rendered progressively over several calls.
bool frame_render(Frame* f, uint32_t sampleCount, uint32_t sampleBegin, uint32_t sampleEnd, uint32_t rowBegin, uint32_t rowEnd, int variant,
                  bool count, void* stream, RenderStats* stats, std::string& err);
// Same, for the rows y with (y / bandRows) % world == rank (one launch covers all bands the rank owns).
bool frame_render_bands(Frame* f, uint32_t sampleCount, uint32_t sampleBegin, uint32_t sampleEnd, uint32_t bandRows, uint32_t rank, uint32_t world,
                        int variant, bool count, void* stream, RenderStats* stats, std::string& err);
// Starts the first logic round of frame_render_bands(f, sampleCount, 0, sampleCount, bandRows, rank, world, kKernelPipe, ...) ahead, on the
// frame's own stream (runtime.cu); the matching render call on the default stream continues from it.
bool frame_prelaunch(Frame* f, uint32_t sampleCount, uint32_t bandRows, uint32_t rank, uint32_t world, std::string& err);
// Progressive accumulation / checkpoint-resume / progress (SURVEY.md section 8f-3, 8f-4); see runtime.cu.
bool frame_write(Frame* f, uint32_t rowBegin, uint32_t rowEnd, const uint16_t* inR, const uint16_t* inG, const uint16_t* inB, void* stream,
                 std::string& err);
bool frame_set_accumulation(Frame* f, int mode, std::string& err);
bool frame_accum_copy(Frame* f, float* host, bool toHost, std::string& err);
bool frame_progress(Frame* f, unsigned long long* done, unsigned long long* total);
// Slices a launch domain is cut into (runtime.cu launch_wavefront): 0 = automatic, k = always k.
void set_slice_count(int k);
// Tracing one round ahead (rt_wavefront.cuh): 0 never, 1 all segments but the camera's, 2 all, -1 automatic.
void set_ahead_mode(int m);
// Skipping the shadow rays of lights on the unseen side of a surface (rt_wavefront.cuh): 1 (default) or 0.  The planes are the same.
void set_cull_hidden_lights(int on);
uint32_t band_owned_rows(uint32_t height, uint32_t bandRows, uint32_t rank, uint32_t world);
// Device -> host copy of ALL rows `rank` owns (bands of bandRows dealt round-robin over world): compacted on the device, one transfer
// into a pinned staging block, scattered to the caller's (pageable) planes by the calling thread.
bool frame_read_bands(Frame* f, uint32_t bandRows, uint32_t rank, uint32_t world, uint16_t* outR, uint16_t* outG, uint16_t* outB,
                      std::string& err);
// Device -> host copy of rows [rowBegin,rowEnd) of the three planes (full-frame sized host arrays).
bool frame_read(Frame* f, uint32_t rowBegin, uint32_t rowEnd, uint16_t* outR, uint16_t* outG, uint16_t* outB, void* stream,
                std::string& err);
// SceneTriangleList::New on CUDA device `device` (grid_builder.cuh); outputs are malloc'ed host arrays, entry-for-entry the host builder's.
bool build_scene_grid_device(int device, int32_t n, uint32_t vertexCount, const float4* vertex, uint32_t triangleCount, const int32_t* triIdx,
                             float4** outBoxMin, uint32_t** outStart, uint32_t** outList, size_t* outListSize, std::string& err);
uint32_t frame_last_launches(const Frame* f);
bool frame_read_ids(Frame* f, uint32_t* ids, std::string& err);
bool frame_read_flags(Frame* f, uint8_t* flags, std::string& err);
// Stores the rows rank owns (bands of bandRows dealt round-robin over world) into the full-frame planes [3][H][W] of every GPU
// listed in peerPlanes (device pointers valid in this process: the rank's own buffer and its NVLink peers').
bool frame_push_rows(Frame* f, uint32_t bandRows, uint32_t rank, uint32_t world, void* const* peerPlanes, void* stream, std::string& err);
// Device pointers of the planes (for NCCL gathers done by the host layer) and of the id plane.
void frame_device_planes(Frame* f, void** r, void** g, void** b);

// Batched ray queries on a resident scene (rt_query.cuh; semantics and preconditions in include/oclr_abi.h): closest hit
// (RayIntersectsTriangles) into hit4 = (as_float(tri), t, abL, acL), and the shadow loop's transmittance into att4 = (rgb,
// as_float(last blocker)).  origin4 / direction4 / hit4 / att4 are 4 floats per ray; excluded may be null.  Rays are processed in
// batches of kQueryBatch: the call's scratch (walk records 64 B, class order 16 B, queue 4 B, excluded triangle 4 B per ray of a batch;
// transmittance adds a second queue, hits and an origin copy, 36 B; host-memory inputs add staging, 52 B) stays below 300 MB.
// deviceMemory: the arrays are device memory of the scene's device, 16-byte aligned (excluded: 4).  Synchronous when `stats` is given,
// for host memory and for transmittance.
enum { kQueryBatch = 1 << 21 };
bool scene_intersect(Scene* s, size_t count, const float* origin4, const float* direction4, const uint32_t* excluded, float* hit4,
                     bool deviceMemory, bool counting, void* stream, RenderStats* stats, std::string& err);
bool scene_transmittance(Scene* s, size_t count, const float* origin4, const float* direction4, const uint32_t* excluded, float* att4,
                         bool deviceMemory, bool counting, void* stream, RenderStats* stats, std::string& err);
// Radiance along caller rays (rt_query.cuh radiance_start_kernel + the frame's logic kernel; semantics in include/oclr_abi.h): the reference's pixel-sample loop
// with the camera segment replaced by the ray, sampleCount samples, rgb4 = (mean rgb, as_float(first hit of sample 0)), flags optional
// (cl_uchar per ray).  `cam` may be null when no material has a BUMP channel.  Rays are processed in batches of kRadianceBatch; the
// call's path state is about 1 KB per ray of a batch with a 12-slot ring (432 B + 48 B per ring slot: ring, shading carry, two ray
// slots, walk records, accumulator), about 1.1 GB for a full batch; host-memory inputs add 53 B per ray of staging.  Synchronous.
enum { kRadianceBatch = 1 << 20 };
bool scene_radiance(Scene* s, const Camera* cam, size_t count, const float* origin4, const float* direction4, const uint32_t* excluded,
                    unsigned long long indexBase, uint32_t sampleCount, float* rgb4, uint8_t* flags, bool deviceMemory, bool counting,
                    void* stream, RenderStats* stats, std::string& err);

}  // namespace oclr
