// tests/hostemu/hostemu_walkgrid.cpp -- TEST INFRASTRUCTURE ONLY.
// The walk grid (rt_types.h: runs of coincident split planes collapsed where their lists agree) in its host form (scene_pack.cpp
// pack_walk_grid), and the trace kernels' packed walk (rt_walk.h) over it, on frames and on caller rays.  Built into tests/_build/ by
// tests/test_collapsed_grid_host.py; never part of, nor reachable from, libopencl_render_b200.so.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include "../../include/oclr_abi.h"
#include "../../opencl_render_b200/csrc/rt_core.h"
#include "../../opencl_render_b200/csrc/runtime.h"

using namespace oclr;

namespace {

HostScene host_scene(const oclr_scene_desc* d) {
    HostScene h;
    h.vertexCount = d->vertexCount; h.vertex = (const float4*)d->vertex;
    h.triangleCount = d->triangleCount; h.triIdx = (const int32_t*)d->triangleVertexIndex; h.triMat = d->triangleMaterialId;
    h.triUv = (const float*)d->triangleUv; h.triNormal = (const float4*)d->triangleNormal;
    h.axesDivCount = d->axesDivCount; h.boxMin = (const float4*)d->sceneBoxMin; h.gridStart = d->scenePixelTriangleListStart;
    h.gridList = d->scenePixelTriangleList; h.materialCount = d->materialCount; h.matSize = (const uint2*)d->materialImageSize;
    h.matStart = d->materialImageStart; h.texturesSize = d->texturesSize; h.textures = (const uchar4*)d->textures;
    h.lightCount = d->lightCount; h.lightType = d->lightType; h.lightPos = (const float4*)d->lightPosition;
    h.lightDir = (const float4*)d->lightDirection; h.lightColour = (const float4*)d->lightColour; h.lightRadius = d->lightRadius;
    h.lightHalf = d->lightHalfAttenuationDistance;
    return h;
}

// The scene as the production trace stage walks it: the walk grid when a run collapses, else the reference grid.
struct WalkScene {
    HostScene h;
    std::vector<float4> geo, shade;
    std::vector<Light> lights;
    PackedGrid ref, walk;
    SceneView S = {};
    bool build(const oclr_scene_desc* d, int threads) {
        h = host_scene(d);
        std::string err;
        if (!validate_scene(h, err) || !pack_grid(h, ref, err) || !pack_walk_grid(h, ref, walk, err)) {
            fprintf(stderr, "hostemu_walkgrid: %s\n", err.c_str());
            return false;
        }
        geo.resize(4 * (size_t)h.triangleCount + 1);
        shade.resize(8 * (size_t)h.triangleCount + 1);
        pack_triangles(h, geo.data(), shade.data(), threads);
        pack_lights(h, lights);
        const PackedGrid& g = walk.n ? walk : ref;
        S.triGeo = geo.data(); S.triShade = shade.data(); S.bricks = g.bricks.data(); S.cellRange = g.cellRange.data();
        S.cellList = ref.cellList.data(); S.faceMask = g.faceMask.data(); S.planes = g.planes.data(); S.matSize = h.matSize;
        S.matStart = h.matStart; S.textures = h.textures; S.lights = lights.data(); S.triangleCount = h.triangleCount;
        S.materialCount = h.materialCount; S.lightCount = h.lightCount; S.n = ref.n; S.nb = ref.nb; S.walkTrim = walk.walkTrim;
        return true;
    }
};

void run_parallel(int threads, const std::function<void(int)>& fn) {
    if (threads <= 1) return fn(0);
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t) pool.emplace_back(fn, t);
    for (auto& t : pool) t.join();
}

}  // namespace

// The walk grid: extents (3 ints), map (3 x n ints, -1 past the extent), planes (3 x (n+1) floats), bricks (16 B each, nb^3),
// ranges / face masks of its non-empty cells (count returned; 0 = no run collapsed, nothing written).
extern "C" long hostemu_walk_grid(const oclr_scene_desc* d, int32_t* extents, int32_t* map, float* planes, void* bricks, void* ranges,
                                  size_t rangesCap, uint32_t* faceMask) {
    WalkScene w;
    if (!w.build(d, 2)) return -1;
    if (!w.walk.n) return 0;
    const int n = w.walk.n;
    for (int a = 0; a < 3; ++a) extents[a] = n - pk_get(w.walk.walkTrim, a);
    memcpy(map, w.walk.cellMap.data(), sizeof(int32_t) * w.walk.cellMap.size());
    memcpy(planes, w.walk.planes.data(), sizeof(float) * w.walk.planes.size());
    memcpy(bricks, w.walk.bricks.data(), sizeof(uint4) * w.walk.bricks.size());
    if (w.walk.cellRange.size() * sizeof(uint2) > rangesCap) return -2;
    memcpy(ranges, w.walk.cellRange.data(), sizeof(uint2) * w.walk.cellRange.size());
    memcpy(faceMask, w.walk.faceMask.data(), sizeof(uint32_t) * w.walk.faceMask.size());
    return (long)w.walk.cellRange.size();
}

// hostemu_render (tests/hostemu/hostemu.cpp) with every walk the packed walk over the walk grid (walk mode 2 of trace_sample).
extern "C" int hostemu_walkgrid_render(const oclr_scene_desc* d, const oclr_camera* cam, const uint32_t* camStart, const uint32_t* camEnd,
                                       const uint32_t* camList, uint32_t sampleCount, uint32_t rowBegin, uint32_t rowEnd, uint16_t* outR,
                                       uint16_t* outG, uint16_t* outB, uint32_t* ids, uint8_t* flags, oclr_counters* counters, int threads) {
    WalkScene w;
    if (!w.build(d, threads)) return 0;
    const SceneView& S = w.S;
    FrameView F = {};
    memcpy(&F.cam, cam, sizeof(Camera));
    F.camStart = camStart; F.camEnd = camEnd; F.camList = camList; F.sampleCount = sampleCount; F.rowBegin = rowBegin; F.rowEnd = rowEnd;
    F.bandWorld = 1; F.ownedRows = rowEnd - rowBegin;
    F.outR = outR; F.outG = outG; F.outB = outB; F.idOut = ids; F.flagOut = flags;
    if (rowEnd > cam->height) rowEnd = cam->height;
    std::atomic<uint32_t> nextRow(rowBegin);
    std::vector<Counters> cnts(threads > 0 ? threads : 1);
    run_parallel(threads, [&](int tid) {
        Counters& cnt = cnts[tid];
        memset(&cnt, 0, sizeof(cnt));
        const float scale = 65535.f / (float)sampleCount;
        for (;;) {
            const uint32_t y = nextRow.fetch_add(1);
            if (y >= rowEnd) break;
            for (uint32_t x = 0; x < cam->width; ++x) {
                const uint32_t pixel = y * cam->width + x;
                uint16_t r = 0, g = 0, b = 0;
                bool undef = false;
                for (uint32_t s = 0; s < sampleCount; ++s) {
                    uint32_t pid;
                    const f3 c = trace_sample<true>(S, F, S.planes, nullptr, nullptr, pixel, s, &pid, undef, &cnt, 2);
                    if (s == 0 && ids) ids[pixel] = pid;
                    r = accumulate16(r, c.x, scale); g = accumulate16(g, c.y, scale); b = accumulate16(b, c.z, scale);
                }
                outR[pixel] = r; outG[pixel] = g; outB[pixel] = b;
                if (flags) flags[pixel] = undef ? 1 : 0;
            }
        }
    });
    if (counters) {
        Counters tot;
        memset(&tot, 0, sizeof(tot));
        unsigned long long* a = (unsigned long long*)&tot;
        for (auto& c : cnts) { const unsigned long long* b = (const unsigned long long*)&c; for (size_t i = 0; i < sizeof(Counters) / 8; ++i) a[i] += b[i]; }
        memcpy(counters, &tot, sizeof(tot));
    }
    return 1;
}

// hostemu_walk_rays (tests/hostemu/hostemu_rays.cpp) with the packed walk over the walk grid.
extern "C" int hostemu_walkgrid_rays(const oclr_scene_desc* d, size_t count, const float* o4, const float* d4, const uint32_t* excl, float* out4,
                                     int threads) {
    WalkScene w;
    if (!w.build(d, threads)) return 0;
    const SceneView& S = w.S;
    std::atomic<size_t> next(0);
    run_parallel(threads, [&](int) {
        for (;;) {
            const size_t first = next.fetch_add(256);
            if (first >= count) break;
            const size_t last = std::min(count, first + 256);
            for (size_t i = first; i < last; ++i) {
                const float* o = o4 + 4 * i;
                const float* r = d4 + 4 * i;
                float t = 0.f, ab = 0.f, ac = 0.f;
                const uint32_t tri = grid_trace_packed<false>(S, S.planes, mk3(o[0], o[1], o[2]), mk3(r[0], r[1], r[2]), o[3], r[3],
                                                              excl ? excl[i] : kNoTriangle, t, ab, ac, nullptr);
                float* out = out4 + 4 * i;
                memcpy(out, &tri, 4);
                out[1] = t;
                out[2] = tri == kNoTriangle ? 0.f : ab;
                out[3] = tri == kNoTriangle ? 0.f : ac;
            }
        }
    });
    return 1;
}
