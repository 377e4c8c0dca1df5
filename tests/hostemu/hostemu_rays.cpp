// tests/hostemu/hostemu_rays.cpp -- TEST INFRASTRUCTURE ONLY.
// The production walk's host form (rt_walk.h / rt_core.h grid_trace_mode, the arithmetic the trace kernels instantiate) on caller
// rays, over the scene as the product's packers lay it out.  Built into tests/_build/ by tests/test_query_host.py; never part of, nor
// reachable from, libopencl_render_b200.so.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <string>
#include <thread>
#include <vector>

#include "../../include/oclr_abi.h"
#include "../../opencl_render_b200/csrc/rt_core.h"
#include "../../opencl_render_b200/csrc/runtime.h"

using namespace oclr;

// RayIntersectsTriangles on caller rays: o4 = (o.xyz, minD), d4 = (d.xyz, maxD), excl = excluded triangle per ray (NULL: none);
// out4 = (as_float(triangle), t, abL, acL), abL / acL 0 on a miss.  Walk mode as in hostemu_render (HOSTEMU_HIERARCHICAL): unset = the
// reference's cell walk, 1 = two-level walk, 2 = the trace kernel's packed walk, 1000 / 1001 = the tail kernels' cooperative bursts over
// cell / brick planes (rt_tail.cuh).
extern "C" int hostemu_walk_rays(const oclr_scene_desc* d, size_t count, const float* o4, const float* d4, const uint32_t* excl, float* out4,
                                 int threads) {
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
    std::string err;
    if (!validate_scene(h, err)) { fprintf(stderr, "hostemu: %s\n", err.c_str()); return 0; }
    std::vector<float4> geo(4 * (size_t)h.triangleCount + 1), shade(8 * (size_t)h.triangleCount + 1);
    pack_triangles(h, geo.data(), shade.data(), threads);
    PackedGrid grid;
    if (!pack_grid(h, grid, err)) { fprintf(stderr, "hostemu: %s\n", err.c_str()); return 0; }
    SceneView S = {};
    S.triGeo = geo.data(); S.triShade = shade.data(); S.bricks = grid.bricks.data(); S.cellRange = grid.cellRange.data();
    S.cellList = grid.cellList.data(); S.faceMask = grid.faceMask.data(); S.planes = grid.planes.data(); S.matSize = h.matSize; S.matStart = h.matStart;
    S.textures = h.textures; S.triangleCount = h.triangleCount; S.materialCount = h.materialCount; S.n = grid.n; S.nb = grid.nb;
    const float* px = S.planes; const float* py = px + (S.n + 1); const float* pz = py + (S.n + 1);
    const int hierEnv = getenv("HOSTEMU_HIERARCHICAL") ? atoi(getenv("HOSTEMU_HIERARCHICAL")) : 0;
    const int mode = getenv("HOSTEMU_HIERARCHICAL") ? (hierEnv >= 2 ? hierEnv : 1) : 0;
    std::atomic<size_t> next(0);
    auto worker = [&]() {
        for (;;) {
            const size_t first = next.fetch_add(256);
            if (first >= count) break;
            const size_t last = std::min(count, first + 256);
            for (size_t i = first; i < last; ++i) {
                const float* o = o4 + 4 * i;
                const float* r = d4 + 4 * i;
                float t = 0.f, ab = 0.f, ac = 0.f;
                const uint32_t tri = grid_trace_mode<false>(mode, S, px, py, pz, mk3(o[0], o[1], o[2]), mk3(r[0], r[1], r[2]), o[3], r[3],
                                                            excl ? excl[i] : kNoTriangle, t, ab, ac, nullptr);
                float* out = out4 + 4 * i;
                memcpy(out, &tri, 4);
                out[1] = t;
                out[2] = tri == kNoTriangle ? 0.f : ab;
                out[3] = tri == kNoTriangle ? 0.f : ac;
            }
        }
    };
    if (threads <= 1) worker();
    else {
        std::vector<std::thread> pool;
        for (int t = 0; t < threads; ++t) pool.emplace_back(worker);
        for (auto& t : pool) t.join();
    }
    return 1;
}
