// scene_pack.cpp -- "scene upload path": repack the reference's flat SoA scene (source/opencl/raytrace.h:58-106) into
// the GPU layout of rt_types.h.  Compiled with g++ -ffp-contract=off: the hoisted per-triangle terms must be the
// exact fp32 values the reference's RayIntersectsTriangle would compute per ray (raytrace_opencl.c:131-149).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <thread>

#include "rt_core.h"
#include "runtime.h"

namespace oclr {

static inline float int_bits_as_float(int32_t i) {
    float f;
    memcpy(&f, &i, 4);
    return f;
}

bool validate_scene(const HostScene& h, std::string& err, bool gridMayBeMissing) {
    if (h.axesDivCount < 1 || (h.axesDivCount & (h.axesDivCount - 1)) != 0) {
        err = "axesDivCount must be a power of two (GetBoxAddress is a binary search, raytrace_opencl.c:174-193)";
        return false;
    }
    if (h.axesDivCount > 1024) {
        err = "axesDivCount > 1024 is not supported";
        return false;
    }
    if ((!h.boxMin || !h.gridStart) && !(gridMayBeMissing && !h.boxMin && !h.gridStart)) {
        err = "scene grid (sceneBoxMin / scenePixelTriangleListStart) is missing";
        return false;
    }
    if (h.triangleCount && (!h.vertex || !h.triIdx || !h.triMat || !h.triUv || !h.triNormal)) {
        err = "triangle arrays missing";
        return false;
    }
    // per-element range checks (vertex indices, material ids, CSR monotonicity, list entries) run in the device packers
    if (h.materialCount && (!h.matSize || !h.matStart)) {
        err = "material tables missing";
        return false;
    }
    for (uint32_t m = 0; m < h.materialCount * kMaterialChannels; ++m) {
        // a channel is present when size.x > 0 (raytrace_opencl.h:14-22, channel_present()); a present channel with size.y == 0 would
        // index the atlas with (float)(size.y - 1u) = 4.29e9 (Get2dTableValue3, :103-122) -- rejected instead of read out of bounds
        if (h.matSize[m].x && !h.matSize[m].y) {
            err = "material image with width > 0 and height 0";
            return false;
        }
        const uint64_t texels = (uint64_t)h.matSize[m].x * h.matSize[m].y;
        if (texels && (!h.textures || h.matStart[m] < 0 || (uint64_t)h.matStart[m] + texels > h.texturesSize)) {
            err = "material image outside the texture atlas";
            return false;
        }
    }
    if (h.lightCount && (!h.lightType || !h.lightPos || !h.lightDir || !h.lightColour || !h.lightRadius || !h.lightHalf)) {
        err = "light arrays missing (lightCount > 0)";
        return false;
    }
    return true;
}

static void pack_range(const HostScene& h, float4* geo, float4* shade, size_t begin, size_t end) {
    for (size_t i = begin; i < end; ++i) {
        const int32_t* vi = h.triIdx + 4 * i;
        const float4 A = h.vertex[vi[0]], B = h.vertex[vi[1]], C = h.vertex[vi[2]];
        const f3 a = mk3(A.x, A.y, A.z), b = mk3(B.x, B.y, B.z), c = mk3(C.x, C.y, C.z);
        const f3 ab = mk3(b.x - a.x, b.y - a.y, b.z - a.z);
        const f3 ac = mk3(c.x - a.x, c.y - a.y, c.z - a.z);
        const f3 n = cross3(ac, ab);
        const float abab = dot3(ab, ab), abac = dot3(ab, ac), acac = dot3(ac, ac);
        const float D = 1.f / (abac * abac - abab * acac);
        float4* g = geo + 4 * i;
        g[0] = make_float4(n.x, n.y, n.z, a.x);
        g[1] = make_float4(a.y, a.z, abab, abac);
        g[2] = make_float4(ab.x, ab.y, ab.z, acac);
        g[3] = make_float4(ac.x, ac.y, ac.z, D);
        const float4 nA = h.triNormal[3 * i + 0], nB = h.triNormal[3 * i + 1], nC = h.triNormal[3 * i + 2];
        const float* uv = h.triUv + 6 * i;
        float4* s = shade + 8 * i;
        s[0] = make_float4(a.x, a.y, a.z, int_bits_as_float(h.triMat[i]));
        s[1] = make_float4(b.x, b.y, b.z, 0.f);
        s[2] = make_float4(c.x, c.y, c.z, 0.f);
        s[3] = make_float4(nA.x, nA.y, nA.z, 0.f);
        s[4] = make_float4(nB.x, nB.y, nB.z, 0.f);
        s[5] = make_float4(nC.x, nC.y, nC.z, 0.f);
        s[6] = make_float4(uv[0], uv[1], uv[2], uv[3]);
        s[7] = make_float4(uv[4], uv[5], 0.f, 0.f);
    }
}

void pack_triangles(const HostScene& h, float4* geo, float4* shade, int threads) {
    const size_t n = h.triangleCount;
    if (threads < 1) threads = 1;
    if (n < 65536 || threads == 1) {
        pack_range(h, geo, shade, 0, n);
        return;
    }
    std::vector<std::thread> pool;
    const size_t chunk = (n + threads - 1) / threads;
    for (int t = 0; t < threads; ++t) {
        const size_t b = (size_t)t * chunk, e = b + chunk < n ? b + chunk : n;
        if (b < e) pool.emplace_back(pack_range, std::cref(h), geo, shade, b, e);
    }
    for (auto& t : pool) t.join();
}

// Bricks {mask, rank base}, ranges and face masks of the cells of a grid over the reference CSR.  map == nullptr: the reference grid.
// Otherwise a walk grid (rt_types.h): walk cell j of axis a stands for reference cell map[a * n + j] (-1: past the axis' extent, no
// cell); face masks are taken against the neighbour in the walk grid.  Same order and arithmetic as the device packers (pack_kernels.cuh).
static bool pack_cells(const HostScene& h, int n, const int32_t* map, PackedGrid& out, std::string& err) {
    const int nb = n >= 4 ? n / 4 : 1;
    const uint32_t total = h.gridStart[(size_t)n * n * n];
    auto ref_id = [&](const int c[3]) -> long long {   // reference cell id of a cell of this grid, or -1
        int q[3] = {c[0], c[1], c[2]};
        for (int a = 0; a < 3; ++a) {
            if (q[a] < 0 || q[a] >= n) return -1;
            if (map && (q[a] = map[a * n + q[a]]) < 0) return -1;
        }
        return (long long)q[0] + (long long)n * q[1] + (long long)n * n * q[2];
    };
    out.bricks.assign((size_t)nb * nb * nb, make_uint4(0, 0, 0, 0));
    out.cellRange.clear();
    out.faceMask.clear();
    const int side = n >= 4 ? 4 : n;
    for (int bz = 0; bz < nb; ++bz)
        for (int by = 0; by < nb; ++by)
            for (int bx = 0; bx < nb; ++bx) {
                uint64_t mask = 0;
                const uint32_t rankBase = (uint32_t)out.cellRange.size();
                for (int z = 0; z < side; ++z)
                    for (int y = 0; y < side; ++y)
                        for (int x = 0; x < side; ++x) {
                            const int c[3] = {bx * 4 + x, by * 4 + y, bz * 4 + z};
                            const long long id = ref_id(c);
                            if (id < 0) continue;
                            const uint32_t s = h.gridStart[id], e = h.gridStart[id + 1];
                            if (e < s || e > total) {
                                err = "scenePixelTriangleListStart is not a monotone CSR";
                                return false;
                            }
                            if (s < e) {
                                mask |= 1ull << (x | (y << 2) | (z << 4));
                                out.cellRange.push_back(make_uint2(s, e));
                                for (int face = 0; face < 6; ++face) {  // face = axis*2 + (entered moving towards +axis)
                                    int q[3] = {c[0], c[1], c[2]};
                                    q[face >> 1] += (face & 1) ? -1 : 1;  // the cell the walk came from
                                    uint32_t m = 0xFFFFFFFFu;
                                    const long long nid = ref_id(q);
                                    if (nid >= 0) {
                                        const uint32_t ns = h.gridStart[nid], ne = h.gridStart[nid + 1];
                                        for (uint32_t k = 0; k < 32 && s + k < e; ++k) {
                                            bool found = false;
                                            for (uint32_t j = ns; j < ne && !found; ++j) found = h.gridList[j] == h.gridList[s + k];
                                            if (found) m &= ~(1u << k);
                                        }
                                    }
                                    out.faceMask.push_back(m);
                                }
                            }
                        }
                out.bricks[(size_t)bx + (size_t)nb * (by + (size_t)nb * bz)] =
                    make_uint4((uint32_t)mask, (uint32_t)(mask >> 32), mask ? rankBase : 0u, 0);   // (.z of an empty brick: flags, rt_walk.h)
            }
    if (out.cellRange.empty()) {
        out.cellRange.push_back(make_uint2(0, 0));
        out.faceMask.assign(6, 0xFFFFFFFFu);
    }
    return true;
}

// CSR over n^3 cells  ->  4x4x4 bricks {mask, rank base} + ranges of the non-empty cells + list in brick-major order.
bool pack_grid(const HostScene& h, PackedGrid& out, std::string& err) {
    const int n = h.axesDivCount;
    const int nb = n >= 4 ? n / 4 : 1;
    const size_t cells = (size_t)n * n * n;
    const uint32_t total = h.gridStart[cells];
    if (total && !h.gridList) {
        err = "scenePixelTriangleList missing";
        return false;
    }
    out.n = n;
    out.nb = nb;
    out.planes.resize(3 * (size_t)(n + 1));
    for (int i = 0; i <= n; ++i) {
        out.planes[i] = h.boxMin[i].x;
        out.planes[(n + 1) + i] = h.boxMin[i].y;
        out.planes[2 * (n + 1) + i] = h.boxMin[i].z;
    }
    out.cellList.assign(h.gridList, h.gridList + total);   // list kept in the reference's order; ranges point into it
    for (uint32_t k = 0; k < total; ++k)
        if (out.cellList[k] >= h.triangleCount) {
            err = "scenePixelTriangleList entry out of range";
            return false;
        }
    if (!pack_cells(h, n, nullptr, out, err)) return false;
    append_super_bricks(out.bricks, n, nb, super_policy(0));   // (the production kernel has no super-brick level: nothing is appended unless asked)
    return true;
}

// ---- walk grid (rt_types.h) -----------------------------------------------------------------------------------------------------
std::vector<WalkRun> walk_runs(const float* planes, int n) {
    std::vector<WalkRun> runs;
    if (n < 4) return runs;   // (no brick level to keep the extent a multiple of 4 for; nothing worth collapsing)
    for (int a = 0; a < 3; ++a) {
        const float* p = planes + (size_t)a * (n + 1);
        for (int c = 0; c < n;) {
            int e = c;
            while (e < n && p[e] == p[e + 1]) ++e;   // cells c .. e-1 have zero width
            if (e - c >= 2) runs.push_back({a, c, e - c});
            c = e > c ? e : c + 1;
        }
    }
    return runs;
}

bool walk_run_collapses(const uint32_t* start, const uint32_t* list, int n, const WalkRun& r) {
    const size_t stride[3] = {1, (size_t)n, (size_t)n * n};
    const uint32_t total = start[(size_t)n * n * n];
    const int u = r.axis == 0 ? 1 : 0, v = r.axis == 2 ? 1 : 2;   // the other two axes
    for (int j = 0; j < n; ++j)
        for (int i = 0; i < n; ++i) {
            const size_t first = (size_t)r.first * stride[r.axis] + (size_t)i * stride[u] + (size_t)j * stride[v];
            const uint32_t s0 = start[first], len = start[first + 1] - s0;
            if (start[first + 1] < s0 || start[first + 1] > total) return false;   // (as run_check_kernel: no entry of a bad range is read)
            for (int k = 1; k < r.count; ++k) {
                const size_t id = first + (size_t)k * stride[r.axis];
                const uint32_t s = start[id];
                if (start[id + 1] < s || start[id + 1] > total || start[id + 1] - s != len) return false;
                for (uint32_t q = 0; q < len; ++q)
                    if (list[s + q] != list[s0 + q]) return false;
            }
        }
    return true;
}

uint32_t walk_cell_map(int n, const std::vector<WalkRun>& runs, const std::vector<uint8_t>& collapses, std::vector<int32_t>& map) {
    std::vector<uint8_t> keep(3 * (size_t)n, 1);
    int removed[3] = {0, 0, 0};
    for (size_t i = 0; i < runs.size(); ++i)
        if (collapses[i]) {
            const WalkRun& r = runs[i];
            for (int k = 1; k < r.count; ++k) keep[(size_t)r.axis * n + r.first + k] = 0;
            removed[r.axis] += r.count - 1;
        }
    // extent up to a multiple of 4 (n is one): cells of collapsed runs kept again, in run order -- each only revisits its run's list
    for (size_t i = 0; i < runs.size(); ++i) {
        const WalkRun& r = runs[i];
        for (int k = 1; collapses[i] && k < r.count && removed[r.axis] % 4 != 0; ++k) {
            keep[(size_t)r.axis * n + r.first + k] = 1;
            removed[r.axis] -= 1;
        }
    }
    map.assign(3 * (size_t)n, -1);
    for (int a = 0; a < 3; ++a) {
        int m = 0;
        for (int c = 0; c < n; ++c)
            if (keep[(size_t)a * n + c]) map[(size_t)a * n + m++] = c;
    }
    return pk_make(removed[0], removed[1], removed[2]);
}

void walk_planes(const float* planes, int n, const int32_t* map, float* out) {
    for (int a = 0; a < 3; ++a) {
        const float* p = planes + (size_t)a * (n + 1);
        float* w = out + (size_t)a * (n + 1);
        int j = 0;
        for (; j < n && map[a * n + j] >= 0; ++j) w[j] = p[map[a * n + j]];   // lower plane of the kept cell
        for (; j <= n; ++j) w[j] = p[n];   // the extent's upper plane, repeated up to the plane stride
    }
}

bool pack_walk_grid(const HostScene& h, const PackedGrid& ref, PackedGrid& walk, std::string& err) {
    const int n = ref.n;
    const std::vector<WalkRun> runs = walk_runs(ref.planes.data(), n);
    std::vector<uint8_t> collapses(runs.size());
    bool any = false;
    for (size_t i = 0; i < runs.size(); ++i) any |= (collapses[i] = walk_run_collapses(h.gridStart, h.gridList, n, runs[i]) ? 1 : 0) != 0;
    walk = PackedGrid();
    if (!any) return true;
    const uint32_t trim = walk_cell_map(n, runs, collapses, walk.cellMap);
    if (!trim) {   // the padding kept every cell again (a run of < 4 cells on a small grid): nothing to walk faster
        walk = PackedGrid();
        return true;
    }
    walk.n = n;
    walk.nb = ref.nb;
    walk.walkTrim = trim;
    walk.planes.resize(ref.planes.size());
    walk_planes(ref.planes.data(), n, walk.cellMap.data(), walk.planes.data());
    return pack_cells(h, n, walk.cellMap.data(), walk, err);
}

// Super-brick level of the three-level walk (rt_walk.h).  Behind the nb^3 brick records: the record {non-empty, 0, 0, 0} of super-brick
// (sx, sy, sz) at nb^3 + sx + nb * (sy + nb * sz) -- the brick strides, so a step updates the record index the same way at every level;
// the slots between them stay zero.  In the record of an EMPTY brick .z (a rank base nobody reads) becomes the flag "my whole
// super-brick is empty: cross it in one step".  Only for power-of-two grids of at least 32 cells per axis.
int super_bricks_per_axis(int n) { return (n >= 32 && (n & (n - 1)) == 0) ? n / 16 : 0; }
size_t super_brick_records(int n) {   // records appended to the brick array
    const size_t ns = (size_t)super_bricks_per_axis(n), nb = (size_t)n / 4;
    return ns * nb * nb;
}

int super_policy(int dflt) {   // (read per scene, not cached: tests switch it between two scenes of one process)
    const char* e = getenv("OCLR_SUPER");
    return e ? atoi(e) : dflt;
}

void append_super_bricks(std::vector<uint4>& bricks, int n, int nb, int policy) {
    const int ns = policy > 0 ? super_bricks_per_axis(n) : 0;
    if (ns == 0) return;
    const size_t nBricks = (size_t)nb * nb * nb;
    bricks.resize(nBricks + super_brick_records(n), make_uint4(0, 0, 0, 0));
    for (int sz = 0; sz < ns; ++sz)
        for (int sy = 0; sy < ns; ++sy)
            for (int sx = 0; sx < ns; ++sx) {
                uint32_t any = 0;
                for (int z = 0; z < 4; ++z)
                    for (int y = 0; y < 4; ++y)
                        for (int x = 0; x < 4; ++x) {
                            const uint4& b = bricks[(size_t)(sx * 4 + x) + (size_t)nb * ((sy * 4 + y) + (size_t)nb * (sz * 4 + z))];
                            any |= b.x | b.y;
                        }
                bricks[nBricks + (size_t)sx + (size_t)nb * (sy + (size_t)nb * sz)] = make_uint4(any ? 1u : 0u, 0, 0, 0);
                if (any) continue;
                for (int z = 0; z < 4; ++z)
                    for (int y = 0; y < 4; ++y)
                        for (int x = 0; x < 4; ++x) bricks[(size_t)(sx * 4 + x) + (size_t)nb * ((sy * 4 + y) + (size_t)nb * (sz * 4 + z))].z = 1u;
            }
}

void pack_lights(const HostScene& h, std::vector<Light>& out) {
    out.resize(h.lightCount ? h.lightCount : 1);
    memset(out.data(), 0, sizeof(Light) * out.size());
    for (uint32_t j = 0; j < h.lightCount; ++j) {
        Light& L = out[j];
        L.type = h.lightType[j];
        L.radius = h.lightRadius[j];
        L.halfDistance = h.lightHalf[j];
        const float4 p = h.lightPos[j], d = h.lightDir[j], c = h.lightColour[j];
        L.pos[0] = p.x; L.pos[1] = p.y; L.pos[2] = p.z;
        L.dir[0] = d.x; L.dir[1] = d.y; L.dir[2] = d.z;
        L.colour[0] = c.x; L.colour[1] = c.y; L.colour[2] = c.z;
        // raytrace_opencl.c:594 -- float argument, double sin * double sqrt, narrowed once
        const float kPi = 3.14159265f;
        const float arg = (L.radius / 2.f) * kPi / 180.f;
        const float dd = dot3(mk3(d.x, d.y, d.z), mk3(d.x, d.y, d.z));
        L.distantRadius = (float)(sin((double)arg) * sqrt((double)dd));
    }
}

}  // namespace oclr
