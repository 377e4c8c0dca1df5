// pack_kernels.cuh -- device half of the "scene upload path": the reference arrays are copied to HBM as they are
// (one cudaMemcpyAsync per array, straight from the caller's memory) and repacked there into the layout of
// rt_types.h.  Same arithmetic as scene_pack.cpp (the host packer the tests use as the checker), compiled with
// -fmad=false so the hoisted per-triangle terms are the exact fp32 values of raytrace_opencl.c:131-149.
#pragma once
#include <cuda_runtime.h>

#include <cub/device/device_scan.cuh>

#include "rt_core.h"

namespace oclr {

enum PackError { kPackOk = 0, kPackBadVertexIndex = 1, kPackBadMaterial = 2, kPackBadCsr = 4, kPackBadListEntry = 8, kPackListTooLong = 16 };
enum { kMaxCellListLength = 1 << 17 };   // wf_pipe_kernel orders the pairs of one drain (<= 127 cells) with a 24-bit index

// One thread per triangle: gathers the 3 vertices (16 B loads), precomputes the plane/Gram terms, writes 4 + 8 float4.
__global__ void __launch_bounds__(256) pack_triangles_kernel(uint32_t triangleCount, uint32_t vertexCount, uint32_t materialCount,
                                                             const float4* __restrict__ vertex, const int4* __restrict__ triIdx,
                                                             const int32_t* __restrict__ triMat, const float2* __restrict__ triUv,
                                                             const float4* __restrict__ triNormal, float4* __restrict__ geo,
                                                             float4* __restrict__ shade, uint32_t* __restrict__ error) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= triangleCount) return;
    const int4 vi = __ldg(triIdx + i);
    const int32_t mat = __ldg(triMat + i);
    if ((uint32_t)vi.x >= vertexCount || (uint32_t)vi.y >= vertexCount || (uint32_t)vi.z >= vertexCount) {
        atomicOr(error, (uint32_t)kPackBadVertexIndex);
        return;
    }
    if (mat >= (int32_t)materialCount) atomicOr(error, (uint32_t)kPackBadMaterial);
    const float4 A = __ldg(vertex + vi.x), B = __ldg(vertex + vi.y), C = __ldg(vertex + vi.z);
    const f3 a = mk3(A.x, A.y, A.z), b = mk3(B.x, B.y, B.z), c = mk3(C.x, C.y, C.z);
    const f3 ab = mk3(b.x - a.x, b.y - a.y, b.z - a.z);
    const f3 ac = mk3(c.x - a.x, c.y - a.y, c.z - a.z);
    const f3 n = cross3(ac, ab);
    const float abab = dot3(ab, ab), abac = dot3(ab, ac), acac = dot3(ac, ac);
    const float D = 1.f / (abac * abac - abab * acac);
    float4* g = geo + 4 * (size_t)i;
    g[0] = make_float4(n.x, n.y, n.z, a.x);
    g[1] = make_float4(a.y, a.z, abab, abac);
    g[2] = make_float4(ab.x, ab.y, ab.z, acac);
    g[3] = make_float4(ac.x, ac.y, ac.z, D);
    const float4 nA = __ldg(triNormal + 3 * (size_t)i), nB = __ldg(triNormal + 3 * (size_t)i + 1), nC = __ldg(triNormal + 3 * (size_t)i + 2);
    const float2 u0 = __ldg(triUv + 3 * (size_t)i), u1 = __ldg(triUv + 3 * (size_t)i + 1), u2 = __ldg(triUv + 3 * (size_t)i + 2);
    float4* s = shade + 8 * (size_t)i;
    s[0] = make_float4(a.x, a.y, a.z, __int_as_float(mat));
    s[1] = make_float4(b.x, b.y, b.z, 0.f);
    s[2] = make_float4(c.x, c.y, c.z, 0.f);
    s[3] = make_float4(nA.x, nA.y, nA.z, 0.f);
    s[4] = make_float4(nB.x, nB.y, nB.z, 0.f);
    s[5] = make_float4(nC.x, nC.y, nC.z, 0.f);
    s[6] = make_float4(u0.x, u0.y, u1.x, u1.y);
    s[7] = make_float4(u2.x, u2.y, 0.f, 0.f);
}

// Reference cell id of cell (x, y, z) of the grid being packed, or -1 when it has none.  map == nullptr: the reference grid itself; else a
// walk grid (rt_types.h): cell j of axis a stands for reference cell map[a * n + j], -1 past the axis' extent (scene_pack.cpp walk_cell_map).
__device__ __forceinline__ long long grid_ref_id(const int32_t* __restrict__ map, int n, int x, int y, int z) {
    if ((unsigned)x >= (unsigned)n || (unsigned)y >= (unsigned)n || (unsigned)z >= (unsigned)n) return -1;
    if (map) {
        x = __ldg(map + x);
        y = __ldg(map + n + y);
        z = __ldg(map + 2 * n + z);
        if ((x | y | z) < 0) return -1;
    }
    return (long long)x + (long long)n * y + (long long)n * n * z;
}

// Pass 1 over the reference CSR (n^3 + 1 starts): one thread per 4x4x4 brick builds its occupancy mask and counts its
// non-empty cells.  Pass 2 (after an exclusive scan of the counts) writes {mask, rank base} and the {begin,end} ranges.
__device__ __forceinline__ uint64_t brick_mask(const uint32_t* __restrict__ start, int n, int nb, uint32_t total, int b, uint32_t* error,
                                               const int32_t* __restrict__ map, uint2* ranges /* nullable */,
                                               uint32_t* cellIds = nullptr /* linear cell id (of this grid) per non-empty cell */) {
    const int side = n >= 4 ? 4 : n;
    const int bx = b % nb, by = (b / nb) % nb, bz = b / (nb * nb);
    uint64_t mask = 0;
    int k = 0;
    for (int z = 0; z < side; ++z)
        for (int y = 0; y < side; ++y)
            for (int x = 0; x < side; ++x) {
                const long long id = grid_ref_id(map, n, bx * 4 + x, by * 4 + y, bz * 4 + z);
                if (id < 0) continue;
                const uint32_t s = __ldg(start + id), e = __ldg(start + id + 1);
                if (e < s || e > total) atomicOr(error, (uint32_t)kPackBadCsr);
                else if (e - s >= (uint32_t)kMaxCellListLength) atomicOr(error, (uint32_t)kPackListTooLong);
                if (s < e) {
                    mask |= 1ull << (x | (y << 2) | (z << 4));
                    if (ranges) ranges[k] = make_uint2(s, e);
                    if (cellIds) cellIds[k] = (uint32_t)((bx * 4 + x) + (size_t)n * (by * 4 + y) + (size_t)n * n * (bz * 4 + z));
                    ++k;
                }
            }
    return mask;
}

__global__ void __launch_bounds__(128) brick_count_kernel(const uint32_t* __restrict__ start, int n, int nb, uint32_t total,
                                                          const int32_t* __restrict__ map, uint32_t* __restrict__ counts, uint32_t* __restrict__ error) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb * nb * nb) return;
    counts[b] = (uint32_t)__popcll(brick_mask(start, n, nb, total, b, error, map, nullptr));
}

__global__ void __launch_bounds__(128) brick_write_kernel(const uint32_t* __restrict__ start, int n, int nb, uint32_t total,
                                                          const int32_t* __restrict__ map, const uint32_t* __restrict__ rankBase, uint4* __restrict__ bricks,
                                                          uint2* __restrict__ cellRange, uint32_t* __restrict__ cellIds,
                                                          uint32_t* __restrict__ error) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb * nb * nb) return;
    const uint32_t base = rankBase[b];
    const uint64_t mask = brick_mask(start, n, nb, total, b, error, map, cellRange + base, cellIds + base);
    bricks[b] = make_uint4((uint32_t)mask, (uint32_t)(mask >> 32), mask ? base : 0u, 0u);   // (.z of an empty brick: flags of the three-level walk, rt_walk.h)
}

// Super-brick level of the three-level walk (rt_walk.h): one 64-thread CTA per super-brick (4x4x4 bricks) writes its record
// {non-empty, 0, 0, 0} behind the nb^3 brick records (at the brick strides; the slots between are zeroed by the caller) and turns .z of
// its EMPTY bricks into the flag "the whole super-brick is empty".  Same result as append_super_bricks (scene_pack.cpp), byte for byte.
__global__ void __launch_bounds__(64) super_brick_kernel(uint4* __restrict__ bricks, int nb, int ns) {
    const int s = blockIdx.x, t = threadIdx.x;
    const int sx = s % ns, sy = (s / ns) % ns, sz = s / (ns * ns);
    const size_t b = (size_t)(sx * 4 + (t & 3)) + (size_t)nb * ((size_t)(sy * 4 + ((t >> 2) & 3)) + (size_t)nb * (size_t)(sz * 4 + (t >> 4)));
    const uint4 br = bricks[b];
    const int any = __syncthreads_or((br.x | br.y) != 0u);
    if (t == 0) bricks[(size_t)nb * nb * nb + (size_t)sx + (size_t)nb * ((size_t)sy + (size_t)nb * (size_t)sz)] = make_uint4(any ? 1u : 0u, 0u, 0u, 0u);
    if (!any) bricks[b].z = 1u;
}

// Face masks (rt_types.h): bit e set = list entry e of the cell is absent from the list of the neighbour the walk comes from (in the
// grid being packed: map as in grid_ref_id).  One thread per (non-empty cell, face): the work of the face masks sits in the ~10 % of
// bricks that hold triangles, so it is spread over cells x faces instead of being done by the brick's thread.  Both lists are
// ascending: one merge pass.
__global__ void __launch_bounds__(256) face_mask_kernel(const uint32_t* __restrict__ start, int n, uint32_t total, uint32_t nonEmpty,
                                                        const int32_t* __restrict__ map, const uint32_t* __restrict__ cellIds,
                                                        const uint2* __restrict__ cellRange, const uint32_t* __restrict__ list,
                                                        uint32_t* __restrict__ faceMask) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nonEmpty * 6u) return;
    const uint32_t k = t / 6u, face = t - 6u * k;   // face = axis*2 + (entered moving towards +axis)
    const uint32_t id = cellIds[k];
    int q[3] = {(int)(id % (uint32_t)n), (int)((id / (uint32_t)n) % (uint32_t)n), (int)(id / ((uint32_t)n * (uint32_t)n))};
    q[face >> 1] += (face & 1) ? -1 : 1;
    uint32_t m = 0xFFFFFFFFu;
    const long long nid = grid_ref_id(map, n, q[0], q[1], q[2]);
    if (nid >= 0) {
        const uint32_t ns = __ldg(start + nid), ne = __ldg(start + nid + 1);
        const uint2 r = cellRange[k];
        if (ns < ne && ne <= total && r.y <= total) {
            uint32_t j = ns;
            uint32_t other = __ldg(list + j);
            for (uint32_t e = 0; e < 32u && r.x + e < r.y; ++e) {
                const uint32_t tri = __ldg(list + r.x + e);
                while (other < tri && j + 1 < ne) other = __ldg(list + (++j));
                if (other == tri) m &= ~(1u << e);
            }
        }
    }
    faceMask[t] = m;
}

// Walk grid (rt_types.h): does run `r` (zero-width cells first .. first + count - 1 of its axis) collapse?  One thread per column across
// the other two axes compares the lists of the run's cells with the first one's; a difference sets bit 0 of differs[r].  Same rule as
// scene_pack.cpp walk_run_collapses.  The grid may be the caller's and is not known to be a CSR yet (brick_mask's flag is read later):
// a cell whose range is not inside the list (end < begin or end > total) counts as a difference, and no entry of it is read.
__global__ void __launch_bounds__(256) run_check_kernel(const uint32_t* __restrict__ start, const uint32_t* __restrict__ list, int n,
                                                        uint32_t total, const int3* __restrict__ runs, uint32_t* __restrict__ differs) {
    const int3 r = runs[blockIdx.y];   // (axis, first, count)
    const uint32_t col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= (uint32_t)n * (uint32_t)n) return;
    const size_t stride[3] = {1, (size_t)n, (size_t)n * n};
    const int u = r.x == 0 ? 1 : 0, v = r.x == 2 ? 1 : 2;
    const size_t first = (size_t)r.y * stride[r.x] + (size_t)(col % (uint32_t)n) * stride[u] + (size_t)(col / (uint32_t)n) * stride[v];
    const uint32_t s0 = __ldg(start + first), e0 = __ldg(start + first + 1);
    bool same = s0 <= e0 && e0 <= total;
    for (int k = 1; same && k < r.z; ++k) {
        const size_t id = first + (size_t)k * stride[r.x];
        const uint32_t s = __ldg(start + id), e = __ldg(start + id + 1);
        same = s <= e && e <= total && e - s == e0 - s0;
        for (uint32_t q = 0; same && q < e0 - s0; ++q) same = __ldg(list + s + q) == __ldg(list + s0 + q);
    }
    if (!same) atomicOr(differs + blockIdx.y, 1u);
}

// Vertex indices of every triangle, checked before the device grid builder gathers vertices by them (the packer checks them too,
// but runs concurrently with the builder's first kernels).
__global__ void __launch_bounds__(256) check_indices_kernel(uint32_t triangleCount, uint32_t vertexCount, const int4* __restrict__ triIdx,
                                                            uint32_t* __restrict__ error) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= triangleCount) return;
    const int4 vi = __ldg(triIdx + i);
    if ((uint32_t)vi.x >= vertexCount || (uint32_t)vi.y >= vertexCount || (uint32_t)vi.z >= vertexCount) atomicOr(error, (uint32_t)kPackBadVertexIndex);
}

// Material ids of the resident triangles (the .w word of triShade record 0, pack_triangles_kernel) against a new material count:
// the same rule as the packer's.
__global__ void __launch_bounds__(256) check_materials_kernel(uint32_t triangleCount, uint32_t materialCount, const float4* __restrict__ shade,
                                                              uint32_t* __restrict__ error) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < triangleCount && __float_as_int(__ldg(shade + 8 * (size_t)i).w) >= (int32_t)materialCount) atomicOr(error, (uint32_t)kPackBadMaterial);
}

__global__ void __launch_bounds__(256) check_list_kernel(const uint32_t* __restrict__ list, uint32_t total, uint32_t triangleCount,
                                                         uint32_t* __restrict__ error) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total && __ldg(list + i) >= triangleCount) atomicOr(error, (uint32_t)kPackBadListEntry);
}

// Caller-supplied camera lists (cameraPixelTriangleListStart / End / list, raytrace.h:58-106): Start <= End <= list size for every
// pixel, every entry a triangle id.  The reference trusts them; a bad entry here would be an illegal address -- a sticky fault for the
// whole process.  Runs on the upload stream in front of the first logic launch (also the one started ahead); no host round trip.
enum { kCamBadRange = 1, kCamBadEntry = 2 };
__global__ void __launch_bounds__(256) check_camera_lists_kernel(const uint32_t* __restrict__ start, const uint32_t* __restrict__ end,
                                                                 const uint32_t* __restrict__ list, uint32_t pixels, uint32_t listSize,
                                                                 uint32_t triangleCount, uint32_t* __restrict__ flag) {
    const uint32_t stride = gridDim.x * blockDim.x;
    uint32_t bad = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < pixels; i += stride) {
        const uint32_t s = __ldg(start + i), e = __ldg(end + i);
        if (s > e || e > listSize) bad |= kCamBadRange;
    }
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < listSize; i += stride)
        if (__ldg(list + i) >= triangleCount) bad |= kCamBadEntry;
    if (bad) atomicOr(flag, bad);
}

// sceneBoxMin (cl_float3 per plane index) -> three contiguous float arrays
__global__ void split_planes_kernel(const float4* __restrict__ boxMin, int n, float* __restrict__ planes) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    const float4 p = boxMin[i];
    planes[i] = p.x;
    planes[(n + 1) + i] = p.y;
    planes[2 * (n + 1) + i] = p.z;
}

}  // namespace oclr
