// rt_types.h -- device-side data layout of the B200 raytrace path (HBM-resident, uploaded once per scene).
//
// The reference hands its kernel 35 flat SoA buffers (source/opencl/raytrace_opencl.c:406-450).  They are
// repacked at upload into the layout below so that every fetch on the hot path is a 128-bit load of data
// that is consumed whole:
//
//   triGeo    4 x float4 per triangle (64 B, two 32 B sectors)
//               q0 = (n.x, n.y, n.z, a.x)   n = cross(ac, ab)          stage 1 (plane distance) needs q0,q1
//               q1 = (a.y, a.z, abab, abac)
//               q2 = (ab.x, ab.y, ab.z, acac)                           stage 2 (barycentrics) needs q2,q3
//               q3 = (ac.x, ac.y, ac.z, D)  D = 1/(abac*abac - abab*acac)
//             All of these are ray-independent sub-expressions of RayIntersectsTriangle
//             (raytrace_opencl.c:131-149) evaluated with the reference's exact fp32 operation order, so
//             hoisting them out of the per-ray test leaves every result bit-identical.
//   triShade  8 x float4 per triangle (128 B): a|mat, b, c, nA, nB, nC, (uv0,uv1), (uv2,-) -- read once per hit.
//   bricks    the reference's 256^3 CSR `Start` array (67 MB, 88 % empty cells) becomes 4x4x4-cell bricks:
//             one uint4 per brick = {occupancy mask lo, hi, rank of the brick's first non-empty cell, 0}
//             (4 MB at 256^3).  A DDA walk reads one 16 B record per brick and then steps through up to
//             ~10 cells of it from registers; empty cells cost one bit test.
//   cellRange one uint2 {begin,end} per NON-EMPTY cell, in brick-major order, into cellList.
//   cellList  the reference's scenePixelTriangleList as uploaded (triangle ids, ascending per cell; the order is
//             observable through the strict `<` closest-hit rule, raytrace_opencl.c:143, 372-377).
//   faceMask  6 x uint32 per non-empty cell, face = axis*2 + (entered moving towards +axis): bit k set when the k-th
//             list entry (k < 32) does not occur in the list of the neighbour cell the DDA just left.  A ray that steps
//             from cell N into cell C has already examined every triangle of N, so only the masked-in entries of C
//             can be new to it -- the trace kernel jumps straight to them instead of scanning the whole list.
//   planes    3 x (n+1) floats (x planes, y planes, z planes) -- copied to shared memory by each CTA.
//
// Walk grid.  The reference puts split plane i at a vertex quantile, so a scene whose vertices sit on few distinct heights (config 2:
// 36 UV spheres, 26 ring heights) repeats planes: 229 of its 256 y layers have zero width, in runs of 8-9.  Where every cell of such a
// run has the same list as the run's first cell in every column (checked at pack time, scene_pack.cpp walk_cell_map), crossing the run
// cell by cell only revisits one list.  The production trace stage therefore walks a second grid over the cells it keeps per axis --
// every positive-width cell, one cell per collapsed run (plus up to 3 duplicates, to make the extent a multiple of 4), every cell of a
// run that did not collapse -- with its own bricks / cellRange / faceMask / planes and the same cellList; planes past the extent repeat
// the last one.  The walk's crossing sequence
// on it is the reference's with runs of equal crossing values shortened, which the tie rule merges in the same order, so it visits the
// same lists in the same order with repeats dropped: the same first hit.  A scene without a collapsible run walks the reference grid.
#pragma once
#include <stdint.h>

#include <vector_functions.h>
#include <vector_types.h>  // float4 / uint4 / uint2 / uchar4 (plain C++ header of the CUDA toolkit)

#if defined(__CUDACC__)
#define OCLR_HD __host__ __device__ __forceinline__
#else
#define OCLR_HD inline
#endif
// Code size of the logic kernel: with everything forced inline it is 7 430 SASS instructions (119 KB against a 32 KB L1.5 instruction
// cache), 40 % of them the 14 inlined copies of the reference's 64-bit RNG, and "no instruction" (instruction-cache misses) is its first
// stall reason (3.7 warp-cycles per issue; the 1 424-instruction trace kernel: 0.2).  OCLR_OUTLINE_LEVEL >= 1 makes rand_f one function,
// >= 2 also sphere_point and the light accumulation (a double-precision pow), >= 3 also the texture lookup (4 020 instructions).  Same
// arithmetic either way.  Default 3 since the end of round 2: config 2 4.31 -> 4.21 ms, config 3 22.53 -> 22.38, config 5 10.88 -> 10.79,
// 1/8 shares unchanged / +1.8 % (profiles/r02_outline_experiment.txt; the first measurement, on the round's earlier code, had been a wash).
#ifndef OCLR_OUTLINE_LEVEL
#define OCLR_OUTLINE_LEVEL 3
#endif
#if defined(__CUDACC__)
#define OCLR_HD_OUT(level) __host__ __device__ OCLR_OUTLINE_##level
#if OCLR_OUTLINE_LEVEL >= 1
#define OCLR_OUTLINE_1 __noinline__
#else
#define OCLR_OUTLINE_1 __forceinline__
#endif
#if OCLR_OUTLINE_LEVEL >= 2
#define OCLR_OUTLINE_2 __noinline__
#else
#define OCLR_OUTLINE_2 __forceinline__
#endif
#if OCLR_OUTLINE_LEVEL >= 3
#define OCLR_OUTLINE_3 __noinline__
#else
#define OCLR_OUTLINE_3 __forceinline__
#endif
#else
#define OCLR_HD_OUT(level) inline
#endif
// Level switches of the walk (rt_walk.h: 3 + 6 IEEE divisions, ~20 % of the trace kernel's code, run by 10 lanes at a time):
// OCLR_OUTLINE_SWITCH=1 makes them real functions (A/B builds).
#ifndef OCLR_OUTLINE_SWITCH
#define OCLR_OUTLINE_SWITCH 0
#endif
#if defined(__CUDACC__) && OCLR_OUTLINE_SWITCH
#define OCLR_HD_SW __host__ __device__ __noinline__
#else
#define OCLR_HD_SW OCLR_HD
#endif

namespace oclr {

enum { kMaterialChannels = 5, kChColor = 0, kChReflection = 1, kChTransparency = 2, kChBump = 3, kChLuminance = 4 };
enum { kRingSize = 12, kMaxBounces = 12 };
enum { kNoTriangle = 0xFFFFFFFFu };

// One light, with the per-light constants of raytrace_opencl.c:594 hoisted (evaluated once at upload in the
// reference's double-precision expression).
struct Light {
    int32_t type;            // _LIGHT_TYPE_* (raytrace_opencl.h:1-12)
    float radius;            // lightRadius[j]
    float halfDistance;      // lightHalfAttenuationDistance[j]
    float distantRadius;     // (float)(sin((radius/2)*M_PIf/180) * sqrt(dot(dir,dir)))   (:594)
    float pos[4];
    float dir[4];
    float colour[4];
};

struct SceneView {
    const float4* triGeo;
    const float4* triShade;
    const uint4* bricks;
    const uint2* cellRange;
    const uint32_t* cellList;
    const uint32_t* faceMask;  // 6 per non-empty cell: bit k of [rank*6 + face] = list entry k is NOT in the face neighbour's list
    const float* planes;      // 3*(n+1)
    const uint2* matSize;     // 5*materialCount
    const int32_t* matStart;  // 5*materialCount+1
    const uchar4* textures;
    const Light* lights;
    uint32_t triangleCount;
    uint32_t materialCount;
    uint32_t lightCount;
    int32_t n;                // axesDivCount (power of two)
    int32_t nb;               // bricks per axis = max(n/4, 1)
    // Extents of the grid the packed walk runs on (rt_walk.h): n minus `walkTrim`'s field of the axis, packed like a cell coordinate
    // (pk_make).  0 = the reference grid (the default, so that a view built without knowing of walk grids is one); non-zero only in a
    // walk grid's view (see the top of this file).  Index space, brick addressing and plane stride stay those of n.
    uint32_t walkTrim = 0;
};

struct Camera {
    uint32_t width, height;
    float eye[4];
    float eyeToTopLeft[4];
    float leftToRight[4];
    float topToBottom[4];
    float pixelSizeInv;
};

struct FrameView {
    Camera cam;
    const uint32_t* camStart;
    const uint32_t* camEnd;
    const uint32_t* camList;
    uint32_t sampleCount;        // S of the whole job: seeds are pixel*S + s+1 and every sample is scaled by 65535/S
    uint32_t sampleBegin, sampleEnd;   // samples rendered by this call (progressive rendering: 0 <= begin < end <= S)
    uint32_t rowBegin, rowEnd;   // rows rendered by this launch when bandWorld <= 1
    // Screen-band partition across GPUs (SURVEY.md section 8e): when bandWorld > 1 the launch covers the rows y with
    // (y / bandRows) % bandWorld == bandRank; `ownedRows` of them exist.  Launch-domain row k maps to frame row map_row(k).
    uint32_t bandRows, bandRank, bandWorld, ownedRows;
    uint16_t* outR;              // full-frame planes, row-major, width*height
    uint16_t* outG;
    uint16_t* outB;
    uint32_t* idOut;             // optional: primary-hit triangle id per pixel (sample 0), or nullptr
    uint8_t* flagOut;            // optional: per pixel, bit 0 = the reference's result is undefined here (rt_core.h triangle_normal)
    // Progressive accumulation (SURVEY.md section 8f-3).  Default (accum == nullptr): the reference's rule, every sample is
    // truncated to an integer and added to the 16-bit planes (raytrace_opencl.c:726-741); sample 0 overwrites, later samples add,
    // so a job can be rendered in several calls over sample ranges.  accum != nullptr: (sum r, sum g, sum b, samples) per pixel
    // in fp32, no per-sample truncation; the planes are resolved from it after the call (resolve_accum_kernel).
    float4* accum;
    unsigned long long* doneCount;   // optional: pixel-samples finished so far by the current render call (progress, raytrace.c:580)
    // optional: non-zero when the caller's camera lists failed the range check (check_camera_lists_kernel, pack_kernels.cuh): the
    // kernels then return without touching the lists and the host reports the error at its next synchronisation
    const uint32_t* camBad;
};

// Launch-domain row k -> frame row (>= height when k is past the owned rows).
OCLR_HD uint32_t map_row(const FrameView& F, uint32_t k) {
    if (F.bandWorld <= 1) return F.rowBegin + k < F.rowEnd ? F.rowBegin + k : 0xFFFFFFFFu;
    if (k >= F.ownedRows) return 0xFFFFFFFFu;
    return (k / F.bandRows) * (F.bandRows * F.bandWorld) + F.bandRank * F.bandRows + (k % F.bandRows);
}
OCLR_HD uint32_t launch_rows(const FrameView& F) { return F.bandWorld <= 1 ? F.rowEnd - F.rowBegin : F.ownedRows; }

// Per-launch event counters for the algorithmic-bytes figure (SURVEY.md section 8d).  Only the counting build
// of the kernel touches them.
struct Counters {
    unsigned long long segments, primCandidates, gridRays, cells, cellsNonEmpty, gridCandidates, shadedHits,
        occluderLookups, bricksLoaded, emptyBrickCells, walkWarpIters, walkLaneIters, testWarpIters, testLaneIters,
        mailboxSkips, coarseSteps, coarseEnters, switchWarpIters, switchLaneIters,
        walkIdleLanes, walkParkedLanes, walkFinishedLanes, walkLowIters, walkExhaustedIters,
        splitAttempts, splitsDone, splitParts, splitCancelled,
        superSteps, superEnters, superRefines,   /* three-level walk: steps / level switches at super-brick granularity */
        /* per-warp timing of the trace kernel, counting build: when warps leave / see the queue dry, 32-us buckets since their start */
        exitHist00, exitHist01, exitHist02, exitHist03, exitHist04, exitHist05, exitHist06, exitHist07, exitHist08, exitHist09, exitHist10, exitHist11, exitHist12, exitHist13, exitHist14, exitHist15, exhaustHist00, exhaustHist01, exhaustHist02, exhaustHist03, exhaustHist04, exhaustHist05, exhaustHist06, exhaustHist07, exhaustHist08, exhaustHist09, exhaustHist10, exhaustHist11, exhaustHist12, exhaustHist13, exhaustHist14, exhaustHist15, warpOuterItersMax, warpOuterItersSum, warpsRun;   // lanes of a walk iteration that were not walking, by reason
};

}  // namespace oclr
