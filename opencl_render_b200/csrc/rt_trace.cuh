// rt_trace.cuh -- production trace stage of the wavefront pipeline: a setup kernel + a persistent trace kernel organised as a
// warp-level pipeline (rt_wavefront.cuh has the logic kernel).
//
// What ncu said about the first-generation trace kernel, in which a lane owned a ray from queue to result
// (profiles/r01_wf_trace_cfg2_*; the kernel itself is retired, git history has it): issue-bound (66-69 % of issue slots) with 14 of 32
// lanes active per instruction.  By phase: the walk ran at ~21 lanes, but "open the cell + scan its list + test" -- 37 % of all
// instructions -- ran with 5-6 lanes, the level switches of the two-level walk with <2, and every refill ran
// BindInCube/GetBoxAddress with a handful of lanes.  Hence:
//
//   wf_setup_kernel   one thread per queued ray, all lanes busy: BindInCube + GetBoxAddress + first crossings
//                     (raytrace_opencl.c:350-362), written as 64-byte records in QUEUE order, so the trace kernel's refill is
//                     four coalesced 128-bit loads per lane instead of a gather plus ~400 divergent instructions.
//   wf_pipe_kernel    see the comment above the kernel.
//
// Results are bit-identical to the other kernels by construction (same rt_core.h / rt_walk.h arithmetic; tests assert it).
#pragma once
#include "rt_wavefront.cuh"

namespace oclr {

#ifndef OCLR_TRACE_MIN_CTAS
#define OCLR_TRACE_MIN_CTAS 8
#endif
// Scheduling knobs of wf_pipe_kernel (run-time tunable through OCLR_DRAIN_MIN / OCLR_WALK_MIN3 / OCLR_SWITCH_MIN / OCLR_REFILL_MIN /
// OCLR_TAIL_DRAIN / OCLR_HIERARCHICAL; the defaults are the measured optimum on config 2, flat within a few per cent).
struct TraceTuning {
    int refillMin;     // refill from the queue once this many lanes are idle
    int hierarchical;  // 1: cross empty 4x4x4 bricks at brick granularity (exact two-level walk); 2: and empty super-bricks in one step
    int tailDrain;     // queue dry: drain only once this many cells wait (latency of the last long rays)
    int drainMin;      // drain the warp's cell queue at this size
    int walkMin3;      // end a walk burst below this many walking lanes
    int switchMin;     // run parked level switches once this many lanes wait for one
    int splitMin;      // queue dry: a walk with at least this many cells to go is cut into parts for the warp's idle lanes (0 = never)
    int splitPart;     // ... of at least this many cells each
    int splitEarly;    // > 0: also before the queue is dry, for a ray that has been with the warp for that many outer iterations
    int handoffAfter;  // HANDOFF instantiation: outer iterations a ray has been with its warp before the warp gives it up (queue dry; rt_tail.cuh)
    int handoffMode;   // 1 / 3: to a burst walker, one ray per warp (brick planes / cell planes); 2: back into a queue of walk records for a second pass
    int handoffLanes;  // a warp gives its rays up once at most this many of its lanes still hold one (32: whatever it holds)
    int handoffBurst;  // HANDOFF: with the queue dry a walk burst ends after this many iterations at the latest (tail mode would let a lone
                       // ray that crosses empty space -- no cell to drain -- walk to its end inside ONE burst, out of the hand-off's reach)
};

// Rays a launch's pipe kernel gives up in its tail (HANDOFF instantiation, small launch domains; rt_tail.cuh).
struct TailQueue {
    uint4* entries;     // modes 1, 3: {ray index (slot * Q + path), current cell (not yet examined) / empty brick, entry face, level}
    uint32_t* count;    // rays given up by the pipe kernel of this round; {count, 0, 0, 0} doubles as the class counts of the second pass
    uint32_t* cursor;   // next entry to take
    uint32_t capacity;
    // mode 2: the rays as walk records (the setup kernel's format, resumed from the cell the lane stood in) + identity order
    float4* o;
    float4* d;
    float4* s0;
    uint4* s1;
    uint32_t* order;
};

// Walk records written by wf_setup_kernel, indexed by queue slot, and the order in which the trace kernel takes them.
enum { kLengthClasses = 4, kRoundLogSize = 64 };
struct WalkRecords {
    float4* o;    // (o.xyz, minD)
    float4* d;    // (r.xyz, maxD)
    float4* s0;   // (tx, ty, tz, as_float(cpk))
    uint4* s1;    // (epk, excl, path, coarseOk)
    // Longest-first scheduling: a trace launch cannot end before its longest walk does, and one lane walking 500 cells alone
    // takes ~0.3 ms -- if that ray is taken from the queue last it is all tail.  The setup kernel therefore sorts the queue
    // slots into length classes (estimated cells between start and end / exit cell) and the trace kernel drains the classes
    // longest first.  order[c * Q + k] = k-th queue slot of class c; classCount[c] = slots in class c.
    uint32_t* order;
    uint32_t* classCount;
    uint32_t Q;
};

// Estimated number of cells between the start cell and the end cell (finite rays) or the cell where the ray leaves the grid.
// Only used to ORDER the work, never for a result: approximate arithmetic is fine here.
// On a walk grid (trim != 0, SceneView::walkTrim) the exit cell is clamped to the extents like pwalk_setup's cells.
__device__ __forceinline__ int walk_length_estimate(const PackedWalk& g, int n, uint32_t trim, const float* px, const float* py, const float* pz) {
    int ex, ey, ez;
    if (g.epk != kPkNone) {
        ex = pk_get(g.epk, 0);
        ey = pk_get(g.epk, 1);
        ez = pk_get(g.epk, 2);
    } else {
        const float bx = g.r.x >= 0.f ? px[n] : px[0], by = g.r.y >= 0.f ? py[n] : py[0], bz = g.r.z >= 0.f ? pz[n] : pz[0];
        float t = OCLR_INF;
        if (g.r.x != 0.f) t = fminf(t, (bx - g.o.x) / g.r.x);
        if (g.r.y != 0.f) t = fminf(t, (by - g.o.y) / g.r.y);
        if (g.r.z != 0.f) t = fminf(t, (bz - g.o.z) / g.r.z);
        if (!(t < OCLR_INF) || t < 0.f) t = 0.f;
        box_address(n, px, py, pz, mk3(g.o.x + t * g.r.x, g.o.y + t * g.r.y, g.o.z + t * g.r.z), ex, ey, ez);
        ex = pwalk_clamp_cell(ex, n, trim, 0);
        ey = pwalk_clamp_cell(ey, n, trim, 1);
        ez = pwalk_clamp_cell(ez, n, trim, 2);
    }
    const int sh = 2 * g.level;   // (level 1: brick coordinates, level 2: super-brick coordinates)
    return abs(ex - (pk_get(g.cpk, 0) << sh)) + abs(ey - (pk_get(g.cpk, 1) << sh)) + abs(ez - (pk_get(g.cpk, 2) << sh));
}

__global__ void __launch_bounds__(256) wf_setup_kernel(SceneView S, WfState w, WalkRecords rec) {
    extern __shared__ float shPlanes[];
    __shared__ uint32_t shCount[kLengthClasses], shBase[kLengthClasses];
    const uint32_t count = *w.queueCount;
    if (blockIdx.x == 0 && threadIdx.x == 0 && w.roundIndex < kRoundLogSize) w.roundLog[w.roundIndex] = count;
    if (blockIdx.x * blockDim.x >= count) return;
    load_planes(shPlanes, S);
    const int n = S.n;
    const int lane = threadIdx.x & 31;
    const float* px = shPlanes;
    const float* py = shPlanes + (n + 1);
    const float* pz = shPlanes + 2 * (n + 1);
    const int span = n - (int)min(S.walkTrim & kPkMask, min((S.walkTrim >> kPkBits) & kPkMask, (S.walkTrim >> (2 * kPkBits)) & kPkMask));
    for (uint32_t base = blockIdx.x * blockDim.x; base < count; base += gridDim.x * blockDim.x) {
        const uint32_t idx = base + threadIdx.x;
        const bool valid = idx < count;
        int cls = -1;
        if (valid) {
            const uint32_t path = w.queue[idx];
            const float4 ro = w.rayO[path], rd = w.rayD[path];
            PackedWalk g;
            pwalk_setup(g, n, S.nb, S.walkTrim, px, py, pz, mk3(ro.x, ro.y, ro.z), mk3(rd.x, rd.y, rd.z), ro.w, rd.w);
            rec.o[idx] = ro;
            rec.d[idx] = rd;
            rec.s0[idx] = make_float4(g.tx, g.ty, g.tz, __uint_as_float(g.cpk));
            rec.s1[idx] = make_uint4(g.epk, w.rayExcl[path], path, g.coarseOk ? 1u : 0u);
            const int len = walk_length_estimate(g, n, S.walkTrim, px, py, pz);
            // classes by quarters of the longest extent (n on the reference grid), longest first (a walk can be up to 3n cells long; 8
            // classes measured no better than 4)
            cls = kLengthClasses - 1 - min(kLengthClasses - 1, (len * kLengthClasses) / (span > 0 ? span : 1));
        }
        // one global atomic per CTA, class and iteration (the warps' counts are first summed in shared memory)
        if (threadIdx.x < kLengthClasses) shCount[threadIdx.x] = 0u;
        __syncthreads();
        uint32_t within = 0;
#pragma unroll
        for (int c = 0; c < kLengthClasses; ++c) {
            const unsigned m = __ballot_sync(0xFFFFFFFFu, cls == c);
            if (m == 0u) continue;
            uint32_t pos = 0;
            if (lane == 0) pos = atomicAdd(&shCount[c], (uint32_t)__popc(m));
            pos = __shfl_sync(0xFFFFFFFFu, pos, 0);
            if (cls == c) within = pos + (uint32_t)__popc(m & ((1u << lane) - 1u));
        }
        __syncthreads();
        if (threadIdx.x < kLengthClasses) shBase[threadIdx.x] = shCount[threadIdx.x] ? atomicAdd(rec.classCount + threadIdx.x, shCount[threadIdx.x]) : 0u;
        __syncthreads();
        if (cls >= 0) rec.order[(size_t)cls * rec.Q + shBase[cls] + within] = idx;
    }
}

enum { kWsNone = 0, kWsRun = 1, kWsRefine = 2, kWsEnter = 3, kWsFinished = 4, kWsHeld = 5, kWsPartDone = 6 };

// ---- wf_pipe_kernel: warp-level pipeline ----------------------------------------------------------------------------------
// ncu on the lane-owned trace kernels: 37 % of all instructions are the
// lane-owned test work (open cell, scan its list, test) executed with 5-6 of 32 lanes, because at any moment only a few of a
// warp's rays sit on a cell with untested triangles.  Only the WALK is inherently per-ray; opening a cell and testing a
// (ray, triangle) pair are independent work items, so they are decoupled from the lane that owns the ray:
//
//   WALK    lanes own rays; an occupied cell is appended to the WARP's cell queue {rank, entry face, owner lane, seq}
//           (one ballot + one store); seq = position of the cell along that ray's walk within the current batch;
//   OPEN    any lane takes any queued cell: range + face mask, then the warp enumerates the untested entries round by round
//           into the warp's pair queue {triangle, owner, seq};
//   TEST    any lane takes any pair: ray constants from the owner's row of a shared table, the full test against the ray's
//           ORIGINAL (minD, maxD), result folded with a 64-bit shared atomicMin on key = seq | t | pair index.  That is the
//           reference's rule exactly: first cell (in walk order) with any hit wins (:380); inside a cell the in-cell bound
//           shrinks with a strict `<` (:143, :372-377), i.e. smallest t, earliest list entry on ties -- pair indices grow in
//           list order.  t > 0 (minD >= 0 for every ray the path produces), so the float's bit pattern orders like the value;
//   RESOLVE after a drain every owner looks at its key: hit -> write (tri, t, abL, acL) and free the lane; walk finished and
//           nothing found -> miss.  Rays keep walking between drains (bounded speculation: a batch is ~one cell per lane).
//
//   SPLIT   (tail of the launch: the ray queue is dry and lanes sit idle) a launch cannot end before its longest walk does, and one
//           lane stepping through several hundred cells alone is ~0.3 ms that nothing hides -- the floor that capped strong scaling
//           at 0.50 on 8 GPUs.  The warp therefore cuts the longest walk it still holds into parts along its dominant axis
//           (pwalk_split_plan): the owner keeps the first part, idle lanes start the others from the exact state pwalk_jump computes
//           at each stop plane (binary search over the crossing values, no walking; exactness: tests/test_hostemu_parity.py
//           test_run_time_split_is_exact).  Parts are ordinary lane-owned walks with their own best-hit keys; a group record per
//           head lane (hit / miss bit per part) gives the ray's result by the reference's rule -- the first part in walk order with
//           a hit wins once every part before it has finished without one; a hit cancels the parts behind it.
//
// No mailbox here: pairs of one ray are tested concurrently, and face masks already remove the repeats between adjacent cells
// (a per-lane mailbox removed 6 % more in the lane-owned kernel).
// Super-brick level of the walk (rt_walk.h, three-level walk): exact, and measured -- it removes 37 % of config 3's brick-level steps
// and 10 % of config 2's, but the kernel sits exactly at its 64-register cap: compiled in, the level costs 5 % more executed
// instructions and spills into the loops (long-scoreboard stalls 1.6 -> 2.6 per issue), config 2 -7 %, config 3 -3 % even when it is
// used (profiles/r02_super_level.txt).  Off in the production build; `-DOCLR_SUPER_LEVEL=1` builds the variant the tests exercise.
#ifndef OCLR_SUPER_LEVEL
#define OCLR_SUPER_LEVEL 0
#endif
#ifndef OCLR_END_KEY
#define OCLR_END_KEY 1
#endif
// 1: the walk reads origin / direction of the stepped axis from the warp's shared ray table (the tests read it from there anyway)
// instead of holding all six components in registers through every phase of the kernel; the signs of the direction stay in a register
#ifndef OCLR_RAY_IN_SMEM
#define OCLR_RAY_IN_SMEM 1
#endif
#ifndef OCLR_CELLQ_CAP
#define OCLR_CELLQ_CAP 96
#endif
enum { kCellQCap = OCLR_CELLQ_CAP, kPairQCap = 64 };

struct WarpPipe {
    float ray[8][32];               // [o.x o.y o.z r.x r.y r.z minD maxD][owner lane] (a miss reports maxD from here: no register for it)
    uint32_t excl[32];
    unsigned long long bestKey[32];
    uint32_t bestTri[32];
    float bestAB[32], bestAC[32];
    uint32_t cellQ[2][kCellQCap];   // [0] rank | face << 29, [1] owner | seq << 8
    uint32_t pairQ[2][kPairQCap];   // [0] triangle, [1] owner | seq << 8
    // run-time split of long walks (SPLIT above)
    uint32_t grp[32];               // per lane: 0 = a whole ray; else 1 << 31 | head lane | part index << 8
    uint32_t gHit[32], gMiss[32];   // per group, indexed by head lane: bit j = part j holds a hit / finished without one (bit 31 of gMiss: result written)
    uint32_t gParts[32];            // parts of the group
    uint32_t groups;                // live groups of this warp
    uint32_t birth[32];             // outer iteration in which the lane took its ray (early split: only rays that HAVE walked are cut)
    int sParts, sAxis, sCut[kMaxWalkParts];   // plan of the split in progress
};

// Next list entry at or after k that this ray still has to test: entries whose face-mask bit is clear were in the cell the walk
// just left (already examined).  Lists longer than 32 entries are scanned in full beyond the mask.  (A variant with one bit
// per list entry -- no 32-entry limit -- measured 7 % slower on configs 2-3 and saved only 9 % of the tests on config 4, whose
// neighbouring cells share few triangles; it was dropped.)
__device__ __forceinline__ uint32_t next_entry(uint32_t begin, uint32_t end, uint32_t fm, uint32_t k) {
    const uint32_t rel = k - begin;
    if (rel < 32u) {
        const uint32_t mm = fm >> rel;
        k = mm ? k + (uint32_t)(__ffs((int)mm) - 1) : begin + 32u;
    }
    return k < end ? k : end;
}

// WALKGRID: the scene view is a walk grid (rt_types.h, SceneView::walkTrim != 0) and a step's exit test reads the axis' extent; without it
// the test is the reference grid's `cn >= n >> level`, so a scene that has no walk grid runs the instructions it ran before walk grids.
template <bool COUNT, bool SPLIT, bool HANDOFF = false, bool WALKGRID = false>
__global__ void __launch_bounds__(128, OCLR_TRACE_MIN_CTAS) wf_pipe_kernel(SceneView S, WfState w, WalkRecords rec, TraceTuning tune,
                                                                            Counters* gcnt, TailQueue tq) {
    extern __shared__ float shPlanes[];
    __shared__ WarpPipe pipes[4];
    __shared__ uint32_t classOff[kLengthClasses];   // first queue position of each length class (longest class first)
    if (blockIdx.x * 128u >= *w.queueCount) return;   // launched with the full persistent grid: the host does not know the count
    if (threadIdx.x == 0) {
        uint32_t acc = 0;
        for (int c = 0; c < kLengthClasses; ++c) {
            classOff[c] = acc;
            acc += rec.classCount[c];
        }
    }
    load_planes(shPlanes, S);   // (ends with __syncthreads)
    const int lane = threadIdx.x & 31;
    WarpPipe& P = pipes[threadIdx.x >> 5];
    const unsigned ltMask = (1u << lane) - 1u;
    const uint32_t count = *w.queueCount;
    const int n = S.n;
    const int nbShift = 31 - __clz(S.nb);
    const unsigned long long kEmptyKey = ~0ull;


    if (SPLIT) {
        P.grp[lane] = 0u;
        P.gParts[lane] = 0u;
        P.birth[lane] = 0u;
        if (lane == 0) P.groups = 0u;
        __syncwarp();
    }
    int splitWait = 0;   // warp-uniform: outer iterations until the next split attempt
    uint32_t iter = 0;   // warp-uniform: outer iterations so far
    const float* px = shPlanes;
    const float* py = shPlanes + (n + 1);
    const float* pz = shPlanes + 2 * (n + 1);

    Counters cnt = {};
    unsigned long long tWarpStart = 0, outerIters = 0;
    bool exhaustSeen = false;
    if (COUNT) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tWarpStart));
    PackedWalk g;
    g.level = 0;
    uint32_t path = 0;
    int ws = kWsNone;
    bool exhausted = false;
    int face = kFaceNone, lastAxis = 0;
    uint32_t sgn = 0;       // bit a: direction component a is >= 0 (the walk goes up along that axis)
    float lastE = 0.f;
    uint32_t seqNext = 0;   // cells this ray has in the current batch
    uint32_t cq = 0;        // warp-uniform: cells queued

    for (;;) {
        // ---- SPLIT: idle lanes take parts of the longest whole walk this warp holds (queue dry; or, early mode, a ray that has been
        //      walking for tune.splitEarly outer iterations already -- in FRONT of the refill, which takes what idle lanes are left) -----
        ++iter;
        if (SPLIT && tune.splitMin > 0 && (exhausted || tune.splitEarly > 0) && --splitWait < 0) {
            const unsigned idleNow = __ballot_sync(0xFFFFFFFFu, ws == kWsNone);
            int best = 0, who = lane;
            if (idleNow != 0u) {
                if (COUNT && lane == 0) cnt.splitAttempts++;
                // a whole ray (at either level of the walk) whose group record is free (a lane that headed a group before keeps that record until
                // the group has its result), old enough when the queue still has rays
                if (ws == kWsRun && g.coarseOk && P.grp[lane] == 0u && P.gParts[lane] == 0u &&
                    (exhausted || iter - P.birth[lane] >= (uint32_t)tune.splitEarly))
                {
#if OCLR_RAY_IN_SMEM
                    g.o = mk3(P.ray[0][lane], P.ray[1][lane], P.ray[2][lane]);   // (the estimate and the plan below read the ray from the walk state)
                    g.r = mk3(P.ray[3][lane], P.ray[4][lane], P.ray[5][lane]);
#endif
                    best = walk_length_estimate(g, n, WALKGRID ? S.walkTrim : 0u, px, py, pz);
                }
#pragma unroll
                for (int off = 16; off; off >>= 1) {
                    const int ob = __shfl_xor_sync(0xFFFFFFFFu, best, off), ow = __shfl_xor_sync(0xFFFFFFFFu, who, off);
                    if (ob > best || (ob == best && ow < who)) {
                        best = ob;
                        who = ow;
                    }
                }
            }
            if (best < tune.splitMin) {
                splitWait = 4;   // nothing worth cutting (or nobody to take a part): look again a few drains later
            } else {
                const int cand = who;
                if (lane == cand) {
                    int axis = 0, cut[kMaxWalkParts];
                    const int parts = pwalk_split_plan(g, n, px, py, pz, __popc(idleNow) + 1, tune.splitPart, axis, cut);
                    P.sParts = parts;
                    P.sAxis = axis;
#pragma unroll
                    for (int j = 0; j < kMaxWalkParts; ++j) P.sCut[j] = cut[j];
                    if (parts >= 2) {
                        P.gHit[cand] = 0u;
                        P.gMiss[cand] = 0u;
                        P.gParts[cand] = (uint32_t)parts;
                        P.groups += 1u;
                        if (COUNT) {
                            cnt.splitsDone++;
                            cnt.splitParts += (unsigned long long)parts;
                        }
                    }
                }
                __syncwarp();
                const int parts = P.sParts;
                if (parts >= 2) {
                    const int axis = P.sAxis;
                    int cut[kMaxWalkParts];
#pragma unroll
                    for (int j = 0; j < kMaxWalkParts; ++j) cut[j] = P.sCut[j];
                    PackedWalk head;   // what pwalk_split_part needs of the interrupted walk
                    head.o = mk3(P.ray[0][cand], P.ray[1][cand], P.ray[2][cand]);
                    head.r = mk3(P.ray[3][cand], P.ray[4][cand], P.ray[5][cand]);
                    head.cpk = __shfl_sync(0xFFFFFFFFu, g.cpk, cand);
                    head.level = __shfl_sync(0xFFFFFFFFu, g.level, cand);
                    head.epk = __shfl_sync(0xFFFFFFFFu, g.epk, cand);
                    head.endBrick = __shfl_sync(0xFFFFFFFFu, g.endBrick, cand);
                    const uint32_t headPath = __shfl_sync(0xFFFFFFFFu, path, cand);
                    const int myPart = __popc(idleNow & ltMask) + 1;
                    if (ws == kWsNone && myPart < parts) {
                        PackedWalk part;
                        if (pwalk_split_part(part, head, n, S.nb, px, py, pz, axis, cut, parts, myPart)) {
                            g = part;
                            pwalk_load_brick(g, S.bricks);
                            const float minD = P.ray[6][cand];
                            const float maxD = P.ray[7][cand];
                            P.ray[0][lane] = head.o.x;
                            P.ray[1][lane] = head.o.y;
                            P.ray[2][lane] = head.o.z;
                            P.ray[3][lane] = head.r.x;
                            P.ray[4][lane] = head.r.y;
                            P.ray[5][lane] = head.r.z;
                            P.ray[6][lane] = minD;
                            P.ray[7][lane] = maxD;
                            P.excl[lane] = P.excl[cand];
                            P.bestKey[lane] = kEmptyKey;
                            P.grp[lane] = 0x80000000u | (uint32_t)cand | ((uint32_t)myPart << 8);
                            sgn = (0 <= head.r.x ? 1u : 0u) | (0 <= head.r.y ? 2u : 0u) | (0 <= head.r.z ? 4u : 0u);
                            path = headPath;
                            ws = kWsRun;
                            face = kFaceNone;
                            seqNext = 0;
                            if (COUNT) cnt.bricksLoaded++;
                        } else {
                            atomicOr(&P.gMiss[cand], 1u << myPart);   // the walk leaves the grid before this part begins
                        }
                    }
                    if (lane == cand) {
                        pwalk_split_head(g, axis, cut);
                        P.grp[lane] = 0x80000000u | (uint32_t)cand;
                    }
                    __syncwarp();
                } else {
                    splitWait = 4;
                }
            }
        }

        if (HANDOFF && !exhausted) {
            // a warp learns that the queue is dry when it asks for more -- and a warp whose 32 rays are all long (the queue is sorted
            // longest first) does not ask for a long time.  Small launches look: one read of the cursor per outer iteration
            uint32_t cur = 0;
            if (lane == 0) cur = *(volatile uint32_t*)w.queueCursor;
            exhausted = __shfl_sync(0xFFFFFFFFu, cur, 0) >= count;
        }
        // ---- refill idle lanes: one atomic per warp, records read in queue order ----
        const unsigned idle = __ballot_sync(0xFFFFFFFFu, ws == kWsNone);
        if (idle != 0u && !exhausted && (idle == 0xFFFFFFFFu || __popc(idle) >= tune.refillMin)) {
            const int nIdle = __popc(idle);
            const int leader = __ffs(idle) - 1;
            uint32_t base = 0;
            if (lane == leader) base = atomicAdd(w.queueCursor, (uint32_t)nIdle);
            base = __shfl_sync(0xFFFFFFFFu, base, leader);
            if (base + (uint32_t)nIdle >= count) exhausted = true;
            if (ws == kWsNone) {
                const uint32_t pos = base + (uint32_t)__popc(idle & ltMask);
                if (pos < count) {
                    uint32_t cls = 0;
#pragma unroll
                    for (int c = 1; c < kLengthClasses; ++c) cls += pos >= classOff[c];
                    const uint32_t idx = rec.order[(size_t)cls * rec.Q + (pos - classOff[cls])];
                    const float4 ro = rec.o[idx], rd = rec.d[idx], s0 = rec.s0[idx];
                    const uint4 s1 = rec.s1[idx];
#if OCLR_RAY_IN_SMEM
                    sgn = (0 <= rd.x ? 1u : 0u) | (0 <= rd.y ? 2u : 0u) | (0 <= rd.z ? 4u : 0u);
#else
                    g.o = mk3(ro.x, ro.y, ro.z);
                    g.r = mk3(rd.x, rd.y, rd.z);
#endif
                    P.ray[0][lane] = ro.x;
                    P.ray[1][lane] = ro.y;
                    P.ray[2][lane] = ro.z;
                    P.ray[3][lane] = rd.x;
                    P.ray[4][lane] = rd.y;
                    P.ray[5][lane] = rd.z;
                    P.ray[6][lane] = ro.w;
                    P.ray[7][lane] = rd.w;
                    P.excl[lane] = s1.y;
                    P.bestKey[lane] = kEmptyKey;
                    g.tx = s0.x;
                    g.ty = s0.y;
                    g.tz = s0.z;
                    g.cpk = __float_as_uint(s0.w);
                    g.epk = s1.x;
                    path = s1.z;
                    g.coarseOk = s1.w != 0u;
                    g.level = 0;
                    g.brick = ((pk_get(g.cpk, 0) >> 2) + (((pk_get(g.cpk, 1) >> 2) + ((pk_get(g.cpk, 2) >> 2) << nbShift)) << nbShift));
                    g.endBrick = pwalk_end_key(g.epk, nbShift);   // (the hot loop below reads this word, never the end cell itself)
                    pwalk_load_brick(g, S.bricks);
                    ws = kWsRun;
                    face = kFaceNone;
                    seqNext = 0;
                    if (SPLIT || HANDOFF) P.birth[lane] = iter;
                    if (COUNT) {
                        cnt.gridRays++;
                        cnt.bricksLoaded++;
                    }
                }
            }
        }
        if (__ballot_sync(0xFFFFFFFFu, ws != kWsNone) == 0u) break;
        __syncwarp();
        if (COUNT) {
            ++outerIters;
            if (exhausted && !exhaustSeen && lane == 0) {   // when this warp learnt that the queue is dry
                unsigned long long t;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
                const unsigned long long b = (t - tWarpStart) >> 15;
                atomicAdd(&gcnt->exhaustHist00 + (b < 15 ? b : 15), 1ull);
            }
            exhaustSeen = exhausted;
        }

        // ---- WALK burst: step every walking lane until the cell queue is worth draining or too few lanes still walk ----------------
        int burstIters = 0;   // (HANDOFF only)
        for (;;) {
            const bool walking = ws == kWsRun;
            if (COUNT) {
                if (lane == 0) cnt.walkWarpIters++;
                if (walking) cnt.walkLaneIters++;
                if (ws == kWsNone) cnt.walkIdleLanes++;
                if ((ws == kWsRefine) | (ws == kWsEnter)) cnt.walkParkedLanes++;
                if (ws == kWsFinished) cnt.walkFinishedLanes++;
                if (lane == 0 && exhausted) cnt.walkExhaustedIters++;
            }
            if (COUNT) {
                const int nw = __popc(__ballot_sync(0xFFFFFFFFu, walking));
                if (lane == 0 && nw <= 8) cnt.walkLowIters++;
            }
            bool occupied = false;
            int bit = 0;
            if (walking) {
                bit = pwalk_bit(g.cpk);
                occupied = (g.level == 0) & pwalk_occupied(g, bit);
            }
            const unsigned occ = __ballot_sync(0xFFFFFFFFu, occupied);
            if (occupied) {
                const uint32_t pos = cq + (uint32_t)__popc(occ & ltMask);
                P.cellQ[0][pos] = pwalk_rank(g, bit) | ((uint32_t)face << 29);
                P.cellQ[1][pos] = (uint32_t)lane | (seqNext << 8);
                ++seqNext;
                if (COUNT) cnt.cellsNonEmpty++;
            }
            cq += (uint32_t)__popc(occ);
            if (walking) {
                const bool coarse = g.level != 0;
                const bool brickEmpty = (g.maskLo | g.maskHi) == 0u;
                const bool inEnd = pwalk_in_end(g);   // (level 2: both are super-brick records, rt_walk.h)
                if (COUNT && !coarse) {
                    cnt.cells++;
                    if (brickEmpty) cnt.emptyBrickCells++;
                }
#if OCLR_END_KEY
                const bool atEnd = (!coarse) & pwalk_at_end(g, bit);
#else
                const bool atEnd = (!coarse) & (g.cpk == g.epk);   // (A/B build: the end cell stays live through the loop -- and is spilled)
#endif
                const bool needRefine = coarse & ((!brickEmpty) | inEnd);
                // one level up: from the cells of an empty brick; from brick level when the record of the empty brick says that its whole
                // super-brick is empty (bit 0 of what is the rank base of other bricks; super-brick records never carry it)
                const bool up2 = OCLR_SUPER_LEVEL && ((g.rankBase & 1u) != 0u) & (tune.hierarchical >= 2) & !(SPLIT && pk_is_stop(g.epk));
                const bool needEnter = brickEmpty & g.coarseOk & (!inEnd) & (tune.hierarchical != 0) & ((!coarse) | up2);
                if (atEnd) {
                    ws = kWsFinished;
                } else if (needRefine | needEnter) {
                    ws = needRefine ? kWsRefine : kWsEnter;
                } else {
                    int up;
                    bool crossed;
                    if (COUNT && coarse) cnt.coarseSteps++;
                    if (COUNT && g.level == 2) cnt.superSteps++;
#if OCLR_RAY_IN_SMEM
                    lastAxis = pwalk_step_axis(g, lastE);
                    up = (int)((sgn >> lastAxis) & 1u);
                    const bool inside = pwalk_step_along(g, n, WALKGRID ? S.walkTrim : 0u, nbShift, shPlanes, lastAxis, P.ray[lastAxis][lane], P.ray[3 + lastAxis][lane], up, crossed);
#else
                    const bool inside = pwalk_step(g, n, WALKGRID ? S.walkTrim : 0u, nbShift, shPlanes, lastAxis, up, lastE, crossed);
#endif
                    if (!inside) {
                        ws = kWsFinished;
                    } else if (SPLIT && pk_is_stop(g.epk) && pwalk_stopped(g, lastAxis, up)) {
                        ws = kWsFinished;   // this part of a cut walk ends here; the cell just entered belongs to the next part
                    } else {
                        face = coarse ? (int)kFaceNone : lastAxis * 2 + up;
                        if (crossed) {
                            pwalk_load_brick(g, S.bricks);
                            if (COUNT) cnt.bricksLoaded++;
                        }
                    }
                }
                if ((ws == kWsFinished) & (seqNext == 0u)) {  // walk over and nothing of this ray awaits a test: miss
                    if (!SPLIT || P.grp[lane] == 0u) {        // (a part of a cut walk reports to its group in RESOLVE instead)
                        w.hit[path] = make_float4(__uint_as_float(kNoTriangle), P.ray[7][lane], 0.f, 0.f);
                        ws = kWsNone;
                    }
                }
            }
            const int nSwitch = __popc(__ballot_sync(0xFFFFFFFFu, (ws == kWsRefine) | (ws == kWsEnter)));
            const int nWalk = __popc(__ballot_sync(0xFFFFFFFFu, ws == kWsRun));
            if (cq >= (uint32_t)tune.drainMin) break;   // (checked before anything that loops back: the queue holds drainMin + 31 cells)
            if (HANDOFF && exhausted && ++burstIters >= tune.handoffBurst) break;
            // Tail of the launch (queue dry, a few long rays left): the launch cannot end before its longest walk does, so what
            // counts now is that ray's latency.  Draining after every step would put a full open + test round trip between two
            // steps; let a few cells accumulate instead (they are opened and tested side by side in one drain).
            const bool tail = exhausted & (nWalk != 0) & (cq < (uint32_t)tune.tailDrain);
            if (nSwitch != 0 && (nSwitch >= tune.switchMin || nWalk < tune.walkMin3)) {
                // ---- SWITCH: parked level switches of the two-level walk, run together
                if (COUNT) {
                    if (lane == 0) cnt.switchWarpIters++;
                    if ((ws == kWsRefine) | (ws == kWsEnter)) cnt.switchLaneIters++;
                }
#if OCLR_RAY_IN_SMEM
                if ((ws == kWsEnter) | (ws == kWsRefine)) {   // the level switches divide along all three axes
                    g.o = mk3(P.ray[0][lane], P.ray[1][lane], P.ray[2][lane]);
                    g.r = mk3(P.ray[3][lane], P.ray[4][lane], P.ray[5][lane]);
                }
#endif
                if (ws == kWsEnter) {
                    if (g.level == 0) {
                        pwalk_enter_coarse(g, n, nbShift, shPlanes);
                        if (COUNT) cnt.coarseEnters++;
                    }
                    if (OCLR_SUPER_LEVEL && tune.hierarchical >= 2 && (g.rankBase & 1u) != 0u) {   // (straight on to level 2 when the flag says so)
                        if (pwalk_super_allowed(g)) {
                            pwalk_enter_coarse(g, n, nbShift, shPlanes);
                            if (COUNT) cnt.superEnters++;
                        } else {
                            g.rankBase = 0u;   // the end cell's super-brick: brick by brick (the next brick's record asks again)
                        }
                    }
                    ws = kWsRun;
                } else if (ws == kWsRefine) {
                    pwalk_refine(g, n, nbShift, shPlanes, lastAxis, lastE);
                    if (OCLR_SUPER_LEVEL && g.level == 1) {   // back from the super-brick level: the brick the walk stands in is new to it
                        pwalk_load_brick(g, S.bricks);
                        if (COUNT) {
                            cnt.bricksLoaded++;
                            cnt.superRefines++;
                        }
                    }
                    face = kFaceNone;
                    ws = kWsRun;
                }
                continue;
            }
            if (nWalk < tune.walkMin3 && !tail) break;
        }

        // ---- DRAIN: open every queued cell, test every pair, any lane for any ray ---------------------------------------------------
        if (cq != 0u) {
            __syncwarp();
            uint32_t pqHead = 0, pqTail = 0;   // absolute pair indices of this drain (warp-uniform)
            // TEST round: lanes [0, take) each take one (ray, triangle) pair
            auto test_round = [&](uint32_t take) {
                __syncwarp();
                bool hit = false;
                unsigned long long key = kEmptyKey;
                uint32_t owner = 0, ptri = 0;
                float ab = 0.f, ac = 0.f;
                if (COUNT) {
                    if (lane == 0) cnt.testWarpIters++;
                    if ((uint32_t)lane < take) {
                        cnt.testLaneIters++;
                        cnt.gridCandidates++;
                    }
                }
                if ((uint32_t)lane < take) {
                    const uint32_t pidx = pqHead + (uint32_t)lane;
                    ptri = P.pairQ[0][pidx & (kPairQCap - 1)];
                    const uint32_t os = P.pairQ[1][pidx & (kPairQCap - 1)];
                    owner = os & 31u;
                    const f3 o = mk3(P.ray[0][owner], P.ray[1][owner], P.ray[2][owner]);
                    const f3 r = mk3(P.ray[3][owner], P.ray[4][owner], P.ray[5][owner]);
                    float t;
                    hit = tri_test(S.triGeo + 4 * (size_t)ptri, o, r, P.ray[6][owner], P.ray[7][owner], t, ab, ac);
                    if (hit) {
                        key = ((unsigned long long)(os >> 8) << 56) | ((unsigned long long)__float_as_uint(t) << 24) |
                              (unsigned long long)(pidx & 0xFFFFFFu);
                        atomicMin(&P.bestKey[owner], key);
                    }
                }
                __syncwarp();
                if (hit && P.bestKey[owner] == key) {
                    P.bestTri[owner] = ptri;
                    P.bestAB[owner] = ab;
                    P.bestAC[owner] = ac;
                }
                pqHead += take;
            };
            for (uint32_t base = 0; base < cq; base += 32u) {
                uint32_t k = 0, kEnd = 0, kBegin = 0, fm = 0, ownerSeq = 0, excl = kNoTriangle;
                if (base + (uint32_t)lane < cq) {  // OPEN one cell per lane
                    const uint32_t e = P.cellQ[0][base + lane];
                    ownerSeq = P.cellQ[1][base + lane];
                    const uint32_t rank = e & 0x1FFFFFFFu, f = e >> 29;
                    const uint2 range = __ldg(S.cellRange + rank);
                    // entries shared with the cell the walk came from were examined there (exact, rt_types.h faceMask)
                    fm = f != (uint32_t)kFaceNone ? __ldg(S.faceMask + 6 * (size_t)rank + f) : 0xFFFFFFFFu;
                    excl = P.excl[ownerSeq & 31u];
                    kBegin = range.x;
                    kEnd = range.y;
                    k = next_entry(kBegin, kEnd, fm, kBegin);
                }
                // enumerate the untested entries, one per lane per round, into the pair queue (list order per cell)
                while (__any_sync(0xFFFFFFFFu, k < kEnd)) {
                    const bool more = k < kEnd;
                    uint32_t tri = 0;
                    if (more) tri = __ldg(S.cellList + k);
                    const bool valid = more & (tri != excl);
                    const unsigned vb = __ballot_sync(0xFFFFFFFFu, valid);
                    if (valid) {
                        const uint32_t pos = (pqTail + (uint32_t)__popc(vb & ltMask)) & (kPairQCap - 1);
                        P.pairQ[0][pos] = tri;
                        P.pairQ[1][pos] = ownerSeq;
                    }
                    pqTail += (uint32_t)__popc(vb);
                    if (more) k = next_entry(kBegin, kEnd, fm, k + 1u);
                    if (pqTail - pqHead >= 32u) test_round(32u);
                }
            }
            while (pqTail != pqHead) test_round(pqTail - pqHead < 32u ? pqTail - pqHead : 32u);
            __syncwarp();
            cq = 0;
        }

        // ---- RESOLVE ----------------------------------------------------------------------------------------------------------------
        if (!SPLIT || P.groups == 0u) {   // (warp-uniform; the only case outside the tail of a launch)
            if (ws != kWsNone) {
                const unsigned long long key = P.bestKey[lane];
                if (key != kEmptyKey) {  // first cell with any hit wins (:380); whatever the walker found beyond it is dropped
                    w.hit[path] = make_float4(__uint_as_float(P.bestTri[lane]), __uint_as_float((uint32_t)(key >> 24)), P.bestAB[lane], P.bestAC[lane]);
                    ws = kWsNone;
                } else if (ws == kWsFinished) {
                    w.hit[path] = make_float4(__uint_as_float(kNoTriangle), P.ray[7][lane], 0.f, 0.f);
                    ws = kWsNone;
                }
                seqNext = 0;
            }
        } else {
            // some walks of this warp are cut into parts: a part reports to its group, the group decides
            const uint32_t grp = ws != kWsNone ? P.grp[lane] : 0u;
            const uint32_t headLane = grp & 31u, order = (grp >> 8) & 15u;
            const unsigned long long key = P.bestKey[lane];
            if (ws != kWsNone) {
                if (grp == 0u) {   // a whole ray: as above
                    if (key != kEmptyKey) {
                        w.hit[path] = make_float4(__uint_as_float(P.bestTri[lane]), __uint_as_float((uint32_t)(key >> 24)), P.bestAB[lane], P.bestAC[lane]);
                        ws = kWsNone;
                    } else if (ws == kWsFinished) {
                        w.hit[path] = make_float4(__uint_as_float(kNoTriangle), P.ray[7][lane], 0.f, 0.f);
                        ws = kWsNone;
                    }
                } else if (ws != kWsHeld) {
                    if (key != kEmptyKey) {   // this part's first cell with a hit: held until every part before it has finished
                        atomicOr(&P.gHit[headLane], 1u << order);
                        ws = kWsHeld;
                    } else if (ws == kWsFinished) {
                        atomicOr(&P.gMiss[headLane], 1u << order);
                        ws = kWsPartDone;
                    }
                }
                seqNext = 0;
            }
            __syncwarp();
            bool closes = false;   // this lane wrote its group's result
            if (grp != 0u) {
                const uint32_t hm = P.gHit[headLane], mm = P.gMiss[headLane];
                const uint32_t firstHit = hm ? (uint32_t)(__ffs((int)hm) - 1) : 32u;
                const uint32_t below = (1u << order) - 1u;
                if (order > firstHit) {   // a part before this one has a hit: nothing found here can matter
                    ws = kWsNone;
                    P.grp[lane] = 0u;
                    if (COUNT) cnt.splitCancelled++;
                } else if (ws == kWsHeld) {
                    if ((mm & below) == below) {   // every part before it finished without a hit: this is the ray's result
                        w.hit[path] = make_float4(__uint_as_float(P.bestTri[lane]), __uint_as_float((uint32_t)(key >> 24)), P.bestAB[lane], P.bestAC[lane]);
                        ws = kWsNone;
                        P.grp[lane] = 0u;
                        atomicSub(&P.groups, 1u);
                        closes = true;
                    }
                } else if (ws == kWsPartDone) {   // (its miss is on the group's record: the lane is free again)
                    const uint32_t all = (1u << P.gParts[headLane]) - 1u;
                    if (hm == 0u && (mm & all) == all && (atomicOr(&P.gMiss[headLane], 0x80000000u) >> 31) == 0u) {
                        w.hit[path] = make_float4(__uint_as_float(kNoTriangle), P.ray[7][lane], 0.f, 0.f);   // the last parts to finish: one of them says so
                        atomicSub(&P.groups, 1u);
                        closes = true;
                    }
                    ws = kWsNone;
                    P.grp[lane] = 0u;
                }
            }
            __syncwarp();
            if (closes) P.gParts[headLane] = 0u;   // the head lane's group record is free again
            __syncwarp();
        }

        // ---- HANDOFF (small launches only): the queue has been dry for a while and what this warp still walks is the launch's tail ---
        if (HANDOFF && exhausted && __popc(__ballot_sync(0xFFFFFFFFu, ws != kWsNone)) <= tune.handoffLanes) {
            // a lane walking at cell level with nothing pending (cells drained, keys resolved just above) gives its ray up, to go on
            // from the cell it stands in: mode 1 in wf_tail_kernel, one warp to the ray; mode 2 in a second pass of this kernel over
            // the rays given up, which fills its warps densely again (rt_tail.cuh)
            // ... and that has been with this warp for handoffAfter outer iterations (~12 cells each) already: a LONG walk, which is what
            // a launch with the queue dry is waiting for -- the many medium ones finish where they are
            // (mode 1, the brick-plane burst walker, also takes a ray that is crossing an empty brick at brick level -- the long walks
            // through empty space spend most of their time there; mode 3 = the cell-plane burst walker)
            const bool atCells = g.level == 0;
            const bool inEmptyBrick = (tune.handoffMode == 1) & (g.level == 1) & ((g.maskLo | g.maskHi) == 0u) & !pwalk_in_end(g);
            const bool give = (ws == kWsRun) & (atCells | inEmptyBrick) & (tune.handoffMode == 2 || g.coarseOk) & (!SPLIT || P.grp[lane] == 0u) &
                              (iter - P.birth[lane] >= (uint32_t)tune.handoffAfter);
            const unsigned gm = __ballot_sync(0xFFFFFFFFu, give);
            if (gm != 0u) {
                const int leader = __ffs(gm) - 1;
                uint32_t base = 0;
                if (lane == leader) base = atomicAdd(tq.count, (uint32_t)__popc(gm));
                base = __shfl_sync(0xFFFFFFFFu, base, leader);
                if (give) {
                    const uint32_t pos = base + (uint32_t)__popc(gm & ltMask);
                    if (pos < tq.capacity) {   // (a full list: the lane keeps its ray)
                        if (tune.handoffMode == 2) {   // a walk record like the setup kernel's: the state of a walk at cell level IS (cell, crossings)
                            tq.o[pos] = make_float4(P.ray[0][lane], P.ray[1][lane], P.ray[2][lane], P.ray[6][lane]);
                            tq.d[pos] = make_float4(P.ray[3][lane], P.ray[4][lane], P.ray[5][lane], P.ray[7][lane]);
                            tq.s0[pos] = make_float4(g.tx, g.ty, g.tz, __uint_as_float(g.cpk));
                            tq.s1[pos] = make_uint4(g.epk, P.excl[lane], path, g.coarseOk ? 1u : 0u);
                            tq.order[pos] = pos;
                        } else {
                            tq.entries[pos] = make_uint4(path, g.cpk, (uint32_t)face, (uint32_t)g.level);
                        }
                        ws = kWsNone;
                    }
                }
            }
        }
    }
    if (COUNT) {
        flush_counters(cnt, gcnt);
        if (lane == 0) {   // when this warp left (32.768-us buckets since its start; all CTAs of the persistent grid start together)
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            const unsigned long long b = (t - tWarpStart) >> 15;
            atomicAdd(&gcnt->exitHist00 + (b < 15 ? b : 15), 1ull);
            atomicMax(&gcnt->warpOuterItersMax, outerIters);
            atomicAdd(&gcnt->warpOuterItersSum, outerIters);
            atomicAdd(&gcnt->warpsRun, 1ull);
        }
    }
}

}  // namespace oclr
