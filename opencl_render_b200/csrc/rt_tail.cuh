// rt_tail.cuh -- the tail of a small trace launch: ONE ray per warp, walked by cooperative bursts.
//
// A trace launch cannot end before its longest walk does.  On a whole 1080p frame that tail is 6 % of the walk iterations; on the 1/8
// share an 8-GPU run gives each GPU it is 38 %, and the launch takes 0.38 ms where its throughput bound is 0.11 ms -- the floor that
// holds strong scaling of small frames at 0.5 (DESIGN.md section 5).  The rays in that tail are few and long (a ray skimming the floor
// quad crosses several hundred occupied cells), and a lane walks them one dependent step at a time, ~1 000 cycles per cell.
//
// wf_pipe_kernel<., ., HANDOFF = true> (chosen by the host for SMALL launch domains only: the whole-frame kernel stays as it is) gives
// such rays up: a warp that has spent a few outer iterations with the queue dry writes {ray, current cell, entry face} of every lane
// that is walking at cell level with nothing pending into a hand-off list and is done with them.  This kernel picks them up, a warp
// per ray.  One burst = 32 lanes take the next 11 / 11 / 10 plane crossings of the x / y / z axis (one division each); the merge
// order of the reference's walk (:387-398) gives every crossing its position directly (rt_walk.h, coop_burst_serial: the host form the
// tests compare with the reference's cell walk), so ~25 cells are classified per burst with no serial dependency; their bricks are
// looked up side by side, the occupied ones are opened and their (ray, triangle) pairs tested 32 at a time exactly as in the pipe
// kernel's drain -- key = position of the cell in the walk | t | pair index, smallest key wins = the reference's first-cell-wins rule.
// A 600-cell walk is ~25 bursts of a few hundred instructions instead of 600 dependent steps.
//
// Result (round 2, sessions n / o): bit-exact on every golden case with the hand-off forced as early as possible -- and not faster.  ncu
// on a 1/8 share of config 2: the two ray-carrying pipe launches take 0.49 + 0.26 ms for 305 M + 102 M warp instructions (68 % / 43 %
// of the whole-frame issue rate); handing rays off 4 outer iterations after the queue runs dry shortens them to 0.43-0.47 + 0.22 ms
// and adds 0.05 + 0.075 ms of tail kernel (5 M + 21 M warp instructions): what a small launch loses is the decaying lane fill of
// EVERY warp's last batch, thousands of medium rays, not a handful of very long ones.  And where only the longest walks are left -- a
// 17-row share still needs 0.31 + 0.23 ms for its two trace launches -- giving up rays by their AGE is no faster either (0.556 -> 0.59 ms):
// those rays cross mostly empty space, which the lane's two-level walk takes four cells at a step, while a burst works at cell
// granularity.  The next step would be the burst over BRICK planes.  Off by default (OCLR_HANDOFF_MAX_PATHS = 0);
// tests/test_gpu_progressive.py::test_tail_handoff_is_invisible keeps it exact.
#pragma once
#include "rt_trace.cuh"

namespace oclr {

struct TailWarp {
    float t[3][11];                  // crossing values of the burst's candidates
    uint32_t slotCell[32];           // cells of the burst in walk order
    uint32_t slotFace[32];
    uint32_t pairTri[kPairQCap], pairSeq[kPairQCap];
    unsigned long long bestKey;
    uint32_t bestTri;
    float bestAB, bestAC;
};

__global__ void __launch_bounds__(128) wf_tail_kernel(SceneView S, WfState w, TailQueue tq) {
    extern __shared__ float shPlanes[];
    __shared__ TailWarp warps[4];
    const uint32_t total = min(*tq.count, tq.capacity);
    if (total == 0u) return;   // (the usual case on a whole frame: nothing was handed off)
    load_planes(shPlanes, S);
    const int lane = threadIdx.x & 31;
    TailWarp& T = warps[threadIdx.x >> 5];
    const unsigned ltMask = (1u << lane) - 1u;
    const int n = S.n, nb = S.nb;
    const float* px = shPlanes;
    const float* py = shPlanes + (n + 1);
    const float* pz = shPlanes + 2 * (n + 1);
    const unsigned long long kEmptyKey = ~0ull;

    for (;;) {
        uint32_t idx = 0;
        if (lane == 0) idx = atomicAdd(tq.cursor, 1u);
        idx = __shfl_sync(0xFFFFFFFFu, idx, 0);
        if (idx >= total) break;
        const uint4 e = tq.entries[idx];
        const uint32_t path = e.x;
        const float4 ro = w.rayO[path], rd = w.rayD[path];
        const uint32_t excl = w.rayExcl[path];
        const f3 o = mk3(ro.x, ro.y, ro.z), r = mk3(rd.x, rd.y, rd.z);
        const float minD = ro.w, maxD = rd.w;
        CoopRay ray;
        ray.o = o;
        ray.r = r;
        {   // the end cell, as wf_setup_kernel computed it (raytrace_opencl.c:357-361)
            PackedWalk s;
            pwalk_setup(s, n, nb, S.walkTrim, px, py, pz, o, r, minD, maxD);
            ray.epk = s.epk;
        }
        ray.c0[0] = pk_get(e.y, 0);
        ray.c0[1] = pk_get(e.y, 1);
        ray.c0[2] = pk_get(e.y, 2);
        if (lane == 0) {
            T.bestKey = kEmptyKey;
            T.slotCell[0] = e.y;
            T.slotFace[0] = e.z;
        }
        __syncwarp();

        // opens the cells in slots [0, count) -- walk order -- and tests their untested list entries against the ray
        auto process_cells = [&](uint32_t count) {
            uint32_t k = 0, kEnd = 0, kBegin = 0, fm = 0;
            if ((uint32_t)lane < count) {
                const uint32_t cell = T.slotCell[lane], face = T.slotFace[lane];
                const int cx = pk_get(cell, 0), cy = pk_get(cell, 1), cz = pk_get(cell, 2);
                const uint4 br = __ldg(S.bricks + ((cx >> 2) + nb * ((cy >> 2) + nb * (cz >> 2))));
                const int bit = pwalk_bit(cell);
                const uint64_t mask = (uint64_t)br.x | ((uint64_t)br.y << 32);
                if ((mask >> bit) & 1ull) {
                    const uint32_t rank = br.z + (uint32_t)__popcll(mask & ((1ull << bit) - 1ull));
                    const uint2 range = __ldg(S.cellRange + rank);
                    fm = face != (uint32_t)kFaceNone ? __ldg(S.faceMask + 6 * (size_t)rank + face) : 0xFFFFFFFFu;
                    kBegin = range.x;
                    kEnd = range.y;
                    k = next_entry(kBegin, kEnd, fm, kBegin);
                }
            }
            uint32_t pqHead = 0, pqTail = 0;
            auto test_round = [&](uint32_t take) {
                __syncwarp();
                bool hit = false;
                unsigned long long key = kEmptyKey;
                uint32_t tri = 0;
                float ab = 0.f, ac = 0.f;
                if ((uint32_t)lane < take) {
                    const uint32_t pidx = pqHead + (uint32_t)lane;
                    tri = T.pairTri[pidx & (kPairQCap - 1)];
                    const uint32_t seq = T.pairSeq[pidx & (kPairQCap - 1)];
                    float t;
                    hit = tri_test(S.triGeo + 4 * (size_t)tri, o, r, minD, maxD, t, ab, ac);
                    if (hit) {
                        key = ((unsigned long long)seq << 56) | ((unsigned long long)__float_as_uint(t) << 24) | (unsigned long long)(pidx & 0xFFFFFFu);
                        atomicMin(&T.bestKey, key);
                    }
                }
                __syncwarp();
                if (hit && T.bestKey == key) {
                    T.bestTri = tri;
                    T.bestAB = ab;
                    T.bestAC = ac;
                }
                pqHead += take;
            };
            while (__any_sync(0xFFFFFFFFu, k < kEnd)) {
                const bool more = k < kEnd;
                uint32_t tri = 0;
                if (more) tri = __ldg(S.cellList + k);
                const bool valid = more & (tri != excl);
                const unsigned vb = __ballot_sync(0xFFFFFFFFu, valid);
                if (valid) {
                    const uint32_t pos = (pqTail + (uint32_t)__popc(vb & ltMask)) & (kPairQCap - 1);
                    T.pairTri[pos] = tri;
                    T.pairSeq[pos] = (uint32_t)lane;   // position of the cell in the walk: the first cell with a hit wins (:380)
                }
                pqTail += (uint32_t)__popc(vb);
                if (more) k = next_entry(kBegin, kEnd, fm, k + 1u);
                if (pqTail - pqHead >= 32u) test_round(32u);
            }
            while (pqTail != pqHead) test_round(pqTail - pqHead < 32u ? pqTail - pqHead : 32u);
            __syncwarp();
        };
        auto finish = [&](bool hit) {
            if (lane == 0) {
                const unsigned long long key = T.bestKey;
                w.hit[path] = hit ? make_float4(__uint_as_float(T.bestTri), __uint_as_float((uint32_t)(key >> 24)), T.bestAB, T.bestAC)
                                  : make_float4(__uint_as_float(kNoTriangle), maxD, 0.f, 0.f);
            }
            __syncwarp();
        };

        // the cell the lane stood in when it gave the ray up has not been examined yet
        process_cells(1u);
        if (T.bestKey != kEmptyKey) {
            finish(true);
            continue;
        }
        if (e.y == ray.epk) {
            finish(false);
            continue;
        }
        for (;;) {
            // ---- one burst (rt_walk.h coop_burst_serial, one virtual lane per real lane) ------------------------------------------
            const int a = lane % 3, kc = lane / 3;
            int kmaxA;
            const float tv = coop_crossing(ray, n, shPlanes, a, kc, kmaxA);
            __syncwarp();
            T.t[a][kc] = tv;
            __syncwarp();
            int cnt[3];
            int rank = kc;
#pragma unroll
            for (int b = 0; b < 3; ++b) {
                if (b == a) {
                    cnt[b] = kc + 1;
                    continue;
                }
                int c = 0;
                for (int kk = 0; kk < coop_candidates(b); ++kk) c += coop_precedes(b, T.t[b][kk], a, tv) ? 1 : 0;
                cnt[b] = c;
                rank += c;
            }
            const bool present = kc <= kmaxA;
            const int kBig = 1 << 20;
            // crossings with rank < R are certain: no crossing beyond the candidates can precede them
            const int R = __reduce_min_sync(0xFFFFFFFFu, (kc == coop_candidates(a) - 1 && kmaxA >= coop_candidates(a)) ? rank + 1 : kCoopLanes);
            const int exitRank = __reduce_min_sync(0xFFFFFFFFu, (present && kc == kmaxA) ? rank : kBig);
            const float rx = ray.r.x, ry = ray.r.y, rz = ray.r.z;
            const int cx = ray.c0[0] + ((0 <= rx) ? cnt[0] : -cnt[0]);
            const int cy = ray.c0[1] + ((0 <= ry) ? cnt[1] : -cnt[1]);
            const int cz = ray.c0[2] + ((0 <= rz) ? cnt[2] : -cnt[2]);
            const uint32_t cellV = (present && kc < kmaxA) ? pk_make(cx & kPkMask, cy & kPkMask, cz & kPkMask) : (uint32_t)kPkNone;
            const int endRank = __reduce_min_sync(0xFFFFFFFFu, (cellV != (uint32_t)kPkNone && cellV == ray.epk) ? rank : kBig);
            int limit = R;
            bool finished = false;
            if (exitRank < limit) {   // the crossing that leaves the grid enters no cell
                limit = exitRank;
                finished = true;
            }
            if (endRank < limit) {   // the end cell is visited, then the walk stops (:381)
                limit = endRank + 1;
                finished = true;
            }
            if (rank < limit) {
                const float ra = a == 0 ? rx : (a == 1 ? ry : rz);
                T.slotCell[rank] = cellV;
                T.slotFace[rank] = (uint32_t)(a * 2 + ((0 <= ra) ? 1 : 0));
            }
            __syncwarp();
            if (limit > 0) {
                process_cells((uint32_t)limit);
                const uint32_t last = T.slotCell[limit - 1];
                ray.c0[0] = pk_get(last, 0);
                ray.c0[1] = pk_get(last, 1);
                ray.c0[2] = pk_get(last, 2);
            }
            if (T.bestKey != kEmptyKey) {
                finish(true);
                break;
            }
            if (finished) {
                finish(false);
                break;
            }
        }
    }
}

// ---- the same, one level up: bursts over BRICK planes ------------------------------------------------------------------------------
// The rays a small launch waits for cross mostly empty space, which a lane's two-level walk takes four cells at a step; a burst at
// cell granularity is no faster than that (measured above).  Result of THIS kernel (profiles/r02_super_level.txt, sessions u - z2): exact
// on every golden case; with bursts of the HANDOFF instantiation that end and warps that look at the queue cursor (two reasons why long
// walks never reached the hand-off before) a 17-row share of config 2 goes 0.56 -> 0.52 ms, a 1/8 share stays at 0.94.  Off by default.
// (Host form: rt_walk.h grid_trace_coop_bricks, compared with the reference's cell walk by tests/test_hostemu_parity.py::
// test_brick_plane_bursts_are_exact; the counting build does not count what the tail kernels do.)
// Here the 32 lanes take the next 11 / 11 / 10 crossings of every 4th plane:
// each certain crossing enters one 4x4x4 brick, its lane rebuilds the exact cell state at that entry (pwalk_refine, the very function
// the lanes' two-level walk uses) and walks the brick's cells on its own -- up to 10 dependent steps, 32 bricks side by side, nothing at
// all for an empty brick that does not hold the ray's end cell.  Occupied cells go to a list with their position in the walk
// (brick slot, step inside the brick); the list is opened and tested as in the pipe kernel's drain, smallest key wins; cells behind
// the end cell are dropped.  Slot 0 of the first burst is the rest of the brick the ray was given up in.
enum { kTailCellCap = 33 * 12 };
struct TailBrickWarp {
    float t[3][11];
    uint32_t cellRank[kTailCellCap];   // index of an occupied cell among the scene's non-empty cells
    uint32_t cellMeta[kTailCellCap];   // seq << 3 | entry face, seq = brick slot << 4 | step inside the brick
    uint32_t cells;                    // entries of the list
    uint32_t stopSeq;                  // seq of the ray's end cell once a lane has reached it
    uint32_t pairTri[kPairQCap], pairSeq[kPairQCap];
    unsigned long long bestKey;
    uint32_t bestTri;
    float bestAB, bestAC;
};

__global__ void __launch_bounds__(128) wf_tail_brick_kernel(SceneView S, WfState w, TailQueue tq) {
    extern __shared__ float shPlanes[];
    __shared__ TailBrickWarp warps[4];
    const uint32_t total = min(*tq.count, tq.capacity);
    if (total == 0u) return;
    load_planes(shPlanes, S);
    const int lane = threadIdx.x & 31;
    TailBrickWarp& T = warps[threadIdx.x >> 5];
    const unsigned ltMask = (1u << lane) - 1u;
    const int n = S.n, nb = S.nb;
    const int nbShift = 31 - __clz(nb);
    const float* px = shPlanes;
    const float* py = shPlanes + (n + 1);
    const float* pz = shPlanes + 2 * (n + 1);
    const unsigned long long kEmptyKey = ~0ull;

    for (;;) {
        uint32_t idx = 0;
        if (lane == 0) idx = atomicAdd(tq.cursor, 1u);
        idx = __shfl_sync(0xFFFFFFFFu, idx, 0);
        if (idx >= total) break;
        const uint4 e = tq.entries[idx];
        const uint32_t path = e.x;
        const float4 ro = w.rayO[path], rd = w.rayD[path];
        const uint32_t excl = w.rayExcl[path];
        const f3 o = mk3(ro.x, ro.y, ro.z), r = mk3(rd.x, rd.y, rd.z);
        const float minD = ro.w, maxD = rd.w;
        uint32_t epk;
        {
            PackedWalk s;
            pwalk_setup(s, n, nb, S.walkTrim, px, py, pz, o, r, minD, maxD);
            epk = s.epk;
        }
        const uint32_t endBrickPk = epk == (uint32_t)kPkNone ? (uint32_t)kPkNone : ((epk >> 2) & 0x0FF3FCFFu);
        // brick the walk stands in: given up at cell level (the rest of that brick is slot 0 of the first burst) or while crossing an
        // empty brick at brick level (nothing left to visit in it)
        const int lsh0 = e.w ? 0 : 2;
        int bc0[3] = {pk_get(e.y, 0) >> lsh0, pk_get(e.y, 1) >> lsh0, pk_get(e.y, 2) >> lsh0};
        const int upx = (0 <= r.x) ? 1 : 0, upy = (0 <= r.y) ? 1 : 0, upz = (0 <= r.z) ? 1 : 0;
        if (lane == 0) T.bestKey = kEmptyKey;
        bool first = true;
        bool done = false;
        while (!done) {
            if (lane == 0) {
                T.cells = 0u;
                T.stopSeq = 0xFFFFFFFFu;
            }
            // ---- brick-level burst: which bricks does the walk enter next, in which order? ---------------------------------------
            const int a = lane % 3, kc = lane / 3;
            const float oa = a == 0 ? o.x : (a == 1 ? o.y : o.z), ra = a == 0 ? r.x : (a == 1 ? r.y : r.z);
            const int upa = a == 0 ? upx : (a == 1 ? upy : upz);
            const int kmaxA = upa ? (nb - 1 - bc0[a]) : bc0[a];   // brick-plane crossings that stay inside the grid; crossing kmaxA leaves it
            const float tv = kc > kmaxA ? OCLR_INF : (shPlanes[a * (n + 1) + ((bc0[a] + upa + (upa ? kc : -kc)) << 2)] - oa) / ra;
            __syncwarp();
            T.t[a][kc] = tv;
            __syncwarp();
            int cnt[3];
            int rank = kc;
#pragma unroll
            for (int b = 0; b < 3; ++b) {
                if (b == a) {
                    cnt[b] = kc + 1;
                    continue;
                }
                int c = 0;
                for (int kk = 0; kk < coop_candidates(b); ++kk) c += coop_precedes(b, T.t[b][kk], a, tv) ? 1 : 0;
                cnt[b] = c;
                rank += c;
            }
            const bool present = kc <= kmaxA;
            const int kBig = 1 << 20;
            const int R = __reduce_min_sync(0xFFFFFFFFu, (kc == coop_candidates(a) - 1 && kmaxA >= coop_candidates(a)) ? rank + 1 : kCoopLanes);
            const int exitRank = __reduce_min_sync(0xFFFFFFFFu, (present && kc == kmaxA) ? rank : kBig);
            const int bx = bc0[0] + (upx ? cnt[0] : -cnt[0]), by = bc0[1] + (upy ? cnt[1] : -cnt[1]), bz = bc0[2] + (upz ? cnt[2] : -cnt[2]);
            const bool entersBrick = present && kc < kmaxA;
            const uint32_t brickPk = entersBrick ? pk_make(bx & kPkMask, by & kPkMask, bz & kPkMask) : (uint32_t)kPkNone;
            // the end cell's brick is walked cell by cell whatever it holds, and nothing behind it belongs to this burst
            const int endRank = __reduce_min_sync(0xFFFFFFFFu, (entersBrick && brickPk == endBrickPk) ? rank : kBig);
            int limit = R;
            bool finished = false;
            if (exitRank < limit) {
                limit = exitRank;
                finished = true;
            }
            if (endRank < limit) limit = endRank + 1;
            // ---- every brick of the burst is walked by the lane that holds its crossing; slot 0 (first burst only, lane 0 before its
            //      own brick) = the rest of the brick the ray was given up in ------------------------------------------------------------
            auto walk_cells = [&](PackedWalk& g, const uint4 br, uint32_t slot, int face) {
                const uint64_t mask = (uint64_t)br.x | ((uint64_t)br.y << 32);
                for (uint32_t step = 0; step < 16u; ++step) {
                    const int bit = pwalk_bit(g.cpk);
                    const uint32_t seq = (slot << 4) | step;
                    if ((mask >> bit) & 1ull) {
                        const uint32_t pos = atomicAdd(&T.cells, 1u);
                        if (pos < (uint32_t)kTailCellCap) {
                            T.cellRank[pos] = br.z + (uint32_t)__popcll(mask & ((1ull << bit) - 1ull));
                            T.cellMeta[pos] = (seq << 3) | (uint32_t)face;
                        }
                    }
                    if (g.cpk == epk) {   // the end cell is visited, then the walk stops (:381)
                        atomicMin(&T.stopSeq, seq);
                        break;
                    }
                    int axis, up;
                    float tE;
                    bool crossed;
                    if (!pwalk_step(g, n, S.walkTrim, nbShift, shPlanes, axis, up, tE, crossed)) break;   // left the grid (the exit crossing says "finished")
                    if (crossed) break;                                                          // left the brick: the next slot's business
                    face = axis * 2 + up;
                }
            };
            if (first && lane == 0 && e.w == 0u) {
                PackedWalk g;
                g.o = o;
                g.r = r;
                g.epk = epk;
                g.endBrick = (int)kEndNone;
                g.coarseOk = true;
                g.level = 0;
                g.cpk = e.y;
                const int cx = pk_get(e.y, 0), cy = pk_get(e.y, 1), cz = pk_get(e.y, 2);
                g.tx = (px[cx + upx] - o.x) / r.x;
                g.ty = (py[cy + upy] - o.y) / r.y;
                g.tz = (pz[cz + upz] - o.z) / r.z;
                g.brick = bc0[0] + ((bc0[1] + (bc0[2] << nbShift)) << nbShift);
                walk_cells(g, __ldg(S.bricks + g.brick), 0u, (int)e.z);
            }
            if (rank < limit) {
                // (the record first: an empty brick that does not hold the end cell has nothing to visit -- no crossings, no refinement)
                const int brick = bx + ((by + (bz << nbShift)) << nbShift);
                const uint4 br = __ldg(S.bricks + brick);
                if ((br.x | br.y) != 0u || brickPk == endBrickPk) {
                    PackedWalk g;
                    g.o = o;
                    g.r = r;
                    g.epk = epk;
                    g.endBrick = (int)kEndNone;
                    g.coarseOk = true;
                    g.level = 1;
                    g.cpk = brickPk;
                    g.tx = (px[(bx + upx) << 2] - o.x) / r.x;
                    g.ty = (py[(by + upy) << 2] - o.y) / r.y;
                    g.tz = (pz[(bz + upz) << 2] - o.z) / r.z;
                    g.brick = brick;
                    pwalk_refine(g, n, nbShift, shPlanes, a, tv);
                    g.brick = brick;
                    walk_cells(g, br, (uint32_t)rank + 1u, (int)kFaceNone);
                }
            }
            __syncwarp();
            const uint32_t nCells = min(T.cells, (uint32_t)kTailCellCap);
            const uint32_t stopSeq = T.stopSeq;
            // ---- open the listed cells (any order: the key carries the position in the walk) and test their pairs ------------------
            uint32_t pqHead = 0, pqTail = 0;
            auto test_round = [&](uint32_t take) {
                __syncwarp();
                bool hit = false;
                unsigned long long key = kEmptyKey;
                uint32_t tri = 0;
                float ab = 0.f, ac = 0.f;
                if ((uint32_t)lane < take) {
                    const uint32_t pidx = pqHead + (uint32_t)lane;
                    tri = T.pairTri[pidx & (kPairQCap - 1)];
                    const uint32_t seq = T.pairSeq[pidx & (kPairQCap - 1)];
                    float t;
                    hit = tri_test(S.triGeo + 4 * (size_t)tri, o, r, minD, maxD, t, ab, ac);
                    if (hit) {
                        key = ((unsigned long long)seq << 54) | ((unsigned long long)__float_as_uint(t) << 22) | (unsigned long long)(pidx & 0x3FFFFFu);
                        atomicMin(&T.bestKey, key);
                    }
                }
                __syncwarp();
                if (hit && T.bestKey == key) {
                    T.bestTri = tri;
                    T.bestAB = ab;
                    T.bestAC = ac;
                }
                pqHead += take;
            };
            for (uint32_t base = 0; base < nCells; base += 32u) {
                uint32_t k = 0, kEnd = 0, kBegin = 0, fm = 0, seq = 0;
                if (base + (uint32_t)lane < nCells) {
                    const uint32_t rankC = T.cellRank[base + lane], meta = T.cellMeta[base + lane];
                    seq = meta >> 3;
                    if (seq <= stopSeq) {   // (a cell behind the end cell is not part of the walk)
                        const uint32_t face = meta & 7u;
                        const uint2 range = __ldg(S.cellRange + rankC);
                        fm = face != (uint32_t)kFaceNone ? __ldg(S.faceMask + 6 * (size_t)rankC + face) : 0xFFFFFFFFu;
                        kBegin = range.x;
                        kEnd = range.y;
                        k = next_entry(kBegin, kEnd, fm, kBegin);
                    }
                }
                while (__any_sync(0xFFFFFFFFu, k < kEnd)) {
                    const bool more = k < kEnd;
                    uint32_t tri = 0;
                    if (more) tri = __ldg(S.cellList + k);
                    const bool valid = more & (tri != excl);
                    const unsigned vb = __ballot_sync(0xFFFFFFFFu, valid);
                    if (valid) {
                        const uint32_t pos = (pqTail + (uint32_t)__popc(vb & ltMask)) & (kPairQCap - 1);
                        T.pairTri[pos] = tri;
                        T.pairSeq[pos] = seq;
                    }
                    pqTail += (uint32_t)__popc(vb);
                    if (more) k = next_entry(kBegin, kEnd, fm, k + 1u);
                    if (pqTail - pqHead >= 32u) test_round(32u);
                }
            }
            while (pqTail != pqHead) test_round(pqTail - pqHead < 32u ? pqTail - pqHead : 32u);
            __syncwarp();
            const unsigned long long key = T.bestKey;
            if (key != kEmptyKey) {
                if (lane == 0) w.hit[path] = make_float4(__uint_as_float(T.bestTri), __uint_as_float((uint32_t)(key >> 22)), T.bestAB, T.bestAC);
                done = true;
            } else if (finished || stopSeq != 0xFFFFFFFFu) {
                if (lane == 0) w.hit[path] = make_float4(__uint_as_float(kNoTriangle), maxD, 0.f, 0.f);
                done = true;
            } else {   // go on from the last brick entered (limit >= 1 here: no exit, no end cell, so R >= 1 crossings were certain)
                const int src = __ffs(__ballot_sync(0xFFFFFFFFu, rank == limit - 1)) - 1;
                bc0[0] = __shfl_sync(0xFFFFFFFFu, bx, src);
                bc0[1] = __shfl_sync(0xFFFFFFFFu, by, src);
                bc0[2] = __shfl_sync(0xFFFFFFFFu, bz, src);
            }
            first = false;
            __syncwarp();
        }
    }
}

}  // namespace oclr
