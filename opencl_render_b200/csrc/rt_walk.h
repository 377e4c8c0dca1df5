// rt_walk.h -- the grid walk of raytrace_opencl.c:324-401 in the form the production trace kernel runs it: packed cell
// coordinates, one select-based step that serves both levels of the two-level walk, incremental brick addressing.
//
// Same contract as rt_core.h: `__host__ __device__`, the reference's fp32 operation order, IEEE division, no FMA
// contraction; tests/hostemu compiles grid_trace_packed() for the host and compares it with the reference walk cell by cell
// (tests/test_hostemu_parity.py).  The exactness argument of the two-level walk is the one written above
// walk_enter_coarse() in rt_core.h; this file only changes the bookkeeping:
//
//   cpk     cell coordinates (level 0), 4x4x4-brick coordinates (level 1) or super-brick coordinates (level 2: 4x4x4 bricks =
//           16x16x16 cells), 10 bits per axis: x | y << 10 | z << 20 (axesDivCount <= 1024; the plugin passes 256, render.cpp:1334);
//   brick   linear id of the brick the walk is in, updated by +-nb^axis only when a step crosses a brick face, so the
//           16-byte brick record is fetched exactly once per brick;
//   step    axis = argmin of the three next-crossing values with the reference's tie rule (x only if strictly smallest,
//           else y if strictly smaller than z, else z; NaNs fall through to z), then ONE plane fetch + ONE division.
#pragma once
#include "rt_core.h"

namespace oclr {

enum { kPkBits = 10, kPkMask = 1023, kPkNone = 0xFFFFFFFFu };
enum { kFaceNone = 7 };

OCLR_HD uint32_t pk_make(int x, int y, int z) { return (uint32_t)x | ((uint32_t)y << kPkBits) | ((uint32_t)z << (2 * kPkBits)); }
OCLR_HD int pk_get(uint32_t pk, int axis) { return (int)((pk >> (axis * kPkBits)) & kPkMask); }

// A walk that is one PART of a longer walk (see pwalk_jump) ends at a plane instead of a cell: PackedWalk::epk then holds
// 10b | axis << 10 | cell index -- the part is over the moment a step along `axis` enters that cell index (the cell belongs to
// the next part).  The index is the first cell of its brick in travel direction, so a brick-level step lands on it too.
OCLR_HD uint32_t pk_stop(int axis, int cellIndex) { return 0x80000000u | ((uint32_t)axis << kPkBits) | (uint32_t)cellIndex; }
OCLR_HD bool pk_is_stop(uint32_t epk) { return (epk >> 30) == 2u; }

// Three-level walk.  The argument that makes the brick-level walk exact (rt_core.h, walk_enter_coarse: the walk is a 3-way merge of
// per-axis crossing sequences whose order depends on values and the tie rule alone, so the merge of every 4th plane visits the bricks
// the cell walk visits, in its order, with the same crossing values) holds for any subsequence of the planes, hence also for every
// 16th: an entirely empty SUPER-BRICK (4x4x4 bricks) is crossed in one step and the brick-level state is rebuilt on entering a
// super-brick that holds triangles -- or the ray's end cell -- by the same refinement that rebuilds the cell state inside a brick.
//
// Kept out of the hot loop (a first version that told the levels apart there cost config 2, whose super-bricks are all occupied, 5 %):
//   * super-brick records {non-empty, 0, 0, 0} live behind the nb^3 brick records of the same array at the BRICK strides -- record of
//     super-brick (sx, sy, sz) = nb^3 + sx + nb * (sy + nb * sz) -- so the incremental id update of a step is the same at every level;
//   * an EMPTY brick's record carries in .z (the rank base nobody reads: the brick has no cells to rank) bit 0 = "my whole super-brick
//     is empty"; pack_grid / super_brick_kernel decide, the walk only obeys, and the flag is never set on a grid without this level;
//   * while the walk is at level 2 `endBrick` holds the record index of the END CELL's super-brick (swapped on the level switch), so
//     "never skip the end" is the same comparison at every level.
// Config 3: 65 of 130 steps per path are brick-level steps, 41 with this level (config 2: 39 of 106, 35).
struct PackedWalk {
    f3 o, r;
    float tx, ty, tz;    // next crossing per axis at the current level
    uint32_t cpk;        // current cell (level 0) / brick (level 1) / super-brick (level 2)
    uint32_t epk;        // end cell, or kPkNone
    int brick;           // index of the current brick's record; level 2: of the current super-brick's record
    int endBrick;        // where the walk ends, as one word (pwalk_end_key): record index of the end cell's brick (level 2: super-brick)
                         // -- walked at the finer level, never skipped -- | the cell's bit inside the brick << 25; or kEndNone
    uint32_t maskLo, maskHi, rankBase;   // record of `brick`; empty brick: bit 0 of rankBase = the whole super-brick is empty
    int level;           // 0: cells, 1: bricks, 2: super-bricks
    bool coarseOk;       // all direction components non-zero and n >= 4
};

// Super-brick coordinates (packed, 10-bit fields) of a packed cell / brick coordinate.
OCLR_HD uint32_t pk_super_of_cell(uint32_t pk) { return (pk >> 4) & 0x03F0FC3Fu; }
OCLR_HD uint32_t pk_super_of_brick(uint32_t pk) { return (pk >> 2) & 0x0FF3FCFFu; }
// Index of a super-brick's record in the brick array (nb = 1 << nbShift bricks per axis; brick strides, see above).
OCLR_HD int pk_super_record(uint32_t spk, int nbShift) {
    return (1 << (3 * nbShift)) + (int)((spk & kPkMask) + ((((spk >> kPkBits) & kPkMask) + (((spk >> (2 * kPkBits)) & kPkMask) << nbShift)) << nbShift));
}
OCLR_HD int pk_brick_record(uint32_t cellPk, int nbShift) {
    return (pk_get(cellPk, 0) >> 2) + (((pk_get(cellPk, 1) >> 2) + ((pk_get(cellPk, 2) >> 2) << nbShift)) << nbShift);
}
// Bit of a cell inside its brick's occupancy mask: (x & 3) | (y & 3) << 2 | (z & 3) << 4.
OCLR_HD int pwalk_bit(uint32_t cpk) {
    const uint32_t t = cpk & 0x00300C03u;
    return (int)((t | (t >> 8) | (t >> 16)) & 63u);
}
// The end of a bounded walk as ONE word, so that the trace kernel's hot loop needs neither the end cell nor a second comparison (ncu:
// at 64 registers the end cell was the value ptxas spilled, and every walk iteration began with its reload from local memory):
//   record index of the end cell's brick (< 2^25: nb^3 brick + nb^3 / 4 super-brick records, nb <= 256) | bit of the end cell << 25
// "in the end brick" = the low 25 bits (and bit 31) agree with `brick`; "on the end cell" = the whole word equals brick | bit << 25.
// kEndNone (bit 31): no end cell -- an unbounded ray, or a part of a cut walk, which ends at a plane.
enum : uint32_t { kEndNone = 0x80000000u, kEndBrickMask = 0x81FFFFFFu };
enum { kEndBitShift = 25 };
OCLR_HD int pwalk_end_key(uint32_t epk, int nbShift) {
    if ((epk >> 31) != 0u) return (int)kEndNone;   // kPkNone / a stop plane
    return pk_brick_record(epk, nbShift) | (pwalk_bit(epk) << kEndBitShift);
}

// Ray -> initial walk state: raytrace_opencl.c:350-362 (BindInCube on start and end, GetBoxAddress) + the first three crossing values.
// Cell index along `axis` on a grid of n - (trim's field) cells per axis (SceneView::walkTrim).  On a walk grid the planes past its
// extent repeat its last plane, so a point beyond that plane addresses a padded cell: the grid's last cell stands for it (its list is
// the list of every reference cell past the last kept plane, a collapsed run).  The reference grid: box_address's own answer.
OCLR_HD int pwalk_clamp_cell(int c, int n, uint32_t trim, int axis) {
    const int last = n - 1 - (int)((trim >> (axis * kPkBits)) & kPkMask);
    return c < last ? c : last;
}

OCLR_HD void pwalk_setup(PackedWalk& w, int n, int nb, uint32_t trim, const float* px, const float* py, const float* pz, f3 o, f3 r, float minD,
                         float maxD) {
    w.o = o;
    w.r = r;
    const f3 lo = mk3(px[0], py[0], pz[0]);
    const f3 hi = mk3(px[n], py[n], pz[n]);
    f3 start = mk3(o.x + minD * r.x, o.y + minD * r.y, o.z + minD * r.z);
    bind_in_cube(start, r, lo, hi);
    int cx, cy, cz;
    box_address(n, px, py, pz, start, cx, cy, cz);
    cx = pwalk_clamp_cell(cx, n, trim, 0);
    cy = pwalk_clamp_cell(cy, n, trim, 1);
    cz = pwalk_clamp_cell(cz, n, trim, 2);
    w.cpk = pk_make(cx, cy, cz);
    w.epk = kPkNone;
    w.endBrick = (int)kEndNone;
    if (maxD < OCLR_INF) {
        f3 end = mk3(o.x + maxD * r.x, o.y + maxD * r.y, o.z + maxD * r.z);
        bind_in_cube(end, r, lo, hi);
        int ex, ey, ez;
        box_address(n, px, py, pz, end, ex, ey, ez);
        ex = pwalk_clamp_cell(ex, n, trim, 0);
        ey = pwalk_clamp_cell(ey, n, trim, 1);
        ez = pwalk_clamp_cell(ez, n, trim, 2);
        w.epk = pk_make(ex, ey, ez);
        w.endBrick = ((ex >> 2) + nb * ((ey >> 2) + nb * (ez >> 2))) | (pwalk_bit(w.epk) << kEndBitShift);
    }
    w.tx = (px[cx + (0 <= r.x)] - o.x) / r.x;
    w.ty = (py[cy + (0 <= r.y)] - o.y) / r.y;
    w.tz = (pz[cz + (0 <= r.z)] - o.z) / r.z;
    w.brick = (cx >> 2) + nb * ((cy >> 2) + nb * (cz >> 2));
    w.level = 0;
    w.coarseOk = (n >= 4) & (r.x != 0.f) & (r.y != 0.f) & (r.z != 0.f);
    w.maskLo = w.maskHi = w.rankBase = 0;
}

OCLR_HD void pwalk_load_brick(PackedWalk& w, const uint4* bricks) {
    const uint4 br = OCLR_LDG(bricks + w.brick);
    w.maskLo = br.x;
    w.maskHi = br.y;
    w.rankBase = br.z;
}
// At level 1 in an empty brick whose record says "the whole super-brick is empty": may the walk go on super-brick by super-brick?
// Not through the super-brick that holds the end cell (it would be skipped), and not as a part of a cut walk (a part ends at a plane
// only brick-level steps are sure to land on).  kPkNone gives a coordinate only a 1024^3 grid has: a refusal too many there.
OCLR_HD bool pwalk_super_allowed(const PackedWalk& w) {
    return (pk_super_of_brick(w.cpk) != pk_super_of_cell(w.epk)) & !pk_is_stop(w.epk);
}

OCLR_HD bool pwalk_in_end(const PackedWalk& w) { return ((uint32_t)(w.endBrick ^ w.brick) & kEndBrickMask) == 0u; }
OCLR_HD bool pwalk_at_end(const PackedWalk& w, int bit) { return (uint32_t)w.endBrick == ((uint32_t)w.brick | ((uint32_t)bit << kEndBitShift)); }
OCLR_HD bool pwalk_occupied(const PackedWalk& w, int bit) {
    const uint32_t half = (bit & 32) ? w.maskHi : w.maskLo;
    return ((half >> (bit & 31)) & 1u) != 0u;
}
// Index of the current (occupied) cell among the non-empty cells of the scene, brick-major.
OCLR_HD uint32_t pwalk_rank(const PackedWalk& w, int bit) {
    const uint64_t m = (uint64_t)w.maskLo | ((uint64_t)w.maskHi << 32);
    return w.rankBase + (uint32_t)OCLR_POPCLL(m & ((1ull << bit) - 1ull));
}

// One step at the current level (:383-398), in two halves so that a caller that keeps the ray somewhere else than in registers (the
// trace kernel: its shared-memory ray table -- six registers less in a loop that sits at the register cap) fetches the origin and
// direction component of the stepped axis only.
// First half: the axis whose crossing comes next and its value.  (x only if strictly smallest, else y if strictly smaller than z, else z)
OCLR_HD int pwalk_step_axis(const PackedWalk& w, float& tEvent) {
    const bool xmin = (w.tx < w.ty) & (w.tx < w.tz);
    const bool ymin = (!xmin) & (w.ty < w.tz);
    tEvent = xmin ? w.tx : (ymin ? w.ty : w.tz);
    return xmin ? 0 : (ymin ? 1 : 2);
}
// Second half: the step along `axis` (oo, rr = origin / direction component of that axis, up = (0 <= rr)).  Returns false when the walk
// left the grid -- n - (trim's field of the axis) cells, SceneView::walkTrim; a multiple of 4 whenever the brick level runs;
// `crossed` is set when the step entered another brick (always above level 0).
OCLR_HD bool pwalk_step_along(PackedWalk& w, int n, uint32_t trim, int nbShift, const float* planes, int axis, float oo, float rr, int up,
                              bool& crossed) {
    const int sh = axis * kPkBits;
    const int c = (int)((w.cpk >> sh) & kPkMask);
    const int dir = up ? 1 : -1;
    const int cn = c + dir;
    const int lsh = 2 * w.level;
    crossed = false;
    if ((uint32_t)cn >= (uint32_t)((n - (int)((trim >> sh) & kPkMask)) >> lsh)) return false;
    const float t = (planes[axis * (n + 1) + ((cn + up) << lsh)] - oo) / rr;
    w.cpk += (uint32_t)dir << sh;   // two's complement: -1 << sh subtracts one from the axis' field
    w.tx = axis == 0 ? t : w.tx;
    w.ty = axis == 1 ? t : w.ty;
    w.tz = axis == 2 ? t : w.tz;
    crossed = (w.level != 0) | (((c ^ cn) & ~3) != 0);
    if (crossed) w.brick += dir * (1 << (axis * nbShift));   // (the same at level 2: super-brick records sit at the brick strides)
    return true;
}
// Both halves, the ray taken from the walk state.  `axis`, `up` and `tEvent` describe the crossing taken.
OCLR_HD bool pwalk_step(PackedWalk& w, int n, uint32_t trim, int nbShift, const float* planes, int& axis, int& up, float& tEvent, bool& crossed) {
    axis = pwalk_step_axis(w, tEvent);
    const float rr = axis == 0 ? w.r.x : (axis == 1 ? w.r.y : w.r.z);
    const float oo = axis == 0 ? w.o.x : (axis == 1 ? w.o.y : w.o.z);
    up = (0 <= rr) ? 1 : 0;
    return pwalk_step_along(w, n, trim, nbShift, planes, axis, oo, rr, up, crossed);
}

// After a successful step along `axis`: did the walk just cross into the cell index at which this part ends?
OCLR_HD bool pwalk_stopped(const PackedWalk& w, int axis, int up) {
    if (!pk_is_stop(w.epk) || (int)((w.epk >> kPkBits) & 3u) != axis) return false;
    const int c = pk_get(w.cpk, axis), lsh = 2 * w.level;
    const int cell = up ? (c << lsh) : (c << lsh) + (1 << lsh) - 1;
    return cell == (int)(w.epk & kPkMask);
}

// One level up inside an empty brick (0 -> 1) / an empty super-brick (1 -> 2): coordinates become those of the coarser level, the
// heads become the crossings that leave the brick / super-brick.
OCLR_HD_SW void pwalk_enter_coarse(PackedWalk& w, int n, int nbShift, const float* planes) {
    w.cpk = (w.cpk >> 2) & 0x0FF3FCFFu;
    w.level += 1;
    const int lsh = 2 * w.level;
    const float* px = planes;
    const float* py = planes + (n + 1);
    const float* pz = planes + 2 * (n + 1);
    w.tx = (px[(pk_get(w.cpk, 0) + (0 <= w.r.x)) << lsh] - w.o.x) / w.r.x;
    w.ty = (py[(pk_get(w.cpk, 1) + (0 <= w.r.y)) << lsh] - w.o.y) / w.r.y;
    w.tz = (pz[(pk_get(w.cpk, 2) + (0 <= w.r.z)) << lsh] - w.o.z) / w.r.z;
    if (w.level == 2) {   // (its record says "empty", like the masks the walk holds)
        w.brick = pk_super_record(w.cpk, nbShift);
        w.endBrick = (w.epk >> 31) != 0u ? (int)kEndNone : pk_super_record(pk_super_of_cell(w.epk), nbShift);
        w.rankBase = 0u;
    }
}

// One axis of the refinement, select-only form of refine_axis() / the entry-axis case of walk_refine() (rt_core.h): every lane of a
// warp runs the same instructions whatever axis its ray entered the brick along (the branchy form ran with 2.2 of 32 lanes active,
// profiles/r01d_wf_pipe_cfg2_phases.txt).  For the entry axis the answer is "first cell in travel direction, next crossing = the
// plane that cell is left through" -- exactly what the probe sequence yields when both probes are forced to "not before E" (the
// second probe then reads crossing 0, the very plane the entry case divides by), so forcing the predicates is all it takes.
// `psh`: the planes of the level being entered are every (1 << psh)-th cell plane (0: cells inside a brick, 2: bricks inside a super-brick).
OCLR_HD void prefine_axis(bool entry, int b, float tExit, float o, float r, const float* p, float E, bool strict, int psh, int& cell, float& tNext) {
    const int up = (0 <= r) ? 1 : 0;
    const int base = b << 2;
    const float t1 = (p[(base + 2) << psh] - o) / r;
    const bool pre1 = (!entry) & (strict ? (t1 < E) : (t1 <= E));
    const int p2 = (pre1 == (up != 0)) ? base + 3 : base + 1;   // pre1: crossing 2 (up: base+3, down: base+1); else crossing 0 (up: base+1, down: base+3)
    const float t2 = (p[p2 << psh] - o) / r;
    const bool pre2 = (!entry) & (strict ? (t2 < E) : (t2 <= E));
    const int j = (pre1 ? 2 : 0) + (pre2 ? 1 : 0);
    tNext = pre1 ? (pre2 ? tExit : t2) : (pre2 ? t1 : t2);
    cell = up ? base + j : base + 3 - j;
}

// One level down after the step along `axis` (crossing value E) entered a brick that has to be walked cell by cell (1 -> 0) / a
// super-brick that has to be walked brick by brick (2 -> 1): the exact state the finer walk would have on entering it (rt_core.h:
// walk_refine).  Arriving at level 1 the brick id is recomputed; its record is the caller's to load.
OCLR_HD_SW void pwalk_refine(PackedWalk& w, int n, int nbShift, const float* planes, int axis, float E) {
    const float* px = planes;
    const float* py = planes + (n + 1);
    const float* pz = planes + 2 * (n + 1);
    const int psh = 2 * (w.level - 1);
    int cx, cy, cz;
    float tx, ty, tz;
    prefine_axis(axis == 0, pk_get(w.cpk, 0), w.tx, w.o.x, w.r.x, px, E, true, psh, cx, tx);       // x precedes y / z crossings only when strictly smaller
    prefine_axis(axis == 1, pk_get(w.cpk, 1), w.ty, w.o.y, w.r.y, py, E, axis == 2, psh, cy, ty);  // y: "<= E" against x, "< E" against z
    prefine_axis(axis == 2, pk_get(w.cpk, 2), w.tz, w.o.z, w.r.z, pz, E, false, psh, cz, tz);      // z wins ties against x and y
    w.cpk = pk_make(cx, cy, cz);
    w.tx = tx;
    w.ty = ty;
    w.tz = tz;
    w.level -= 1;
    if (w.level == 1) {
        w.brick = cx + ((cy + (cz << nbShift)) << nbShift);
        w.endBrick = pwalk_end_key(w.epk, nbShift);
    }
}

// Position of the k-th still-untested list entry at or after `k` (rt_wavefront.cuh next_candidate, serial form without a mailbox).
OCLR_HD uint32_t pwalk_next_entry(uint32_t begin, uint32_t end, uint32_t faceBits, uint32_t k) {
    const uint32_t rel = k - begin;
    if (rel < 32u) {
        const uint32_t mm = faceBits >> rel;
        if (mm == 0u) return begin + 32u < end ? begin + 32u : end;
        uint32_t s = 0;
        while (((mm >> s) & 1u) == 0u) ++s;
        k += s;
    }
    return k < end ? k : end;
}

// ---- exact random access into the walk --------------------------------------------------------------------------------------------
// The walk is a 3-way merge of per-axis crossing sequences t_b(k) = (plane_b[k] - o_b) / r_b (rt_core.h, walk_enter_coarse).
// With all direction components non-zero the merge order of two crossings of DIFFERENT axes is decided by their values and the
// reference's tie rule alone (:387-398): an x crossing goes first only when strictly smaller; y goes before z only when strictly
// smaller; otherwise the later axis goes first.  So the state of the walk right after it crosses into cell index B along axis a
// (crossing value E) is known without walking: along every other axis b it has taken exactly the crossings that precede E,
// a monotone predicate over the sorted planes -> binary search, one division per probe (walk_refine is the 4-plane case).
// Used to cut a long walk into parts that different lanes walk concurrently (rt_trace.cuh, wf_setup_kernel).

// Number of crossings of axis b, starting in cell c0, that precede the crossing value E of another axis.  `exits`: the crossing
// that leaves the grid precedes E too (the walk ends before E).
OCLR_HD int pwalk_count_before(int n, const float* pb, float o, float r, int c0, float E, bool strict, bool& exits) {
    const int up = (0 <= r) ? 1 : 0;
    const int kmax = up ? (n - 1 - c0) : c0;   // crossings 0 .. kmax-1 stay inside the grid, crossing kmax leaves it
    int lo = 0, hi = kmax + 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const float t = (pb[c0 + up + (up ? mid : -mid)] - o) / r;
        const bool pre = strict ? (t < E) : (t <= E);
        if (pre) lo = mid + 1; else hi = mid;
    }
    exits = lo > kmax;
    return lo;
}

// State of the walk that started in cell (c0x, c0y, c0z) right after it crosses into cell index B along `axis`.
// Returns false when the walk leaves the grid before that crossing.  Requires r.x, r.y, r.z != 0.
OCLR_HD bool pwalk_jump(PackedWalk& w, int n, int nb, const float* px, const float* py, const float* pz, f3 o, f3 r, int c0x, int c0y,
                        int c0z, int axis, int B) {
    const float* pa = axis == 0 ? px : (axis == 1 ? py : pz);
    const float oa = axis == 0 ? o.x : (axis == 1 ? o.y : o.z), ra = axis == 0 ? r.x : (axis == 1 ? r.y : r.z);
    const int upa = (0 <= ra) ? 1 : 0;
    const float E = (pa[B + (upa ? 0 : 1)] - oa) / ra;
    int c[3] = {c0x, c0y, c0z};
    bool exits = false;
    if (axis != 0) {  // x goes before y / z only when strictly smaller
        const int k = pwalk_count_before(n, px, o.x, r.x, c0x, E, true, exits);
        if (exits) return false;
        c[0] = c0x + ((0 <= r.x) ? k : -k);
    }
    if (axis != 1) {  // y: before x on ties, before z only when strictly smaller
        const int k = pwalk_count_before(n, py, o.y, r.y, c0y, E, axis == 2, exits);
        if (exits) return false;
        c[1] = c0y + ((0 <= r.y) ? k : -k);
    }
    if (axis != 2) {  // z wins ties against x and y
        const int k = pwalk_count_before(n, pz, o.z, r.z, c0z, E, false, exits);
        if (exits) return false;
        c[2] = c0z + ((0 <= r.z) ? k : -k);
    }
    c[axis] = B;
    w.o = o;
    w.r = r;
    w.cpk = pk_make(c[0], c[1], c[2]);
    w.tx = (px[c[0] + (0 <= r.x)] - o.x) / r.x;
    w.ty = (py[c[1] + (0 <= r.y)] - o.y) / r.y;
    w.tz = (pz[c[2] + (0 <= r.z)] - o.z) / r.z;
    w.brick = (c[0] >> 2) + nb * ((c[1] >> 2) + nb * (c[2] >> 2));
    w.level = 0;
    w.coarseOk = (n >= 4);
    w.maskLo = w.maskHi = w.rankBase = 0;
    return true;
}

// Cuts of one walk into parts along its dominant axis: at most kMaxWalkParts parts of about `partCells` cells (Manhattan
// estimate between the start cell and (ex, ey, ez) = end cell or estimated exit cell).  cutIndex[j] (j >= 1) = cell index along
// `axis` whose entry starts part j (and ends part j - 1, pk_stop).
enum { kMaxWalkParts = 8 };
OCLR_HD int pwalk_plan_parts(int c0x, int c0y, int c0z, int ex, int ey, int ez, int partCells, int& axis, int cutIndex[kMaxWalkParts]) {
    const int dx = ex - c0x, dy = ey - c0y, dz = ez - c0z;
    const int ax = dx < 0 ? -dx : dx, ay = dy < 0 ? -dy : dy, az = dz < 0 ? -dz : dz;
    axis = (ax >= ay && ax >= az) ? 0 : (ay >= az ? 1 : 2);
    const int span = axis == 0 ? ax : (axis == 1 ? ay : az), sgn = (axis == 0 ? dx : (axis == 1 ? dy : dz)) < 0 ? -1 : 1;
    const int c0 = axis == 0 ? c0x : (axis == 1 ? c0y : c0z), e = c0 + sgn * span;
    int want = (ax + ay + az + partCells - 1) / partCells;
    if (want > kMaxWalkParts) want = kMaxWalkParts;
    cutIndex[0] = c0;
    int parts = 1;
    for (int j = 1; j < want; ++j) {
        int B = c0 + sgn * (int)(((long long)span * j) / want);
        B = sgn > 0 ? (B & ~3) : (B | 3);   // first cell of its brick in travel direction: brick-level steps land on it
        // strictly between the previous cut and the end, in travel order
        const bool ok = sgn > 0 ? (B > cutIndex[parts - 1] && B < e) : (B < cutIndex[parts - 1] && B > e);
        if (ok) cutIndex[parts++] = B;
    }
    return parts;
}

// The walk proper from an initialised state (brick record not yet loaded).  Serial form of the trace kernel's per-ray logic
// (test infrastructure for the host; the kernel runs the same functions with the work of 32 rays interleaved).  Face masks skip
// entries shared with the cell just left; a small direct-mapped mailbox skips triangles this ray already tested -- both exact
// (rt_wavefront.cuh).
// A walk interrupted between two cells (wf_pipe_kernel splits long walks at run time, see pwalk_split_plan): everything the walk
// carries from cell to cell.  The current cell w.cpk has NOT been examined yet.
enum : uint32_t { kWalkPaused = 0xFFFFFFFEu };
struct WalkPause {
    PackedWalk w;
    int face, lastAxis;
    float lastE;
};

// `pauseAfter` >= 0: the walk stops at the top of its loop -- at either level -- after that many iterations, stores its state in *pause
// and returns kWalkPaused (test infrastructure for the run-time split).  `resume`: the state a paused walk continues from.
template <bool COUNT>
OCLR_HD uint32_t grid_walk_packed(const SceneView& S, const float* planes, PackedWalk w, float minD, float maxD, uint32_t excl, float& outT,
                                  float& outAB, float& outAC, Counters* cnt, int pauseAfter = -1, WalkPause* pause = nullptr,
                                  const WalkPause* resume = nullptr) {
    const int n = S.n;
    int nbShift = 0;
    while ((1 << nbShift) < S.nb) ++nbShift;
    const f3 o = w.o, r = w.r;
    if (!resume) {
        pwalk_load_brick(w, S.bricks);
        if (COUNT) cnt->bricksLoaded++;
    }
    uint32_t mailbox[16];
    for (int k = 0; k < 16; ++k) mailbox[k] = kNoTriangle;
    int face = resume ? resume->face : (int)kFaceNone, lastAxis = resume ? resume->lastAxis : 0;
    float lastE = resume ? resume->lastE : 0.f;
    outT = maxD;
    for (;;) {
        if (pauseAfter >= 0 && pauseAfter-- == 0) {
            pause->w = w;
            pause->face = face;
            pause->lastAxis = lastAxis;
            pause->lastE = lastE;
            return kWalkPaused;
        }
        if (w.level == 0) {
            const int bit = pwalk_bit(w.cpk);
            if (COUNT) {
                cnt->cells++;
                if ((w.maskLo | w.maskHi) == 0u) cnt->emptyBrickCells++;
            }
            if (pwalk_occupied(w, bit)) {
                const uint32_t rank = pwalk_rank(w, bit);
                const uint2 range = OCLR_LDG(S.cellRange + rank);
                const uint32_t fm = face != kFaceNone ? OCLR_LDG(S.faceMask + 6 * (size_t)rank + face) : 0xFFFFFFFFu;
                if (COUNT) cnt->cellsNonEmpty++;
                uint32_t closest = kNoTriangle;
                outT = maxD;
                for (uint32_t k = pwalk_next_entry(range.x, range.y, fm, range.x); k < range.y; k = pwalk_next_entry(range.x, range.y, fm, k + 1)) {
                    const uint32_t tri = OCLR_LDG(S.cellList + k);
                    if (tri == excl) continue;
                    if (mailbox[tri & 15u] == tri) {
                        if (COUNT) cnt->mailboxSkips++;
                        continue;
                    }
                    mailbox[tri & 15u] = tri;
                    float t, ab, ac;
                    if (COUNT) cnt->gridCandidates++;
                    if (tri_test(S.triGeo + 4 * (size_t)tri, o, r, minD, outT, t, ab, ac)) {
                        closest = tri;
                        outT = t;
                        outAB = ab;
                        outAC = ac;
                    }
                }
                if (closest != kNoTriangle) return closest;
            }
            if (pwalk_at_end(w, bit)) break;
            if (((w.maskLo | w.maskHi) == 0u) & w.coarseOk & !pwalk_in_end(w)) {
                pwalk_enter_coarse(w, n, nbShift, planes);
                if (COUNT) cnt->coarseEnters++;
                continue;
            }
        } else if (((w.maskLo | w.maskHi) != 0u) | pwalk_in_end(w)) {
            pwalk_refine(w, n, nbShift, planes, lastAxis, lastE);
            if (w.level == 1) {
                pwalk_load_brick(w, S.bricks);
                if (COUNT) {
                    cnt->bricksLoaded++;
                    cnt->superRefines++;
                }
            }
            face = kFaceNone;
            continue;
        } else if ((w.rankBase & 1u) != 0u) {   // (level 1, empty brick: the flag of its record)
            if (pwalk_super_allowed(w)) {
                pwalk_enter_coarse(w, n, nbShift, planes);
                if (COUNT) cnt->superEnters++;
                continue;
            }
            w.rankBase = 0u;   // refused: through this brick at brick level (its neighbour's record raises the question again)
        }
        int up;
        bool crossed;
        if (COUNT && w.level) cnt->coarseSteps++;
        if (COUNT && w.level == 2) cnt->superSteps++;
        if (!pwalk_step(w, n, S.walkTrim, nbShift, planes, lastAxis, up, lastE, crossed)) break;
        if (pwalk_stopped(w, lastAxis, up)) break;   // this part of the walk ends here; the cell belongs to the next part
        face = w.level ? (int)kFaceNone : lastAxis * 2 + up;
        if (crossed) {
            pwalk_load_brick(w, S.bricks);
            if (COUNT) cnt->bricksLoaded++;
        }
    }
    outT = maxD;
    return kNoTriangle;
}

template <bool COUNT>
OCLR_HD uint32_t grid_trace_packed(const SceneView& S, const float* planes, f3 o, f3 r, float minD, float maxD, uint32_t excl,
                                   float& outT, float& outAB, float& outAC, Counters* cnt) {
    const int n = S.n;
    PackedWalk w;
    pwalk_setup(w, n, S.nb, S.walkTrim, planes, planes + (n + 1), planes + 2 * (n + 1), o, r, minD, maxD);
    if (COUNT) cnt->gridRays++;
    return grid_walk_packed<COUNT>(S, planes, w, minD, maxD, excl, outT, outAB, outAC, cnt);
}

// Approximate cell where an unbounded ray leaves the grid (ordering / planning only, never a result).
OCLR_HD void pwalk_exit_estimate(int n, const float* px, const float* py, const float* pz, f3 o, f3 r, int& ex, int& ey, int& ez) {
    const float bx = r.x >= 0.f ? px[n] : px[0], by = r.y >= 0.f ? py[n] : py[0], bz = r.z >= 0.f ? pz[n] : pz[0];
    float t = OCLR_INF;
    if (r.x != 0.f) { const float q = (bx - o.x) / r.x; t = q < t ? q : t; }
    if (r.y != 0.f) { const float q = (by - o.y) / r.y; t = q < t ? q : t; }
    if (r.z != 0.f) { const float q = (bz - o.z) / r.z; t = q < t ? q : t; }
    if (!(t < OCLR_INF) || t < 0.f) t = 0.f;
    box_address(n, px, py, pz, mk3(o.x + t * r.x, o.y + t * r.y, o.z + t * r.z), ex, ey, ez);
}

// The same traversal with the walk cut into parts (the trace stage's way of bounding the longest work item): every part is
// walked on its own, the first part (in walk order) with a hit gives the result.  Exactly the uncut walk (tests assert it).
template <bool COUNT>
OCLR_HD uint32_t grid_trace_split(const SceneView& S, const float* planes, f3 o, f3 r, float minD, float maxD, uint32_t excl, float& outT,
                                  float& outAB, float& outAC, Counters* cnt, int partCells) {
    const int n = S.n;
    const float* px = planes;
    const float* py = planes + (n + 1);
    const float* pz = planes + 2 * (n + 1);
    PackedWalk first;
    pwalk_setup(first, n, S.nb, S.walkTrim, px, py, pz, o, r, minD, maxD);
    if (COUNT) cnt->gridRays++;
    const bool splittable = (n >= 4) & (r.x != 0.f) & (r.y != 0.f) & (r.z != 0.f);
    if (!splittable) return grid_walk_packed<COUNT>(S, planes, first, minD, maxD, excl, outT, outAB, outAC, cnt);
    const int c0x = pk_get(first.cpk, 0), c0y = pk_get(first.cpk, 1), c0z = pk_get(first.cpk, 2);
    int ex, ey, ez;
    if (first.epk != kPkNone) {
        ex = pk_get(first.epk, 0);
        ey = pk_get(first.epk, 1);
        ez = pk_get(first.epk, 2);
    } else {
        pwalk_exit_estimate(n, px, py, pz, o, r, ex, ey, ez);
    }
    int axis, cut[kMaxWalkParts];
    const int parts = pwalk_plan_parts(c0x, c0y, c0z, ex, ey, ez, partCells, axis, cut);
    for (int j = 0; j < parts; ++j) {
        PackedWalk part = first;
        // a part starts where the walk crosses into its cut (state computed without walking); when the walk leaves the grid
        // before that crossing there is nothing left to visit
        if (j > 0 && !pwalk_jump(part, n, S.nb, px, py, pz, o, r, c0x, c0y, c0z, axis, cut[j])) break;
        if (j + 1 < parts) {  // ends at the next cut
            part.epk = pk_stop(axis, cut[j + 1]);
            part.endBrick = (int)kEndNone;
        } else {  // last part: the ray's own end condition
            part.epk = first.epk;
            part.endBrick = first.endBrick;
        }
        const uint32_t hit = grid_walk_packed<COUNT>(S, planes, part, minD, maxD, excl, outT, outAB, outAC, cnt);
        if (hit != kNoTriangle) return hit;
    }
    outT = maxD;
    return kNoTriangle;
}

// ---- run-time split of a walk in progress (wf_pipe_kernel, tail of a launch) -------------------------------------------------------
// A trace launch cannot end before its longest walk does, and a lone lane stepping through several hundred cells is ~0.3 ms of
// latency that nothing else hides once the ray queue is dry.  Cutting walks by their ESTIMATED length before they start was tried
// and backed out (most long-looking rays end at a nearby hit).  Here the cut is made at run time, for a ray that HAS walked into the
// tail: the lane that owns it keeps the first part and idle lanes of the same warp take the others, every part starting from the
// exact state pwalk_jump computes at its stop plane.  The first part (in walk order) with a hit gives the ray's result.
//
// Plan for the remaining walk of `w` (either level, all direction components non-zero, current cell not yet examined): at most
// `maxParts` parts of equal length along the dominant axis of the way to the end cell / the estimated exit cell.  Returns the number
// of parts (1 = not worth cutting); cut[j] (j >= 1) = cell index along `axis` whose entry starts part j.
// Cell index along `axis` from which the crossings still ahead of the walk are counted: the current cell at level 0; at level 1 (the
// walk is somewhere inside an empty brick) the brick's first cell in travel direction -- every plane before it has been crossed, and
// pwalk_count_before is a search over a monotone predicate, so a lower bound is all it needs.
OCLR_HD int pwalk_floor_cell(const PackedWalk& w, int axis) {
    const int c = pk_get(w.cpk, axis);
    if (w.level == 0) return c;
    const float r = axis == 0 ? w.r.x : (axis == 1 ? w.r.y : w.r.z);
    const int lsh = 2 * w.level;
    return (c << lsh) + ((0 <= r) ? 0 : (1 << lsh) - 1);
}

OCLR_HD int pwalk_split_plan(const PackedWalk& w, int n, const float* px, const float* py, const float* pz, int maxParts, int minPartCells,
                             int& axis, int cut[kMaxWalkParts]) {
    if (w.level == 2) return 1;   // (a part ends at a plane super-brick steps can jump: the walk is cut once it is back at brick level)
    const int c0x = pwalk_floor_cell(w, 0), c0y = pwalk_floor_cell(w, 1), c0z = pwalk_floor_cell(w, 2);
    int ex, ey, ez;
    if (w.epk != kPkNone && !pk_is_stop(w.epk)) {
        ex = pk_get(w.epk, 0);
        ey = pk_get(w.epk, 1);
        ez = pk_get(w.epk, 2);
    } else {
        pwalk_exit_estimate(n, px, py, pz, w.o, w.r, ex, ey, ez);
    }
    const int dx = ex - c0x, dy = ey - c0y, dz = ez - c0z;
    const int len = (dx < 0 ? -dx : dx) + (dy < 0 ? -dy : dy) + (dz < 0 ? -dz : dz);
    int want = len / (minPartCells > 0 ? minPartCells : 1);
    if (want > maxParts) want = maxParts;
    if (want > kMaxWalkParts) want = kMaxWalkParts;
    if (want < 2) return 1;
    return pwalk_plan_parts(c0x, c0y, c0z, ex, ey, ez, (len + want - 1) / want, axis, cut);
}

// Part j >= 1 of that plan: the state right after the walk crosses into cut[j] (false: the walk leaves the grid first -- the part
// does not exist), with the part's own end condition.  Part 0 is the interrupted walk itself with pwalk_split_head() applied.
OCLR_HD bool pwalk_split_part(PackedWalk& part, const PackedWalk& w, int n, int nb, const float* px, const float* py, const float* pz, int axis,
                              const int cut[kMaxWalkParts], int parts, int j) {
    if (!pwalk_jump(part, n, nb, px, py, pz, w.o, w.r, pwalk_floor_cell(w, 0), pwalk_floor_cell(w, 1), pwalk_floor_cell(w, 2), axis, cut[j])) return false;
    if (j + 1 < parts) {
        part.epk = pk_stop(axis, cut[j + 1]);
        part.endBrick = (int)kEndNone;
    } else {
        part.epk = w.epk;
        part.endBrick = w.endBrick;
    }
    return true;
}
OCLR_HD void pwalk_split_head(PackedWalk& w, int axis, const int cut[kMaxWalkParts]) {
    w.epk = pk_stop(axis, cut[1]);
    w.endBrick = (int)kEndNone;
}

// Host form of the whole thing (tests/hostemu): walk `walkFirst` cells the ordinary way, then cut the rest into up to `maxParts` parts.
template <bool COUNT>
OCLR_HD uint32_t grid_trace_split_mid(const SceneView& S, const float* planes, f3 o, f3 r, float minD, float maxD, uint32_t excl, float& outT,
                                      float& outAB, float& outAC, Counters* cnt, int walkFirst, int maxParts, int minPartCells) {
    const int n = S.n;
    const float* px = planes;
    const float* py = planes + (n + 1);
    const float* pz = planes + 2 * (n + 1);
    PackedWalk first;
    pwalk_setup(first, n, S.nb, S.walkTrim, px, py, pz, o, r, minD, maxD);
    if (COUNT) cnt->gridRays++;
    WalkPause pause;
    uint32_t hit = grid_walk_packed<COUNT>(S, planes, first, minD, maxD, excl, outT, outAB, outAC, cnt, walkFirst, &pause);
    if (hit != kWalkPaused) return hit;
    PackedWalk head = pause.w;
    int axis = 0, cut[kMaxWalkParts];
    const int parts = head.coarseOk ? pwalk_split_plan(head, n, px, py, pz, maxParts, minPartCells, axis, cut) : 1;
    if (parts < 2) return grid_walk_packed<COUNT>(S, planes, head, minD, maxD, excl, outT, outAB, outAC, cnt, -1, nullptr, &pause);
    for (int j = 0; j < parts; ++j) {
        PackedWalk part = head;
        if (j == 0) {
            pwalk_split_head(part, axis, cut);
            hit = grid_walk_packed<COUNT>(S, planes, part, minD, maxD, excl, outT, outAB, outAC, cnt, -1, nullptr, &pause);
        } else {
            if (!pwalk_split_part(part, head, n, S.nb, px, py, pz, axis, cut, parts, j)) break;
            hit = grid_walk_packed<COUNT>(S, planes, part, minD, maxD, excl, outT, outAB, outAC, cnt);
        }
        if (hit != kNoTriangle) return hit;
    }
    outT = maxD;
    return kNoTriangle;
}

// ---- warp-cooperative walk of ONE ray ------------------------------------------------------------------------------------------
// (Groundwork, exercised by the host tests only: a first wiring into wf_pipe_kernel's tail mode was bit-exact but no faster --
// at the low occupancy of a launch's tail a burst costs about as much latency as the steps it replaces; DESIGN.md section 5.)
// A lone lane stepping through 500 cells is the critical path of a trace launch (~0.3 ms): each step is ~170 dependent
// instructions.  When few rays are left, the warp can walk one ray together instead: 32 lanes take the next 11 / 11 / 10 plane
// crossings of the x / y / z axis (one division each), and the merge order of the reference's walk gives every crossing its
// position directly -- crossing (a, k) is preceded by its own k predecessors plus, per other axis b, the b-crossings t' with
// t' < t, or t' == t and b > a (the tie rule of :387-398; see pwalk_jump).  The cell entered by a crossing follows from the same
// counts, so ~25 cells are classified per burst with no serial dependency.  Requires all direction components non-zero.
//
// The arithmetic below is per crossing ("virtual lane" v = 0..31: axis v % 3, index v / 3) so that the kernel (one real lane per
// crossing) and the host emulation (a loop) share it.
enum { kCoopLanes = 32 };
OCLR_HD int coop_candidates(int axis) { return axis == 2 ? 10 : 11; }   // lanes 0..31: axis = lane % 3

struct CoopRay {   // what every lane knows about the ray being walked
    f3 o, r;
    int c0[3];      // current cell (already classified)
    uint32_t epk;   // end cell / stop plane / none
};

// Crossing value of candidate (axis, k): the k-th next crossing of that axis; +inf when the walk has left the grid before it.
// kmax = crossings that stay inside the grid; crossing kmax itself is the one that leaves it.
OCLR_HD float coop_crossing(const CoopRay& ray, int n, const float* planes, int axis, int k, int& kmax) {
    const float o = axis == 0 ? ray.o.x : (axis == 1 ? ray.o.y : ray.o.z), r = axis == 0 ? ray.r.x : (axis == 1 ? ray.r.y : ray.r.z);
    const int up = (0 <= r) ? 1 : 0, c0 = ray.c0[axis];
    kmax = up ? (n - 1 - c0) : c0;
    if (k > kmax) return OCLR_INF;
    return (planes[axis * (n + 1) + c0 + up + (up ? k : -k)] - o) / r;
}
// does a crossing of axis b with value tb precede a crossing of axis a (a != b) with value ta?
OCLR_HD bool coop_precedes(int b, float tb, int a, float ta) { return (tb < ta) | ((tb == ta) & (b > a)); }

// Serial emulation of one burst (test infrastructure): appends the cells the walk enters, in order, to cells[] / faces[]
// (at most 31); returns their number.  `finished`: the walk ended inside the burst (left the grid, reached its end cell or its
// stop plane).  On return ray.c0 is the last cell entered (when the walk goes on).
OCLR_HD int coop_burst_serial(CoopRay& ray, int n, const float* planes, uint32_t* cells, int* faces, bool& finished) {
    float t[3][11];
    int kmax[3];
    for (int a = 0; a < 3; ++a)
        for (int k = 0; k < 11; ++k) t[a][k] = k < coop_candidates(a) ? coop_crossing(ray, n, planes, a, k, kmax[a]) : OCLR_INF;
    int rank[kCoopLanes], cnt[kCoopLanes][3];
    int R = kCoopLanes, exitRank = 1 << 20, endRank = 1 << 20;
    uint32_t cellOf[kCoopLanes];
    for (int v = 0; v < kCoopLanes; ++v) {
        const int a = v % 3, k = v / 3;
        rank[v] = k;
        for (int b = 0; b < 3; ++b) {
            cnt[v][b] = b == a ? k + 1 : 0;
            if (b == a) continue;
            for (int kk = 0; kk < coop_candidates(b); ++kk) cnt[v][b] += coop_precedes(b, t[b][kk], a, t[a][k]) ? 1 : 0;
            rank[v] += cnt[v][b];
        }
        const bool present = k <= kmax[a];
        if (k == coop_candidates(a) - 1 && kmax[a] >= coop_candidates(a) && rank[v] + 1 < R) R = rank[v] + 1;   // more crossings of a may follow
        if (present && k == kmax[a] && rank[v] < exitRank) exitRank = rank[v];
        int c[3];
        for (int b = 0; b < 3; ++b) {
            const float rb = b == 0 ? ray.r.x : (b == 1 ? ray.r.y : ray.r.z);
            c[b] = ray.c0[b] + ((0 <= rb) ? cnt[v][b] : -cnt[v][b]);
        }
        cellOf[v] = present && k < kmax[a] ? pk_make(c[0] & kPkMask, c[1] & kPkMask, c[2] & kPkMask) : kPkNone;
        bool ends = false;
        if (present && k < kmax[a]) {
            if (pk_is_stop(ray.epk)) {   // this part of a cut walk is over when a step along the stop axis enters the stop index
                ends = (int)((ray.epk >> kPkBits) & 3u) == a && c[a] == (int)(ray.epk & kPkMask);
                if (ends && rank[v] < exitRank) exitRank = rank[v];   // like leaving the grid: the cell is not visited
                ends = false;
            } else {
                ends = cellOf[v] == ray.epk;
            }
        }
        if (ends && rank[v] < endRank) endRank = rank[v];
    }
    // crossings with rank < R are certain (no crossing beyond the candidates can precede them); an exit / end crossing only
    // counts when it lies inside that prefix
    int limit = R;
    finished = false;
    if (exitRank < limit) {
        limit = exitRank;   // the crossing that leaves the grid (or enters the stop index) enters no cell
        finished = true;
    }
    if (endRank < limit) {
        limit = endRank + 1;   // the end cell is visited, then the walk stops (:381)
        finished = true;
    }
    int count = 0;
    for (int q = 0; q < limit; ++q)
        for (int v = 0; v < kCoopLanes; ++v)
            if (rank[v] == q && cellOf[v] != kPkNone) {
                cells[count] = cellOf[v];
                faces[count] = (v % 3) * 2 + ((0 <= ((v % 3) == 0 ? ray.r.x : ((v % 3) == 1 ? ray.r.y : ray.r.z))) ? 1 : 0);
                ++count;
            }
    if (count > 0) {
        ray.c0[0] = pk_get(cells[count - 1], 0);
        ray.c0[1] = pk_get(cells[count - 1], 1);
        ray.c0[2] = pk_get(cells[count - 1], 2);
    }
    return count;
}

// The traversal walked entirely by cooperative bursts (host test of the burst arithmetic against the reference's cell walk).
template <bool COUNT>
OCLR_HD uint32_t grid_trace_coop(const SceneView& S, const float* planes, f3 o, f3 r, float minD, float maxD, uint32_t excl, float& outT,
                                 float& outAB, float& outAC, Counters* cnt) {
    const int n = S.n;
    PackedWalk w;
    pwalk_setup(w, n, S.nb, S.walkTrim, planes, planes + (n + 1), planes + 2 * (n + 1), o, r, minD, maxD);
    if (!w.coarseOk) return grid_trace_packed<COUNT>(S, planes, o, r, minD, maxD, excl, outT, outAB, outAC, cnt);
    if (COUNT) cnt->gridRays++;
    auto test_cell = [&](uint32_t cpk, int face, uint32_t& closest) {
        const int cx = pk_get(cpk, 0), cy = pk_get(cpk, 1), cz = pk_get(cpk, 2);
        const uint4 br = OCLR_LDG(S.bricks + ((cx >> 2) + S.nb * ((cy >> 2) + S.nb * (cz >> 2))));
        PackedWalk b;
        b.maskLo = br.x;
        b.maskHi = br.y;
        b.rankBase = br.z;
        const int bit = pwalk_bit(cpk);
        if (COUNT) cnt->cells++;
        if (!pwalk_occupied(b, bit)) return;
        const uint32_t rank = pwalk_rank(b, bit);
        const uint2 range = OCLR_LDG(S.cellRange + rank);
        const uint32_t fm = face != kFaceNone ? OCLR_LDG(S.faceMask + 6 * (size_t)rank + face) : 0xFFFFFFFFu;
        if (COUNT) cnt->cellsNonEmpty++;
        outT = maxD;
        for (uint32_t k = pwalk_next_entry(range.x, range.y, fm, range.x); k < range.y; k = pwalk_next_entry(range.x, range.y, fm, k + 1)) {
            const uint32_t tri = OCLR_LDG(S.cellList + k);
            if (tri == excl) continue;
            float t, ab, ac;
            if (COUNT) cnt->gridCandidates++;
            if (tri_test(S.triGeo + 4 * (size_t)tri, o, r, minD, outT, t, ab, ac)) {
                closest = tri;
                outT = t;
                outAB = ab;
                outAC = ac;
            }
        }
    };
    uint32_t closest = kNoTriangle;
    test_cell(w.cpk, kFaceNone, closest);   // the start cell
    if (closest != kNoTriangle) return closest;
    if (w.cpk == w.epk) {
        outT = maxD;
        return kNoTriangle;
    }
    CoopRay ray;
    ray.o = o;
    ray.r = r;
    ray.c0[0] = pk_get(w.cpk, 0);
    ray.c0[1] = pk_get(w.cpk, 1);
    ray.c0[2] = pk_get(w.cpk, 2);
    ray.epk = w.epk;
    for (;;) {
        uint32_t cells[kCoopLanes];
        int faces[kCoopLanes];
        bool finished;
        const int count = coop_burst_serial(ray, n, planes, cells, faces, finished);
        for (int q = 0; q < count; ++q) {
            test_cell(cells[q], faces[q], closest);
            if (closest != kNoTriangle) return closest;
        }
        if (finished) break;
    }
    outT = maxD;
    return kNoTriangle;
}

// ---- the cooperative walk one level up: bursts over BRICK planes (host form of rt_tail.cuh's wf_tail_brick_kernel) --------------------
// The 32 virtual lanes take the next 11 / 11 / 10 crossings of every 4th plane; each certain crossing enters one 4x4x4 brick.  An empty
// brick that does not hold the ray's end cell has nothing to visit; for any other the exact cell state at the entry is rebuilt with
// pwalk_refine -- the function the two-level walk uses -- and the brick's cells are walked one by one until the walk leaves the brick.
// Cells are tested in (brick, step) order, the first cell with a hit wins, the end cell stops the walk.  The walk starts in the middle
// of a brick: its rest is walked first.  Requires all direction components non-zero and n >= 4.
template <bool COUNT>
OCLR_HD uint32_t grid_trace_coop_bricks(const SceneView& S, const float* planes, f3 o, f3 r, float minD, float maxD, uint32_t excl, float& outT,
                                        float& outAB, float& outAC, Counters* cnt) {
    const int n = S.n, nb = S.nb;
    const float* px = planes;
    const float* py = planes + (n + 1);
    const float* pz = planes + 2 * (n + 1);
    PackedWalk start;
    pwalk_setup(start, n, nb, S.walkTrim, px, py, pz, o, r, minD, maxD);
    if (!start.coarseOk) return grid_trace_packed<COUNT>(S, planes, o, r, minD, maxD, excl, outT, outAB, outAC, cnt);
    if (COUNT) cnt->gridRays++;
    int nbShift = 0;
    while ((1 << nbShift) < nb) ++nbShift;
    const uint32_t epk = start.epk;
    const uint32_t endBrickPk = epk == kPkNone ? (uint32_t)kPkNone : pk_super_of_brick(epk);   // (>> 2 per field: the end cell's brick)
    const int up[3] = {(0 <= r.x) ? 1 : 0, (0 <= r.y) ? 1 : 0, (0 <= r.z) ? 1 : 0};
    const float oc[3] = {o.x, o.y, o.z}, rc[3] = {r.x, r.y, r.z};
    uint32_t closest = kNoTriangle;
    bool stop = false;   // the end cell has been visited
    // the cells of one brick from the state `g` (level 0) on, until the walk leaves the brick / the grid, finds a hit or reaches the end cell
    auto walk_brick = [&](PackedWalk& g, int face) {
        const uint4 br = OCLR_LDG(S.bricks + g.brick);
        g.maskLo = br.x;
        g.maskHi = br.y;
        g.rankBase = br.z;
        for (;;) {
            const int bit = pwalk_bit(g.cpk);
            if (COUNT) cnt->cells++;
            if (pwalk_occupied(g, bit)) {
                const uint32_t rank = pwalk_rank(g, bit);
                const uint2 range = OCLR_LDG(S.cellRange + rank);
                const uint32_t fm = face != kFaceNone ? OCLR_LDG(S.faceMask + 6 * (size_t)rank + face) : 0xFFFFFFFFu;
                if (COUNT) cnt->cellsNonEmpty++;
                outT = maxD;
                for (uint32_t k = pwalk_next_entry(range.x, range.y, fm, range.x); k < range.y; k = pwalk_next_entry(range.x, range.y, fm, k + 1)) {
                    const uint32_t tri = OCLR_LDG(S.cellList + k);
                    if (tri == excl) continue;
                    float t, ab, ac;
                    if (COUNT) cnt->gridCandidates++;
                    if (tri_test(S.triGeo + 4 * (size_t)tri, o, r, minD, outT, t, ab, ac)) {
                        closest = tri;
                        outT = t;
                        outAB = ab;
                        outAC = ac;
                    }
                }
                if (closest != kNoTriangle) return;
            }
            if (g.cpk == epk) {
                stop = true;
                return;
            }
            int axis, upA;
            float tE;
            bool crossed;
            if (!pwalk_step(g, n, S.walkTrim, nbShift, planes, axis, upA, tE, crossed)) return;
            if (crossed) return;
            face = axis * 2 + upA;
        }
    };
    int bc0[3] = {pk_get(start.cpk, 0) >> 2, pk_get(start.cpk, 1) >> 2, pk_get(start.cpk, 2) >> 2};
    {   // the rest of the brick the walk starts in
        PackedWalk g = start;
        walk_brick(g, kFaceNone);
        if (closest != kNoTriangle) return closest;
        if (stop) {
            outT = maxD;
            return kNoTriangle;
        }
    }
    for (;;) {
        float t[3][11];
        int kmax[3];
        for (int a = 0; a < 3; ++a) {
            kmax[a] = up[a] ? (nb - 1 - bc0[a]) : bc0[a];
            for (int k = 0; k < 11; ++k)
                t[a][k] = (k < coop_candidates(a) && k <= kmax[a]) ? (planes[a * (n + 1) + ((bc0[a] + up[a] + (up[a] ? k : -k)) << 2)] - oc[a]) / rc[a]
                                                                  : OCLR_INF;
        }
        int rank[kCoopLanes], cntv[kCoopLanes][3];
        int R = kCoopLanes, exitRank = 1 << 20, endRank = 1 << 20;
        for (int v = 0; v < kCoopLanes; ++v) {
            const int a = v % 3, k = v / 3;
            rank[v] = k;
            for (int b = 0; b < 3; ++b) {
                cntv[v][b] = b == a ? k + 1 : 0;
                if (b == a) continue;
                for (int kk = 0; kk < coop_candidates(b); ++kk) cntv[v][b] += coop_precedes(b, t[b][kk], a, t[a][k]) ? 1 : 0;
                rank[v] += cntv[v][b];
            }
            const bool present = k <= kmax[a];
            if (k == coop_candidates(a) - 1 && kmax[a] >= coop_candidates(a) && rank[v] + 1 < R) R = rank[v] + 1;
            if (present && k == kmax[a] && rank[v] < exitRank) exitRank = rank[v];
            if (present && k < kmax[a]) {
                const uint32_t bpk = pk_make((bc0[0] + (up[0] ? cntv[v][0] : -cntv[v][0])) & kPkMask, (bc0[1] + (up[1] ? cntv[v][1] : -cntv[v][1])) & kPkMask,
                                             (bc0[2] + (up[2] ? cntv[v][2] : -cntv[v][2])) & kPkMask);
                if (bpk == endBrickPk && rank[v] < endRank) endRank = rank[v];
            }
        }
        int limit = R;
        bool finished = false;
        if (exitRank < limit) {
            limit = exitRank;
            finished = true;
        }
        if (endRank < limit) limit = endRank + 1;   // nothing behind the end cell's brick belongs to this burst
        for (int q = 0; q < limit; ++q)
            for (int v = 0; v < kCoopLanes; ++v) {
                if (rank[v] != q) continue;
                const int a = v % 3;
                const int bx = bc0[0] + (up[0] ? cntv[v][0] : -cntv[v][0]), by = bc0[1] + (up[1] ? cntv[v][1] : -cntv[v][1]),
                          bz = bc0[2] + (up[2] ? cntv[v][2] : -cntv[v][2]);
                const int brick = bx + ((by + (bz << nbShift)) << nbShift);
                const uint4 br = OCLR_LDG(S.bricks + brick);
                if (COUNT) cnt->bricksLoaded++;
                if ((br.x | br.y) != 0u || pk_make(bx, by, bz) == endBrickPk) {
                    PackedWalk g;
                    g.o = o;
                    g.r = r;
                    g.epk = epk;
                    g.endBrick = (int)kEndNone;
                    g.coarseOk = true;
                    g.level = 1;
                    g.cpk = pk_make(bx, by, bz);
                    g.tx = (px[(bx + up[0]) << 2] - o.x) / r.x;
                    g.ty = (py[(by + up[1]) << 2] - o.y) / r.y;
                    g.tz = (pz[(bz + up[2]) << 2] - o.z) / r.z;
                    g.brick = brick;
                    pwalk_refine(g, n, nbShift, planes, a, t[a][v / 3]);
                    g.brick = brick;
                    walk_brick(g, kFaceNone);
                    if (closest != kNoTriangle) return closest;
                    if (stop) {
                        outT = maxD;
                        return kNoTriangle;
                    }
                }
                if (q == limit - 1) {
                    bc0[0] = bx;
                    bc0[1] = by;
                    bc0[2] = bz;
                }
            }
        if (finished) break;
    }
    outT = maxD;
    return kNoTriangle;
}

}  // namespace oclr
