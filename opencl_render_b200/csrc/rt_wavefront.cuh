// rt_wavefront.cuh -- the production form of the raytrace path on B200: a wavefront pipeline.
//
// Why: ncu on the one-thread-per-pixel kernel (profiles/r01_simple_kernel_cfg2_details.txt) shows 5.65 active threads
// per warp instruction -- ray/triangle tests run with ~3 lanes because at any DDA step only ~9 % of the cells a warp
// looks at hold triangles, and every lane waits for the longest of three consecutive grid walks.  The path is issue-
// bound with the working set in L2 (DRAM traffic 118 MB per frame), so the cure is lane utilisation, not bytes.
//
//   wf_logic_kernel   (this file) one thread per pixel-sample "path".  Runs the reference's per-pixel control flow
//                     (raytrace_opencl.c:452-742: ray-gen, camera-list scan, shading, light sampling, bounce ring, RNG
//                     in the reference's draw order) as a resumable state machine and SUSPENDS at every call of
//                     RayIntersectsTriangles (:530 closest hit of a ring segment, :611 shadow/occluder ray), appending
//                     the path to a ray queue.  Path state lives in HBM as SoA float4 planes: ring (12 slots x 48 B),
//                     shading carry (112 B), ray (36 B), hit (16 B), rng (8 B), colour (16 B).
//   wf_setup_kernel / wf_pipe_kernel   (rt_trace.cuh) drain the queue: the trace stage.
//
// The host enqueues rounds of (logic, setup, trace) ahead until a round finds no path waiting; the arithmetic is rt_core.h /
// rt_walk.h, identical to the simple kernel, so results are bit-identical by construction (tests assert it).
//
// Running one trace ahead.  In the reference a ring segment is finished (:639-722: colour, then the spawn of the diffuse / mirror /
// glass segments) only after the shadow rays of all its lights have returned, and only then is the next segment popped and traced.
// But the spawn depends on nothing the shadow rays return (weights = segment multiplier x texture x reflectance/transparency; the
// bounce direction = the next RNG draws, and the shadow loop :608-627 draws none), and the next segment's closest-hit query depends
// only on the ring.  So when a path suspends for the shadow ray of its LAST light it performs the spawn at once (same RNG position
// as the reference: right after that light's sample draws) and, if the ring then holds a next non-camera segment, queues that
// segment's closest-hit ray in the same round through a second ray slot.  When the shadow result arrives the segment's colour is
// accumulated (the only thing that needed it) and the next segment continues with its hit already there.  A diffuse frame needs
// 2 trace rounds instead of 3 (shadow + bounce | bounce's shadow), a mirror chain of depth d about d instead of 2d; fewer, fuller
// trace launches and one pass less of the logic kernel over the path state.
#pragma once
#include <cuda_runtime.h>

#include <string>

#include "rt_kernels.cuh"

namespace oclr {

enum WfStage { kWfDone = 0, kWfNew = 1, kWfWaitClosest = 2, kWfWaitShadow = 3 };
enum : uint32_t { kCtlSpawned = 1u << 28, kCtlAhead = 1u << 29 };   // ctl = stage | begin << 4 | end << 8 | flags
enum { kCarryParts = 7, kRingParts = 3 };

// Path state (device pointers; Q = paths in the launch domain).  All float4 planes are [part][Q].
struct WfState {
    uint32_t Q;
    uint32_t* ctl;       // stage | begin << 4 | end << 8 | flags
    uint64_t* rng;
    float4* colour;
    float4* ring;        // [slot * 3 + part][Q], slot < ringSlots
    uint32_t ringSlots;  // kRingSize, or 2 for a scene without mirror / glass materials (runtime.cu, Scene::ringSlots)
    float4* carry;       // [part][Q], part < 7; part 6's w = the light a kWfWaitShadow path waits on (any uint32_t lightCount)
    // two ray slots per path, slot-major [slot * Q + path]: slot 0 = the query the path is suspended on, slot 1 = the closest-hit
    // query of the NEXT ring segment traced one round ahead.  Queue entries are these flat indices (the trace stage knows no paths).
    float4* rayO;        // (o.xyz, minD)
    float4* rayD;        // (d.xyz, maxD)
    uint32_t* rayExcl;
    float4* hit;         // (as_float(tri), t, abL, acL)
    uint32_t* queue;     // ray indices waiting for a trace (up to 2 Q)
    uint32_t* queueCount;
    uint32_t* queueCursor;
    uint32_t* roundLog;  // rays queued per round of the current sample (written by the setup kernel): tells the host how many rounds
    uint32_t roundIndex; // the sample really needed, so that the next one enqueues exactly that many ahead
};

struct Segment {
    f3 o, v, mul;
    float minD;
    int maxB;
    uint32_t excl;
    bool cam;
};

__device__ __forceinline__ void ring_store(const WfState& w, uint32_t q, int slot, const Segment& s) {
    if ((uint32_t)slot >= w.ringSlots) __trap();   // (unreachable: the slot count follows from the material table the spawn rules read)
    float4* p = w.ring + (size_t)(slot * kRingParts) * w.Q + q;
    p[0] = make_float4(s.o.x, s.o.y, s.o.z, s.v.x);
    p[w.Q] = make_float4(s.v.y, s.v.z, s.mul.x, s.mul.y);
    p[2 * (size_t)w.Q] = make_float4(s.mul.z, s.minD, __int_as_float((s.maxB & 0xFFFF) | (s.cam ? 0x10000 : 0)), __uint_as_float(s.excl));
}

__device__ __forceinline__ Segment ring_load(const WfState& w, uint32_t q, int slot) {
    const float4* p = w.ring + (size_t)(slot * kRingParts) * w.Q + q;
    const float4 a = p[0], b = p[w.Q], c = p[2 * (size_t)w.Q];
    Segment s;
    s.o = mk3(a.x, a.y, a.z);
    s.v = mk3(a.w, b.x, b.y);
    s.mul = mk3(b.z, b.w, c.x);
    s.minD = c.y;
    const int packed = __float_as_int(c.z);
    s.maxB = (int)(short)(packed & 0xFFFF);
    s.cam = (packed & 0x10000) != 0;
    s.excl = __float_as_uint(c.w);
    return s;
}

// Appends ray index q (slot 0) and / or Q + q (slot 1) to the ray queue.  One atomic per CTA: the 16 k CTAs of a pass all bump the
// same counter, and with one returning atomic per WARP the logic kernel spent 9 % of its stall samples waiting for them (ncu,
// profiles/README.md).  Must be reached by every thread of the CTA (two barriers).
// `finished` / doneCount: the progress counter (pixel-samples finished) rides on the same CTA-level sums.
__device__ __forceinline__ void enqueue(const WfState& w, uint32_t q, bool want0, bool want1, bool finished, unsigned long long* doneCount) {
    __shared__ uint32_t warpCount0[4], warpCount1[4], warpDone[4], ctaBase;
    const unsigned m0 = __ballot_sync(0xFFFFFFFFu, want0), m1 = __ballot_sync(0xFFFFFFFFu, want1);
    const unsigned md = __ballot_sync(0xFFFFFFFFu, finished);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        warpCount0[warp] = (uint32_t)__popc(m0);
        warpCount1[warp] = (uint32_t)__popc(m1);
        warpDone[warp] = (uint32_t)__popc(md);
    }
    __syncthreads();
    const uint32_t total0 = warpCount0[0] + warpCount0[1] + warpCount0[2] + warpCount0[3];
    if (threadIdx.x == 0) {
        const uint32_t total = total0 + warpCount1[0] + warpCount1[1] + warpCount1[2] + warpCount1[3];
        ctaBase = total ? atomicAdd(w.queueCount, total) : 0u;
        const uint32_t done = warpDone[0] + warpDone[1] + warpDone[2] + warpDone[3];
        if (doneCount && done) atomicAdd(doneCount, (unsigned long long)done);
    }
    __syncthreads();
    // the CTA's slot-0 rays (shadow / closest of a 16x8 pixel tile) first, then its slot-1 rays (bounce rays traced ahead): the trace
    // kernel takes consecutive queue entries into one warp, and rays of one kind from one tile walk the grid together
    uint32_t base0 = ctaBase, base1 = ctaBase + total0;
    for (int k = 0; k < warp; ++k) {
        base0 += warpCount0[k];
        base1 += warpCount1[k];
    }
    const unsigned lt = (1u << lane) - 1u;
    if (want0) w.queue[base0 + __popc(m0 & lt)] = q;
    if (want1) w.queue[base1 + __popc(m1 & lt)] = w.Q + q;
}

// ---- logic kernel -----------------------------------------------------------------------------------------------------
// Thread -> path mapping keeps a warp on an 8x4 pixel tile, so queue entries appended by a warp are spatially coherent.
#ifndef OCLR_LOGIC_MIN_CTAS
#define OCLR_LOGIC_MIN_CTAS 5   /* 94 registers, no spills; 6 (80 registers) spills and measures slower */
#endif
template <bool COUNT>
__global__ void __launch_bounds__(128, OCLR_LOGIC_MIN_CTAS) wf_logic_kernel(SceneView S, FrameView F, WfState w, uint32_t sampleIdx, uint32_t startSample,
                                                       const uint32_t* prevCount, Counters* gcnt, int aheadMode, bool cullHidden) {
    // Rounds are enqueued ahead without a host round trip; a round whose predecessor traced no ray has nothing to resume.
    if (prevCount != nullptr && *prevCount == 0u) return;
    if (F.camBad != nullptr && *F.camBad != 0u) return;   // caller's camera lists failed the range check: nothing is read from them
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t x = blockIdx.x * 16 + (warp & 1) * 8 + (lane & 7);
    const uint32_t k = blockIdx.y * 8 + (warp >> 1) * 4 + (lane >> 3);
    const uint32_t y = map_row(F, k);
    const bool valid = x < F.cam.width && y < F.cam.height;
    const uint32_t q = k * F.cam.width + x;
    const uint32_t pixel = valid ? y * F.cam.width + x : 0;
    uint32_t ctl = valid ? (startSample ? (uint32_t)kWfNew : w.ctl[q]) : (uint32_t)kWfDone;
    int stage = (int)(ctl & 7u);
    bool want = false, wantAhead = false, finished = false;
    if (stage != kWfDone) {
        Counters cnt = {};
        const Camera& cam = F.cam;
        int begin = (int)((ctl >> 4) & 15u), end = (int)((ctl >> 8) & 15u);
        uint32_t j = 0;   // the light loop's index: set by GO_SHADE, or from the carry on a shadow resume
        bool spawned = (ctl & kCtlSpawned) != 0u;   // the current segment's spawn (:656-722) was done ahead of its shadow result
        bool ahead = (ctl & kCtlAhead) != 0u;       // slot 1 holds (or is about to receive) the next segment's closest hit
        uint64_t rng;
        f3 colour;
        Segment seg;
        uint32_t hit = kNoTriangle, tri2 = 0;
        float hitT = 0.f, hitAB = 0.f, hitAC = 0.f;
        // shading state
        f3 loc, nrm, tex, transp, refl, lum, att;
        f3 face[2];
        LightRay lr;
        bool undef = false;
        bool first = (stage == kWfNew);
        enum { GO_SEGMENT, GO_SHADE, GO_LIGHTS, GO_FINISH, GO_SPAWN, GO_POP, GO_EXIT } go;
        bool suspendAfterSpawn = false;

        if (stage == kWfNew) {
            rng = (uint64_t)pixel * (uint64_t)F.sampleCount + (uint64_t)(sampleIdx + 1u);
            colour = mk3(0.f, 0.f, 0.f);
            const float fx = (float)(pixel % cam.width), fy = (float)(pixel / cam.width);
            seg.maxB = kMaxBounces;
            seg.excl = kNoTriangle;
            seg.o = mk3(cam.eye);
            seg.v = mk3(cam.eyeToTopLeft);
            float tmp = fx + rand_f(rng, 0.f, 1.f);
            seg.v.x += cam.leftToRight[0] * tmp;
            seg.v.y += cam.leftToRight[1] * tmp;
            seg.v.z += cam.leftToRight[2] * tmp;
            tmp = fy + rand_f(rng, 0.f, 1.f);
            seg.v.x += cam.topToBottom[0] * tmp;
            seg.v.y += cam.topToBottom[1] * tmp;
            seg.v.z += cam.topToBottom[2] * tmp;
            seg.mul = mk3(1.f, 1.f, 1.f);
            seg.cam = true;
            seg.minD = 0.f;
            begin = 0;
            end = 1;
            ring_store(w, q, 0, seg);
            go = GO_SEGMENT;
        } else {
            rng = w.rng[q];
            const float4 c4 = w.colour[q];
            colour = mk3(c4.x, c4.y, c4.z);
            seg = ring_load(w, q, begin);
            const float4 h = w.hit[q];
            hit = __float_as_uint(h.x);
            if (stage == kWfWaitClosest) {
                hitT = h.y;
                hitAB = h.z;
                hitAC = h.w;
                go = (hit == kNoTriangle) ? GO_POP : GO_SHADE;
            } else {  // kWfWaitShadow: the occluder query of light j returned
                const float4* cp = w.carry + q;
                const float4 k0 = cp[0], k1 = cp[w.Q], k2 = cp[2 * (size_t)w.Q], k3 = cp[3 * (size_t)w.Q], k4 = cp[4 * (size_t)w.Q],
                             k5 = cp[5 * (size_t)w.Q], k6 = cp[6 * (size_t)w.Q];
                nrm = mk3(k0.x, k0.y, k0.z);
                hitT = k0.w;
                tex = mk3(k1.x, k1.y, k1.z);
                const uint32_t shaded = __float_as_uint(k1.w);
                j = __float_as_uint(k6.w);
                refl = mk3(k2.x, k2.y, k2.z);
                transp = mk3(k2.w, k3.x, k3.y);
                lum = mk3(k3.z, k3.w, k4.x);
                att = mk3(k4.y, k4.z, k4.w);
                face[0] = mk3(k5.x, k5.y, k5.z);
                face[1] = mk3(k6.x, k6.y, k6.z);
                const float4 ro4 = w.rayO[q], rd4 = w.rayD[q];
                loc = mk3(ro4.x, ro4.y, ro4.z);
                lr.dir = mk3(rd4.x, rd4.y, rd4.z);
                lr.minLen = ro4.w;
                lr.maxLen = rd4.w;
                const uint32_t occ = hit;
                hit = shaded;
                bool again = false;
                if (occ != kNoTriangle) {  // raytrace_opencl.c:613-625
                    int om;
                    float u0, v0, u1, v1, u2, v2;
                    load_mat_uv(S, occ, om, u0, v0, u1, v1, u2, v2);
                    f3 tr = mk3(0.f, 0.f, 0.f);
                    uint2 sz;
                    if (channel_present(S, om, kChTransparency, sz)) {
                        if (COUNT) cnt.occluderLookups++;
                        const int start = __ldg(S.matStart + kMaterialChannels * om + kChTransparency);
                        tr = table_value(S.textures + start, sz, u0, v0, u1, v1, u2, v2, h.z, h.w);
                    }
                    att.x *= tr.x;
                    att.y *= tr.y;
                    att.z *= tr.z;
                    if (0.f < att.x && 0.f < att.y && 0.f < att.z) {
                        again = true;
                        w.rayO[q] = make_float4(loc.x, loc.y, loc.z, h.y);  // toLightVectorMinLength = mult
                        w.carry[4 * (size_t)w.Q + q] = make_float4(lum.z, att.x, att.y, att.z);
                    }
                }
                if (again) {
                    want = true;
                    go = GO_EXIT;
                } else {
                    light_accumulate(S.lights[j], nrm, lr, att, face);
                    ++j;
                    go = GO_LIGHTS;
                }
            }
        }

        while (go != GO_EXIT) {
            if (go == GO_SEGMENT) {
                if (COUNT) cnt.segments++;
                if (seg.cam) {  // raytrace_opencl.c:514-528
                    hit = kNoTriangle;
                    hitT = OCLR_INF;
                    hitAB = hitAC = 0.f;
                    // The scan is a chain of dependent loads (list entry -> triangle record) and a warp waits for its longest list:
                    // entries are fetched two iterations ahead and the next triangle's record is pulled into L1 meanwhile.
                    const uint32_t e = __ldg(F.camEnd + pixel);
                    uint32_t i = __ldg(F.camStart + pixel);
                    uint32_t tri = i < e ? __ldg(F.camList + i) : 0u;
                    uint32_t tri1 = i + 1u < e ? __ldg(F.camList + i + 1u) : 0u;
                    for (; i < e; ++i, tri = tri1, tri1 = tri2) {
                        tri2 = i + 2u < e ? __ldg(F.camList + i + 2u) : 0u;
                        if (i + 1u < e) asm volatile("prefetch.global.L1 [%0];" ::"l"(S.triGeo + 4 * (size_t)tri1));
                        if (seg.excl != tri) {
                            float t, ab, ac;
                            if (COUNT) cnt.primCandidates++;
                            if (tri_test(S.triGeo + 4 * (size_t)tri, seg.o, seg.v, seg.minD, hitT, t, ab, ac)) {
                                hitT = t;
                                hit = tri;
                                hitAB = ab;
                                hitAC = ac;
                            }
                        }
                    }
                    if (first && F.idOut && sampleIdx == 0) F.idOut[pixel] = hit;
                    first = false;
                    go = (hit == kNoTriangle) ? GO_POP : GO_SHADE;
                } else {
                    w.rayO[q] = make_float4(seg.o.x, seg.o.y, seg.o.z, seg.minD);
                    w.rayD[q] = make_float4(seg.v.x, seg.v.y, seg.v.z, OCLR_INF);
                    w.rayExcl[q] = seg.excl;
                    stage = kWfWaitClosest;
                    want = true;
                    go = GO_EXIT;
                }
            } else if (go == GO_SHADE) {  // :532-561
                if (COUNT) cnt.shadedHits++;
                const TriShade ts = load_shade(S, hit);
                tex = transp = refl = lum = mk3(0.f, 0.f, 0.f);
                face[0] = face[1] = mk3(0.1f, 0.1f, 0.1f);
                loc = mk3(seg.o.x + hitT * seg.v.x, seg.o.y + hitT * seg.v.y, seg.o.z + hitT * seg.v.z);
                nrm = triangle_normal(S, cam, ts, loc, seg.o, seg.v, hitAB, hitAC, undef);
                shade_channels(S, ts, hitAB, hitAC, tex, transp, refl, lum);
                j = 0;
                go = GO_LIGHTS;
            } else if (go == GO_LIGHTS) {  // :563-637, suspended at :611
                // Hidden-side cull: light_accumulate adds light j to face[0 <= dot(nrm, dir)], and GO_FINISH reads only face[front]
                // (nothing else reads face).  A light on the other side changes no output bit, so its shadow ray, the re-traces through
                // transparent occluders and the accumulate are skipped; light_ray still runs, so the RNG draws stay in the reference's
                // order.  Same expressions as light_accumulate and GO_FINISH: NaN, -0 and d == 0 fall on the same side in both.  The
                // counting instantiation keeps every shadow ray: its counters describe the reference's work.
                // hiddenFace = 1 - front, or 2 (no face) without the cull.  A face index rather than a flag tested inside the loop: a
                // loop-invariant test lets the compiler clone the whole light loop (+7 calls, 24 B of spills, config 3 0.8 % slower).
                const int hiddenFace = (!COUNT && cullHidden) ? 1 - (int)(dot3(nrm, seg.v) <= 0.f) : 2;
                go = GO_FINISH;
                while (j < S.lightCount) {
                    att = mk3(1.f, 1.f, 1.f);
                    light_ray(S.lights[j], loc, rng, lr);
                    if ((int)(0.f <= dot3(nrm, lr.dir)) == hiddenFace) {
                        ++j;
                        continue;
                    }
                    if (lr.minLen < lr.maxLen) {
                        w.rayO[q] = make_float4(loc.x, loc.y, loc.z, lr.minLen);
                        w.rayD[q] = make_float4(lr.dir.x, lr.dir.y, lr.dir.z, lr.maxLen);
                        w.rayExcl[q] = hit;
                        float4* cp = w.carry + q;
                        cp[0] = make_float4(nrm.x, nrm.y, nrm.z, hitT);
                        cp[w.Q] = make_float4(tex.x, tex.y, tex.z, __uint_as_float(hit));
                        cp[2 * (size_t)w.Q] = make_float4(refl.x, refl.y, refl.z, transp.x);
                        cp[3 * (size_t)w.Q] = make_float4(transp.y, transp.z, lum.x, lum.y);
                        cp[4 * (size_t)w.Q] = make_float4(lum.z, att.x, att.y, att.z);
                        cp[5 * (size_t)w.Q] = make_float4(face[0].x, face[0].y, face[0].z, 0.f);
                        cp[6 * (size_t)w.Q] = make_float4(face[1].x, face[1].y, face[1].z, __uint_as_float(j));
                        stage = kWfWaitShadow;
                        want = true;
                        // last light: spawn now and trace the next segment one round ahead (aheadMode 2: every segment; 1: all but
                        // camera segments -- on a large diffuse frame the primary hits gain nothing from it, see runtime.cu)
                        if (!spawned && j + 1u == S.lightCount && (aheadMode == 2 || (aheadMode == 1 && !seg.cam))) {
                            suspendAfterSpawn = true;
                            go = GO_SPAWN;
                            break;
                        }
                        go = GO_EXIT;
                        break;
                    }
                    light_accumulate(S.lights[j], nrm, lr, att, face);
                    ++j;
                }
            } else if (go == GO_FINISH) {  // :639-722
                const f3 rm = seg.mul, rv = seg.v;
                colour.x += (1.f - colour.x) * lum.x * rm.x;
                colour.y += (1.f - colour.y) * lum.y * rm.y;
                colour.z += (1.f - colour.z) * lum.z * rm.z;
                const int front = (int)(dot3(nrm, rv) <= 0.f);
                const f3 light = face[front];
                colour.x += (1.f - colour.x) * rm.x * (1.f - transp.x) * tex.x * light.x;
                colour.y += (1.f - colour.y) * rm.y * (1.f - transp.y) * tex.y * light.y;
                colour.z += (1.f - colour.z) * rm.z * (1.f - transp.z) * tex.z * light.z;
                go = spawned ? GO_POP : GO_SPAWN;
                spawned = false;
            } else if (go == GO_SPAWN) {
                // :656-722 -- the segments the current hit spawns.  Reads nothing a shadow ray returns, so it may run before the
                // segment's colour is accumulated ("running one trace ahead" at the top of this file); reached either from GO_FINISH
                // (the reference's order) or from GO_LIGHTS right before the path suspends on its last light's shadow ray.
                if (seg.maxB > 0) {
                    const f3 rm = seg.mul, rv = seg.v;
                    const int front = (int)(dot3(nrm, rv) <= 0.f);
                    float total = (refl.x + transp.x) > (refl.y + transp.y) ? (refl.x + transp.x) : (refl.y + transp.y);
                    total = total > (refl.z + transp.z) ? total : (refl.z + transp.z);
                    f3 diffuse = mk3(0.f, 0.f, 0.f);
                    if (total < 1.f) diffuse = mk3(1.f - total, 1.f - total, 1.f - total);
                    bool full = false;
                    Segment ns;
                    ns.excl = hit;
                    ns.mul = mk3(rm.x * tex.x * diffuse.x, rm.y * tex.y * diffuse.y, rm.z * tex.z * diffuse.z);
                    if (3.f / 256.f <= ns.mul.x + ns.mul.y + ns.mul.z) {  // diffuse bounce
                        f3 d = sphere_point(rng, 1.f);
                        if (front != (int)(0 <= dot3(d, nrm))) d = mk3(-d.x, -d.y, -d.z);
                        ns.maxB = 0;
                        ns.o = loc;
                        ns.v = d;
                        ns.cam = false;
                        ns.minD = 0.f;
                        ring_store(w, q, end, ns);
                        end = (end + 1) % kRingSize;
                        full = ((end + 1) % kRingSize == begin);
                    }
                    if (!full) {
                        ns.mul = mk3(rm.x * tex.x * refl.x, rm.y * tex.y * refl.y, rm.z * tex.z * refl.z);
                        if (3.f / 256.f <= ns.mul.x + ns.mul.y + ns.mul.z) {  // mirror
                            const float tmp = -2.f * dot3(nrm, rv);
                            ns.maxB = seg.maxB - 1;
                            ns.o = loc;
                            ns.v = mk3(rv.x + tmp * nrm.x, rv.y + tmp * nrm.y, rv.z + tmp * nrm.z);
                            ns.cam = false;
                            ns.minD = 0.f;
                            ring_store(w, q, end, ns);
                            end = (end + 1) % kRingSize;
                            full = ((end + 1) % kRingSize == begin);
                        }
                    }
                    if (!full) {
                        ns.mul = mk3(rm.x * tex.x * transp.x, rm.y * tex.y * transp.y, rm.z * tex.z * transp.z);
                        if (3.f / 256.f <= ns.mul.x + ns.mul.y + ns.mul.z) {  // glass
                            ns.maxB = seg.maxB - 1;
                            ns.o = seg.o;
                            ns.v = rv;
                            ns.cam = seg.cam;
                            ns.minD = hitT;
                            ring_store(w, q, end, ns);
                            end = (end + 1) % kRingSize;
                        }
                    }
                }
                if (!suspendAfterSpawn) {
                    spawned = false;
                    go = GO_POP;
                } else {
                    spawned = true;
                    const int nb = (begin + 1) % kRingSize;
                    if (nb != end) {
                        const Segment nx = ring_load(w, q, nb);
                        if (!nx.cam) {   // (a camera segment is resolved from the pixel's list by this kernel: nothing to trace)
                            w.rayO[w.Q + q] = make_float4(nx.o.x, nx.o.y, nx.o.z, nx.minD);
                            w.rayD[w.Q + q] = make_float4(nx.v.x, nx.v.y, nx.v.z, OCLR_INF);
                            w.rayExcl[w.Q + q] = nx.excl;
                            ahead = true;
                            wantAhead = true;
                        }
                    }
                    go = GO_EXIT;
                }
            } else {  // GO_POP
                begin = (begin + 1) % kRingSize;
                if (begin == end) {
                    if (F.accum) {   // float accumulation: no per-sample truncation (resolved by resolve_accum_kernel)
                        float4 a = sampleIdx ? F.accum[pixel] : make_float4(0.f, 0.f, 0.f, 0.f);
                        a.x += colour.x;
                        a.y += colour.y;
                        a.z += colour.z;
                        a.w += 1.f;
                        F.accum[pixel] = a;
                    } else {
                        const float scale = 65535.f / (float)F.sampleCount;
                        const uint16_t pr = sampleIdx ? F.outR[pixel] : (uint16_t)0;
                        const uint16_t pg = sampleIdx ? F.outG[pixel] : (uint16_t)0;
                        const uint16_t pb = sampleIdx ? F.outB[pixel] : (uint16_t)0;
                        F.outR[pixel] = accumulate16(pr, colour.x, scale);
                        F.outG[pixel] = accumulate16(pg, colour.y, scale);
                        F.outB[pixel] = accumulate16(pb, colour.z, scale);
                    }
                    finished = true;
                    stage = kWfDone;
                    go = GO_EXIT;
                } else {
                    seg = ring_load(w, q, begin);
                    if (ahead) {   // this segment's closest hit was traced one round ahead (slot 1)
                        ahead = false;
                        const float4 h2 = w.hit[w.Q + q];
                        hit = __float_as_uint(h2.x);
                        hitT = h2.y;
                        hitAB = h2.z;
                        hitAC = h2.w;
                        if (COUNT) cnt.segments++;
                        go = (hit == kNoTriangle) ? GO_POP : GO_SHADE;
                    } else {
                        stage = kWfWaitClosest;  // provisional; GO_SEGMENT decides
                        go = GO_SEGMENT;
                    }
                }
            }
        }
        if (undef && F.flagOut) F.flagOut[pixel] = 1;
        if (stage != kWfDone) {
            w.rng[q] = rng;
            w.colour[q] = make_float4(colour.x, colour.y, colour.z, 0.f);
        }
        w.ctl[q] = (uint32_t)stage | ((uint32_t)begin << 4) | ((uint32_t)end << 8) | (spawned ? kCtlSpawned : 0u) | (ahead ? kCtlAhead : 0u);
        if (COUNT) flush_counters(cnt, gcnt);
    }
    enqueue(w, q, want, wantAhead, finished, F.doneCount);
}

// Planes from the float accumulator: out = (int)(sum * 65535 / samples so far), the reference's conversion (:726-741) applied once
// to the mean instead of once per sample.  One thread per pixel of the launch domain.
__global__ void resolve_accum_kernel(FrameView F) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t y = map_row(F, blockIdx.y);
    if (x >= F.cam.width || y >= F.cam.height) return;
    const uint32_t pixel = y * F.cam.width + x;
    const float4 a = F.accum[pixel];
    const float scale = 65535.f / (a.w > 0.f ? a.w : 1.f);
    F.outR[pixel] = accumulate16(0, a.x, scale);
    F.outG[pixel] = accumulate16(0, a.y, scale);
    F.outB[pixel] = accumulate16(0, a.z, scale);
}

}  // namespace oclr
