// rt_query.cuh -- batched ray queries on a resident scene: closest hit (RayIntersectsTriangles, raytrace_opencl.c:324-401) and
// shadow transmittance (the occluder loop of raytrace_opencl.c:608-627) for rays the caller supplies (runtime.cu scene_intersect /
// scene_transmittance, include/oclr_abi.h), and the entry / exit of radiance queries (the frame's path state machine started from caller
// rays, runtime.cu scene_radiance; at the end of this file).
//
// The trace itself is the frame's trace stage, unchanged (wf_setup_kernel + wf_pipe_kernel, rt_trace.cuh): it reads rays through
// queue entries from rayO = (o.xyz, minD), rayD = (d.xyz, maxD) and rayExcl and writes (tri, t, abL, acL) to hit[entry].  The caller's
// arrays already have that layout, so the two kernels here only decide which rays go to the trace stage and what to do with its hits:
//
//   query_screen_kernel    one thread per ray: applies the preconditions of the trace stage (below), writes the results of the rays it
//                          keeps back, and appends the traced rays to the queue in the caller's order (enqueue(), rt_wavefront.cuh).
//   query_transmit_kernel  transmittance only, one thread per ray of the previous round's queue: multiplies att by the blocker's
//                          TRANSPARENCY texel and queues the ray again from minD = t while every component is > 0.
//
// Preconditions.  The trace kernel orders the hits of a ray by the bit pattern of t, which orders like the value only for t > 0, i.e.
// minD >= 0 (rt_trace.cuh, TEST phase).  A ray with minD < 0, a NaN range or a non-finite origin / direction component is therefore
// NOT traced: (kNoTriangle, NaN, 0, 0), transmittance NaN.  A ray with !(minD < maxD) or a zero direction meets no triangle in the
// reference (no t passes minD < t < maxD) and is answered as the ordinary miss without a trace: (kNoTriangle, maxD, 0, 0), att (1,1,1).
#pragma once
#include "rt_trace.cuh"

namespace oclr {

// One batch of caller rays (device pointers, `count` rays).
struct QueryBatch {
    const float4* origin;      // caller's (o.xyz, minD)
    const float4* direction;   // caller's (d.xyz, maxD)
    const uint32_t* excluded;  // caller's excluded triangle per ray, or nullptr (= kNoTriangle)
    uint32_t count;
    uint32_t* excl;            // scratch: excluded triangle per ray, what the setup kernel reads
    float4* hit;               // closest hit: the result array; transmittance: scratch
    float4* rayO;              // transmittance: scratch copy of `origin` whose minD advances along the loop; else nullptr
    float4* att;               // transmittance: (att.rgb, as_float(last blocker)); else nullptr
};

__device__ __forceinline__ bool query_finite(float v) { return fabsf(v) < OCLR_INF; }   // (false for NaN)

// 128 threads per CTA (enqueue() sums four warps).  A grid-stride loop whose trip count is uniform per CTA, so that every thread
// reaches enqueue()'s barriers.
__global__ void __launch_bounds__(128) query_screen_kernel(QueryBatch b, WfState w) {
    for (uint32_t base = blockIdx.x * 128u; base < b.count; base += gridDim.x * 128u) {
        const uint32_t i = base + threadIdx.x;
        bool trace = false;
        if (i < b.count) {
            const float nan = __int_as_float(0x7fc00000);
            const float4 o = b.origin[i], d = b.direction[i];
            const bool usable = 0.f <= o.w && d.w == d.w && query_finite(o.x) && query_finite(o.y) && query_finite(o.z) &&
                                query_finite(d.x) && query_finite(d.y) && query_finite(d.z);
            const bool empty = !(o.w < d.w) || (d.x == 0.f && d.y == 0.f && d.z == 0.f);
            trace = usable && !empty;
            b.excl[i] = b.excluded ? b.excluded[i] : kNoTriangle;
            if (b.att) {
                b.att[i] = usable ? make_float4(1.f, 1.f, 1.f, __uint_as_float(kNoTriangle))
                                  : make_float4(nan, nan, nan, __uint_as_float(kNoTriangle));
                if (trace) b.rayO[i] = o;
            } else if (!trace) {
                b.hit[i] = make_float4(__uint_as_float(kNoTriangle), usable ? d.w : nan, 0.f, 0.f);
            }
        }
        enqueue(w, i, trace, false, false, nullptr);
    }
}

// raytrace_opencl.c:613-625 (the logic kernel's kWfWaitShadow branch, rt_wavefront.cuh): `prevQueue` / `prevCount` = the rays traced
// in the round that just ended; w.queue / w.queueCount = the next round's queue.
__global__ void __launch_bounds__(128) query_transmit_kernel(SceneView S, QueryBatch b, const uint32_t* prevQueue, const uint32_t* prevCount,
                                                             WfState w) {
    const uint32_t count = *prevCount;
    for (uint32_t base = blockIdx.x * 128u; base < count; base += gridDim.x * 128u) {
        const uint32_t k = base + threadIdx.x;
        uint32_t i = 0;
        bool again = false;
        if (k < count) {
            i = prevQueue[k];
            const float4 h = b.hit[i];
            const uint32_t occ = __float_as_uint(h.x);
            if (occ != kNoTriangle) {
                int om;
                float u0, v0, u1, v1, u2, v2;
                load_mat_uv(S, occ, om, u0, v0, u1, v1, u2, v2);
                f3 tr = mk3(0.f, 0.f, 0.f);
                uint2 sz;
                if (channel_present(S, om, kChTransparency, sz)) {
                    const int start = __ldg(S.matStart + kMaterialChannels * om + kChTransparency);
                    tr = table_value(S.textures + start, sz, u0, v0, u1, v1, u2, v2, h.z, h.w);
                }
                float4 a = b.att[i];
                a.x *= tr.x;
                a.y *= tr.y;
                a.z *= tr.z;
                a.w = h.x;
                b.att[i] = a;
                if (0.f < a.x && 0.f < a.y && 0.f < a.z) {
                    b.rayO[i].w = h.y;   // toLightVectorMinLength = mult (:624)
                    again = true;
                }
            }
        }
        enqueue(w, i, again, false, false, nullptr);
    }
}

// ---- radiance along caller rays (runtime.cu scene_radiance) ----------------------------------------------------------------------------
// The reference's pixel-sample loop with the camera segment replaced by the caller's ray.  wf_logic_kernel (rt_wavefront.cuh) already
// runs every NON-camera segment through the trace stage, and only its entry state (kWfNew: jitter draws, camera-list scan) is tied to
// pixels.  So the entry is done here instead: radiance_start_kernel builds ring slot 0 from the caller's ray, seeds the RNG, and queues
// the segment's closest hit exactly as the logic kernel's GO_SEGMENT does; after that trace the unchanged logic kernel resumes the path
// at kWfWaitClosest.  Its launch domain is a 16-wide "image" of the batch (F.cam.width = 16, one row per 16 rays), where its pixel
// and path index are both the ray index and a CTA's 8 x 16 tile is 128 consecutive rays; its camera fields are the caller's (bump
// normals read leftToRight / topToBottom / pixelSizeInv), and the ring-end colours go to the fp32 accumulator F.accum.
enum { kRadianceRowWidth = 16 };

// Caller rays of one radiance batch.
struct RayBatch {
    const float4* origin;          // (o.xyz, minD)
    const float4* direction;       // (d.xyz, +inf)
    const uint32_t* excluded;      // or nullptr (= kNoTriangle)
    uint32_t count;
    unsigned long long indexBase;  // global index of the batch's first ray: sample s of ray i is seeded (indexBase + i) * S + s + 1
};

// 0: traced; 1: meets nothing (a zero direction or minD = +inf: no t passes minD < t); 2: not traced, it breaks a precondition
// (minD < 0 or NaN, maxD != +inf -- ring segments have no far limit --, a non-finite origin or direction component).
enum { kRayTraced = 0, kRayEmpty = 1, kRayScreened = 2 };
__device__ __forceinline__ int radiance_ray_class(float4 o, float4 d) {
    if (!(0.f <= o.w && d.w == OCLR_INF && query_finite(o.x) && query_finite(o.y) && query_finite(o.z) && query_finite(d.x) &&
          query_finite(d.y) && query_finite(d.z)))
        return kRayScreened;
    return (o.w == OCLR_INF || (d.x == 0.f && d.y == 0.f && d.z == 0.f)) ? kRayEmpty : kRayTraced;
}

// One thread per path of the launch domain (w.Q), 128 per CTA (enqueue()).  Ring slot 0 = {o, d, minD, excluded, mul (1,1,1),
// kMaxBounces, cam = false} (raytrace_opencl.c:461-472 with no jitter draws); the path then waits for that segment's closest hit.
template <bool COUNT>
__global__ void __launch_bounds__(128) radiance_start_kernel(RayBatch b, WfState w, uint32_t sampleIdx, uint32_t sampleCount, Counters* gcnt) {
    const uint32_t q = blockIdx.x * 128u + threadIdx.x;
    bool trace = false;
    if (q < w.Q) {
        uint32_t ctl = kWfDone;
        if (q < b.count) {
            const float4 o = b.origin[q], d = b.direction[q];
            if (radiance_ray_class(o, d) == kRayTraced) {
                Segment seg;
                seg.o = mk3(o.x, o.y, o.z);
                seg.v = mk3(d.x, d.y, d.z);
                seg.mul = mk3(1.f, 1.f, 1.f);
                seg.minD = o.w;
                seg.maxB = kMaxBounces;
                seg.excl = b.excluded ? b.excluded[q] : kNoTriangle;
                seg.cam = false;
                ring_store(w, q, 0, seg);
                w.rng[q] = (b.indexBase + q) * (uint64_t)sampleCount + (uint64_t)(sampleIdx + 1u);
                w.colour[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                w.rayO[q] = make_float4(seg.o.x, seg.o.y, seg.o.z, seg.minD);   // (GO_SEGMENT of a non-camera segment)
                w.rayD[q] = make_float4(seg.v.x, seg.v.y, seg.v.z, OCLR_INF);
                w.rayExcl[q] = seg.excl;
                ctl = (uint32_t)kWfWaitClosest | (1u << 8);   // begin 0, end 1
                trace = true;
            }
        }
        w.ctl[q] = ctl;
    }
    if (COUNT) {   // (the logic kernel counts the segments it enters; this one is entered here)
        const unsigned m = __ballot_sync(0xFFFFFFFFu, trace);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(&gcnt->segments, (unsigned long long)__popc(m));
    }
    enqueue(w, q, trace, false, false, nullptr);
}

// Sample 0, after the first trace round: the hit of each ray's own segment (slot 0 of the path's ray slots).
__global__ void radiance_first_hit_kernel(uint32_t count, const float4* hit, uint32_t* firstHit) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < count) firstHit[q] = __float_as_uint(hit[q].x);
}

// rgb4[i] = (sum / S, as_float(first hit)) for traced rays, one IEEE division per channel; (0, 0, 0, kNoTriangle) for rays that meet
// nothing and (NaN, NaN, NaN, kNoTriangle) for rays that break a precondition.
__global__ void radiance_resolve_kernel(RayBatch b, const float4* accum, const uint32_t* firstHit, uint32_t sampleCount, float4* rgb4) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= b.count) return;
    const int cls = radiance_ray_class(b.origin[i], b.direction[i]);
    float4 out;
    if (cls == kRayTraced) {
        const float4 a = accum[i];
        const float n = (float)sampleCount;
        out = make_float4(a.x / n, a.y / n, a.z / n, __uint_as_float(firstHit[i]));
    } else {
        const float v = cls == kRayEmpty ? 0.f : __int_as_float(0x7fc00000);
        out = make_float4(v, v, v, __uint_as_float(kNoTriangle));
    }
    rgb4[i] = out;
}

}  // namespace oclr
