// rt_query.cuh -- batched ray queries on a resident scene: closest hit (RayIntersectsTriangles, raytrace_opencl.c:324-401) and
// shadow transmittance (the occluder loop of raytrace_opencl.c:608-627) for rays the caller supplies (runtime.cu scene_intersect /
// scene_transmittance, include/oclr_abi.h).
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

}  // namespace oclr
