/* tests/abi_caller.c -- TEST INFRASTRUCTURE.  Compiled against include/oclr_abi.h (OUR declaration of the boundary): calls
 * RaytraceAll with by-value cl_uint2 / cl_float3 unions carrying vector members, the reference's layout and x86-64 calling
 * convention, the way render.cpp calls it. */
#include "../include/oclr_abi.h"

/* RaytraceAll with every size argument filled in and a caller-chosen computation type: what render.cpp:1314 passes.  Linked against
 * the PRODUCT library by tests/test_gpu_parity.py (computation type 1 = the first CUDA device). */
cl_uint abi_call_by_value_full(cl_uint computationType, const cl_uint* dim, const float* eye, const float* tl, const float* lr, const float* tb,
                               float psi, cl_uint* camStart, cl_uint* camEnd, cl_uint* camList, ptrdiff_t camListSize, cl_uint sampleCount,
                               cl_uint vertexCount, cl_float3* vertex, cl_uint triangleCount, cl_int3* triIdx, cl_int* triMat,
                               cl_float2* triUv, cl_float3* triNormal, cl_int axesDivCount, cl_float3* boxMin, cl_uint* gridStart,
                               cl_uint* gridList, cl_uint materialCount, cl_uint2* matSize, cl_int* matStart, cl_uint texturesSize,
                               cl_uchar3* textures, cl_uint lightCount, cl_int* lightType, cl_float3* lightPos, cl_float3* lightDir,
                               cl_float3* lightColour, cl_float* lightRadius, cl_float* lightHalf, cl_ushort* r, cl_ushort* g, cl_ushort* b) {
    cl_uint2 d;
    cl_float3 e, t, l, bb;
    int i;
    d.s[0] = dim[0];
    d.s[1] = dim[1];
    for (i = 0; i < 3; ++i) {
        e.s[i] = eye[i];
        t.s[i] = tl[i];
        l.s[i] = lr[i];
        bb.s[i] = tb[i];
    }
    e.s[3] = t.s[3] = l.s[3] = bb.s[3] = 0.f;
    return RaytraceAll(computationType, d, e, t, l, bb, psi, camStart, camEnd, camList, camListSize, sampleCount, vertexCount, vertex,
                       triangleCount, triIdx, triMat, triUv, triNormal, axesDivCount, boxMin, gridStart, gridList, materialCount, matSize,
                       matStart, texturesSize, textures, lightCount, lightType, lightPos, lightDir, lightColour, lightRadius, lightHalf, r, g,
                       b);
}

/* by-value helper round trip through OUR exported helpers (abi_helpers.c) is covered from Python via this door */
float abi_dot_by_value(const float* a, const float* b) {
    cl_float3 x, y;
    int i;
    for (i = 0; i < 4; ++i) {
        x.s[i] = i < 3 ? a[i] : 0.f;
        y.s[i] = i < 3 ? b[i] : 0.f;
    }
    return dot(x, y);
}
