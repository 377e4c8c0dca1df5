/* helpers_kat.c -- test driver (not product code): calls the eight host helpers of source/opencl/raytrace.h:37-44 in the shared
 * library given on the command line -- by value, through include/oclr_abi.h's types -- on a fixed pseudo-random + boundary input
 * set and writes every result to stdout as raw 32-bit words.  tests/test_abi_c.py runs it against libopencl_render_b200.so and
 * compares the stream with the reference build's, stored in tests/golden/reference_values.json. */
#include <dlfcn.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../include/oclr_abi.h"

typedef cl_float (*dot_t)(cl_float3, cl_float3);
typedef cl_float3 (*vec2_t)(cl_float3, cl_float3);
typedef cl_float3 (*vec1_t)(cl_float3);
typedef cl_float (*bindf_t)(cl_float, cl_float, cl_float);
typedef cl_float (*p2l_t)(cl_float3, cl_float3, cl_float3);
typedef cl_bool (*hit_t)(cl_float3, cl_float3, cl_float, cl_float, cl_float3, cl_float3, cl_float3, cl_float*, cl_float*, cl_float*);
typedef cl_int3 (*box_t)(cl_int, cl_float3*, cl_float3);

static uint64_t state = 0x9E3779B97F4A7C15ull;
static float rnd(float lo, float hi) {
    state = state * 6364136223846793005ull + 1442695040888963407ull;
    return lo + (hi - lo) * (float)((state >> 40) & 0xFFFFFF) / 16777216.0f;
}
static cl_float3 v3(float x, float y, float z) {
    cl_float3 v;
    v.s[0] = x; v.s[1] = y; v.s[2] = z; v.s[3] = 0.f;
    return v;
}
static cl_float3 rv(float lo, float hi) { return v3(rnd(lo, hi), rnd(lo, hi), rnd(lo, hi)); }
static void put(const void* p, size_t n) { fwrite(p, 1, n, stdout); }
static void putf(float f) { put(&f, 4); }
static void putv(cl_float3 v) { put(v.s, 12); }

int main(int argc, char** argv) {
    if (argc < 2) return 2;
    void* h = dlopen(argv[1], RTLD_NOW | RTLD_LOCAL);
    if (!h) { fprintf(stderr, "%s\n", dlerror()); return 3; }
    dot_t f_dot = (dot_t)dlsym(h, "dot");
    vec2_t f_cross = (vec2_t)dlsym(h, "cross"), f_vector = (vec2_t)dlsym(h, "vector");
    vec1_t f_normalize = (vec1_t)dlsym(h, "normalize");
    bindf_t f_bindf = (bindf_t)dlsym(h, "bindf");
    p2l_t f_p2l = (p2l_t)dlsym(h, "GetPointToLineSqLen");
    hit_t f_hit = (hit_t)dlsym(h, "RayIntersectsTriangle");
    box_t f_box = (box_t)dlsym(h, "GetBoxAddress");
    if (!f_dot || !f_cross || !f_vector || !f_normalize || !f_bindf || !f_p2l || !f_hit || !f_box) return 4;

    /* split planes of a 16-cell grid, non-uniform like the quantile planes of SceneTriangleList::New */
    enum { N = 16 };
    cl_float3 planes[N + 1];
    float x = -3.f, y = -1.f, z = -2.5f;
    for (int i = 0; i <= N; ++i) {
        planes[i] = v3(x, y, z);
        x += 0.05f + 0.6f * (float)((i * 7) % 5) / 5.f;
        y += 0.02f + 0.3f * (float)((i * 3) % 4) / 4.f;
        z += 0.5f;
    }
    for (int k = 0; k < 20000; ++k) {
        const cl_float3 a = rv(-4.f, 4.f), b = rv(-4.f, 4.f), c = rv(-4.f, 4.f);
        putf(f_dot(a, b));
        putv(f_cross(a, b));
        putv(f_vector(a, b));
        putv(f_normalize(a));
        putf(f_bindf(a.s[0], b.s[0], c.s[0]));
        putf(f_p2l(a, b, c));
        /* ray against triangle: origin and direction chosen so that about a third of the rays hit */
        const cl_float3 o = rv(-6.f, 6.f);
        const cl_float3 centre = v3((a.s[0] + b.s[0] + c.s[0]) / 3.f, (a.s[1] + b.s[1] + c.s[1]) / 3.f, (a.s[2] + b.s[2] + c.s[2]) / 3.f);
        const cl_float3 d = v3(centre.s[0] - o.s[0] + rnd(-2.f, 2.f), centre.s[1] - o.s[1] + rnd(-2.f, 2.f), centre.s[2] - o.s[2] + rnd(-2.f, 2.f));
        float t = -1.f, ab = -1.f, ac = -1.f;
        const float lo = (k & 1) ? 0.f : rnd(0.f, 0.5f), hi = (k & 2) ? INFINITY : rnd(0.5f, 2.f);
        const cl_bool hit = f_hit(o, d, lo, hi, a, b, c, &t, &ab, &ac);
        put(&hit, 4);
        putf(t);                      /* written on every call that reaches the plane test (raytrace_opencl.c:141-142) */
        if (hit) { putf(ab); putf(ac); }
        const cl_float3 pos = (k % 50 == 0) ? planes[(k / 50) % (N + 1)] : rv(-5.f, 8.f);   /* every 50th: exactly on a plane */
        const cl_int3 cell = f_box(N, planes, pos);
        put(cell.s, 12);
    }
    /* boundary cases */
    {
        const cl_float3 a = v3(0, 0, 0), b = v3(1, 0, 0), c = v3(0, 1, 0);
        float t, ab, ac;
        cl_bool r;
        t = ab = ac = -7.f; r = f_hit(v3(0.25f, 0.25f, 1.f), v3(0, 0, -1), 0.f, 1.f, a, b, c, &t, &ab, &ac); put(&r, 4); putf(t);        /* t == max: miss (strict) */
        t = ab = ac = -7.f; r = f_hit(v3(0.25f, 0.25f, 1.f), v3(0, 0, -1), 1.f, 2.f, a, b, c, &t, &ab, &ac); put(&r, 4); putf(t);        /* t == min: miss (strict) */
        t = ab = ac = -7.f; r = f_hit(v3(0.5f, 0.5f, 1.f), v3(0, 0, -1), 0.f, 2.f, a, b, c, &t, &ab, &ac); put(&r, 4); putf(t); putf(ab); putf(ac);   /* abL + acL == 1: hit */
        t = ab = ac = -7.f; r = f_hit(v3(0.f, 0.f, 1.f), v3(0, 0, -1), 0.f, 2.f, a, b, c, &t, &ab, &ac); put(&r, 4); putf(t); putf(ab); putf(ac);     /* corner a */
        t = ab = ac = -7.f; r = f_hit(v3(0.25f, 0.25f, 1.f), v3(1, 0, 0), 0.f, 2.f, a, b, c, &t, &ab, &ac); put(&r, 4);                   /* parallel ray: division by zero */
        t = ab = ac = -7.f; r = f_hit(v3(0.25f, 0.25f, 1.f), v3(0, 0, -1), 0.f, 2.f, a, a, c, &t, &ab, &ac); put(&r, 4);                   /* degenerate triangle: NaN -> miss */
        putf(f_bindf(NAN, 0.f, 1.f)); putf(f_bindf(2.f, 0.f, 1.f)); putf(f_bindf(-2.f, 0.f, 1.f)); putf(f_bindf(0.5f, 1.f, 0.f));
        putv(f_normalize(v3(0, 0, 0)));
        putf(f_p2l(a, a, c));
        const cl_float3 below = v3(-100.f, -100.f, -100.f), above = v3(100.f, 100.f, 100.f);
        cl_int3 cell;
        cell = f_box(N, planes, below); put(cell.s, 12);
        cell = f_box(N, planes, above); put(cell.s, 12);
        cell = f_box(N, planes, planes[0]); put(cell.s, 12);
        cell = f_box(N, planes, planes[N]); put(cell.s, 12);
        cell = f_box(1, planes, planes[3]); put(cell.s, 12);
    }
    return 0;
}
