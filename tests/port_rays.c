/* tests/port_rays.c -- TEST INFRASTRUCTURE ONLY: the reference of the batched ray queries (oclr_scene_intersect /
 * oclr_scene_transmittance) on top of the plain-C port of the reference's raytrace path, built by tests/port_rays.py.
 *
 * The port is compiled into this translation unit as it stands, so its walk (port_walk_grid, raytrace_opencl.c:324-401) and its texel
 * lookup are used unchanged.  port_transmit restates the occluder loop of the light loop, raytrace_opencl.c:608-627 -- the port's own
 * copy is inline in port_pixel_sample (raytrace_port.c:352-364); this one differs only in reporting the last blocker it met.
 */
#include "../oracle/raytrace_port.c"

uint32_t port_transmit(const port_job* j, v3 at, v3 to, float near_, float far_, uint32_t skip, v3* through) {
    uint32_t last = NONE;
    if (near_ < far_) {
        for (;;) {
            float tt, b, c;
            v3 pass = V(0, 0, 0);
            const uint32_t* size;
            const uint8_t* image;
            const uint32_t blocker = port_walk_grid(j, at, to, near_, far_, skip, &tt, &b, &c);
            if (blocker == NONE) break;
            last = blocker;
            if (channel(j, j->tri_material[blocker], CH_TRANSPARENCY, &size, &image))
                pass = port_texel(image, size, j->tri_uv + 6 * (size_t)blocker, b, c);
            *through = V(through->x * pass.x, through->y * pass.y, through->z * pass.z);
            if (!(0.f < through->x && 0.f < through->y && 0.f < through->z)) break;
            near_ = tt;
        }
    }
    return last;
}

/* Ray i = origin o4[4i..4i+2], minD o4[4i+3], direction d4[4i..4i+2], maxD d4[4i+3], excluded triangle excl[i] (excl NULL: none).
 *   port_walk_rays:     out4[i] = (as_float(port_walk_grid), t, abL, acL); abL / acL are 0 on a miss.
 *   port_transmit_rays: out4[i] = (att.rgb, as_float(port_transmit)). */
typedef struct {
    const port_job* job;
    size_t count;
    const float *o4, *d4;
    const uint32_t* excl;
    float* out4;
    int transmit;
    volatile size_t* next;
} port_ray_batch;

static void* port_rays_main(void* arg) {
    port_ray_batch* b = (port_ray_batch*)arg;
    for (;;) {
        const size_t first = __sync_fetch_and_add(b->next, (size_t)256), last = first + 256 < b->count ? first + 256 : b->count;
        size_t i;
        if (first >= b->count) break;
        for (i = first; i < last; ++i) {
            const float* o = b->o4 + 4 * i;
            const float* d = b->d4 + 4 * i;
            const uint32_t skip = b->excl ? b->excl[i] : NONE;
            float* out = b->out4 + 4 * i;
            uint32_t tri;
            if (b->transmit) {
                v3 through = V(1, 1, 1);
                tri = port_transmit(b->job, load3(o), load3(d), o[3], d[3], skip, &through);
                out[0] = through.x; out[1] = through.y; out[2] = through.z;
                memcpy(out + 3, &tri, 4);
            } else {
                float t = 0.f, bl = 0.f, cl = 0.f;
                tri = port_walk_grid(b->job, load3(o), load3(d), o[3], d[3], skip, &t, &bl, &cl);
                memcpy(out, &tri, 4);
                out[1] = t; out[2] = bl; out[3] = cl;
            }
        }
    }
    return 0;
}

static void port_rays(const port_job* job, size_t count, const float* o4, const float* d4, const uint32_t* excl, float* out4, int transmit,
                      int threads) {
    volatile size_t next = 0;
    port_ray_batch b;
    pthread_t tid[256];
    int i;
    b.job = job; b.count = count; b.o4 = o4; b.d4 = d4; b.excl = excl; b.out4 = out4; b.transmit = transmit; b.next = &next;
    if (threads > 256) threads = 256;
    if (threads <= 1) { port_rays_main(&b); return; }
    for (i = 0; i < threads; ++i) pthread_create(&tid[i], 0, port_rays_main, &b);
    for (i = 0; i < threads; ++i) pthread_join(tid[i], 0);
}

void port_walk_rays(const port_job* job, size_t count, const float* o4, const float* d4, const uint32_t* excl, float* out4, int threads) {
    port_rays(job, count, o4, d4, excl, out4, 0, threads);
}

void port_transmit_rays(const port_job* job, size_t count, const float* o4, const float* d4, const uint32_t* excl, float* out4, int threads) {
    port_rays(job, count, o4, d4, excl, out4, 1, threads);
}
