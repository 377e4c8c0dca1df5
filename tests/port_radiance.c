/* tests/port_radiance.c -- TEST INFRASTRUCTURE ONLY: the reference of oclr_scene_radiance on top of the plain-C port of the reference's
 * raytrace path, built by tests/port_radiance.py.
 *
 * The port is compiled into this translation unit as it stands (its walk, texel lookup, surface normal, light sampling and RNG are used
 * unchanged).  shade_ring restates the ring loop of port_pixel_sample (raytrace_port.c:289-414, raytrace_opencl.c:452-725) from a given
 * first segment and also reports what the library reports: the first segment's hit, the bump helper-ray miss that makes the reference's
 * own result undefined (rt_core.h triangle_normal), and segment / shaded-hit / grid-walk counts.  Two doors enter it:
 *   port_shade_frame  with the camera segment, exactly as port_pixel_sample builds it: pins this restatement to the port (the planes
 *                     must equal port_render_rows' bit for bit);
 *   port_shade_rays   with the caller's ray as an ordinary grid segment and no jitter draws, seeded (index_base + i) * S + s + 1.
 */
#include "../oracle/raytrace_port.c"

typedef struct {
    unsigned long long segments, shaded, walks;
} shade_counts;

/* The first bump helper ray of a hit (raytrace_opencl.c:244) does not meet the triangle's plane at 0 < t < inf: the reference then reads
 * uninitialised barycentrics.  Same arithmetic as port_hit_triangle's t. */
static int bump_helper_miss(const port_job* j, uint32_t tri, v3 o, v3 d) {
    const uint32_t* size;
    const uint8_t* image;
    float tt, b2 = 0.f, c2 = 0.f;
    if (!channel(j, j->tri_material[tri], CH_BUMP, &size, &image)) return 0;
    port_hit_triangle(o, V(d.x + j->step_down.x, d.y + j->step_down.y, d.z + j->step_down.z), 0.f, INFINITY, tri_vertex(j, tri, 0),
                      tri_vertex(j, tri, 1), tri_vertex(j, tri, 2), &tt, &b2, &c2);
    return !(0.f < tt && tt < INFINITY);
}

/* The ring loop of port_pixel_sample from ring[0] = `first`; `pixel` is read only by camera segments (their list scan). */
static v3 shade_ring(const port_job* j, segment first, uint32_t pixel, uint64_t* rngp, uint32_t* first_hit, int* undef, shade_counts* cnt) {
    uint64_t rng = *rngp;
    segment ring[RING];
    int head = 0, tail = 1, is_first = 1;
    v3 colour = V(0, 0, 0);
    ring[0] = first;
    for (; head != tail; head = (head + 1) % RING) {
        const segment s = ring[head];
        float t = s.hi, bl = 0.f, cl = 0.f;
        uint32_t tri = NONE;
        cnt->segments++;
        if (s.from_camera) {
            uint32_t i;
            for (i = j->cam_start[pixel]; i < j->cam_end[pixel]; ++i) {
                const uint32_t cand = j->cam_list[i];
                float tt, b, c;
                if (cand != s.skip &&
                    port_hit_triangle(s.o, s.d, s.lo, t, tri_vertex(j, cand, 0), tri_vertex(j, cand, 1), tri_vertex(j, cand, 2), &tt, &b, &c)) {
                    t = tt;
                    tri = cand;
                    bl = b;
                    cl = c;
                }
            }
        } else {
            cnt->walks++;
            tri = port_walk_grid(j, s.o, s.d, s.lo, s.hi, s.skip, &t, &bl, &cl);
        }
        if (is_first) {
            *first_hit = tri;
            is_first = 0;
        }
        if (tri == NONE) continue;
        cnt->shaded++;
        {
            const int mat = j->tri_material[tri];
            const float* uv = j->tri_uv + 6 * (size_t)tri;
            const v3 at = along(s.o, t, s.d);
            const v3 n = port_surface_normal(j, at, s.o, s.d, tri, bl, cl);
            v3 albedo = V(0, 0, 0), glass = albedo, mirror = albedo, glow = albedo;
            v3 lit[2] = {{0.1f, 0.1f, 0.1f}, {0.1f, 0.1f, 0.1f}};
            const uint32_t* size;
            const uint8_t* image;
            uint32_t l;
            int facing;
            v3 shade, w;
            float busy;
            *undef |= bump_helper_miss(j, tri, s.o, s.d);
            if (channel(j, mat, CH_COLOR, &size, &image)) albedo = port_texel(image, size, uv, bl, cl);
            if (channel(j, mat, CH_TRANSPARENCY, &size, &image)) glass = port_texel(image, size, uv, bl, cl);
            if (channel(j, mat, CH_REFLECTION, &size, &image)) mirror = port_texel(image, size, uv, bl, cl);
            if (channel(j, mat, CH_LUMINANCE, &size, &image)) glow = port_texel(image, size, uv, bl, cl);
            for (l = 0; l < j->light_count; ++l) {
                v3 to = V(0, 0, 0), through = V(1, 1, 1);
                float near_ = 0.f, far_ = 0.f;
                const int type = j->light_type[l];
                if (type == 1 || type == 2 || type == 7 || type == 8 || type == 9) {
                    const v3 jitter = port_ball_sample(&rng, j->light_radius[l]);
                    float inv;
                    to = V(jitter.x + j->light_pos[4 * l] - at.x, jitter.y + j->light_pos[4 * l + 1] - at.y, jitter.z + j->light_pos[4 * l + 2] - at.z);
                    far_ = (float)sqrt(dot(to, to));
                    inv = 1.f / far_;
                    to = V(to.x * inv, to.y * inv, to.z * inv);
                } else if (type >= 3 && type <= 6) {
                    const v3 dir = load3(j->light_dir + 4 * l);
                    const float spread = (float)(sin((j->light_radius[l] / 2.f) * 3.14159265f / 180.f) * sqrt(dot(dir, dir)));
                    float inv;
                    to = port_ball_sample(&rng, spread);
                    to = sub(to, dir);
                    inv = 1.f / (float)sqrt(dot(to, to));
                    to = V(to.x * inv, to.y * inv, to.z * inv);
                    far_ = INFINITY;
                }
                if (near_ < far_) {
                    for (;;) {
                        float tt, b, c;
                        v3 pass = V(0, 0, 0);
                        uint32_t blocker;
                        cnt->walks++;
                        blocker = port_walk_grid(j, at, to, near_, far_, tri, &tt, &b, &c);
                        if (blocker == NONE) break;
                        if (channel(j, j->tri_material[blocker], CH_TRANSPARENCY, &size, &image))
                            pass = port_texel(image, size, j->tri_uv + 6 * (size_t)blocker, b, c);
                        through = V(through.x * pass.x, through.y * pass.y, through.z * pass.z);
                        if (!(0.f < through.x && 0.f < through.y && 0.f < through.z)) break;
                        near_ = tt;
                    }
                }
                {
                    const float cosine = dot(n, to);
                    const int side = 0.f <= cosine;
                    const float fall = (float)pow(0.5f, far_ / j->light_half[l]);
                    const float e = (float)fabs(cosine) * (fall == fall ? fall : 1.f);
                    lit[side].x += (1.f - lit[side].x) * through.x * e * j->light_colour[4 * l];
                    lit[side].y += (1.f - lit[side].y) * through.y * e * j->light_colour[4 * l + 1];
                    lit[side].z += (1.f - lit[side].z) * through.z * e * j->light_colour[4 * l + 2];
                }
            }
            colour.x += (1.f - colour.x) * glow.x * s.weight.x;
            colour.y += (1.f - colour.y) * glow.y * s.weight.y;
            colour.z += (1.f - colour.z) * glow.z * s.weight.z;
            facing = dot(n, s.d) <= 0.f;
            shade = lit[facing];
            colour.x += (1.f - colour.x) * s.weight.x * (1.f - glass.x) * albedo.x * shade.x;
            colour.y += (1.f - colour.y) * s.weight.y * (1.f - glass.y) * albedo.y * shade.y;
            colour.z += (1.f - colour.z) * s.weight.z * (1.f - glass.z) * albedo.z * shade.z;
            if (s.depth <= 0) continue;

            busy = (mirror.x + glass.x) > (mirror.y + glass.y) ? (mirror.x + glass.x) : (mirror.y + glass.y);
            busy = busy > (mirror.z + glass.z) ? busy : (mirror.z + glass.z);
            busy = busy < 1.f ? 1.f - busy : 0.f;
            w = V(s.weight.x * albedo.x * busy, s.weight.y * albedo.y * busy, s.weight.z * albedo.z * busy);
            if (3.f / 256.f <= w.x + w.y + w.z) {
                segment* q = &ring[tail];
                v3 dir = port_ball_sample(&rng, 1.f);
                if (facing != (0 <= dot(dir, n))) dir = V(-dir.x, -dir.y, -dir.z);
                q->depth = 0; q->skip = tri; q->o = at; q->d = dir; q->weight = w; q->from_camera = 0; q->lo = 0.f; q->hi = INFINITY;
                tail = (tail + 1) % RING;
                if ((tail + 1) % RING == head) continue;
            }
            w = V(s.weight.x * albedo.x * mirror.x, s.weight.y * albedo.y * mirror.y, s.weight.z * albedo.z * mirror.z);
            if (3.f / 256.f <= w.x + w.y + w.z) {
                segment* q = &ring[tail];
                const float twice = -2.f * dot(n, s.d);
                q->depth = s.depth - 1; q->skip = tri; q->o = at; q->d = V(s.d.x + twice * n.x, s.d.y + twice * n.y, s.d.z + twice * n.z);
                q->weight = w; q->from_camera = 0; q->lo = 0.f; q->hi = INFINITY;
                tail = (tail + 1) % RING;
                if ((tail + 1) % RING == head) continue;
            }
            w = V(s.weight.x * albedo.x * glass.x, s.weight.y * albedo.y * glass.y, s.weight.z * albedo.z * glass.z);
            if (3.f / 256.f <= w.x + w.y + w.z) {
                segment* q = &ring[tail];
                q->depth = s.depth - 1; q->skip = tri; q->o = s.o; q->d = s.d; q->weight = w; q->from_camera = s.from_camera; q->lo = t; q->hi = INFINITY;
                tail = (tail + 1) % RING;
                if ((tail + 1) % RING == head) continue;
            }
        }
    }
    *rngp = rng;
    return colour;
}

/* ---- batch doors, one pthread pool each ----------------------------------------------------------------------------------------------- */
typedef struct {
    const port_job* job;
    size_t count;
    const float *o4, *d4;
    const uint32_t* excl;
    unsigned long long index_base;
    uint32_t samples;
    float* out4;
    uint8_t* flags;
    unsigned long long* counts;   /* segments, shaded hits, grid walks */
    volatile size_t* next;
} shade_batch;

static int finite_(float v) { return fabsf(v) < INFINITY; }

/* Ray i: out4[i] = (sum_s colour_s / (float)S, as_float(first hit of sample 0)); rays the library does not trace get its answers
 * ((NaN, NaN, NaN) or (0, 0, 0), with NONE) and count nothing. */
static void* shade_rays_main(void* arg) {
    shade_batch* b = (shade_batch*)arg;
    shade_counts cnt = {0, 0, 0};
    for (;;) {
        const size_t lo = __sync_fetch_and_add(b->next, (size_t)64), hi = lo + 64 < b->count ? lo + 64 : b->count;
        size_t i;
        if (lo >= b->count) break;
        for (i = lo; i < hi; ++i) {
            const float* o = b->o4 + 4 * i;
            const float* d = b->d4 + 4 * i;
            float* out = b->out4 + 4 * i;
            uint32_t tri0 = NONE;
            int undef = 0;
            if (!(0.f <= o[3] && d[3] == INFINITY && finite_(o[0]) && finite_(o[1]) && finite_(o[2]) && finite_(d[0]) && finite_(d[1]) &&
                  finite_(d[2]))) {
                out[0] = out[1] = out[2] = NAN;
            } else if (o[3] == INFINITY || (d[0] == 0.f && d[1] == 0.f && d[2] == 0.f)) {
                out[0] = out[1] = out[2] = 0.f;
            } else {
                v3 sum = V(0.f, 0.f, 0.f);
                uint32_t s;
                segment seg;
                seg.depth = 12;
                seg.skip = b->excl ? b->excl[i] : NONE;
                seg.o = load3(o);
                seg.d = load3(d);
                seg.weight = V(1, 1, 1);
                seg.from_camera = 0;
                seg.lo = o[3];
                seg.hi = INFINITY;
                for (s = 0; s < b->samples; ++s) {
                    uint64_t rng = (uint64_t)(b->index_base + i) * (uint64_t)b->samples + (uint64_t)(s + 1u);
                    uint32_t hit;
                    const v3 c = shade_ring(b->job, seg, 0, &rng, &hit, &undef, &cnt);
                    if (s == 0) tri0 = hit;
                    sum.x += c.x;
                    sum.y += c.y;
                    sum.z += c.z;
                }
                out[0] = sum.x / (float)b->samples;
                out[1] = sum.y / (float)b->samples;
                out[2] = sum.z / (float)b->samples;
            }
            memcpy(out + 3, &tri0, 4);
            if (b->flags) b->flags[i] = (uint8_t)undef;
        }
    }
    __sync_fetch_and_add(&b->counts[0], cnt.segments);
    __sync_fetch_and_add(&b->counts[1], cnt.shaded);
    __sync_fetch_and_add(&b->counts[2], cnt.walks);
    return 0;
}

static void run_pool(void* (*fn)(void*), void* arg, int threads) {
    pthread_t tid[256];
    int i;
    if (threads > 256) threads = 256;
    if (threads <= 1) { fn(arg); return; }
    for (i = 0; i < threads; ++i) pthread_create(&tid[i], 0, fn, arg);
    for (i = 0; i < threads; ++i) pthread_join(tid[i], 0);
}

void port_shade_rays(const port_job* job, size_t count, const float* o4, const float* d4, const uint32_t* excl, unsigned long long index_base,
                     uint32_t samples, float* out4, uint8_t* flags, unsigned long long* counts, int threads) {
    volatile size_t next = 0;
    shade_batch b;
    b.job = job; b.count = count; b.o4 = o4; b.d4 = d4; b.excl = excl; b.index_base = index_base; b.samples = samples; b.out4 = out4;
    b.flags = flags; b.counts = counts; b.next = &next;
    counts[0] = counts[1] = counts[2] = 0;
    run_pool(shade_rays_main, &b, threads);
}

/* The camera door: every pixel-sample of the job, the camera segment built as port_pixel_sample builds it (raytrace_port.c:273-288), its
 * colour added to the planes with the port's own per-sample conversion. */
typedef struct {
    const port_job* job;
    volatile uint32_t* next_row;
} frame_batch;

static void* shade_frame_main(void* arg) {
    frame_batch* fb = (frame_batch*)arg;
    const port_job* j = fb->job;
    shade_counts cnt = {0, 0, 0};
    for (;;) {
        const uint32_t row = __sync_fetch_and_add(fb->next_row, 1u);
        uint32_t x, s;
        if (row >= j->height) break;
        for (x = 0; x < j->width; ++x) {
            const uint32_t pixel = row * j->width + x;
            for (s = 1; s <= j->samples; ++s) {
                uint64_t rng = (uint64_t)pixel * (uint64_t)j->samples + (uint64_t)s;
                segment seg;
                float k;
                uint32_t hit;
                int undef = 0;
                v3 c;
                seg.depth = 12;
                seg.skip = NONE;
                seg.o = j->eye;
                k = (float)(pixel % j->width) + port_rand(&rng, 0.f, 1.f);
                seg.d = V(j->top_left.x + j->step_right.x * k, j->top_left.y + j->step_right.y * k, j->top_left.z + j->step_right.z * k);
                k = (float)(pixel / j->width) + port_rand(&rng, 0.f, 1.f);
                seg.d = V(seg.d.x + j->step_down.x * k, seg.d.y + j->step_down.y * k, seg.d.z + j->step_down.z * k);
                seg.weight = V(1, 1, 1);
                seg.from_camera = 1;
                seg.lo = 0.f;
                seg.hi = INFINITY;
                c = shade_ring(j, seg, pixel, &rng, &hit, &undef, &cnt);
                if (j->primary_id && s == 1) j->primary_id[pixel] = hit;
                {
                    const float scale = (float)0xFFFF / (float)j->samples;
                    j->out_r[pixel] = add16(j->out_r[pixel], c.x, scale);
                    j->out_g[pixel] = add16(j->out_g[pixel], c.y, scale);
                    j->out_b[pixel] = add16(j->out_b[pixel], c.z, scale);
                }
            }
        }
    }
    return 0;
}

void port_shade_frame(const port_job* job, int threads) {
    volatile uint32_t next = 0;
    frame_batch fb;
    fb.job = job;
    fb.next_row = &next;
    run_pool(shade_frame_main, &fb, threads);
}
