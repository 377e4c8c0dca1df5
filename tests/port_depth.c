/* tests/port_depth.c -- TEST INFRASTRUCTURE ONLY: how deep the paths of a scene go, measured on the plain-C port of the reference's
 * raytrace path, built by tests/port_depth.py.
 *
 * depth_ring is shade_ring of tests/port_radiance.c (the ring loop of raytrace_port.c port_pixel_sample, raytrace_opencl.c:452-725) with
 * three more counts: the spawns after which the ring was full (11 live segments: the rule that skips the hit's remaining spawns), and the
 * longest pixel-sample's (or ray-sample's) segment count and sequential grid walks -- its non-camera closest hits plus every shadow-loop
 * step, i.e. the trace rounds the wavefront pipeline needs for it.  The colours it returns are pinned to the port and to port_radiance by
 * tests/test_deep_paths_host.py, so the counts are those of the reference's own control flow.  Two doors, as in port_radiance.c: every
 * pixel-sample of a frame from the camera, and caller rays as ring slot 0 (seeded (index_base + i) * S + s + 1).
 */
#include "port_radiance.c"

typedef struct {
    unsigned long long segments, walks, ring_full, longest_segments, longest_walks;
} depth_counts;

static v3 depth_ring(const port_job* j, segment first, uint32_t pixel, uint64_t* rngp, uint32_t* first_hit, depth_counts* cnt) {
    uint64_t rng = *rngp;
    const unsigned long long segments0 = cnt->segments, walks0 = cnt->walks;
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
                if ((tail + 1) % RING == head) { cnt->ring_full++; continue; }
            }
            w = V(s.weight.x * albedo.x * mirror.x, s.weight.y * albedo.y * mirror.y, s.weight.z * albedo.z * mirror.z);
            if (3.f / 256.f <= w.x + w.y + w.z) {
                segment* q = &ring[tail];
                const float twice = -2.f * dot(n, s.d);
                q->depth = s.depth - 1; q->skip = tri; q->o = at; q->d = V(s.d.x + twice * n.x, s.d.y + twice * n.y, s.d.z + twice * n.z);
                q->weight = w; q->from_camera = 0; q->lo = 0.f; q->hi = INFINITY;
                tail = (tail + 1) % RING;
                if ((tail + 1) % RING == head) { cnt->ring_full++; continue; }
            }
            w = V(s.weight.x * albedo.x * glass.x, s.weight.y * albedo.y * glass.y, s.weight.z * albedo.z * glass.z);
            if (3.f / 256.f <= w.x + w.y + w.z) {
                segment* q = &ring[tail];
                q->depth = s.depth - 1; q->skip = tri; q->o = s.o; q->d = s.d; q->weight = w; q->from_camera = s.from_camera; q->lo = t; q->hi = INFINITY;
                tail = (tail + 1) % RING;
                if ((tail + 1) % RING == head) { cnt->ring_full++; continue; }
            }
        }
    }
    if (cnt->segments - segments0 > cnt->longest_segments) cnt->longest_segments = cnt->segments - segments0;
    if (cnt->walks - walks0 > cnt->longest_walks) cnt->longest_walks = cnt->walks - walks0;
    *rngp = rng;
    return colour;
}

/* counts[5] += / max= one thread's counts */
static void depth_merge(unsigned long long* dst, const depth_counts* c) {
    __sync_fetch_and_add(&dst[0], c->segments);
    __sync_fetch_and_add(&dst[1], c->walks);
    __sync_fetch_and_add(&dst[2], c->ring_full);
    for (;;) {
        const unsigned long long m = dst[3];
        if (c->longest_segments <= m || __sync_bool_compare_and_swap(&dst[3], m, c->longest_segments)) break;
    }
    for (;;) {
        const unsigned long long m = dst[4];
        if (c->longest_walks <= m || __sync_bool_compare_and_swap(&dst[4], m, c->longest_walks)) break;
    }
}

/* ---- the camera door: planes and primary ids as port_shade_frame writes them ------------------------------------------------------------ */
typedef struct {
    const port_job* job;
    volatile uint32_t* next_row;
    unsigned long long* counts;
} depth_frame_batch;

static void* depth_frame_main(void* arg) {
    depth_frame_batch* fb = (depth_frame_batch*)arg;
    const port_job* j = fb->job;
    depth_counts cnt = {0, 0, 0, 0, 0};
    for (;;) {
        const uint32_t row = __sync_fetch_and_add(fb->next_row, 1u);
        uint32_t x, s;
        if (row >= j->height) break;
        for (x = 0; x < j->width; ++x) {
            const uint32_t pixel = row * j->width + x;
            for (s = 1; s <= j->samples; ++s) {
                uint64_t rng = (uint64_t)pixel * (uint64_t)j->samples + (uint64_t)s;
                const float scale = (float)0xFFFF / (float)j->samples;
                segment seg;
                float k;
                uint32_t hit;
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
                c = depth_ring(j, seg, pixel, &rng, &hit, &cnt);
                if (j->primary_id && s == 1) j->primary_id[pixel] = hit;
                j->out_r[pixel] = add16(j->out_r[pixel], c.x, scale);
                j->out_g[pixel] = add16(j->out_g[pixel], c.y, scale);
                j->out_b[pixel] = add16(j->out_b[pixel], c.z, scale);
            }
        }
    }
    depth_merge(fb->counts, &cnt);
    return 0;
}

void port_depth_frame(const port_job* job, unsigned long long* counts, int threads) {
    volatile uint32_t next = 0;
    depth_frame_batch fb;
    fb.job = job;
    fb.next_row = &next;
    fb.counts = counts;
    memset(counts, 0, 5 * sizeof(*counts));
    run_pool(depth_frame_main, &fb, threads);
}

/* ---- the ray door: traced rays only (0 <= minD < inf, maxD = +inf, finite non-zero directions); out4 as port_shade_rays writes it ---- */
typedef struct {
    const port_job* job;
    size_t count;
    const float *o4, *d4;
    unsigned long long index_base;
    uint32_t samples;
    float* out4;
    unsigned long long* counts;
    volatile size_t* next;
} depth_ray_batch;

static void* depth_rays_main(void* arg) {
    depth_ray_batch* b = (depth_ray_batch*)arg;
    depth_counts cnt = {0, 0, 0, 0, 0};
    for (;;) {
        const size_t i = __sync_fetch_and_add(b->next, (size_t)1);
        v3 sum = V(0.f, 0.f, 0.f);
        uint32_t s, tri0 = NONE;
        segment seg;
        float* out;
        if (i >= b->count) break;
        out = b->out4 + 4 * i;
        seg.depth = 12;
        seg.skip = NONE;
        seg.o = load3(b->o4 + 4 * i);
        seg.d = load3(b->d4 + 4 * i);
        seg.weight = V(1, 1, 1);
        seg.from_camera = 0;
        seg.lo = b->o4[4 * i + 3];
        seg.hi = INFINITY;
        for (s = 0; s < b->samples; ++s) {
            uint64_t rng = (uint64_t)(b->index_base + i) * (uint64_t)b->samples + (uint64_t)(s + 1u);
            uint32_t hit;
            const v3 c = depth_ring(b->job, seg, 0, &rng, &hit, &cnt);
            if (s == 0) tri0 = hit;
            sum.x += c.x;
            sum.y += c.y;
            sum.z += c.z;
        }
        out[0] = sum.x / (float)b->samples;
        out[1] = sum.y / (float)b->samples;
        out[2] = sum.z / (float)b->samples;
        memcpy(out + 3, &tri0, 4);
    }
    depth_merge(b->counts, &cnt);
    return 0;
}

void port_depth_rays(const port_job* job, size_t count, const float* o4, const float* d4, unsigned long long index_base, uint32_t samples,
                     float* out4, unsigned long long* counts, int threads) {
    volatile size_t next = 0;
    depth_ray_batch b;
    b.job = job; b.count = count; b.o4 = o4; b.d4 = d4; b.index_base = index_base; b.samples = samples; b.out4 = out4; b.counts = counts;
    b.next = &next;
    memset(counts, 0, 5 * sizeof(*counts));
    run_pool(depth_rays_main, &b, threads);
}
