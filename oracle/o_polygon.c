/*
 * o_polygon.c -- oracle restatement of Polygon/Polygon.zig:50-107 (palette, render_point,
 * create_polygon) applied to a packed batch.  TEST INFRASTRUCTURE ONLY (see mr_oracle.h).
 *
 * One mr_o_tri arena per thread stands in for the single reusable Triangulation the
 * Polygon module owns (Polygon.zig:18,116); polygons are independent, so running them on
 * several threads does not change any result.
 */
#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>
#include "mr_oracle.h"

int mr_o_hardware_threads(void) {
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n > 0 ? (int)n : 1;
}

/* Polygon.zig:50-57 -- channel order is (hex&0xff, hex>>8&0xff, hex>>16&0xff) / 255.0 */
static void color_from_hex(uint32_t hex, float out[3]) {
    out[0] = (float)(hex & 0xffu) / 255.0f;
    out[1] = (float)((hex >> 8) & 0xffu) / 255.0f;
    out[2] = (float)((hex >> 16) & 0xffu) / 255.0f;
}

void mr_o_palette(float rgb_out[12]) { /* Polygon.zig:66-71 */
    static const uint32_t hex[4] = {0x5e315bu, 0xcfff70u, 0x3ca370u, 0x4b5babu};
    int i;
    for (i = 0; i < 4; ++i) color_from_hex(hex[i], &rgb_out[3 * i]);
}

typedef struct sink { /* RenderContext, Polygon.zig:59-63 */
    unsigned char* base; /* start of this polygon's vertex range */
    uint32_t* ids;       /* optional id trace */
    uint32_t len, cap;   /* vertex_array.items.len / capacity */
    uint32_t dropped;
    float b1x, b1y, b2x, b2y;
    const mr_layout* L;
    float pal[12];
} sink;

/* @min/@max for finite floats; ties (+0 vs -0) keep the accumulator */
static float fmin_acc(float acc, float v) {
    if (mr_o_mutant() == MR_O_MUT_BBOX_TIE_REPLACES) return v <= acc ? v : acc;
    return v < acc ? v : acc;
}
static float fmax_acc(float acc, float v) {
    if (mr_o_mutant() == MR_O_MUT_BBOX_TIE_REPLACES) return v >= acc ? v : acc;
    return v > acc ? v : acc;
}

/* render_point, Polygon.zig:65-79 -- including the bbox rule exactly as written:
 * p1.y = min(p1.x, y) and p2.y = max(p2.x, y) use the *x* accumulators. */
static void render_point(void* vctx, uint32_t id, float x, float y) {
    sink* s = (sink*)vctx;
    s->b1x = fmin_acc(s->b1x, x);
    s->b1y = fmin_acc(mr_o_mutant() == MR_O_MUT_BBOX_OWN_Y ? s->b1y : s->b1x, y);
    s->b2x = fmax_acc(s->b2x, x);
    s->b2y = fmax_acc(mr_o_mutant() == MR_O_MUT_BBOX_OWN_Y ? s->b2y : s->b2x, y);
    if (s->len >= s->cap) { /* appendAssumeCapacity past capacity is UB in the reference */
        s->dropped++;
        return;
    }
    {
        unsigned char* v = s->base + (size_t)s->len * s->L->stride;
        const float* c = &s->pal[3u * ((s->len / 3u) % 4u)];
        float xy[2];
        xy[0] = x;
        xy[1] = y;
        memcpy(v + s->L->attr[0].offset, xy, 8);
        if (s->L->nattr > 1) memcpy(v + s->L->attr[1].offset, c, 12);
        if (s->ids) s->ids[s->len] = id;
        s->len++;
    }
}

typedef struct work {
    const mr_polygon_job* job;
    uint32_t* ids_out;
    uint32_t begin, end;
    mr_o_stats stats;
    int want_stats;
} work;

static void run_range(work* w) {
    const mr_polygon_job* j = w->job;
    mr_o_tri* t = mr_o_tri_new();
    uint32_t i;
    memset(&w->stats, 0, sizeof(w->stats));
    for (i = w->begin; i < w->end; ++i) {
        uint64_t p0 = j->first_point[i] - j->point_base;
        uint32_t n = (uint32_t)(j->first_point[i + 1] - j->first_point[i]);
        uint64_t t0 = j->first_tri[i] - j->tri_base;
        uint32_t cap_tri = (uint32_t)(j->first_tri[i + 1] - j->first_tri[i]);
        const float* xy = j->xy + 2u * p0;
        uint32_t status = MR_POLY_OK;
        sink s;
        uint32_t k;
        memset(&s, 0, sizeof(s));
        s.base = (unsigned char*)j->vtx_out + t0 * 3u * j->layout.stride;
        s.ids = w->ids_out ? w->ids_out + t0 * 3u : NULL;
        s.cap = cap_tri * 3u;
        s.L = &j->layout;
        mr_o_palette(s.pal);
        /* the mapped buffer is zero-initialised (WebGPU); unwritten slots stay zero */
        memset(s.base, 0, (size_t)s.cap * j->layout.stride);
        if (s.ids) memset(s.ids, 0xff, (size_t)s.cap * 4u);
        /* boundary_p1 = boundary_p2 = (0,0)  Polygon.zig:87-88 */

        if (n < 3u) {
            status = MR_POLY_DEGENERATE;
        } else if (n > MR_MAX_POLYGON_POINTS) {
            status = MR_POLY_TOO_LARGE;
        } else {
            const uint32_t mut = mr_o_mutant();
            for (k = 0; k < 2u * n; ++k) {
                if (mut == MR_O_MUT_NONFINITE_X_ONLY && (k & 1u)) continue;
                if (mut == MR_O_MUT_NONFINITE_NAN_ONLY ? isnan(xy[k]) : !isfinite(xy[k])) status = MR_POLY_NONFINITE;
            }
        }
        if (status == MR_POLY_OK) {
            mr_o_unirand rng;
            if (j->offset_prime) {
                mr_o_unirand_explicit(&rng, n, j->offset_prime[2u * i], j->offset_prime[2u * i + 1u]);
            } else {
                uint64_t st = mr_o_rng_state0(j->seed, j->poly_index0 + i);
                mr_o_unirand_seed(&rng, n, &st); /* Triangulation.zig:483 */
            }
            status = mr_o_tri_create_polygon(t, xy, n, rng, &s, render_point,
                                             w->want_stats ? &w->stats : NULL);
            if (status & (MR_POLY_NULL_UNWRAP | MR_POLY_ARENA)) {
                /* abandoned polygon: defined as "nothing emitted" */
                memset(s.base, 0, (size_t)s.cap * j->layout.stride);
                if (s.ids) memset(s.ids, 0xff, (size_t)s.cap * 4u);
                s.len = 0;
                s.dropped = 0;
                s.b1x = s.b1y = s.b2x = s.b2y = 0.0f;
            }
            if (s.dropped) status |= MR_POLY_OVERFLOW;
            if (s.len < s.cap) status |= MR_POLY_UNDERFILL;
        }
        if (j->bbox_out) {
            float* b = j->bbox_out + 4u * (size_t)i;
            b[0] = s.b1x;
            b[1] = s.b1y;
            b[2] = s.b2x;
            b[3] = s.b2y;
        }
        if (j->status_out) j->status_out[i] = status;
        if (j->ntri_out) j->ntri_out[i] = s.len / 3u;
    }
    mr_o_tri_destroy(t);
}

/* Timing helper for bench.py's single-polygon line: Polygon.create_polygon's own call shape -- one reusable
 * Triangulation (Polygon.zig:18,116), one polygon per call, render_point writing GPUVertex into a mapped range --
 * timed inside C so that no Python overhead is counted.  Returns the mean seconds per call. */
#include <time.h>
double mr_o_time_create_polygon(const float* xy, uint32_t n, uint32_t offset, uint32_t prime, uint32_t reps) {
    mr_o_tri* t = mr_o_tri_new();
    mr_layout L;
    unsigned char* buf;
    struct timespec a, b;
    uint32_t r;
    if (n < 3u || reps == 0u) return -1.0;
    memset(&L, 0, sizeof(L));
    L.stride = 32;
    L.nattr = 2;
    L.attr[0].offset = 0;
    L.attr[0].ncomp = 2;
    L.attr[1].offset = 16;
    L.attr[1].ncomp = 3;
    buf = (unsigned char*)calloc((size_t)(n - 2u) * 3u, 32);
    clock_gettime(CLOCK_MONOTONIC, &a);
    for (r = 0; r < reps; ++r) {
        sink s;
        mr_o_unirand rng;
        memset(&s, 0, sizeof(s));
        s.base = buf;
        s.cap = (n - 2u) * 3u;
        s.L = &L;
        mr_o_palette(s.pal);
        mr_o_unirand_explicit(&rng, n, offset, prime);
        (void)mr_o_tri_create_polygon(t, xy, n, rng, &s, render_point, NULL);
    }
    clock_gettime(CLOCK_MONOTONIC, &b);
    free(buf);
    mr_o_tri_destroy(t);
    return ((double)(b.tv_sec - a.tv_sec) + 1e-9 * (double)(b.tv_nsec - a.tv_nsec)) / (double)reps;
}

static void* thread_main(void* p) {
    run_range((work*)p);
    return NULL;
}

int mr_o_polygon_batch(const mr_polygon_job* job, uint32_t* ids_out, int nthreads,
                       mr_o_stats* stats_total) {
    int T, i;
    work* ws;
    pthread_t* th;
    uint64_t total_pts, acc;
    uint32_t cursor;
    if (!job || !job->first_point || !job->first_tri || (!job->xy && job->npoly) ||
        (!job->vtx_out && job->npoly))
        return MR_E_BADARG;
    if (job->layout.nattr < 1 || job->layout.stride < 8) return MR_E_BADARG;
    T = nthreads <= 0 ? mr_o_hardware_threads() : nthreads;
    if ((uint32_t)T > job->npoly) T = job->npoly ? (int)job->npoly : 1;
    ws = (work*)calloc((size_t)T, sizeof(work));
    th = (pthread_t*)calloc((size_t)T, sizeof(pthread_t));
    /* static split by point count */
    total_pts = job->first_point[job->npoly] - job->first_point[0];
    cursor = 0;
    for (i = 0; i < T; ++i) {
        uint64_t target = total_pts * (uint64_t)(i + 1) / (uint64_t)T;
        ws[i].job = job;
        ws[i].ids_out = ids_out;
        ws[i].want_stats = stats_total != NULL;
        ws[i].begin = cursor;
        if (i == T - 1) {
            cursor = job->npoly;
        } else {
            while (cursor < job->npoly) {
                acc = job->first_point[cursor + 1] - job->first_point[0];
                if (acc > target) break;
                ++cursor;
            }
        }
        ws[i].end = cursor;
    }
    if (T == 1) {
        run_range(&ws[0]);
    } else {
        for (i = 0; i < T; ++i) pthread_create(&th[i], NULL, thread_main, &ws[i]);
        for (i = 0; i < T; ++i) pthread_join(th[i], NULL);
    }
    if (stats_total) {
        memset(stats_total, 0, sizeof(*stats_total));
        for (i = 0; i < T; ++i) {
            stats_total->nodes += ws[i].stats.nodes;
            stats_total->sum_stack += ws[i].stats.sum_stack;
            stats_total->descent_steps += ws[i].stats.descent_steps;
            stats_total->mountains += ws[i].stats.mountains;
            stats_total->triangles += ws[i].stats.triangles;
            stats_total->not_acute += ws[i].stats.not_acute;
            stats_total->point_steps += ws[i].stats.point_steps;
            stats_total->select_steps += ws[i].stats.select_steps;
            if (ws[i].stats.max_stack > stats_total->max_stack)
                stats_total->max_stack = ws[i].stats.max_stack;
            if (ws[i].stats.max_mountain > stats_total->max_mountain)
                stats_total->max_mountain = ws[i].stats.max_mountain;
        }
    }
    free(ws);
    free(th);
    return MR_OK;
}
