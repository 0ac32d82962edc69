/* o_earclip.c -- CPU checker of mr_triangulate_earclip: the rules of include/myrenderer_b200.h ("ear clipping"), written
 * as a plain sequential loop.  Independent of the kernel: the orientation is always the exact expansion (no filter) and
 * the blocker search scans the whole ring.  The sink restates render_point (Polygon.zig:65-79); mr_o_emit_ids pins that
 * restatement against the reference oracle.  Test infrastructure only. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/myrenderer_b200.h"

static void two_sum(double a, double b, double* s, double* e) {
    const double x = a + b, bv = x - a, av = x - bv;
    *s = x;
    *e = (a - av) + (b - bv);
}

/* sign of the exact (bx-ax)(cy-ay) - (by-ay)(cx-ax) */
int mr_o_orient_sign(const float* abc) {
    const double ax = abc[0], ay = abc[1], bx = abc[2], by = abc[3], cx = abc[4], cy = abc[5];
    const double t[6] = {ax * by, -(ax * cy), bx * cy, -(bx * ay), cx * ay, -(cx * by)};
    double e[6];
    for (int k = 0; k < 6; ++k) {
        double q = t[k];
        for (int i = 0; i < k; ++i) two_sum(q, e[i], &q, &e[i]);
        e[k] = q;
    }
    for (int i = 5; i >= 0; --i)
        if (e[i] != 0.0) return e[i] > 0.0 ? 1 : -1;
    return 0;
}

static int orient(const float* P, uint32_t a, uint32_t b, uint32_t c) {
    const float t[6] = {P[2 * a], P[2 * a + 1], P[2 * b], P[2 * b + 1], P[2 * c], P[2 * c + 1]};
    return mr_o_orient_sign(t);
}
static int same(const float* P, uint32_t a, uint32_t b) { return P[2 * a] == P[2 * b] && P[2 * a + 1] == P[2 * b + 1]; }

/* ---- sink: Polygon.zig:50-57,65-79 ---- */
static const uint32_t PALETTE[4] = {0x5e315b, 0xcfff70, 0x3ca370, 0x4b5bab};
typedef struct {
    unsigned char* base;
    uint32_t cap_vtx, stride, off_x, off_c, len;
    float c1x, c1y, c2x, c2y;
} Sink;
static float fmin_acc(float acc, float v) { return v < acc ? v : acc; }
static float fmax_acc(float acc, float v) { return v > acc ? v : acc; }
static void sink_point(Sink* s, float x, float y) {
    s->c1x = fmin_acc(s->c1x, x);
    s->c1y = fmin_acc(s->c1x, y);
    s->c2x = fmax_acc(s->c2x, x);
    s->c2y = fmax_acc(s->c2x, y);
    if (s->len < s->cap_vtx) {
        unsigned char* v = s->base + (size_t)s->len * s->stride;
        memset(v, 0, s->stride);
        memcpy(v + s->off_x, &x, 4);
        memcpy(v + s->off_x + 4, &y, 4);
        if (s->off_c != 0xFFFFFFFFu) {
            const uint32_t hex = PALETTE[(s->len / 3u) % 4u];
            const float c[3] = {(float)(hex & 0xff) / 255.0f, (float)((hex >> 8) & 0xff) / 255.0f, (float)((hex >> 16) & 0xff) / 255.0f};
            memcpy(v + s->off_c, c, 12);
        }
    }
    ++s->len;
}

typedef struct {
    const float* P;
    uint32_t n;
    const mr_polygon_job* j;
    Sink sink;
    uint32_t cap_tri, t0_out;
} Poly;

static int poly_begin(const mr_polygon_job* j, uint32_t i, Poly* o) {
    const uint64_t p0 = j->first_point[i] - j->point_base, np = j->first_point[i + 1] - j->first_point[i];
    o->j = j;
    o->P = j->xy + 2 * p0;
    o->n = np > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)np;
    o->cap_tri = (uint32_t)(j->first_tri[i + 1] - j->first_tri[i]);
    o->t0_out = (uint32_t)(j->first_tri[i] - j->tri_base);
    memset(&o->sink, 0, sizeof(o->sink));
    o->sink.base = (unsigned char*)j->vtx_out + (size_t)(j->first_tri[i] - j->tri_base) * 3u * j->layout.stride;
    o->sink.cap_vtx = o->cap_tri * 3u;
    o->sink.stride = j->layout.stride;
    o->sink.off_x = j->layout.attr[0].offset;
    o->sink.off_c = j->layout.nattr > 1 ? j->layout.attr[1].offset : 0xFFFFFFFFu;
    return 0;
}

static void poly_end(const mr_polygon_job* j, uint32_t i, Poly* o, uint32_t status, int emitted) {
    uint32_t ntri = 0;
    float b[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    if (emitted) {
        const uint32_t T = o->sink.len / 3u;
        ntri = T < o->cap_tri ? T : o->cap_tri;
        if (T > o->cap_tri) status |= MR_POLY_OVERFLOW;
        if (T < o->cap_tri) status |= MR_POLY_UNDERFILL;
        b[0] = o->sink.c1x;
        b[1] = o->sink.c1y;
        b[2] = o->sink.c2x;
        b[3] = o->sink.c2y;
    }
    const uint32_t from = emitted ? o->sink.len : 0u;
    if (from < o->sink.cap_vtx) memset(o->sink.base + (size_t)from * o->sink.stride, 0, (size_t)(o->sink.cap_vtx - from) * o->sink.stride);
    if (j->status_out) j->status_out[i] = status;
    if (j->ntri_out) j->ntri_out[i] = ntri;
    if (j->bbox_out) memcpy(j->bbox_out + 4 * (size_t)i, b, 16);
}

/* triangle (a, b, c) of the polygon; ids_out (if not NULL) gets the corner ids in the first_tri range */
static void emit(Poly* o, uint32_t a, uint32_t b, uint32_t c, uint32_t* ids_out) {
    const uint32_t t = o->sink.len / 3u, id[3] = {a, b, c};
    for (int k = 0; k < 3; ++k) {
        if (ids_out && t < o->cap_tri) ids_out[3 * ((size_t)o->t0_out + t) + k] = id[k];
        sink_point(&o->sink, o->P[2 * id[k]], o->P[2 * id[k] + 1]);
    }
}

/* The ring walk of the header on one valid polygon; returns MR_POLY_NO_EAR or 0. */
static uint32_t clip(Poly* o, uint32_t* ids_out, uint32_t* prv, uint32_t* nxt, unsigned char* removed) {
    const float* P = o->P;
    const uint32_t n = o->n;
    uint32_t m = 0;
    for (uint32_t i = 1; i < n; ++i)
        if (P[2 * i + 1] < P[2 * m + 1] || (P[2 * i + 1] == P[2 * m + 1] && P[2 * i] < P[2 * m])) m = i;
    int s = 1;
    uint32_t pm = n, nm = n;
    for (uint32_t d = 1; d < n && pm == n; ++d)
        if (!same(P, (m + n - d) % n, m)) pm = (m + n - d) % n;
    for (uint32_t d = 1; d < n && nm == n; ++d)
        if (!same(P, (m + d) % n, m)) nm = (m + d) % n;
    if (pm < n) {
        const int w = orient(P, pm, m, nm);
        if (w) s = w;
    }
    for (uint32_t i = 0; i < n; ++i) {
        prv[i] = i ? i - 1 : n - 1;
        nxt[i] = i + 1 < n ? i + 1 : 0;
        removed[i] = 0;
    }
    uint32_t status = 0, c = 0, stop = 0;
    for (uint32_t k = n; k > 3; --k) {
        for (;;) {
            const uint32_t p = prv[c], q = nxt[c];
            int ear = same(P, c, p) || same(P, c, q);
            if (!ear && s * orient(P, p, c, q) > 0) {
                ear = 1;
                for (uint32_t r = nxt[q]; r != p && ear; r = nxt[r]) {
                    if (s * orient(P, prv[r], r, nxt[r]) > 0) continue;
                    if (same(P, r, p) || same(P, r, c) || same(P, r, q)) continue;
                    if (s * orient(P, p, c, r) >= 0 && s * orient(P, c, q, r) >= 0 && s * orient(P, q, p, r) >= 0) ear = 0;
                }
            }
            if (ear) break;
            c = nxt[c];
            if (c == stop) {
                status = MR_POLY_NO_EAR;
                break;
            }
        }
        const uint32_t p = prv[c], q = nxt[c];
        if (s > 0) emit(o, p, c, q, ids_out);
        else emit(o, q, c, p, ids_out);
        nxt[p] = q;
        prv[q] = p;
        removed[c] = 1;
        c = nxt[q];
        stop = c;
    }
    if (s > 0) emit(o, prv[c], c, nxt[c], ids_out);
    else emit(o, nxt[c], c, prv[c], ids_out);
    return status;
}

/* Whole batch as mr_triangulate_earclip (host pointers).  ids_out: 3 per triangle of the first_tri ranges, or NULL. */
int mr_o_triangulate_earclip(const mr_polygon_job* j, uint32_t* ids_out) {
    uint32_t* prv = malloc(sizeof(uint32_t) * MR_MAX_POLYGON_POINTS);
    uint32_t* nxt = malloc(sizeof(uint32_t) * MR_MAX_POLYGON_POINTS);
    unsigned char* removed = malloc(MR_MAX_POLYGON_POINTS);
    if (!prv || !nxt || !removed) return MR_E_NOMEM;
    for (uint32_t i = 0; i < j->npoly; ++i) {
        Poly o;
        poly_begin(j, i, &o);
        if (o.n < 3) { poly_end(j, i, &o, MR_POLY_DEGENERATE, 0); continue; }
        if (o.n > MR_MAX_POLYGON_POINTS) { poly_end(j, i, &o, MR_POLY_TOO_LARGE, 0); continue; }
        int finite = 1;
        for (uint32_t k = 0; k < 2 * o.n; ++k) finite = finite && isfinite(o.P[k]);
        if (!finite) { poly_end(j, i, &o, MR_POLY_NONFINITE, 0); continue; }
        const uint32_t st = clip(&o, ids_out, prv, nxt, removed);
        poly_end(j, i, &o, st, 1);
    }
    free(prv);
    free(nxt);
    free(removed);
    return MR_OK;
}

/* The sink alone: polygon i's triangles are given as corner ids (3 per triangle of its first_tri range, 0xFFFFFFFF
 * ends the list early); writes the vertex range and bbox_out[i] as the emit sink does.  Pins the restated sink. */
int mr_o_emit_ids(const mr_polygon_job* j, const uint32_t* ids) {
    for (uint32_t i = 0; i < j->npoly; ++i) {
        Poly o;
        poly_begin(j, i, &o);
        const uint32_t* id = ids + 3 * (size_t)o.t0_out;
        for (uint32_t k = 0; k < 3 * o.cap_tri && id[k] != 0xFFFFFFFFu; ++k) sink_point(&o.sink, o.P[2 * id[k]], o.P[2 * id[k] + 1]);
        if (j->bbox_out) {
            const float b[4] = {o.sink.c1x, o.sink.c1y, o.sink.c2x, o.sink.c2y};
            memcpy(j->bbox_out + 4 * (size_t)i, b, 16);
        }
    }
    return MR_OK;
}
