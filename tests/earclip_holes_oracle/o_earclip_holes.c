/* o_earclip_holes.c -- CPU checker of mr_triangulate_earclip_holes: the bridge rule of include/myrenderer_b200.h written
 * as a plain sequential loop (whole-ring scans, the crossing predicate always by its exact expansion), followed by the
 * ear-clipping checker's own ring walk on the merged ring.  That checker is compiled into this library unchanged (its
 * source is included below), so both entry points clip with one restatement of the rules.  Test infrastructure only. */
#include "../earclip_oracle/o_earclip.c"

static void two_prod(double a, double b, double* p, double* e) {
    *p = a * b;
    *e = fma(a, b, -*p);
}

/* sign of the exact (b2y - my) * O(a1, b1, a2) + (my - a2y) * O(a1, b1, b2); q = (a1x, a1y, b1x, b1y, a2x, a2y, b2x, b2y, my).
 * Each of the 24 terms is a product of three floats: the first two multiply exactly in double, the third by two_prod. */
int mr_o_crossing_sign(const float* q) {
    const double a1x = q[0], a1y = q[1], b1x = q[2], b1y = q[3], a2x = q[4], a2y = q[5], b2x = q[6], b2y = q[7], my = q[8];
    const double o1[6] = {a1x * b1y, -(a1x * a2y), b1x * a2y, -(b1x * a1y), a2x * a1y, -(a2x * b1y)};
    const double o2[6] = {a1x * b1y, -(a1x * b2y), b1x * b2y, -(b1x * a1y), b2x * a1y, -(b2x * b1y)};
    const double f1[2] = {b2y, -my}, f2[2] = {my, -a2y};
    double t[48];
    int n = 0;
    for (int k = 0; k < 6; ++k)
        for (int i = 0; i < 2; ++i) {
            two_prod(o1[k], f1[i], &t[n], &t[n + 1]);
            n += 2;
            two_prod(o2[k], f2[i], &t[n], &t[n + 1]);
            n += 2;
        }
    double e[48];
    for (int k = 0; k < 48; ++k) {
        double v = t[k];
        for (int i = 0; i < k; ++i) two_sum(v, e[i], &v, &e[i]);
        e[k] = v;
    }
    for (int i = 47; i >= 0; --i)
        if (e[i] != 0.0) return e[i] > 0.0 ? 1 : -1;
    return 0;
}

static int cross_sign(const float* P, uint32_t a1, uint32_t b1, uint32_t a2, uint32_t b2, float my) {
    const float q[9] = {P[2 * a1], P[2 * a1 + 1], P[2 * b1], P[2 * b1 + 1], P[2 * a2], P[2 * a2 + 1], P[2 * b2], P[2 * b2 + 1], my};
    return mr_o_crossing_sign(q);
}
static int cmp(float a, float b) { return (a > b) - (a < b); }

/* winding of the ring of ids id[0..n-1] by the lowest-vertex rule */
static int ring_winding(const float* P, const uint32_t* id, uint32_t n) {
    uint32_t m = 0;
    for (uint32_t i = 1; i < n; ++i) {
        const float y = P[2 * id[i] + 1], ym = P[2 * id[m] + 1];
        if (y < ym || (y == ym && P[2 * id[i]] < P[2 * id[m]])) m = i;
    }
    uint32_t pm = n, nm = n;
    for (uint32_t d = 1; d < n && pm == n; ++d)
        if (!same(P, id[(m + n - d) % n], id[m])) pm = (m + n - d) % n;
    for (uint32_t d = 1; d < n && nm == n; ++d)
        if (!same(P, id[(m + d) % n], id[m])) nm = (m + d) % n;
    if (pm == n) return 1;
    const int w = orient(P, id[pm], id[m], id[nm]);
    return w ? w : 1;
}

/* Position of the current ring C[0..L-1] (point ids into P) that hole vertex M is bridged to; *bad = no crossing edge. */
static uint32_t bridge_to(const float* P, const uint32_t* C, uint32_t L, uint32_t M, int s, int* bad) {
    const float my = P[2 * M + 1];
    uint32_t e = L;
    for (uint32_t k = 0; k < L; ++k) {
        const uint32_t a = C[k], b = C[(k + 1) % L];
        const float ay = P[2 * a + 1], by = P[2 * b + 1];
        if (s * cmp(by, ay) <= 0 || !(fminf(ay, by) <= my && my <= fmaxf(ay, by))) continue;
        if (s * orient(P, a, b, M) < 0) continue;
        if (e == L || cross_sign(P, C[e], C[(e + 1) % L], a, b, my) > 0) e = k;
    }
    *bad = e == L;
    if (e == L) return 0;
    const uint32_t a = C[e], b = C[(e + 1) % L];
    uint32_t t;
    if (P[2 * a + 1] == my) {
        t = e;
    } else if (P[2 * b + 1] == my) {
        t = (e + 1) % L;
    } else {
        t = P[2 * a] >= P[2 * b] ? e : (e + 1) % L;
        const int u = P[2 * C[t] + 1] > my ? 1 : -1;
        const uint32_t pt = C[t];
        for (uint32_t r = 0; r < L; ++r) {
            const uint32_t v = C[r];
            if (same(P, v, M) || s * orient(P, C[(r + L - 1) % L], v, C[(r + 1) % L]) > 0) continue;
            if (u * cmp(P[2 * v + 1], my) < 0 || s * orient(P, a, b, v) < 0 || u * orient(P, M, pt, v) > 0) continue;
            const int w = u * orient(P, M, v, C[t]);
            if (w > 0 || (w == 0 && P[2 * v] < P[2 * C[t]])) t = r;
        }
    }
    const uint32_t T = C[t];
    for (uint32_t k = 0; k < L; ++k) {
        if (!same(P, C[k], T)) continue;
        const uint32_t pp = C[(k + L - 1) % L], pn = C[(k + 1) % L];
        const int o1 = s * orient(P, pp, T, M), o2 = s * orient(P, T, pn, M);
        if (s * orient(P, pp, T, pn) > 0 ? (o1 > 0 && o2 > 0) : (o1 > 0 || o2 > 0)) return k;
    }
    return t;
}

/* Whole batch as mr_triangulate_earclip_holes (host pointers).  ids_out: 3 per triangle of the first_tri ranges (point
 * ids relative to the polygon's first point), or NULL. */
int mr_o_triangulate_earclip_holes(const mr_polygon_job* j, const mr_polygon_rings* rg, uint32_t* ids_out) {
    const uint32_t CAP = MR_MAX_POLYGON_POINTS;
    uint32_t* prv = malloc(sizeof(uint32_t) * CAP);
    uint32_t* nxt = malloc(sizeof(uint32_t) * CAP);
    uint32_t* ring = malloc(sizeof(uint32_t) * CAP);
    uint32_t* hid = malloc(sizeof(uint32_t) * CAP);
    uint32_t* hs = malloc(sizeof(uint32_t) * (CAP + 1));
    float* Q = malloc(sizeof(float) * 2 * CAP);
    unsigned char* removed = malloc(CAP);
    if (!prv || !nxt || !ring || !hid || !hs || !Q || !removed) return MR_E_NOMEM;
    for (uint32_t i = 0; i < j->npoly; ++i) {
        Poly o;
        poly_begin(j, i, &o);
        const uint64_t N = j->first_point[i + 1] - j->first_point[i];
        const uint64_t r0 = rg->first_ring[i], R = rg->first_ring[i + 1] - r0;
        if (R == 0 || R > N) { poly_end(j, i, &o, MR_POLY_DEGENERATE, 0); continue; }
        const uint32_t H = (uint32_t)(R - 1);
        if (N + 2 * (uint64_t)H > CAP) { poly_end(j, i, &o, MR_POLY_TOO_LARGE, 0); continue; }
        /* hs[h] = start of ring h relative to the polygon, hs[H+1] = N */
        int ok = rg->ring_start[r0 - rg->ring_base] == j->first_point[i];
        for (uint32_t h = 0; h <= H && ok; ++h) {
            const uint64_t a = rg->ring_start[r0 + h - rg->ring_base] - j->first_point[i];
            const uint64_t b = h < H ? rg->ring_start[r0 + h + 1 - rg->ring_base] - j->first_point[i] : N;
            ok = a < b && b - a >= 3 && b <= N;
            hs[h] = (uint32_t)a;
        }
        if (!ok) { poly_end(j, i, &o, MR_POLY_DEGENERATE, 0); continue; }
        hs[H + 1] = (uint32_t)N;
        int finite = 1;
        for (uint64_t k = 0; k < 2 * N; ++k) finite = finite && isfinite(o.P[k]);
        if (!finite) { poly_end(j, i, &o, MR_POLY_NONFINITE, 0); continue; }
        const float* P = o.P;
        uint32_t L = hs[1], status = 0;
        for (uint32_t k = 0; k < L; ++k) {
            ring[k] = k;
            hid[k] = k;
        }
        const int s = ring_winding(P, ring, L);
        /* hole order: decreasing (x, y) of M, equal M in hole order (insertion sort, stable) */
        uint32_t order[MR_MAX_POLYGON_POINTS / 3 + 1], mv[MR_MAX_POLYGON_POINTS / 3 + 1];
        for (uint32_t h = 1; h <= H; ++h) {
            uint32_t m = hs[h];
            for (uint32_t k = hs[h] + 1; k < hs[h + 1]; ++k)
                if (P[2 * k] > P[2 * m] || (P[2 * k] == P[2 * m] && P[2 * k + 1] > P[2 * m + 1])) m = k;
            mv[h - 1] = m;
            uint32_t at = h - 1;
            while (at > 0) {
                const uint32_t pm = mv[order[at - 1]];
                if (P[2 * m] > P[2 * pm] || (P[2 * m] == P[2 * pm] && P[2 * m + 1] > P[2 * pm + 1])) {
                    order[at] = order[at - 1];
                    --at;
                } else {
                    break;
                }
            }
            order[at] = h - 1;
        }
        for (uint32_t z = 0; z < H; ++z) {
            const uint32_t h = order[z] + 1, M = mv[h - 1], a = hs[h], n = hs[h + 1] - hs[h];
            int bad = 0;
            const uint32_t k = bridge_to(P, ring, L, M, s, &bad);
            if (bad) status |= MR_POLY_BAD_HOLE;
            for (uint32_t v = 0; v < n; ++v) hid[v] = a + v;
            const int rev = ring_winding(P, hid, n) == s;
            memmove(ring + k + 1 + n + 2, ring + k + 1, sizeof(uint32_t) * (L - k - 1));
            const uint32_t jm = M - a;
            for (uint32_t d = 0; d < n; ++d) ring[k + 1 + d] = a + (rev ? (jm + n - d) % n : (jm + d) % n);
            ring[k + 1 + n] = M;
            ring[k + 2 + n] = ring[k];
            L += n + 2;
        }
        for (uint32_t k = 0; k < L; ++k) {
            Q[2 * k] = P[2 * ring[k]];
            Q[2 * k + 1] = P[2 * ring[k] + 1];
        }
        o.P = Q;
        o.n = L;
        status |= clip(&o, ids_out, prv, nxt, removed);
        if (ids_out) { /* clip wrote merged-ring positions: turn them into point ids */
            const uint32_t T = L - 2 < o.cap_tri ? L - 2 : o.cap_tri;
            for (size_t k = 3 * (size_t)o.t0_out; k < 3 * ((size_t)o.t0_out + T); ++k) ids_out[k] = ring[ids_out[k]];
        }
        poly_end(j, i, &o, status, 1);
    }
    free(prv);
    free(nxt);
    free(ring);
    free(hid);
    free(hs);
    free(Q);
    free(removed);
    return MR_OK;
}
