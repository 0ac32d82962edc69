// earclip.cu -- ear-clipping triangulation (mr_triangulate_earclip) for sm_100a.
//
// The rules are those of the header, restated by tests/earclip_oracle/o_earclip.c and tests/_earclip.py.  One warp per
// polygon; the ring (points, prev/next links, a flag byte per point) and the list of vertices that can block an ear
// live in shared memory, 15 bytes per point.  Polygons are pulled largest first from four size classes.  The ring walk
// is warp-uniform (every lane holds the same cursor); the blocker scan of a candidate runs lane-parallel over the list
// of non-convex vertices, behind an exact bounding-box reject.  mr_triangulate_earclip_holes first bridges a polygon's
// holes into its outer ring in the same workspace (merge_holes) and then runs the same ring walk on the merged ring.
// mr_triangulate_earclip_indexed runs the same walks in instantiations of their own that also (or, without a vertex
// buffer, only) store each triangle's three point indices.
#include "common.cuh"

namespace {
#include "polygon_sink.cuh"

constexpr int EC_CLASSES = 4;
__host__ __device__ constexpr uint32_t ec_nmax(int c) { return c == 0 ? 64u : c == 1 ? 256u : c == 2 ? 1024u : MR_MAX_POLYGON_POINTS; }
// warps per block: the 4096-point class fits three 61 KB workspaces per SM
__host__ __device__ constexpr int ec_wpb(int c) { return c == EC_CLASSES - 1 ? 3 : 4; }
// per warp: xy 8 B | prev 2 B | next 2 B | blocker list 2 B [| position -> point id map 2 B] | flags 1 B, per point (15
// and 17 times nmax are multiples of 16).  Only the indexed holes instantiation keeps the map: there the clip reuses the
// blocker list that merge_holes built the merged ring's point ids in; in every other one position = id.
__host__ __device__ constexpr size_t ec_ws_bytes(uint32_t nmax, bool map = false) { return (size_t)nmax * (map ? 17u : 15u); }

constexpr uint8_t F_NONCONVEX = 1;  // s * orient(prev, v, next) <= 0 in the current ring
constexpr uint8_t F_REMOVED = 2;    // clipped
constexpr uint8_t F_LISTED = 4;     // present in the blocker list (entries are never removed; the scan skips dead ones)

struct EcArgs {
    const float* xy;
    const uint64_t* first_point;
    uint64_t point_base;
    unsigned char* vtx_out;
    const uint64_t* first_tri;
    uint64_t tri_base;
    float* bbox_out;
    uint32_t* status_out;
    uint32_t* ntri_out;
    uint32_t stride, off_x, off_c;  // off_c == 0xFFFFFFFF: no colour attribute
    int fast32;                     // stride 32, offsets {0,16} in either order, 32B-aligned base
    const uint32_t* order;          // polygon ids, largest first
    const uint32_t* cursor;         // cursor[b] = polygons of size >= b (mr_polygon_size_sort)
    uint32_t* queue_head;           // EC_CLASSES
};

// ring description of mr_triangulate_earclip_holes (device pointers)
struct RingArgs {
    const uint64_t* first_ring;
    uint64_t ring_base;
    const uint64_t* ring_start;
};

// index output of mr_triangulate_earclip_indexed (device pointer)
struct IdxArgs {
    uint32_t* idx_out;
    uint64_t index_base;
};

// ---- exact orientation ---------------------------------------------------------------------------------------
__device__ __forceinline__ void two_sum(double a, double b, double& s, double& e) {
    s = __dadd_rn(a, b);
    const double bv = __dsub_rn(s, a);
    const double av = __dsub_rn(s, bv);
    e = __dadd_rn(__dsub_rn(a, av), __dsub_rn(b, bv));
}

// Sign of ax*by - ax*cy + bx*cy - bx*ay + cx*ay - cx*by: each product of two floats is exact in double; the six are
// summed into a non-overlapping expansion (grow-expansion, increasing magnitude) whose last nonzero component has the
// sign of the exact sum.
__device__ __noinline__ int orient_exact(float ax, float ay, float bx, float by, float cx, float cy) {
    const double t[6] = {__dmul_rn(ax, by), -__dmul_rn(ax, cy), __dmul_rn(bx, cy),
                         -__dmul_rn(bx, ay), __dmul_rn(cx, ay), -__dmul_rn(cx, by)};
    double e[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        double q = t[k];
#pragma unroll
        for (int i = 0; i < k; ++i) two_sum(q, e[i], q, e[i]);
        e[k] = q;
    }
#pragma unroll
    for (int i = 5; i >= 0; --i)
        if (e[i] != 0.0) return e[i] > 0.0 ? 1 : -1;
    return 0;
}

// Exact sign of (b-a) x (c-a).  Filter: the determinant in double with Shewchuk's orient2d bound (the differences of two
// floats and their products neither overflow nor underflow in double, so the bound holds); both products zero means the
// exact value is zero.
__device__ __forceinline__ int orient(float2 a, float2 b, float2 c) {
    const double l = __dmul_rn(__dsub_rn(a.x, c.x), __dsub_rn(b.y, c.y));
    const double r = __dmul_rn(__dsub_rn(a.y, c.y), __dsub_rn(b.x, c.x));
    const double det = __dsub_rn(l, r);
    const double bound = (3.0 + 16.0 * 0x1p-53) * 0x1p-53 * __dadd_rn(fabs(l), fabs(r));
    if (det > bound) return 1;
    if (-det > bound) return -1;
    if (l == 0.0 && r == 0.0) return 0;
    return orient_exact(a.x, a.y, b.x, b.y, c.x, c.y);
}

__device__ __forceinline__ bool same_pt(float2 a, float2 b) { return a.x == b.x && a.y == b.y; }
__device__ __forceinline__ bool below_yx(float2 a, float2 b) { return a.y < b.y || (a.y == b.y && a.x < b.x); }

struct Ring {
    MR_SPAN(float2) P;
    MR_SPAN(uint16_t) prv;
    MR_SPAN(uint16_t) nxt;
    MR_SPAN(uint16_t) lst;
    MR_SPAN(uint8_t) flg;
};

// nearest ring neighbour of m (dir -1: predecessors, +1: successors) whose point differs from P[m]; n when there is none
__device__ uint32_t distinct_neighbour(const Ring& R, uint32_t m, uint32_t n, int dir, uint32_t lane) {
    const float2 pm = R.P[m];
    for (uint32_t base = 1; base < n; base += 32) {
        const uint32_t d = base + lane;
        const uint32_t i = dir < 0 ? (m + n - d % n) % n : (m + d) % n;
        const uint32_t hit = __ballot_sync(0xFFFFFFFFu, d < n && !same_pt(R.P[i], pm));
        if (hit) {
            const uint32_t dd = base + __ffs(hit) - 1u;
            return dir < 0 ? (m + n - dd) % n : (m + dd) % n;
        }
    }
    return n;
}

// c is an ear of the current ring (rules (a) and (b) of the header); warp-uniform result
__device__ bool is_ear(const Ring& R, uint32_t p, uint32_t c, uint32_t q, int s, uint32_t nlist, uint32_t lane) {
    const float2 Pp = R.P[p], Pc = R.P[c], Pq = R.P[q];
    if (same_pt(Pc, Pp) || same_pt(Pc, Pq)) return true;
    if (R.flg[c] & F_NONCONVEX) return false;
    const float x0 = fminf(fminf(Pp.x, Pc.x), Pq.x), x1 = fmaxf(fmaxf(Pp.x, Pc.x), Pq.x);
    const float y0 = fminf(fminf(Pp.y, Pc.y), Pq.y), y1 = fmaxf(fmaxf(Pp.y, Pc.y), Pq.y);
    for (uint32_t base = 0; base < nlist; base += 32) {
        const uint32_t j = base + lane;
        bool blocks = false;
        if (j < nlist) {
            const uint32_t r = R.lst[j];
            if ((R.flg[r] & (F_NONCONVEX | F_REMOVED)) == F_NONCONVEX && r != p && r != c && r != q) {
                const float2 Pr = R.P[r];
                if (Pr.x >= x0 && Pr.x <= x1 && Pr.y >= y0 && Pr.y <= y1 && !same_pt(Pr, Pp) && !same_pt(Pr, Pc) &&
                    !same_pt(Pr, Pq))
                    blocks = s * orient(Pp, Pc, Pr) >= 0 && s * orient(Pc, Pq, Pr) >= 0 && s * orient(Pq, Pp, Pr) >= 0;
            }
        }
        if (__any_sync(0xFFFFFFFFu, blocks)) return false;
    }
    return true;
}

// What the indexed instantiations add to Emit: the polygon's index range, the index of its point 0, the position ->
// point id map of a merged ring (null: position = id) and whether there is a vertex buffer (warp-uniform).  Empty
// otherwise, so that Emit<false> is the plain emitter.
template <bool IDX>
struct EmitIdx {
    static constexpr bool vtx = true;
};
template <>
struct EmitIdx<true> {
    uint32_t* idx;
    uint32_t ibase;
    MR_SPAN(uint16_t) map;
    bool vtx;
};

template <bool IDX>
struct Emit : EmitIdx<IDX> {
    Sink sink;
    uint32_t cap_tri, t;
    float mn, mx, lasty;
    // triangle (x0, x1, x2) as the next one of the polygon; lanes 0..2 store its vertices and indices
    __device__ __forceinline__ void tri(const Ring& R, uint32_t x0, uint32_t x1, uint32_t x2, uint32_t lane) {
        const float2 v0 = R.P[x0], v1 = R.P[x1], v2 = R.P[x2];
        mn = fmin_acc(fmin_acc(fmin_acc(mn, v0.x), v1.x), v2.x);
        mx = fmax_acc(fmax_acc(fmax_acc(mx, v0.x), v1.x), v2.x);
        lasty = v2.y;
        if (t < cap_tri && lane < 3u) {
            if (this->vtx) sink.write(3u * t + lane, lane == 0u ? v0 : lane == 1u ? v1 : v2);
            if constexpr (IDX) {
                const uint32_t x = lane == 0u ? x0 : lane == 1u ? x1 : x2;
                this->idx[3u * t + lane] = this->ibase + (MR_SPAN_IS_NULL(this->map) ? x : (uint32_t)this->map[x]);
            }
        }
        ++t;
    }
    // zero the range from vertex / index k0 on
    __device__ __forceinline__ void zero_from(uint32_t k0, uint32_t lane) {
        if (this->vtx) sink.zero(k0, sink.cap_vtx, lane);
        if constexpr (IDX)
            for (uint32_t k = k0 + lane; k < sink.cap_vtx; k += 32) this->idx[k] = 0u;
    }
};

// Runs the ring walk of one valid polygon (3 <= n, finite points loaded into R.P); returns MR_POLY_NO_EAR or 0.
template <class EM>
__device__ uint32_t clip_ring(const Ring& R, uint32_t n, EM& em, uint32_t lane) {
    // winding s from the lowest point (first index smallest in (y, x)) and its nearest distinct neighbours
    uint32_t m = 0;
    for (uint32_t i = lane; i < n; i += 32)
        if (i == lane ? true : below_yx(R.P[i], R.P[m])) m = i;
    if (lane >= n) m = 0;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const uint32_t o = __shfl_xor_sync(0xFFFFFFFFu, m, d);
        const float2 po = R.P[o], pm = R.P[m];
        if (below_yx(po, pm) || (!below_yx(pm, po) && o < m)) m = o;
    }
    int s = 1;
    const uint32_t pm = distinct_neighbour(R, m, n, -1, lane);
    if (pm < n) {
        const uint32_t nm = distinct_neighbour(R, m, n, +1, lane);
        const int o = orient(R.P[pm], R.P[m], R.P[nm]);
        if (o != 0) s = o;
    }

    // ring, convexity, blocker list (non-convex vertices in index order)
    for (uint32_t i = lane; i < n; i += 32) {
        R.prv[i] = (uint16_t)(i ? i - 1u : n - 1u);
        R.nxt[i] = (uint16_t)(i + 1u < n ? i + 1u : 0u);
    }
    uint32_t nlist = 0;
    for (uint32_t base = 0; base < n; base += 32) {
        const uint32_t i = base + lane;
        bool nc = false;
        if (i < n) nc = s * orient(R.P[i ? i - 1u : n - 1u], R.P[i], R.P[i + 1u < n ? i + 1u : 0u]) <= 0;
        if (i < n) R.flg[i] = nc ? (uint8_t)(F_NONCONVEX | F_LISTED) : (uint8_t)0;
        const uint32_t b = __ballot_sync(0xFFFFFFFFu, nc);
        if (nc) R.lst[nlist + __popc(b & ((1u << lane) - 1u))] = (uint16_t)i;
        nlist += __popc(b);
    }
    __syncwarp();

    uint32_t status = 0, c = 0, stop = 0;
    for (uint32_t k = n; k > 3u; --k) {
        uint32_t p = R.prv[c], q = R.nxt[c];
        while (!is_ear(R, p, c, q, s, nlist, lane)) {
            c = q;
            if (c == stop) {  // a whole lap without an ear: clip the vertex the lap started from
                status = MR_POLY_NO_EAR;
                p = R.prv[c];
                q = R.nxt[c];
                break;
            }
            p = R.prv[c];
            q = R.nxt[c];
        }
        if (s > 0) em.tri(R, p, c, q, lane);
        else em.tri(R, q, c, p, lane);
        __syncwarp();
        if (lane == 0) {
            R.nxt[p] = (uint16_t)q;
            R.prv[q] = (uint16_t)p;
            R.flg[c] |= F_REMOVED;
        }
        __syncwarp();
        // only p and q changed neighbours: refresh their convexity; a vertex that turns non-convex joins the list
        bool add = false;
        uint32_t v = 0;
        if (lane < 2u) {
            v = lane ? q : p;
            const bool nc = s * orient(R.P[R.prv[v]], R.P[v], R.P[R.nxt[v]]) <= 0;
            const uint8_t f = R.flg[v];
            add = nc && !(f & F_LISTED);
            R.flg[v] = (uint8_t)((f & ~F_NONCONVEX) | (nc ? F_NONCONVEX : 0) | (add ? F_LISTED : 0));
        }
        const uint32_t b = __ballot_sync(0xFFFFFFFFu, add);
        if (add) R.lst[nlist + __popc(b & ((1u << lane) - 1u))] = (uint16_t)v;
        nlist += __popc(b);
        __syncwarp();
        c = R.nxt[q];
        stop = c;
    }
    const uint32_t p = R.prv[c], q = R.nxt[c];
    if (s > 0) em.tri(R, p, c, q, lane);
    else em.tri(R, q, c, p, lane);
    return status;
}

// ---- holes: the crossing predicate and the bridge merge (mr_triangulate_earclip_holes) ------------------------------
__device__ __forceinline__ void two_prod(double a, double b, double& p, double& e) {
    p = __dmul_rn(a, b);
    e = __fma_rn(a, b, -p);
}

// Sign of (b2y - my)*O(a1,b1,a2) + (my - a2y)*O(a1,b1,b2) expanded into 24 products of three floats: the first two
// multiply exactly in double, the third by two_prod; the 48 terms are summed by grow-expansion.
__device__ __noinline__ int cross_exact(float2 a1, float2 b1, float2 a2, float2 b2, float my) {
    const double o1[6] = {__dmul_rn(a1.x, b1.y), -__dmul_rn(a1.x, a2.y), __dmul_rn(b1.x, a2.y),
                          -__dmul_rn(b1.x, a1.y), __dmul_rn(a2.x, a1.y), -__dmul_rn(a2.x, b1.y)};
    const double o2[6] = {__dmul_rn(a1.x, b1.y), -__dmul_rn(a1.x, b2.y), __dmul_rn(b1.x, b2.y),
                          -__dmul_rn(b1.x, a1.y), __dmul_rn(b2.x, a1.y), -__dmul_rn(b2.x, b1.y)};
    const double f1[2] = {b2.y, -(double)my}, f2[2] = {my, -(double)a2.y};
    double e[48];
    int n = 0;
    for (int k = 0; k < 6; ++k)
        for (int i = 0; i < 2; ++i) {
            double t[4];
            two_prod(o1[k], f1[i], t[0], t[1]);
            two_prod(o2[k], f2[i], t[2], t[3]);
            for (int u = 0; u < 4; ++u) {
                double q = t[u];
                for (int m = 0; m < n; ++m) two_sum(q, e[m], q, e[m]);
                e[n++] = q;
            }
        }
    for (int i = 47; i >= 0; --i)
        if (e[i] != 0.0) return e[i] > 0.0 ? 1 : -1;
    return 0;
}

// Exact sign of the crossing comparison of the header.  Filter: the value in double, with the differences of floats
// and the two orient determinants rounded once each; its error is below 8 * 2^-53 * S (S the sum of the magnitudes of
// the two products), nothing underflows (every nonzero term is at least 2^-447) and S == 0 means the value is 0.
__device__ __forceinline__ int cross_sign(float2 a1, float2 b1, float2 a2, float2 b2, float my) {
    const double l1 = __dmul_rn(__dsub_rn(a1.x, a2.x), __dsub_rn(b1.y, a2.y)), r1 = __dmul_rn(__dsub_rn(a1.y, a2.y), __dsub_rn(b1.x, a2.x));
    const double l2 = __dmul_rn(__dsub_rn(a1.x, b2.x), __dsub_rn(b1.y, b2.y)), r2 = __dmul_rn(__dsub_rn(a1.y, b2.y), __dsub_rn(b1.x, b2.x));
    const double f1 = __dsub_rn(b2.y, my), f2 = __dsub_rn(my, a2.y);
    const double d = __dadd_rn(__dmul_rn(f1, __dsub_rn(l1, r1)), __dmul_rn(f2, __dsub_rn(l2, r2)));
    const double S = __dadd_rn(__dmul_rn(fabs(f1), __dadd_rn(fabs(l1), fabs(r1))), __dmul_rn(fabs(f2), __dadd_rn(fabs(l2), fabs(r2))));
    const double bound = 16.0 * 0x1p-53 * S;
    if (d > bound) return 1;
    if (-d > bound) return -1;
    if (S == 0.0) return 0;
    return cross_exact(a1, b1, a2, b2, my);
}

__device__ __forceinline__ int cmpf(float a, float b) { return (a > b) - (a < b); }
__device__ __forceinline__ bool above_xy(float2 a, float2 b) { return a.x > b.x || (a.x == b.x && a.y > b.y); }
__device__ __forceinline__ uint32_t wrap(uint32_t k, uint32_t L) { return k >= L ? k - L : k; }

// winding of the ring R.P[a .. a+n) by the lowest-vertex rule (warp-uniform)
__device__ int ring_winding(const Ring& R, uint32_t a, uint32_t n, uint32_t lane) {
    uint32_t m = 0;
    for (uint32_t i = lane; i < n; i += 32)
        if (i == lane || below_yx(R.P[a + i], R.P[a + m])) m = i;
    if (lane >= n) m = 0;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const uint32_t o = __shfl_xor_sync(0xFFFFFFFFu, m, d);
        const float2 po = R.P[a + o], pm = R.P[a + m];
        if (below_yx(po, pm) || (!below_yx(pm, po) && o < m)) m = o;
    }
    const float2 pmv = R.P[a + m];
    uint32_t nb[2] = {n, n};
    for (int dir = 0; dir < 2; ++dir)
        for (uint32_t base = 1; base < n; base += 32) {
            const uint32_t dd = base + lane;
            const uint32_t i = dir == 0 ? (m + n - dd % n) % n : (m + dd) % n;
            const uint32_t hit = __ballot_sync(0xFFFFFFFFu, dd < n && !same_pt(R.P[a + i], pmv));
            if (hit) {
                const uint32_t k = base + __ffs(hit) - 1u;
                nb[dir] = dir == 0 ? (m + n - k) % n : (m + k) % n;
                break;
            }
        }
    if (nb[0] == n) return 1;
    const int o = orient(R.P[a + nb[0]], pmv, R.P[a + nb[1]]);
    return o ? o : 1;
}

// Position of the current ring (point ids R.lst[0..L), points R.P) that the hole vertex M is bridged to (steps 1-3 of the
// header); bad = no edge crosses the ray.  Warp-uniform.
__device__ uint32_t bridge_pos(const Ring& R, uint32_t L, float2 M, int s, uint32_t lane, bool& bad) {
    constexpr uint32_t NONE = 0xFFFFFFFFu;
    const float my = M.y;
    // 1. nearest crossing edge: lane-local scan in position order, then a butterfly under (crossing x, position)
    uint32_t e = NONE;
    float2 ea = M, eb = M;
    for (uint32_t k = lane; k < L; k += 32) {
        const float2 a = R.P[R.lst[k]], b = R.P[R.lst[wrap(k + 1u, L)]];
        if (s * cmpf(b.y, a.y) <= 0 || !(fminf(a.y, b.y) <= my && my <= fmaxf(a.y, b.y)) || s * orient(a, b, M) < 0) continue;
        if (e == NONE || cross_sign(ea, eb, a, b, my) > 0) {
            e = k;
            ea = a;
            eb = b;
        }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const uint32_t o = __shfl_xor_sync(0xFFFFFFFFu, e, d);
        const float2 oa = make_float2(__shfl_xor_sync(0xFFFFFFFFu, ea.x, d), __shfl_xor_sync(0xFFFFFFFFu, ea.y, d));
        const float2 ob = make_float2(__shfl_xor_sync(0xFFFFFFFFu, eb.x, d), __shfl_xor_sync(0xFFFFFFFFu, eb.y, d));
        if (o == NONE) continue;
        int w = 1;
        if (e != NONE) {
            w = cross_sign(ea, eb, oa, ob, my);
            if (w == 0) w = o < e ? 1 : -1;
        }
        if (w > 0) {
            e = o;
            ea = oa;
            eb = ob;
        }
    }
    bad = e == NONE;
    if (bad) return 0;
    // 2. target
    uint32_t t;
    if (ea.y == my) {
        t = e;
    } else if (eb.y == my) {
        t = wrap(e + 1u, L);
    } else {
        t = ea.x >= eb.x ? e : wrap(e + 1u, L);
        const float2 Pt = R.P[R.lst[t]];
        const int u = Pt.y > my ? 1 : -1;
        uint32_t c = NONE;
        float2 pc = M;
        for (uint32_t k = lane; k < L; k += 32) {
            const float2 pr = R.P[R.lst[k]];
            if (same_pt(pr, M) || s * orient(R.P[R.lst[k ? k - 1u : L - 1u]], pr, R.P[R.lst[wrap(k + 1u, L)]]) > 0) continue;
            if (u * cmpf(pr.y, my) < 0 || s * orient(ea, eb, pr) < 0 || u * orient(M, Pt, pr) > 0) continue;
            int w = 1;
            if (c != NONE) {
                w = u * orient(M, pr, pc);
                if (w == 0) w = cmpf(pc.x, pr.x);
            }
            if (w > 0) {
                c = k;
                pc = pr;
            }
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            const uint32_t o = __shfl_xor_sync(0xFFFFFFFFu, c, d);
            const float2 po = make_float2(__shfl_xor_sync(0xFFFFFFFFu, pc.x, d), __shfl_xor_sync(0xFFFFFFFFu, pc.y, d));
            if (o == NONE) continue;
            int w = 1;
            if (c != NONE) {
                w = u * orient(M, po, pc);
                if (w == 0) w = cmpf(pc.x, po.x);
                if (w == 0) w = o < c ? 1 : -1;
            }
            if (w > 0) {
                c = o;
                pc = po;
            }
        }
        if (c != NONE) {
            const int w = u * orient(M, pc, Pt);
            if (w > 0 || (w == 0 && pc.x < Pt.x)) t = c;
        }
    }
    // 3. the first copy of the target point whose wedge contains M
    const float2 T = R.P[R.lst[t]];
    for (uint32_t base = 0; base < L; base += 32) {
        const uint32_t k = base + lane;
        bool ok = false;
        if (k < L && same_pt(R.P[R.lst[k]], T)) {
            const float2 pp = R.P[R.lst[k ? k - 1u : L - 1u]], pn = R.P[R.lst[wrap(k + 1u, L)]];
            const int o1 = s * orient(pp, T, M), o2 = s * orient(T, pn, M);
            ok = s * orient(pp, T, pn) > 0 ? (o1 > 0 && o2 > 0) : (o1 > 0 || o2 > 0);
        }
        const uint32_t hit = __ballot_sync(0xFFFFFFFFu, ok);
        if (hit) return base + __ffs(hit) - 1u;
    }
    return t;
}

// Merges the H holes of a polygon into its outer ring (step 4 of the header).  On entry R.P[0..N) holds the polygon's
// points and hs(h) gives the start of ring h relative to the polygon (hs(H + 1) = N); on exit R.P[0..N+2H) holds the
// merged ring.  Meanwhile R.lst holds the merged ring as point ids and R.prv / R.nxt each hole's M and the merge order.
// Returns MR_POLY_BAD_HOLE or 0.
template <class HS>
__device__ uint32_t merge_holes(const Ring& R, const float2* src, uint32_t N, uint32_t H, const HS& hs, uint32_t lane) {
    const uint32_t N0 = hs(1u);
    const int s = ring_winding(R, 0, N0, lane);
    for (uint32_t h = lane; h < H; h += 32) {
        const uint32_t a = hs(h + 1u), b = hs(h + 2u);
        uint32_t m = a;
        for (uint32_t k = a + 1u; k < b; ++k)
            if (above_xy(R.P[k], R.P[m])) m = k;
        R.prv[h] = (uint16_t)m;
    }
    __syncwarp();
    // merge order: decreasing (x, y) of M, equal M in hole order
    for (uint32_t h = lane; h < H; h += 32) {
        const float2 pm = R.P[R.prv[h]];
        uint32_t rank = 0;
        for (uint32_t g = 0; g < H; ++g) {
            const float2 pg = R.P[R.prv[g]];
            rank += above_xy(pg, pm) || (same_pt(pg, pm) && g < h);
        }
        R.nxt[rank] = (uint16_t)h;
    }
    for (uint32_t k = lane; k < N0; k += 32) R.lst[k] = (uint16_t)k;
    __syncwarp();
    uint32_t L = N0, status = 0;
    for (uint32_t z = 0; z < H; ++z) {
        const uint32_t h = R.nxt[z], M = R.prv[h], a = hs(h + 1u), n = hs(h + 2u) - a;
        bool bad;
        const uint32_t k = bridge_pos(R, L, R.P[M], s, lane, bad);
        if (bad) status = MR_POLY_BAD_HOLE;
        const bool rev = ring_winding(R, a, n, lane) == s;
        // open a gap of n + 2 after position k (from the end, a chunk of 32 read before it is written)
        const uint32_t d = n + 2u;
        for (uint32_t end = L; end > k + 1u;) {
            const uint32_t start = end - (k + 1u) > 32u ? end - 32u : k + 1u;
            const uint32_t i = start + lane;
            const uint16_t v = i < end ? R.lst[i] : (uint16_t)0;
            __syncwarp();
            if (i < end) R.lst[i + d] = v;
            __syncwarp();
            end = start;
        }
        const uint32_t jm = M - a;
        for (uint32_t dd = lane; dd < n; dd += 32) R.lst[k + 1u + dd] = (uint16_t)(a + (rev ? (jm + n - dd) % n : (jm + dd) % n));
        if (lane == 0) {
            R.lst[k + 1u + n] = (uint16_t)M;
            R.lst[k + 2u + n] = R.lst[k];
        }
        __syncwarp();
        L += d;
    }
    // the merged ring's points, from the caller's array (R.P still holds the input order until here)
    for (uint32_t k = lane; k < L; k += 32) R.P[k] = __ldg(src + R.lst[k]);
    __syncwarp();
    return status;
}

// The ring checks of mr_triangulate_earclip_holes, in the header's order; H = the number of holes when they pass.
__device__ uint32_t ring_status(const EcArgs& a, const RingArgs& rg, uint32_t pi, uint64_t r0, uint64_t np64, uint32_t& H,
                                uint32_t lane) {
    const uint64_t nr = rg.first_ring[pi + 1] - r0;
    if (nr == 0 || nr > np64) return MR_POLY_DEGENERATE;
    if (np64 + 2u * (nr - 1u) > MR_MAX_POLYGON_POINTS) return MR_POLY_TOO_LARGE;
    H = (uint32_t)(nr - 1u);
    bool ok = true;
    for (uint32_t h = lane; h <= H; h += 32) {
        const uint64_t s0 = rg.ring_start[r0 + h - rg.ring_base] - a.first_point[pi];
        const uint64_t s1 = h < H ? rg.ring_start[r0 + h + 1u - rg.ring_base] - a.first_point[pi] : np64;
        ok = ok && (h || s0 == 0) && s0 < s1 && s1 - s0 >= 3u && s1 <= np64;
    }
    return __all_sync(0xFFFFFFFFu, ok) ? MR_POLY_OK : MR_POLY_DEGENERATE;
}

// One polygon of mr_triangulate_earclip (HOLES false; rg unused) or mr_triangulate_earclip_holes; with IDX, of
// mr_triangulate_earclip_indexed (map: the position -> point id map of the holes case; ix and map unused otherwise).
template <bool HOLES, bool IDX>
__device__ void earclip_polygon(const EcArgs& a, const RingArgs& rg, const IdxArgs& ix, MR_SPAN(uint16_t) map, uint32_t pi,
                                const Ring& R, uint32_t lane) {
    const uint64_t p0 = a.first_point[pi] - a.point_base;
    const uint64_t np64 = a.first_point[pi + 1] - a.first_point[pi];
    const uint64_t t0 = a.first_tri[pi] - a.tri_base;
    const uint32_t cap_tri = (uint32_t)(a.first_tri[pi + 1] - a.first_tri[pi]);
    const uint32_t n = (uint32_t)(np64 > 0xFFFFFFFFull ? 0xFFFFFFFFull : np64);

    Emit<IDX> em;
    if constexpr (IDX) {
        em.idx = ix.idx_out + t0 * 3u;
        em.ibase = (uint32_t)(a.first_point[pi] - ix.index_base);
        em.map = HOLES ? map : MR_SPAN_NULL(uint16_t);
        em.vtx = a.vtx_out != nullptr;
    }
    em.sink.base = a.vtx_out + t0 * 3u * a.stride;
    em.sink.cap_vtx = cap_tri * 3u;
    em.sink.stride = a.stride;
    em.sink.off_x = a.off_x;
    em.sink.off_c = a.off_c;
    em.sink.fast32 = a.fast32;
    em.cap_tri = cap_tri;
    em.t = 0;
    em.mn = em.mx = em.lasty = 0.0f;

    uint32_t status = MR_POLY_OK, ntri = 0;
    float b1y = 0.0f, b2y = 0.0f;
    uint32_t H = 0;
    const uint64_t r0 = HOLES ? rg.first_ring[pi] : 0;
    if (!HOLES && n < 3u) {
        status = MR_POLY_DEGENERATE;
    } else if (!HOLES && n > MR_MAX_POLYGON_POINTS) {
        status = MR_POLY_TOO_LARGE;
    } else if (HOLES && (status = ring_status(a, rg, pi, r0, np64, H, lane)) != MR_POLY_OK) {
        // rejected by the ring checks
    } else {
        bool finite = true;
        const float2* src = reinterpret_cast<const float2*>(a.xy) + p0;
        for (uint32_t i = lane; i < n; i += 32) {
            const float2 v = __ldg(src + i);
            R.P[i] = v;
            finite = finite && isfinite(v.x) && isfinite(v.y);
        }
        __syncwarp();
        if (!__all_sync(0xFFFFFFFFu, finite)) {
            status = MR_POLY_NONFINITE;
        } else {
            uint32_t L = n;
            if constexpr (HOLES) {
                if (H) {
                    const uint64_t fp = a.first_point[pi];
                    auto hs = [&](uint32_t h) -> uint32_t {
                        return h > H ? n : h ? (uint32_t)(rg.ring_start[r0 + h - rg.ring_base] - fp) : 0u;
                    };
                    status = merge_holes(R, src, n, H, hs, lane);
                    L = n + 2u * H;
                }
                if constexpr (IDX) {  // keep the merged ring's point ids through the clip, which reuses R.lst
                    for (uint32_t k = lane; k < L; k += 32) map[k] = H ? R.lst[k] : (uint16_t)k;
                    __syncwarp();
                }
            }
            status |= clip_ring(R, L, em, lane);
            const uint32_t T = L - 2u;
            ntri = T < cap_tri ? T : cap_tri;
            if (T > cap_tri) status |= MR_POLY_OVERFLOW;
            if (T < cap_tri) {
                status |= MR_POLY_UNDERFILL;
                em.zero_from(3u * T, lane);
            }
            b1y = fmin_acc(em.mn, em.lasty);
            b2y = fmax_acc(em.mx, em.lasty);
        }
    }
    if (status & (MR_POLY_DEGENERATE | MR_POLY_TOO_LARGE | MR_POLY_NONFINITE)) em.zero_from(0, lane);
    if (lane == 0) {
        if (a.status_out) a.status_out[pi] = status;
        if (a.ntri_out) a.ntri_out[pi] = ntri;
        if (a.bbox_out) *reinterpret_cast<float4*>(a.bbox_out + 4 * (size_t)pi) = make_float4(em.mn, b1y, em.mx, b2y);
    }
}

// size class C: polygons of ec_nmax(C-1)+1 .. ec_nmax(C) points (class 0 also takes every invalid size); with holes the
// size is that of the merged ring, N + 2H
template <bool HOLES, bool IDX, int C>
__device__ __forceinline__ void earclip_class(const EcArgs& a, const RingArgs& rg, const IdxArgs& ix) {
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr uint32_t NMAX = ec_nmax(C);
    constexpr bool MAP = HOLES && IDX;
    const uint32_t lane = threadIdx.x & 31u;
    unsigned char* ws = smem + (size_t)(threadIdx.x >> 5) * ec_ws_bytes(NMAX, MAP);
    Ring R;
    R.P = MR_MAKE_SPAN(float2, reinterpret_cast<float2*>(ws), NMAX);
    R.prv = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + 8u * NMAX), NMAX);
    R.nxt = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + 10u * NMAX), NMAX);
    R.lst = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + 12u * NMAX), NMAX);
    R.flg = MR_MAKE_SPAN(uint8_t, ws + (MAP ? 16u : 14u) * NMAX, NMAX);
    MR_SPAN(uint16_t) map = MAP ? MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + 14u * NMAX), NMAX) : MR_SPAN_NULL(uint16_t);
    const uint32_t begin = C == EC_CLASSES - 1 ? 0u : a.cursor[NMAX + 1u];
    const uint32_t end = a.cursor[C == 0 ? 0u : ec_nmax(C - 1) + 1u];
    for (;;) {
        uint32_t idx = 0;
        if (lane == 0) idx = atomicAdd(&a.queue_head[C], 1u);
        idx = __shfl_sync(0xFFFFFFFFu, idx, 0);
        if (idx >= end - begin) break;
        earclip_polygon<HOLES, IDX>(a, rg, ix, map, a.order[begin + idx], R, lane);
        __syncwarp();
    }
}

template <int C>
__global__ void __launch_bounds__(ec_wpb(C) * 32) earclip_k(const EcArgs a) { earclip_class<false, false, C>(a, RingArgs{}, IdxArgs{}); }

template <int C>
__global__ void __launch_bounds__(ec_wpb(C) * 32) earclip_holes_k(const EcArgs a, const RingArgs rg) {
    earclip_class<true, false, C>(a, rg, IdxArgs{});
}

// at the 72 registers earclip_k<0..2> compiles to, 7 blocks per SM (the occupancy the latency-bound ring walk needs);
// class 3 is held to one block per SM by its workspace
template <int C>
__global__ void __launch_bounds__(ec_wpb(C) * 32, C == EC_CLASSES - 1 ? 1 : 7) earclip_idx_k(const EcArgs a, const IdxArgs ix) {
    earclip_class<false, true, C>(a, RingArgs{}, ix);
}

template <int C>
__global__ void __launch_bounds__(ec_wpb(C) * 32) earclip_holes_idx_k(const EcArgs a, const RingArgs rg, const IdxArgs ix) {
    earclip_class<true, true, C>(a, rg, ix);
}

__global__ void __launch_bounds__(256) selftest_orient_k(const float* __restrict__ abc, uint64_t count, int8_t* __restrict__ out) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
        const float* t = abc + 6 * i;
        out[i] = (int8_t)orient(make_float2(t[0], t[1]), make_float2(t[2], t[3]), make_float2(t[4], t[5]));
    }
}

__global__ void __launch_bounds__(256) selftest_crossing_k(const float* __restrict__ q, uint64_t count, int8_t* __restrict__ out) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
        const float* t = q + 9 * i;
        out[i] = (int8_t)cross_sign(make_float2(t[0], t[1]), make_float2(t[2], t[3]), make_float2(t[4], t[5]),
                                    make_float2(t[6], t[7]), t[8]);
    }
}

// rg == nullptr: without holes; ix == nullptr: without indices
template <int C>
int launch_class(mr_context* ctx, const EcArgs& a, const RingArgs* rg, const IdxArgs* ix, uint32_t npoly) {
    const int wpb = ec_wpb(C);
    const size_t smem = (size_t)wpb * ec_ws_bytes(ec_nmax(C), rg && ix);
    const void* fn = ix ? (rg ? reinterpret_cast<const void*>(earclip_holes_idx_k<C>) : reinterpret_cast<const void*>(earclip_idx_k<C>))
                        : (rg ? reinterpret_cast<const void*>(earclip_holes_k<C>) : reinterpret_cast<const void*>(earclip_k<C>));
    MR_CUDA(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    MR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, wpb * 32, smem));
    uint64_t grid = (uint64_t)ctx->sm_count * (per_sm < 1 ? 1 : per_sm);
    const uint64_t need = ((uint64_t)npoly + wpb - 1) / wpb;
    if (need < grid) grid = need;
    if (ix && rg) {
        earclip_holes_idx_k<C><<<(unsigned)grid, wpb * 32, smem, ctx->stream>>>(a, *rg, *ix);
        MR_LAUNCH_CHECK(ctx, "earclip_holes_idx_k");
    } else if (ix) {
        earclip_idx_k<C><<<(unsigned)grid, wpb * 32, smem, ctx->stream>>>(a, *ix);
        MR_LAUNCH_CHECK(ctx, "earclip_idx_k");
    } else if (rg) {
        earclip_holes_k<C><<<(unsigned)grid, wpb * 32, smem, ctx->stream>>>(a, *rg);
        MR_LAUNCH_CHECK(ctx, "earclip_holes_k");
    } else {
        earclip_k<C><<<(unsigned)grid, wpb * 32, smem, ctx->stream>>>(a);
        MR_LAUNCH_CHECK(ctx, "earclip_k");
    }
    return MR_OK;
}
}  // namespace

namespace {
int earclip_run(mr_context* ctx, const mr_polygon_job* j, const mr_polygon_rings* rings, const mr_polygon_indices* indices) {
    // all pointers in *j, *rings and *indices are device pointers here (staging happened in api.cu)
    const uint32_t npoly = j->npoly;
    if (npoly == 0) return MR_OK;
    // work list: hist | cursor | class ranges of the reference path (unused) | queue heads | order [| merged sizes].  A
    // scratch slot of its own, so that the reference path's work-list header (mr_triangulate_tier_counts) stays as it was.
    constexpr size_t ZERO_WORDS = 2 * (size_t)MR_SIZE_BINS + 64 + EC_CLASSES;
    const size_t order_bytes = ((ZERO_WORDS + npoly) * 4 + 7) / 8 * 8;
    void* work = nullptr;
    int rc = mr_scratch(ctx, MR_SLOT_EC_WORK, order_bytes + (rings ? ((size_t)npoly + 1) * 8 : 0), &work);
    if (rc) return rc;
    uint32_t* w = static_cast<uint32_t*>(work);
    uint32_t* hist = w;
    uint32_t* cursor = hist + MR_SIZE_BINS;
    uint32_t* classes = cursor + MR_SIZE_BINS;
    uint32_t* heads = classes + 64;
    uint32_t* order = heads + EC_CLASSES;
    MR_CUDA(ctx, cudaMemsetAsync(w, 0, ZERO_WORDS * 4, ctx->stream));
    // with holes the classes key on the merged size N + 2H: a prefix sum of it stands in for first_point
    const uint64_t* sizes = j->first_point;
    if (rings) {
        uint64_t* msz = reinterpret_cast<uint64_t*>(static_cast<unsigned char*>(work) + order_bytes);
        rc = mr_polygon_ring_counts(ctx, j->first_point, rings->first_ring, npoly, 0, msz);
        if (rc) return rc;
        sizes = msz;
    }
    rc = mr_polygon_size_sort(ctx, sizes, npoly, hist, cursor, classes, classes + 32, order);
    if (rc) return rc;

    EcArgs a;
    a.xy = j->xy;
    a.first_point = j->first_point;
    a.point_base = j->point_base;
    a.vtx_out = static_cast<unsigned char*>(j->vtx_out);
    a.first_tri = j->first_tri;
    a.tri_base = j->tri_base;
    a.bbox_out = j->bbox_out;
    a.status_out = j->status_out;
    a.ntri_out = j->ntri_out;
    if (a.vtx_out) {
        sink_layout(a, j->layout, a.vtx_out);
    } else {  // indices only: the layout is not read
        a.stride = a.off_x = 0;
        a.off_c = 0xFFFFFFFFu;
        a.fast32 = 0;
    }
    a.order = order;
    a.cursor = cursor;
    a.queue_head = heads;
    RingArgs rg{};
    if (rings) rg = RingArgs{rings->first_ring, rings->ring_base, rings->ring_start};
    const RingArgs* rp = rings ? &rg : nullptr;
    IdxArgs ix{};
    if (indices) ix = IdxArgs{indices->idx_out, indices->index_base};
    const IdxArgs* xp = indices ? &ix : nullptr;
    // largest class first
    if ((rc = launch_class<3>(ctx, a, rp, xp, npoly))) return rc;
    if ((rc = launch_class<2>(ctx, a, rp, xp, npoly))) return rc;
    if ((rc = launch_class<1>(ctx, a, rp, xp, npoly))) return rc;
    return launch_class<0>(ctx, a, rp, xp, npoly);
}
}  // namespace

int mr_triangulate_earclip_impl(mr_context* ctx, const mr_polygon_job* j) { return earclip_run(ctx, j, nullptr, nullptr); }

int mr_triangulate_earclip_holes_impl(mr_context* ctx, const mr_polygon_job* j, const mr_polygon_rings* rings) {
    return earclip_run(ctx, j, rings, nullptr);
}

int mr_triangulate_earclip_indexed_impl(mr_context* ctx, const mr_polygon_job* j, const mr_polygon_rings* rings,
                                        const mr_polygon_indices* indices) {
    return earclip_run(ctx, j, rings, indices);
}

int mr_selftest_crossing_impl(mr_context* ctx, const float* q, uint64_t count, int8_t* sign_out) {
    if (count == 0) return MR_OK;
    const unsigned blocks = (unsigned)std::min<uint64_t>((count + 255) / 256, (uint64_t)ctx->sm_count * 16);
    selftest_crossing_k<<<blocks, 256, 0, ctx->stream>>>(q, count, sign_out);
    MR_LAUNCH_CHECK(ctx, "selftest_crossing_k");
    return MR_OK;
}

int mr_selftest_orient_impl(mr_context* ctx, const float* abc, uint64_t count, int8_t* sign_out) {
    if (count == 0) return MR_OK;
    const unsigned blocks = (unsigned)std::min<uint64_t>((count + 255) / 256, (uint64_t)ctx->sm_count * 16);
    selftest_orient_k<<<blocks, 256, 0, ctx->stream>>>(abc, count, sign_out);
    MR_LAUNCH_CHECK(ctx, "selftest_orient_k");
    return MR_OK;
}
