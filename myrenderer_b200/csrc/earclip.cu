// earclip.cu -- ear-clipping triangulation (mr_triangulate_earclip) for sm_100a.
//
// The rules are those of the header, restated by tests/earclip_oracle/o_earclip.c and tests/_earclip.py.  One warp per
// polygon; the ring (points, prev/next links, a flag byte per point) and the list of vertices that can block an ear
// live in shared memory, 15 bytes per point.  Polygons are pulled largest first from four size classes.  The ring walk
// is warp-uniform (every lane holds the same cursor); the blocker scan of a candidate runs lane-parallel over the list
// of non-convex vertices, behind an exact bounding-box reject.
#include "common.cuh"

namespace {
#include "polygon_sink.cuh"

constexpr int EC_CLASSES = 4;
__host__ __device__ constexpr uint32_t ec_nmax(int c) { return c == 0 ? 64u : c == 1 ? 256u : c == 2 ? 1024u : MR_MAX_POLYGON_POINTS; }
// warps per block: the 4096-point class fits three 61 KB workspaces per SM
__host__ __device__ constexpr int ec_wpb(int c) { return c == EC_CLASSES - 1 ? 3 : 4; }
// per warp: xy 8 B | prev 2 B | next 2 B | blocker list 2 B | flags 1 B, per point (15 * nmax is a multiple of 16)
__host__ __device__ constexpr size_t ec_ws_bytes(uint32_t nmax) { return (size_t)nmax * 15u; }

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

struct Emit {
    Sink sink;
    uint32_t cap_tri, t;
    float mn, mx, lasty;
    // triangle (x0, x1, x2) as the next one of the polygon; lanes 0..2 store its vertices
    __device__ __forceinline__ void tri(const Ring& R, uint32_t x0, uint32_t x1, uint32_t x2, uint32_t lane) {
        const float2 v0 = R.P[x0], v1 = R.P[x1], v2 = R.P[x2];
        mn = fmin_acc(fmin_acc(fmin_acc(mn, v0.x), v1.x), v2.x);
        mx = fmax_acc(fmax_acc(fmax_acc(mx, v0.x), v1.x), v2.x);
        lasty = v2.y;
        if (t < cap_tri && lane < 3u) sink.write(3u * t + lane, lane == 0u ? v0 : lane == 1u ? v1 : v2);
        ++t;
    }
};

// Runs the ring walk of one valid polygon (3 <= n, finite points loaded into R.P); returns MR_POLY_NO_EAR or 0.
__device__ uint32_t clip_ring(const Ring& R, uint32_t n, Emit& em, uint32_t lane) {
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

__device__ void earclip_polygon(const EcArgs& a, uint32_t pi, const Ring& R, uint32_t lane) {
    const uint64_t p0 = a.first_point[pi] - a.point_base;
    const uint64_t np64 = a.first_point[pi + 1] - a.first_point[pi];
    const uint64_t t0 = a.first_tri[pi] - a.tri_base;
    const uint32_t cap_tri = (uint32_t)(a.first_tri[pi + 1] - a.first_tri[pi]);
    const uint32_t n = (uint32_t)(np64 > 0xFFFFFFFFull ? 0xFFFFFFFFull : np64);

    Emit em;
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
    if (n < 3u) {
        status = MR_POLY_DEGENERATE;
    } else if (n > MR_MAX_POLYGON_POINTS) {
        status = MR_POLY_TOO_LARGE;
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
            status = clip_ring(R, n, em, lane);
            const uint32_t T = n - 2u;
            ntri = T < cap_tri ? T : cap_tri;
            if (T > cap_tri) status |= MR_POLY_OVERFLOW;
            if (T < cap_tri) {
                status |= MR_POLY_UNDERFILL;
                em.sink.zero(3u * T, em.sink.cap_vtx, lane);
            }
            b1y = fmin_acc(em.mn, em.lasty);
            b2y = fmax_acc(em.mx, em.lasty);
        }
    }
    if (status & (MR_POLY_DEGENERATE | MR_POLY_TOO_LARGE | MR_POLY_NONFINITE)) em.sink.zero(0, em.sink.cap_vtx, lane);
    if (lane == 0) {
        if (a.status_out) a.status_out[pi] = status;
        if (a.ntri_out) a.ntri_out[pi] = ntri;
        if (a.bbox_out) *reinterpret_cast<float4*>(a.bbox_out + 4 * (size_t)pi) = make_float4(em.mn, b1y, em.mx, b2y);
    }
}

// size class C: polygons of ec_nmax(C-1)+1 .. ec_nmax(C) points (class 0 also takes every invalid size)
template <int C>
__global__ void __launch_bounds__(ec_wpb(C) * 32) earclip_k(const EcArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr uint32_t NMAX = ec_nmax(C);
    const uint32_t lane = threadIdx.x & 31u;
    unsigned char* ws = smem + (size_t)(threadIdx.x >> 5) * ec_ws_bytes(NMAX);
    Ring R;
    R.P = MR_MAKE_SPAN(float2, reinterpret_cast<float2*>(ws), NMAX);
    R.prv = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + 8u * NMAX), NMAX);
    R.nxt = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + 10u * NMAX), NMAX);
    R.lst = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + 12u * NMAX), NMAX);
    R.flg = MR_MAKE_SPAN(uint8_t, ws + 14u * NMAX, NMAX);
    const uint32_t begin = C == EC_CLASSES - 1 ? 0u : a.cursor[NMAX + 1u];
    const uint32_t end = a.cursor[C == 0 ? 0u : ec_nmax(C - 1) + 1u];
    for (;;) {
        uint32_t idx = 0;
        if (lane == 0) idx = atomicAdd(&a.queue_head[C], 1u);
        idx = __shfl_sync(0xFFFFFFFFu, idx, 0);
        if (idx >= end - begin) break;
        earclip_polygon(a, a.order[begin + idx], R, lane);
        __syncwarp();
    }
}

__global__ void __launch_bounds__(256) selftest_orient_k(const float* __restrict__ abc, uint64_t count, int8_t* __restrict__ out) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
        const float* t = abc + 6 * i;
        out[i] = (int8_t)orient(make_float2(t[0], t[1]), make_float2(t[2], t[3]), make_float2(t[4], t[5]));
    }
}

template <int C>
int launch_class(mr_context* ctx, const EcArgs& a, uint32_t npoly) {
    const int wpb = ec_wpb(C);
    const size_t smem = (size_t)wpb * ec_ws_bytes(ec_nmax(C));
    MR_CUDA(ctx, cudaFuncSetAttribute(earclip_k<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    MR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, earclip_k<C>, wpb * 32, smem));
    uint64_t grid = (uint64_t)ctx->sm_count * (per_sm < 1 ? 1 : per_sm);
    const uint64_t need = ((uint64_t)npoly + wpb - 1) / wpb;
    if (need < grid) grid = need;
    earclip_k<C><<<(unsigned)grid, wpb * 32, smem, ctx->stream>>>(a);
    MR_LAUNCH_CHECK(ctx, "earclip_k");
    return MR_OK;
}
}  // namespace

int mr_triangulate_earclip_impl(mr_context* ctx, const mr_polygon_job* j) {
    // all pointers in *j are device pointers here (staging happened in api.cu)
    const uint32_t npoly = j->npoly;
    if (npoly == 0) return MR_OK;
    // work list: hist | cursor | class ranges of the reference path (unused) | queue heads | order.  A scratch slot of
    // its own, so that the reference path's work-list header (mr_triangulate_tier_counts) stays as it was.
    constexpr size_t ZERO_WORDS = 2 * (size_t)MR_SIZE_BINS + 64 + EC_CLASSES;
    void* work = nullptr;
    int rc = mr_scratch(ctx, 13, (ZERO_WORDS + npoly) * 4, &work);
    if (rc) return rc;
    uint32_t* w = static_cast<uint32_t*>(work);
    uint32_t* hist = w;
    uint32_t* cursor = hist + MR_SIZE_BINS;
    uint32_t* classes = cursor + MR_SIZE_BINS;
    uint32_t* heads = classes + 64;
    uint32_t* order = heads + EC_CLASSES;
    MR_CUDA(ctx, cudaMemsetAsync(w, 0, ZERO_WORDS * 4, ctx->stream));
    rc = mr_polygon_size_sort(ctx, j->first_point, npoly, hist, cursor, classes, classes + 32, order);
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
    a.stride = j->layout.stride;
    a.off_x = j->layout.attr[0].offset;
    a.off_c = j->layout.nattr > 1 ? j->layout.attr[1].offset : 0xFFFFFFFFu;
    a.fast32 = (a.stride == 32 && j->layout.nattr == 2 && ((a.off_x == 0 && a.off_c == 16) || (a.off_x == 16 && a.off_c == 0)) &&
                reinterpret_cast<uintptr_t>(a.vtx_out) % 32 == 0)
                   ? 1
                   : 0;
    a.order = order;
    a.cursor = cursor;
    a.queue_head = heads;
    // largest class first
    if ((rc = launch_class<3>(ctx, a, npoly))) return rc;
    if ((rc = launch_class<2>(ctx, a, npoly))) return rc;
    if ((rc = launch_class<1>(ctx, a, npoly))) return rc;
    return launch_class<0>(ctx, a, npoly);
}

int mr_selftest_orient_impl(mr_context* ctx, const float* abc, uint64_t count, int8_t* sign_out) {
    if (count == 0) return MR_OK;
    const unsigned blocks = (unsigned)std::min<uint64_t>((count + 255) / 256, (uint64_t)ctx->sm_count * 16);
    selftest_orient_k<<<blocks, 256, 0, ctx->stream>>>(abc, count, sign_out);
    MR_LAUNCH_CHECK(ctx, "selftest_orient_k");
    return MR_OK;
}
