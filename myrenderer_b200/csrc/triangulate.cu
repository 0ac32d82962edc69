// triangulate.cu -- batched polygon triangulation for sm_100a, bit-compatible with
// Polygon/Triangulation.zig (Seidel-style trapezoidation -> monotone mountains -> fan emission)
// and with the emit sink of Polygon/Polygon.zig:65-79.
//
// Execution model: one warp per polygon, polygons pulled from per-size-class queues by
// persistent warps.  The polygon's points, its trapezoid DAG (12-byte nodes, 16-bit ids) and the
// segment-search stack live in shared memory (tier 0).  A polygon that outgrows its tier-0 arena
// is re-queued to tier 1, the same code over a per-warp global-memory arena sized to the
// contract caps MR_NODE_CAP / MR_STACK_CAP.  The trapezoidation is inherently serial (the output
// order depends on the node allocation counter, Triangulation.zig:510), so it runs warp-uniform:
// all lanes execute the same instruction stream on broadcast shared-memory reads.  The mountain
// phase is restated in a data-parallel form that produces the same sequence of emits:
//   scan nodes in id order (ballot compaction)           Triangulation.zig:510-540
//   mountain = edge id, rank = first appearance            :49-62
//   stable sort of every mountain list by (y, x, append)   :555
//   tail loop == "for j = len-1 .. 2: if L[j]!=L[j-1] and L[j]!=L[0] emit(L[j],L[j-1],L[0])"  :558-586
// The last equivalence holds whenever push_triangle_if_acute (:398-425) returns true, which is
// checked per triangle with a musl-exact atan2f; if any check fails the polygon falls back to a
// literal restatement of the loop.
#include <algorithm>
#include "common.cuh"
#include "unirand.cuh"

namespace {

constexpr uint32_t NIL = 0xFFFFu;
enum : uint32_t { T_POINT = 0, T_SEGMENT = 1, T_TRAPEZOID = 2 };
constexpr int NUM_CLASSES = 12;  // classes 0..10: shared-memory workspaces (see class_nmax); 11: up to MR_MAX (global memory)
constexpr int XL_CLASS = 10;     // 1025..3072 points: one polygon per SM; no contract-cap tier fits shared memory, so a
                                 // polygon that outgrows the typical-case arenas goes to the global-memory general path
constexpr int CLASS_SLOTS = 16; // header words reserved per per-class array
constexpr int NBINS = MR_MAX_POLYGON_POINTS + 1;  // polygons are queued by exact size, largest first
constexpr int MAX_WARPS_PER_BLOCK = 4;

// Largest polygon of shared-memory class c.  Above 64 points a class is bound by the polygons whose workspaces
// (~73 bytes per point, fast_layout) fit the SM's 228 KB, so the boundaries sit where one more polygon fits:
// 1024 points -> 3 per SM, 768 -> 4, 608 -> 5, 504 -> 6, 368 -> 8, 288 -> 10, 216 -> 13, 168 -> 16, 128 -> 20;
// 3072 points (220 KB) -> one per SM.
__host__ __device__ inline uint32_t class_nmax(int c) {
    switch (c) {
        case 0: return 64u;
        case 1: return 128u;
        case 2: return 168u;
        case 3: return 216u;
        case 4: return 288u;
        case 5: return 368u;
        case 6: return 504u;
        case 7: return 608u;
        case 8: return 768u;
        case 9: return 1024u;
        default: return 3072u;
    }
}
// warps cooperating on one polygon in the first (typical-case) pass of class c; 1 = independent warps
// (3/4/4/6/8 warps for the 368/504/608/768/1024-point classes -- at most 24 warps of 80 registers per SM; up to 288
// points independent warps; too wide a team loses polygons in flight to the register file)
inline int team_warps(int c) {  // keep in step with the kernel tables in mr_triangulate_impl
    const uint32_t nmax = class_nmax(c);
    return nmax <= 288u ? 1 : nmax == 368u ? 3 : nmax <= 608u ? 4 : nmax == 768u ? 6 : 8;  // 1024 and 3072: 8
}
__host__ __device__ inline int class_of(uint32_t n) {
    int c = 0;
    while (c < NUM_CLASSES - 1 && n > class_nmax(c)) ++c;
    return c;
}

// ---- per-warp workspace -------------------------------------------------------------------
struct Caps {
    uint32_t nmax;       // points
    uint32_t node_cap;   // nodes
    uint32_t stack_cap;  // u16 entries
    uint32_t add_cap;    // mountain adds
};

__host__ __device__ inline Caps tier1_caps(uint32_t nmax) {
    Caps k;
    k.nmax = nmax;
    k.node_cap = MR_NODE_CAP(nmax);
    k.stack_cap = MR_STACK_CAP(nmax);
    k.add_cap = 2u * k.node_cap;
    return k;
}
__host__ __device__ inline size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

struct WsLayout {
    size_t pts, nodes, stack, add_pp, add_key, efirst, add_m, mcount, mstart, sortbuf, total;
};
// alias_sort: sorted lists reuse the node arena (tier 0); otherwise they get their own space.
__host__ __device__ inline WsLayout ws_layout(const Caps& k, bool alias_sort) {
    WsLayout L;
    size_t o = 0;
    L.pts = o;     o += align16((size_t)k.nmax * 8);
    L.nodes = o;   o += align16((size_t)k.node_cap * 12);
    L.stack = o;   o += align16((size_t)k.stack_cap * 2);
    L.add_pp = o;  o += align16((size_t)k.add_cap * 4);
    L.add_key = o; o += align16((size_t)k.add_cap * 4);   // (p1,p2) of the key node
    L.efirst = o;  o += align16((size_t)k.nmax * 2);      // first add of each polygon-edge key
    L.add_m = o;   o += align16((size_t)k.add_cap * 4);   // first add with the same key, then mountain rank
    L.mcount = o;  o += align16((size_t)k.add_cap * 4);
    L.mstart = o;  o += align16((size_t)(k.add_cap + 1) * 4);
    if (alias_sort) {
        L.sortbuf = L.nodes;
    } else {
        L.sortbuf = o;
        o += align16((size_t)k.add_cap * 2 * 14 + 64);
    }
    L.total = o;
    return L;
}

struct BatchArgs {
    const float* xy;
    const uint64_t* first_point;
    uint64_t point_base;
    uint32_t npoly;
    const uint32_t* offset_prime;
    uint64_t seed, poly_index0;
    unsigned char* vtx_out;
    const uint64_t* first_tri;
    uint64_t tri_base;
    float* bbox_out;
    uint32_t* status_out;
    uint32_t* ntri_out;
    uint32_t stride, off_x, off_c;  // off_c == 0xFFFFFFFF: no colour attribute
    int fast32;                     // stride 32, offsets {0,16} in either order, 32B-aligned base
    // work lists
    const uint32_t* order;        // polygon ids grouped by class
    const uint32_t* class_begin;  // NUM_CLASSES: first position of the class in `order` (sorted by size, descending)
    const uint32_t* class_end;    // NUM_CLASSES
    uint32_t* queue_head;         // [c]: first pass of class c; [NUM_CLASSES + c]: its spec tier; [2*NUM_CLASSES + which]: general
    uint32_t* spec_list;          // npoly, class c's overflow at class_begin[c]..
    uint32_t* spec_count;         // NUM_CLASSES
    uint32_t* general_list;       // npoly
    uint32_t* general_count;
    unsigned char* tier1_ws;
    size_t tier1_ws_stride;
    unsigned char* par_ws;  // n <= 64 kernel: PAR_GL_BYTES of global scratch per warp of its grid
};

// ---- the per-polygon state machine ----------------------------------------------------------
struct Poly {
    const float2* pts;
    uint32_t* nodes;
    uint16_t* stack;
    uint32_t n, nnodes, nstack;
    uint32_t status;
    uint32_t tier_node_cap, tier_stack_cap;
    uint32_t spec_node_cap, spec_stack_cap;
    bool requeue;

    __device__ __forceinline__ uint32_t w0(uint32_t id) const { return nodes[3 * id]; }      // child1 | child2<<16
    __device__ __forceinline__ uint32_t w1(uint32_t id) const { return nodes[3 * id + 1]; }  // point1 | point2<<16
    __device__ __forceinline__ uint32_t w2(uint32_t id) const { return nodes[3 * id + 2]; }  // crumb | type<<16
    __device__ __forceinline__ void set_w0(uint32_t id, uint32_t v) { nodes[3 * id] = v; }
    __device__ __forceinline__ void set_w1(uint32_t id, uint32_t v) { nodes[3 * id + 1] = v; }
    __device__ __forceinline__ void set_w2(uint32_t id, uint32_t v) { nodes[3 * id + 2] = v; }

    // Triangulation.zig:102-115 with the contract cap and the tier cap
    __device__ __forceinline__ uint32_t alloc() {
        if (nnodes >= spec_node_cap) {
            status |= MR_POLY_ARENA;
            return NIL;
        }
        if (nnodes >= tier_node_cap) {
            requeue = true;
            return NIL;
        }
        return nnodes++;
    }

    // Triangulation.zig:117-126 -- separately rounded products and difference
    __device__ __forceinline__ bool is_left_of(uint32_t p, uint32_t s1, uint32_t s2) const {
        const float2 P = pts[p], A = pts[s1], B = pts[s2];
        const float mul1 = __fmul_rn(__fsub_rn(B.x, A.x), __fsub_rn(P.y, A.y));
        const float mul2 = __fmul_rn(__fsub_rn(B.y, A.y), __fsub_rn(P.x, A.x));
        return __fsub_rn(mul1, mul2) > 0.0f;
    }
    // Triangulation.zig:128-136
    __device__ __forceinline__ bool above(uint32_t l, uint32_t r) const {
        const float2 L = pts[l], R = pts[r];
        return (L.y < R.y) || (L.y == R.y && L.x < R.x);
    }

    __device__ __forceinline__ bool fail_unwrap() {
        status |= MR_POLY_NULL_UNWRAP;
        return false;
    }

    // Triangulation.zig:139-196
    __device__ bool add_point(uint32_t pid) {
        uint32_t base = 0;  // root_node is always node 0 (:479)
        for (;;) {
            const uint32_t t = w2(base) >> 16;
            if (t == T_TRAPEZOID) break;
            const uint32_t ch = w0(base), pp = w1(base);
            bool first;
            if (t == T_POINT) {
                const uint32_t pc = pp & 0xFFFFu;
                if (pc == pid) return true;  // :149-152
                if (pc == NIL) return fail_unwrap();
                first = above(pid, pc);
            } else {
                const uint32_t s1 = pp & 0xFFFFu, s2 = pp >> 16;
                if (s1 == NIL || s2 == NIL) return fail_unwrap();
                first = is_left_of(pid, s1, s2);
            }
            const uint32_t next = first ? (ch & 0xFFFFu) : (ch >> 16);
            if (next == NIL) return fail_unwrap();
            base = next;
        }
        // :178-179 clone lower first, then upper
        const uint32_t b0 = w0(base), b1 = w1(base), b2 = w2(base);
        const uint32_t lower = alloc();
        const uint32_t upper = alloc();
        if (lower == NIL || upper == NIL) return false;
        // :191-192 with the clones' other fields copied from the found trapezoid
        set_w0(lower, b0);
        set_w1(lower, (b1 & 0xFFFF0000u) | pid);  // point1 = pid
        set_w2(lower, b2);
        set_w0(upper, b0);
        set_w1(upper, (b1 & 0x0000FFFFu) | (pid << 16));  // point2 = pid
        set_w2(upper, b2);
        // :183-188 the trapezoid becomes the point node in place
        set_w0(base, upper | (lower << 16));
        set_w1(base, pid | (NIL << 16));
        set_w2(base, NIL | (T_POINT << 16));
        return true;
    }

    __device__ __forceinline__ bool push(uint32_t id) {
        if (nstack >= spec_stack_cap) {
            status |= MR_POLY_ARENA;
            return false;
        }
        if (nstack >= tier_stack_cap) {
            requeue = true;
            return false;
        }
        stack[nstack++] = (uint16_t)id;
        return true;
    }

    // Triangulation.zig:215-396
    __device__ bool add_segment(uint32_t point1, uint32_t point2) {
        uint32_t up, lo;
        if (above(point1, point2)) {
            up = point1;
            lo = point2;
        } else {
            up = point2;
            lo = point1;
        }
        uint32_t base = 0, breadcrumb = NIL;
        nstack = 0;
        for (;;) {      // loop1 :231
            for (;;) {  // loop :232
                const uint32_t tw = w2(base);
                const uint32_t t = tw >> 16;
                if (t == T_TRAPEZOID) break;
                const uint32_t ch = w0(base), pp = w1(base);
                if (t == T_POINT) {  // :234-259
                    const uint32_t pc = pp & 0xFFFFu;
                    if (pc == NIL) return fail_unwrap();
                    uint32_t next;
                    if (up == pc) {
                        next = ch >> 16;
                    } else if (lo == pc) {
                        next = ch & 0xFFFFu;
                    } else {
                        const bool bottom_point_is_above = above(lo, pc);
                        const bool top_point_is_below = above(pc, up);
                        if (top_point_is_below) {
                            next = ch >> 16;
                        } else if (bottom_point_is_above) {
                            next = ch & 0xFFFFu;
                        } else {  // :252-257 breadcrumb, then child1
                            set_w2(base, breadcrumb | (T_POINT << 16));
                            breadcrumb = base;
                            next = ch & 0xFFFFu;
                        }
                    }
                    if (next == NIL) return fail_unwrap();
                    base = next;
                } else {  // segment :260-296
                    const uint32_t o1 = pp & 0xFFFFu, o2 = pp >> 16;
                    if (o1 == NIL || o2 == NIL) return fail_unwrap();
                    bool is_left;
                    if (up == o2 || up == o1) {
                        is_left = is_left_of(lo, o1, o2);
                    } else if (lo == o1 || lo == o2) {
                        is_left = is_left_of(up, o1, o2);
                    } else {
                        const bool top_is_above = above(up, o1);
                        const bool bottom_is_below = above(lo, o2);
                        if (top_is_above && bottom_is_below)
                            is_left = !is_left_of(o1, up, lo);
                        else if (top_is_above && !bottom_is_below)
                            is_left = is_left_of(lo, o1, o2);
                        else
                            is_left = is_left_of(up, o1, o2);
                    }
                    const uint32_t next = is_left ? (ch & 0xFFFFu) : (ch >> 16);
                    if (next == NIL) return fail_unwrap();
                    base = next;
                }
            }
            if (!push(base)) return false;  // :302
            if (breadcrumb != NIL) {        // :306-313
                const uint32_t crumb = breadcrumb;
                breadcrumb = w2(crumb) & 0xFFFFu;
                set_w2(crumb, NIL | (T_POINT << 16));
                const uint32_t next = w0(crumb) >> 16;
                if (next == NIL) return fail_unwrap();
                base = next;
            } else {
                break;
            }
        }

        // pass 2 :316-395
        uint32_t left_trap = alloc();
        if (left_trap == NIL) return false;
        set_w0(left_trap, NIL | (NIL << 16));
        set_w1(left_trap, up | (NIL << 16));
        set_w2(left_trap, NIL | (T_TRAPEZOID << 16));
        uint32_t right_trap = alloc();
        if (right_trap == NIL) return false;
        set_w0(right_trap, NIL | (NIL << 16));
        set_w1(right_trap, up | (NIL << 16));
        set_w2(right_trap, NIL | (T_TRAPEZOID << 16));

        const uint32_t crumb_left = (point1 == up);  // :351-355
        while (nstack > 0) {                          // :325
            uint32_t base_index = 0, base_id = stack[0], low_point = lo;
            for (uint32_t i = 0; i < nstack; ++i) {  // :329-337
                const uint32_t node = stack[i];
                const uint32_t np = w1(node) >> 16;
                if (np == NIL) return fail_unwrap();
                if (above(np, low_point)) {
                    low_point = np;
                    base_index = i;
                    base_id = node;
                }
            }
            // :347-360
            const uint32_t bch = w0(base_id);
            set_w0(left_trap, (w0(left_trap) & 0xFFFF0000u) | (bch & 0xFFFFu));   // left.child1 = base.child1
            set_w0(right_trap, (w0(right_trap) & 0x0000FFFFu) | (bch & 0xFFFF0000u));  // right.child2 = base.child2
            set_w0(base_id, left_trap | (right_trap << 16));
            set_w2(base_id, (crumb_left ? left_trap : right_trap) | (T_SEGMENT << 16));
            set_w1(base_id, up | (lo << 16));

            if (lo == low_point) {  // :366-373
                set_w0(left_trap, (w0(left_trap) & 0x0000FFFFu) | (base_id << 16));  // left.child2 = base
                set_w1(left_trap, (w1(left_trap) & 0x0000FFFFu) | (low_point << 16));
                set_w0(right_trap, (w0(right_trap) & 0xFFFF0000u) | base_id);  // right.child1 = base
                set_w1(right_trap, (w1(right_trap) & 0x0000FFFFu) | (low_point << 16));
                break;
            } else if (is_left_of(low_point, up, lo)) {  // :375-382
                set_w0(left_trap, (w0(left_trap) & 0x0000FFFFu) | (base_id << 16));
                set_w1(left_trap, (w1(left_trap) & 0x0000FFFFu) | (low_point << 16));
                left_trap = alloc();
                if (left_trap == NIL) return false;
                set_w0(left_trap, NIL | (NIL << 16));
                set_w1(left_trap, low_point | (NIL << 16));
                set_w2(left_trap, NIL | (T_TRAPEZOID << 16));
            } else {  // :383-391
                set_w0(right_trap, (w0(right_trap) & 0xFFFF0000u) | base_id);
                set_w1(right_trap, (w1(right_trap) & 0x0000FFFFu) | (low_point << 16));
                right_trap = alloc();
                if (right_trap == NIL) return false;
                set_w0(right_trap, NIL | (NIL << 16));
                set_w1(right_trap, low_point | (NIL << 16));
                set_w2(right_trap, NIL | (T_TRAPEZOID << 16));
            }
            stack[base_index] = stack[nstack - 1];  // :394 swapRemove
            --nstack;
        }
        return true;
    }
};

// ---- std.math.atan2 (f32): musl algorithm, every operation separately rounded ---------------
__device__ __forceinline__ float dev_atanf(float x) {
    const float hi[4] = {__uint_as_float(0x3eed6338u), __uint_as_float(0x3f490fdau),
                         __uint_as_float(0x3f7b985eu), __uint_as_float(0x3fc90fdau)};
    const float lo[4] = {__uint_as_float(0x31ac3769u), __uint_as_float(0x33222168u),
                         __uint_as_float(0x33140fb4u), __uint_as_float(0x33a22168u)};
    const float aT0 = 3.3333328366e-01f, aT1 = -1.9999158382e-01f, aT2 = 1.4253635705e-01f,
                aT3 = -1.0648017377e-01f, aT4 = 6.1687607318e-02f;
    uint32_t ix = __float_as_uint(x);
    const uint32_t sign = ix >> 31;
    ix &= 0x7fffffffu;
    int id;
    if (ix >= 0x4c800000u) {
        if (ix > 0x7f800000u) return x;
        const float z = __fadd_rn(hi[3], 7.5231638453e-37f);
        return sign ? -z : z;
    }
    if (ix < 0x3ee00000u) {
        if (ix < 0x39800000u) return x;
        id = -1;
    } else {
        x = __uint_as_float(ix);
        if (ix < 0x3f980000u) {
            if (ix < 0x3f300000u) {
                id = 0;
                x = __fdiv_rn(__fsub_rn(__fmul_rn(2.0f, x), 1.0f), __fadd_rn(2.0f, x));
            } else {
                id = 1;
                x = __fdiv_rn(__fsub_rn(x, 1.0f), __fadd_rn(x, 1.0f));
            }
        } else {
            if (ix < 0x401c0000u) {
                id = 2;
                x = __fdiv_rn(__fsub_rn(x, 1.5f), __fadd_rn(1.0f, __fmul_rn(1.5f, x)));
            } else {
                id = 3;
                x = __fdiv_rn(-1.0f, x);
            }
        }
    }
    const float z = __fmul_rn(x, x);
    const float w = __fmul_rn(z, z);
    const float s1 = __fmul_rn(z, __fadd_rn(aT0, __fmul_rn(w, __fadd_rn(aT2, __fmul_rn(w, aT4)))));
    const float s2 = __fmul_rn(w, __fadd_rn(aT1, __fmul_rn(w, aT3)));
    if (id < 0) return __fsub_rn(x, __fmul_rn(x, __fadd_rn(s1, s2)));
    const float r = __fsub_rn(hi[id], __fsub_rn(__fsub_rn(__fmul_rn(x, __fadd_rn(s1, s2)), lo[id]), x));
    return sign ? -r : r;
}

__device__ __forceinline__ float dev_atan2f(float y, float x) {
    const float pi = __uint_as_float(0x40490fdbu);
    const float pi_lo = __uint_as_float(0xb3bbbd2eu);
    uint32_t ix = __float_as_uint(x), iy = __float_as_uint(y);
    if ((ix & 0x7fffffffu) > 0x7f800000u || (iy & 0x7fffffffu) > 0x7f800000u) return __fadd_rn(x, y);
    if (ix == 0x3f800000u) return dev_atanf(y);
    const uint32_t m = ((iy >> 31) & 1u) | ((ix >> 30) & 2u);
    ix &= 0x7fffffffu;
    iy &= 0x7fffffffu;
    if (iy == 0u) {
        switch (m) {
            case 0:
            case 1: return y;
            case 2: return pi;
            default: return -pi;
        }
    }
    if (ix == 0u) return (m & 1u) ? __fdiv_rn(-pi, 2.0f) : __fdiv_rn(pi, 2.0f);
    if (ix == 0x7f800000u) {
        if (iy == 0x7f800000u) {
            switch (m) {
                case 0: return __fdiv_rn(pi, 4.0f);
                case 1: return __fdiv_rn(-pi, 4.0f);
                case 2: return __fdiv_rn(__fmul_rn(3.0f, pi), 4.0f);
                default: return __fdiv_rn(__fmul_rn(-3.0f, pi), 4.0f);
            }
        } else {
            switch (m) {
                case 0: return 0.0f;
                case 1: return -0.0f;
                case 2: return pi;
                default: return -pi;
            }
        }
    }
    if (ix + (26u << 23) < iy || iy == 0x7f800000u) return (m & 1u) ? __fdiv_rn(-pi, 2.0f) : __fdiv_rn(pi, 2.0f);
    float z;
    if ((m & 2u) && iy + (26u << 23) < ix)
        z = 0.0f;
    else
        z = dev_atanf(fabsf(__fdiv_rn(y, x)));
    switch (m) {
        case 0: return z;
        case 1: return -z;
        case 2: return __fsub_rn(pi, __fsub_rn(z, pi_lo));
        default: return __fsub_rn(__fsub_rn(z, pi_lo), pi);
    }
}

// Triangulation.zig:399-403
__device__ __forceinline__ bool is_acute(const float2* pts, uint32_t point, uint32_t axis1, uint32_t axis2) {
    const float2 P = pts[point], A1 = pts[axis1], A2 = pts[axis2];
    const float a = dev_atan2f(__fsub_rn(P.y, A1.y), __fsub_rn(P.x, A1.x));
    const float b = dev_atan2f(__fsub_rn(P.y, A2.y), __fsub_rn(P.x, A2.x));
    return fabsf(__fsub_rn(a, b)) < __uint_as_float(0x40490fdbu);
}

// atan2f(dy, dx) certainly lies in [0, pi - 7e-7]: the vector points into the upper half-plane (or along +x) and makes
// an angle of more than 1e-6 with the negative x axis.  (atan2f's error is an ulp or two, 2.4e-7 near pi.)
__device__ __forceinline__ bool angle_clear_of_pi(float dy, float dx) {
    return (dy > 0.0f && (dx >= 0.0f || dy > __fmul_rn(1e-6f, -dx))) || (dy == 0.0f && dx > 0.0f);
}
// Same value as is_acute.  When both angles are certainly in [0, pi - 7e-7], |a - b| <= max(a, b) < (f32)pi without
// evaluating them -- the case of every triangle of a sorted mountain (SURVEY 8-c) except a centre that sees a neighbour
// within 1e-6 rad of the negative x axis, which takes the exact evaluation.
__device__ __forceinline__ bool is_acute_shortcut(const float2* pts, uint32_t point, uint32_t axis1, uint32_t axis2) {
    const float2 P = pts[point], A1 = pts[axis1], A2 = pts[axis2];
    if (angle_clear_of_pi(__fsub_rn(P.y, A1.y), __fsub_rn(P.x, A1.x)) &&
        angle_clear_of_pi(__fsub_rn(P.y, A2.y), __fsub_rn(P.x, A2.x)))
        return true;
    return is_acute(pts, point, axis1, axis2);
}

// emit order of Triangulation.zig:405-422; returns ids packed, count in *cnt (3, or 1 when an
// axis equals the centre -- cannot happen after the equality checks, kept for fidelity)
__device__ __forceinline__ void triangle_order(uint32_t point, uint32_t axis1, uint32_t axis2, uint32_t out[3],
                                               uint32_t* cnt) {
    out[0] = point;
    *cnt = 3;
    if ((axis1 > point && axis2 > point) || (axis1 < point && axis2 < point)) {
        if (axis1 > axis2) {
            out[1] = axis2;
            out[2] = axis1;
        } else {
            out[1] = axis1;
            out[2] = axis2;
        }
    } else if (axis2 > point) {
        out[1] = axis2;
        out[2] = axis1;
    } else if (axis1 > point) {
        out[1] = axis1;
        out[2] = axis2;
    } else {
        *cnt = 1;
    }
}

#include "polygon_sink.cuh"

// Result of one polygon
struct Result {
    uint32_t status;
    uint32_t ntri;
    float b1x, b1y, b2x, b2y;
    bool requeue;
};

// Processes polygon `pi` with workspace `ws` (shared or global memory).  All 32 lanes call it.
__device__ void process_polygon(const BatchArgs& a, uint32_t pi, unsigned char* ws, const Caps caps,
                                const WsLayout L, bool is_tier1, Result* res) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t p0 = a.first_point[pi] - a.point_base;
    const uint64_t np64 = a.first_point[pi + 1] - a.first_point[pi];
    const uint64_t t0 = a.first_tri[pi] - a.tri_base;
    const uint32_t cap_tri = (uint32_t)(a.first_tri[pi + 1] - a.first_tri[pi]);
    const uint32_t n = (uint32_t)(np64 > 0xFFFFFFFFull ? 0xFFFFFFFFull : np64);

    Sink sink;
    sink.base = a.vtx_out + t0 * 3u * a.stride;
    sink.cap_vtx = cap_tri * 3u;
    sink.stride = a.stride;
    sink.off_x = a.off_x;
    sink.off_c = a.off_c;
    sink.fast32 = a.fast32;

    res->status = MR_POLY_OK;
    res->ntri = 0;
    res->b1x = res->b1y = res->b2x = res->b2y = 0.0f;
    res->requeue = false;

    if (n < 3u) {
        res->status = MR_POLY_DEGENERATE;
        sink.zero(0, sink.cap_vtx, lane);
        return;
    }
    if (n > MR_MAX_POLYGON_POINTS) {
        res->status = MR_POLY_TOO_LARGE;
        sink.zero(0, sink.cap_vtx, lane);
        return;
    }
    if (n > caps.nmax) {  // cannot happen: classes are chosen by n
        res->requeue = true;
        return;
    }

    float2* pts = reinterpret_cast<float2*>(ws + L.pts);
    // ---- load points, check finiteness -------------------------------------------------
    bool finite = true;
    {
        const float2* src = reinterpret_cast<const float2*>(a.xy) + p0;
        for (uint32_t i = lane; i < n; i += 32) {
            const float2 v = __ldg(src + i);
            pts[i] = v;
            finite = finite && isfinite(v.x) && isfinite(v.y);
        }
    }
    __syncwarp();
    if (!__all_sync(0xFFFFFFFFu, finite)) {
        res->status = MR_POLY_NONFINITE;
        sink.zero(0, sink.cap_vtx, lane);
        return;
    }

    // ---- unirand (unirand.zig:12-50) -------------------------------------------------------
    uint32_t ur_offset, ur_prime;
    if (a.offset_prime) {
        ur_offset = __ldg(a.offset_prime + 2 * (size_t)pi);
        ur_prime = __ldg(a.offset_prime + 2 * (size_t)pi + 1);
    } else {
        unirand_seed_warp(n, a.seed, a.poly_index0 + pi, lane, &ur_offset, &ur_prime);
    }

    // ---- part 1: trapezoidation (warp-uniform) ------------------------------------------
    Poly P;
    P.pts = pts;
    P.nodes = reinterpret_cast<uint32_t*>(ws + L.nodes);
    P.stack = reinterpret_cast<uint16_t*>(ws + L.stack);
    P.n = n;
    P.nnodes = 0;
    P.nstack = 0;
    P.status = MR_POLY_OK;
    P.spec_node_cap = MR_NODE_CAP(n);
    P.spec_stack_cap = MR_STACK_CAP(n);
    P.tier_node_cap = caps.node_cap;
    P.tier_stack_cap = caps.stack_cap;
    P.requeue = false;
    {
        const uint32_t root = P.alloc();  // :479
        P.set_w0(root, NIL | (NIL << 16));
        P.set_w1(root, NIL | (NIL << 16));
        P.set_w2(root, NIL | (T_TRAPEZOID << 16));
    }
    bool ok = true;
    for (uint32_t at = 0; at < n && ok; ++at) {  // :484-494, unirand.zig:12-21 (u32 arithmetic)
        const uint32_t edge = (uint32_t)(at * ur_prime + ur_offset) % n;
        const uint32_t p1 = edge;
        const uint32_t p2 = (edge + 1u) % n;
        ok = P.add_point(p1) && P.add_point(p2) && P.add_segment(p1, p2);
    }
    if (P.requeue) {
        res->requeue = true;
        return;
    }
    if (!ok) {
        res->status = P.status;
        sink.zero(0, sink.cap_vtx, lane);
        res->status |= (sink.cap_vtx ? MR_POLY_UNDERFILL : 0u);
        return;
    }
    __syncwarp();

    // ---- part 2: inside trapezoids -> adds, in node id order (:510-540) -------------------
    uint32_t* add_pp = reinterpret_cast<uint32_t*>(ws + L.add_pp);
    uint32_t* add_key = reinterpret_cast<uint32_t*>(ws + L.add_key);
    uint16_t* efirst = reinterpret_cast<uint16_t*>(ws + L.efirst);
    uint32_t* add_m = reinterpret_cast<uint32_t*>(ws + L.add_m);
    uint32_t* mcount = reinterpret_cast<uint32_t*>(ws + L.mcount);
    uint32_t* mstart = reinterpret_cast<uint32_t*>(ws + L.mstart);
    const uint32_t lt_mask = (1u << lane) - 1u;

    uint32_t A = 0;
    bool bad = false, over = false;
    for (uint32_t b = 0; b < P.nnodes; b += 32) {
        const uint32_t id = b + lane;
        uint32_t cnt = 0, k0 = 0, k1 = 0, mypp = 0;
        bool lane_bad = false;
        if (id < P.nnodes) {
            const uint32_t tw = P.w2(id);
            if ((tw >> 16) == T_TRAPEZOID) {
                const uint32_t ch = P.w0(id);
                const uint32_t c1 = ch & 0xFFFFu, c2 = ch >> 16;
                if (c1 != NIL) {  // :516
                    const uint32_t c1_crumb = P.w2(c1) & 0xFFFFu;
                    const uint32_t c1_child2 = P.w0(c1) >> 16;
                    if (c1_crumb == c1_child2) {  // :517 is_inside
                        mypp = P.w1(id);
                        if ((mypp & 0xFFFFu) == NIL || (mypp >> 16) == NIL || c2 == NIL) {
                            lane_bad = true;  // :524-527
                        } else {
                            const uint32_t c2pp = P.w1(c2), c1pp = P.w1(c1);
                            if (mypp == c2pp) {  // :528
                                cnt = 1;
                                k0 = c1pp;
                            } else if (mypp == c1pp) {  // :531
                                cnt = 1;
                                k0 = c2pp;
                            } else {  // :534-538
                                cnt = 2;
                                k0 = c1pp;
                                k1 = c2pp;
                            }
                            // MountainList.add_point :56-58 unwraps the key's points
                            if ((k0 & 0xFFFFu) == NIL || (k0 >> 16) == NIL) lane_bad = true;
                            if (cnt == 2 && ((k1 & 0xFFFFu) == NIL || (k1 >> 16) == NIL)) lane_bad = true;
                        }
                    }
                }
            }
        }
        if (__any_sync(0xFFFFFFFFu, lane_bad)) {
            bad = true;
            break;
        }
        const uint32_t m1 = __ballot_sync(0xFFFFFFFFu, cnt >= 1);
        const uint32_t m2 = __ballot_sync(0xFFFFFFFFu, cnt == 2);
        const uint32_t off = A + __popc(m1 & lt_mask) + __popc(m2 & lt_mask);
        const uint32_t total = __popc(m1) + __popc(m2);
        if (A + total > caps.add_cap) {
            over = true;
            break;
        }
        if (cnt >= 1) {
            add_key[off] = k0;  // mountains are keyed by the key node's (point1, point2)  (:52)
            add_pp[off] = mypp;
        }
        if (cnt == 2) {
            add_key[off + 1] = k1;
            add_pp[off + 1] = mypp;
        }
        A += total;
    }
    if (over) {
        if (is_tier1) {  // cannot happen: tier-1 add_cap is 2*node_cap
            res->status = MR_POLY_ARENA;
            sink.zero(0, sink.cap_vtx, lane);
        } else {
            res->requeue = true;
        }
        return;
    }
    if (bad) {
        res->status = MR_POLY_NULL_UNWRAP | (sink.cap_vtx ? MR_POLY_UNDERFILL : 0u);
        sink.zero(0, sink.cap_vtx, lane);
        return;
    }
    __syncwarp();

    // ---- mountains: rank by first appearance, sizes -----------------------------------------
    // A key is normally a segment node, i.e. (upper, lower) of polygon edge e -> table lookup by e.
    // In inconsistent DAG states the reference can leave a non-segment node in a trapezoid's
    // child1/child2; such a key is an arbitrary pair and is matched by scanning the earlier adds.
    for (uint32_t i = lane; i < n; i += 32) efirst[i] = (uint16_t)NIL;
    __syncwarp();
    uint32_t M = 0;
    for (uint32_t b = 0; b < A; b += 32) {
        const uint32_t ai = b + lane;
        const bool valid = ai < A;
        const uint32_t key = valid ? add_key[ai] : 0u;
        const uint32_t ku = key & 0xFFFFu, kl = key >> 16;
        uint32_t e = NIL;  // polygon edge id when the key is (upper, lower) of an edge
        if (valid && ku < n && kl < n && P.above(ku, kl)) {
            if ((ku + 1u == n ? 0u : ku + 1u) == kl) e = ku;
            else if ((kl + 1u == n ? 0u : kl + 1u) == ku) e = kl;
        }
        const uint32_t same = __match_any_sync(0xFFFFFFFFu, valid ? key : (0xFFFF0000u + lane));
        const bool leader = valid && ((same & lt_mask) == 0u);
        uint32_t first = ai;
        if (leader) {
            if (e != NIL) {
                const uint32_t f = efirst[e];
                if (f != NIL) first = f; else efirst[e] = (uint16_t)ai;
            } else {
                for (uint32_t h = 0; h < b; ++h)  // rare: non-edge key
                    if (add_key[h] == key) {
                        first = h;
                        break;
                    }
            }
        }
        first = __shfl_sync(0xFFFFFFFFu, first, __ffs(same) - 1);  // every lane takes its leader's answer
        const bool isfirst = valid && first == ai;
        const uint32_t fm = __ballot_sync(0xFFFFFFFFu, isfirst);
        // first adds store their mountain rank (flag bit 31); the others store the first add's index
        if (valid) add_m[ai] = isfirst ? (0x80000000u | (M + __popc(fm & lt_mask))) : first;
        M += __popc(fm);
        __syncwarp();
    }
    for (uint32_t ai = lane; ai < A; ai += 32) {  // resolve: every add -> mountain rank
        const uint32_t v = add_m[ai];
        if (!(v & 0x80000000u)) add_m[ai] = add_m[v] & 0x7FFFFFFFu;  // add_m[v] is a first add: never rewritten here
    }
    __syncwarp();
    for (uint32_t ai = lane; ai < A; ai += 32) add_m[ai] &= 0x7FFFFFFFu;
    __syncwarp();
    for (uint32_t i = lane; i < M; i += 32) mcount[i] = 0u;
    __syncwarp();
    // entries per mountain (2 per add)
    for (uint32_t ai = lane; ai < A; ai += 32) atomicAdd(&mcount[add_m[ai]], 2u);
    __syncwarp();
    // exclusive scan of mcount over M mountains -> mstart[0..M]
    {
        uint32_t run = 0;
        for (uint32_t b = 0; b < M; b += 32) {
            const uint32_t i = b + lane;
            const uint32_t v = i < M ? mcount[i] : 0u;
            uint32_t inc = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, d);
                if ((int)lane >= d) inc += t;
            }
            if (i < M) mstart[i] = run + inc - v;
            run += __shfl_sync(0xFFFFFFFFu, inc, 31);
        }
        if (lane == 0) mstart[M] = run;
    }
    __syncwarp();
    for (uint32_t i = lane; i < M; i += 32) mcount[i] = 0u;  // reuse as scatter cursor
    __syncwarp();

    // ---- group entries by mountain, then stable sort by (y, x, append position) --------------
    // sortbuf: Gpos[2A] u32, cum[2A] u32, Gid[2A] u16, Gm[2A] u16, S[2A] u16   (aliases nodes in tier 0)
    const uint32_t E = 2u * A;
    const size_t ecap = (size_t)caps.add_cap * 2;
    uint32_t* Gpos = reinterpret_cast<uint32_t*>(ws + L.sortbuf);
    uint32_t* cum = Gpos + ecap;
    uint16_t* Gid = reinterpret_cast<uint16_t*>(cum + ecap);
    uint16_t* Gm = Gid + ecap;
    uint16_t* S = Gm + ecap;
    for (uint32_t ai = lane; ai < A; ai += 32) {
        const uint32_t m = add_m[ai];
        const uint32_t pp = add_pp[ai];
        const uint32_t slot = mstart[m] + atomicAdd(&mcount[m], 2u);
        Gpos[slot] = 2u * ai;  // p1 appended first (:60)
        Gid[slot] = (uint16_t)(pp & 0xFFFFu);
        Gpos[slot + 1] = 2u * ai + 1u;  // then p2 (:61)
        Gid[slot + 1] = (uint16_t)(pp >> 16);
        Gm[slot] = (uint16_t)m;
        Gm[slot + 1] = (uint16_t)m;
    }
    __syncwarp();
    for (uint32_t g = lane; g < E; g += 32) {
        const uint32_t m = Gm[g];
        const uint32_t s = mstart[m], t = mstart[m + 1];
        const uint32_t myid = Gid[g], mypos = Gpos[g];
        const float2 mp = pts[myid];
        uint32_t rank = 0;
        for (uint32_t h = s; h < t; ++h) {
            const float2 op = pts[Gid[h]];
            const bool o_above = (op.y < mp.y) || (op.y == mp.y && op.x < mp.x);
            const bool me_above = (mp.y < op.y) || (mp.y == op.y && mp.x < op.x);
            rank += (o_above || (!me_above && Gpos[h] < mypos)) ? 1u : 0u;
        }
        S[s + rank] = (uint16_t)myid;
    }
    __syncwarp();

    // ---- triangles: valid j, acute check, slots ------------------------------------------------
    uint32_t running = 0;
    bool all_acute = true;
    for (uint32_t b = 0; b < E; b += 32) {
        const uint32_t g = b + lane;
        bool valid = false;
        if (g < E) {
            const uint32_t m = Gm[g];  // entries are grouped, so Gm[g] is the mountain of sorted slot g too
            const uint32_t s = mstart[m];
            if (g >= s + 2u) {
                const uint32_t c = S[g], a1 = S[g - 1], a2 = S[s];
                valid = (c != a1) && (c != a2);
                if (valid && !is_acute(pts, c, a1, a2)) all_acute = false;
            }
        }
        const uint32_t vm = __ballot_sync(0xFFFFFFFFu, valid);
        if (g < E) cum[g] = running + __popc(vm & (lt_mask | (1u << lane)));
        running += __popc(vm);
    }
    all_acute = __all_sync(0xFFFFFFFFu, all_acute);
    __syncwarp();

    float b1x = 0.0f, b2x = 0.0f, lasty = 0.0f;
    bool has_last = false;
    uint32_t ntri_emitted = 0, status = MR_POLY_OK;
    if (all_acute) {
        const uint32_t T = running;
        float mn = 0.0f, mx = 0.0f;
        for (uint32_t g = lane; g < E; g += 32) {
            const uint32_t m = Gm[g];
            const uint32_t s = mstart[m], t = mstart[m + 1];
            if (g < s + 2u) continue;
            const uint32_t c = S[g], a1 = S[g - 1], a2 = S[s];
            if (c == a1 || c == a2) continue;
            // mountains in rank order, inside a mountain from the tail down
            const uint32_t before = s ? cum[s - 1] : 0u;
            const uint32_t slot = before + (cum[t - 1] - cum[g]);
            uint32_t ids[3], cnt;
            triangle_order(c, a1, a2, ids, &cnt);
            const float2 q0 = pts[ids[0]], q1 = pts[ids[1]], q2 = pts[ids[2]];
            mn = fmin_acc(fmin_acc(fmin_acc(mn, q0.x), q1.x), q2.x);
            mx = fmax_acc(fmax_acc(fmax_acc(mx, q0.x), q1.x), q2.x);
            if (slot == T - 1u) {
                lasty = q2.y;
                has_last = true;
            }
            if (slot < cap_tri) {
                sink.write(3u * slot, q0);
                sink.write(3u * slot + 1u, q1);
                sink.write(3u * slot + 2u, q2);
            }
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            mn = fmin_acc(mn, __shfl_xor_sync(0xFFFFFFFFu, mn, d));
            mx = fmax_acc(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, d));
        }
        {  // exactly one lane holds the last triangle (slot T-1), if there is one
            const uint32_t lm = __ballot_sync(0xFFFFFFFFu, has_last);
            lasty = lm ? __shfl_sync(0xFFFFFFFFu, lasty, __ffs(lm) - 1) : 0.0f;
        }
        b1x = mn;
        b2x = mx;
        ntri_emitted = T < cap_tri ? T : cap_tri;
        if (T > cap_tri) status |= MR_POLY_OVERFLOW;
        if (T < cap_tri) {
            status |= MR_POLY_UNDERFILL;
            sink.zero(3u * T, sink.cap_vtx, lane);
        }
        if (T == 0) lasty = 0.0f;
        res->b1x = b1x;
        res->b2x = b2x;
        res->b1y = T ? fmin_acc(b1x, lasty) : 0.0f;
        res->b2y = T ? fmax_acc(b2x, lasty) : 0.0f;
        res->status = status;
        res->ntri = ntri_emitted;
        return;
    }

    // ---- fallback: literal restatement of :553-587 on the sorted lists (warp-uniform) ---------
    {
        uint32_t len_v = 0;  // vertices appended (vertex_array.items.len)
        uint32_t dropped = 0;
        float c1x = 0.0f, c1y = 0.0f, c2x = 0.0f, c2y = 0.0f;
        bool stuck = false;
        for (uint32_t m = 0; m < M; ++m) {
            const uint32_t s = mstart[m];
            uint32_t len = mstart[m + 1] - s;
            uint16_t* Lst = S + s;
            while (len > 2u) {
                uint32_t q1 = len - 2u, q2 = len - 1u, q3 = 0;
                bool progressed = false;
                for (uint32_t item = 1; item < len; ++item) {
                    uint32_t rm = 0xFFFFFFFFu;
                    if (Lst[q1] == Lst[q2]) {
                        rm = q1;
                    } else if (Lst[q2] == Lst[q3]) {
                        rm = q2;
                    } else if (is_acute(pts, Lst[q2], Lst[q1], Lst[q3])) {
                        uint32_t ids[3], cnt;
                        triangle_order(Lst[q2], Lst[q1], Lst[q3], ids, &cnt);
                        for (uint32_t k = 0; k < cnt; ++k) {  // render_point, Polygon.zig:73-78
                            const float2 q = pts[ids[k]];
                            c1x = fmin_acc(c1x, q.x);
                            c1y = fmin_acc(c1x, q.y);
                            c2x = fmax_acc(c2x, q.x);
                            c2y = fmax_acc(c2x, q.y);
                            if (len_v < sink.cap_vtx) {
                                if (lane == 0) sink.write(len_v, q);
                                ++len_v;
                            } else {
                                ++dropped;
                            }
                        }
                        rm = q2;
                    }
                    if (rm != 0xFFFFFFFFu) {  // orderedRemove
                        __syncwarp();
                        if (lane == 0)
                            for (uint32_t k = rm; k + 1u < len; ++k) Lst[k] = Lst[k + 1];
                        __syncwarp();
                        --len;
                        progressed = true;
                        break;
                    }
                    q1 = q2;
                    q2 = q3;
                    q3 = item;
                }
                if (!progressed) {
                    stuck = true;
                    break;
                }
            }
        }
        status = (stuck ? MR_POLY_STUCK : 0u) | (dropped ? MR_POLY_OVERFLOW : 0u);
        if (len_v < sink.cap_vtx) {
            status |= MR_POLY_UNDERFILL;
            __syncwarp();
            sink.zero(len_v, sink.cap_vtx, lane);
        }
        res->status = status;
        res->ntri = len_v / 3u;
        res->b1x = c1x;
        res->b1y = c1y;
        res->b2x = c2x;
        res->b2y = c2y;
    }
}

__device__ __forceinline__ void write_result(const BatchArgs& a, uint32_t pi, const Result& r) {
    if ((threadIdx.x & 31u) == 0) {
        if (a.status_out) a.status_out[pi] = r.status;
        if (a.ntri_out) a.ntri_out[pi] = r.ntri;
        if (a.bbox_out) {
            float4 b = make_float4(r.b1x, r.b1y, r.b2x, r.b2y);
            *reinterpret_cast<float4*>(a.bbox_out + 4 * (size_t)pi) = b;
        }
    }
}

#include "triangulate_fast.cuh"

// ---- kernels ----------------------------------------------------------------------------------
// Fast path, class c, shared-memory workspace.  spec == 0: the class's polygons with arenas sized for
// the typical case; spec == 1: the polygons that outgrew those, with arenas at the contract caps.
// CLS >= 0: the first pass of class CLS, with class and tier known at compile time (caps and layout fold to constants:
// the n <= 64 kernel needs 64 registers instead of 96); CLS < 0: class and tier from the arguments (retry tiers).
// (No minimum-blocks hint: ptxas picks 72 registers for the n <= 64 instantiation on its own; forcing 64, 80 or 96
// through __launch_bounds__ was measured 15-35 % slower.)
template <bool ITEMS, int CLS>
__global__ void __launch_bounds__(MAX_WARPS_PER_BLOCK * 32) triangulate_fast_k(const BatchArgs a, int c_arg, int spec_arg) {
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr bool CLASS0 = CLS == 0;
    const int c = CLS >= 0 ? CLS : c_arg, spec = CLS >= 0 ? 0 : spec_arg;
    const FCaps caps = fast_caps(c, spec != 0);
    const FLayout L = fast_layout(caps);
    unsigned char* ws = smem + (size_t)(threadIdx.x >> 5) * L.total;  // blockDim.x/32 warps per block
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t begin = a.class_begin[c];
    const uint32_t count = spec ? a.spec_count[c] : (a.class_end[c] - begin);
    const uint32_t* list = spec ? a.spec_list : a.order;
    uint32_t* head = spec ? &a.queue_head[NUM_CLASSES + c] : &a.queue_head[c];
    if (count == 0) return;  // empty class: no queue traffic
    unsigned char* const par_gl =
        CLASS0 && a.par_ws ? a.par_ws + (size_t)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * PAR_GL_BYTES : nullptr;
    for (;;) {
        uint32_t idx = 0;
        if (lane == 0) idx = atomicAdd(head, 1u);
        idx = __shfl_sync(0xFFFFFFFFu, idx, 0);
        if (idx >= count) break;
        const uint32_t pi = list[begin + idx];
        Result r;
        int rc = process_polygon_fast<1, ITEMS>(a, pi, ws, caps, L, &r, nullptr, par_gl);
        if (rc == F_REQUEUE_SPEC && spec) rc = F_REQUEUE_GENERAL;  // the spec tier has no bigger shared-memory tier
        if (rc == F_DONE) {
            write_result(a, pi, r);
        } else if (lane == 0) {
            if (rc == F_REQUEUE_SPEC)
                a.spec_list[begin + atomicAdd(&a.spec_count[c], 1u)] = pi;
            else
                a.general_list[atomicAdd(a.general_count, 1u)] = pi;
        }
        __syncwarp();
    }
}

// Fast path for the large classes: one polygon per block, W warps per polygon (see "warp teams" in
// triangulate_fast.cuh).  Typical-case arenas only; overflow goes to the spec tier of triangulate_fast_k.
template <int W>
__global__ void __launch_bounds__(W * 32) triangulate_team_k(const BatchArgs a, int c) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ TeamShared ts;
    const FCaps caps = fast_caps(c, false);
    const FLayout L = fast_layout(caps);
    const uint32_t lane = threadIdx.x & 31u;
    const bool main_warp = threadIdx.x < 32u;
    const uint32_t begin = a.class_begin[c];
    const uint32_t count = a.class_end[c] - begin;
    if (count == 0) return;  // empty class: no queue traffic
    for (;;) {
        if (threadIdx.x == 0) ts.qidx = atomicAdd(&a.queue_head[c], 1u);
        __syncthreads();
        const uint32_t idx = ts.qidx;
        if (idx >= count) break;
        const uint32_t pi = a.order[begin + idx];
        if (main_warp) {
            Result r;
            const int rc = process_polygon_fast<W, true>(a, pi, smem, caps, L, &r, &ts);
            if (lane == 0) ts.cmd = TEAM_STOP;
            team_bar<W>();
            if (rc == F_DONE) {
                write_result(a, pi, r);
            } else if (lane == 0) {
                // (the XL class has no contract-cap tier: both kinds of hand-over go to its slice of spec_list, which
                // the global-memory general kernel of the > 1024-point polygons consumes)
                if (rc == F_REQUEUE_SPEC || c == XL_CLASS)
                    a.spec_list[begin + atomicAdd(&a.spec_count[c], 1u)] = pi;
                else
                    a.general_list[atomicAdd(a.general_count, 1u)] = pi;
            }
        } else {
            team_helper<W>(a, pi, smem, caps, L, &ts);
        }
    }
}

// General path (float compares, 12-byte nodes, literal fallback loop), global-memory workspace:
// which == 0: polygons handed over by the fast path (coincident points, not-acute corner, oversized
// mountain lists; n <= 1024); which == 1: the last class (3072 < n <= MR_MAX_POLYGON_POINTS), then the polygons the
// XL class (1025..3072) handed over.
__global__ void __launch_bounds__(MAX_WARPS_PER_BLOCK * 32) triangulate_general_k(const BatchArgs a, uint32_t nmax, int which) {
    const Caps caps = tier1_caps(nmax);
    const WsLayout L = ws_layout(caps, false);
    const uint32_t warp_global = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    unsigned char* ws = a.tier1_ws + (size_t)warp_global * a.tier1_ws_stride;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t c = NUM_CLASSES - 1;
    const uint32_t begin = a.class_begin[c], end = a.class_end[c];
    const uint32_t xl_begin = a.class_begin[XL_CLASS];
    const uint32_t total = which == 0 ? *a.general_count : (end - begin) + a.spec_count[XL_CLASS];
    for (;;) {
        uint32_t idx = 0;
        if (lane == 0) idx = atomicAdd(&a.queue_head[2 * NUM_CLASSES + which], 1u);
        idx = __shfl_sync(0xFFFFFFFFu, idx, 0);
        if (idx >= total) break;
        const uint32_t pi = which == 0 ? a.general_list[idx]
                                       : (idx < end - begin ? a.order[begin + idx] : a.spec_list[xl_begin + (idx - (end - begin))]);
        Result r;
        process_polygon(a, pi, ws, caps, L, true, &r);
        write_result(a, pi, r);
        __syncwarp();
    }
}

// work lists: polygons sorted by size, largest first (counting sort on n), so that every tier's queue
// hands out its most expensive polygons first and the kernel tail consists of the cheapest ones
__device__ __forceinline__ uint32_t size_bin(uint64_t n) { return n > MR_MAX_POLYGON_POINTS ? 0u : (uint32_t)n; }  // invalid sizes ride in bin 0

__global__ void __launch_bounds__(256) size_hist_k(const uint64_t* __restrict__ first_point, uint32_t npoly,
                                                  uint32_t* __restrict__ hist) {
    __shared__ uint32_t local[NBINS];
    for (uint32_t b = threadIdx.x; b < NBINS; b += blockDim.x) local[b] = 0;
    __syncthreads();
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npoly; i += gridDim.x * blockDim.x)
        atomicAdd(&local[size_bin(first_point[i + 1] - first_point[i])], 1u);
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < NBINS; b += blockDim.x)
        if (local[b]) atomicAdd(&hist[b], local[b]);
}

// one block: cursor[b] = number of polygons with a size larger than b (descending order); class ranges
__global__ void __launch_bounds__(1024) size_scan_k(const uint32_t* __restrict__ hist, uint32_t* __restrict__ cursor,
                                                   uint32_t* __restrict__ class_begin, uint32_t* __restrict__ class_end) {
    __shared__ uint32_t part[1024];
    constexpr int PER = (NBINS + 1023) / 1024;
    // thread t owns bins NBINS-1-t*PER ... (descending)
    uint32_t sum = 0;
    for (int k = 0; k < PER; ++k) {
        const int b = NBINS - 1 - (int)(threadIdx.x * PER + k);
        if (b >= 0) sum += hist[b];
    }
    part[threadIdx.x] = sum;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {  // inclusive scan
        const uint32_t v = threadIdx.x >= (unsigned)d ? part[threadIdx.x - d] : 0u;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t run = part[threadIdx.x] - sum;
    for (int k = 0; k < PER; ++k) {
        const int b = NBINS - 1 - (int)(threadIdx.x * PER + k);
        if (b >= 0) {
            cursor[b] = run;
            run += hist[b];
        }
    }
    __syncthreads();
    if (threadIdx.x < NUM_CLASSES) {
        const int c = threadIdx.x;
        const uint32_t hi = c == NUM_CLASSES - 1 ? MR_MAX_POLYGON_POINTS : class_nmax(c);  // largest size of the class
        const uint32_t lo = c == 0 ? 0u : class_nmax(c - 1) + 1u;                          // smallest size
        class_begin[c] = cursor[hi];
        class_end[c] = cursor[lo] + hist[lo];
    }
}

__global__ void size_scatter_k(const uint64_t* __restrict__ first_point, uint32_t npoly,
                               uint32_t* __restrict__ cursor, uint32_t* __restrict__ order) {
    // warp-aggregated: one atomic per distinct size per warp (a batch of small polygons has only a few dozen sizes)
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t step = gridDim.x * blockDim.x;
    for (uint32_t i0 = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); i0 < npoly; i0 += step) {
        const uint32_t i = i0 + lane;
        const bool valid = i < npoly;
        const uint32_t bin = valid ? size_bin(first_point[i + 1] - first_point[i]) : 0xFFFFFFFFu;
        const uint32_t same = __match_any_sync(0xFFFFFFFFu, bin);
        const uint32_t leader = __ffs(same) - 1u;
        uint32_t base = 0;
        if (valid && lane == leader) base = atomicAdd(&cursor[bin], (uint32_t)__popc(same));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (valid) order[base + __popc(same & ((1u << lane) - 1u))] = i;
    }
}

__global__ void polygon_offsets_k(const uint64_t* __restrict__ first_point, uint32_t npoly,
                                  uint64_t* __restrict__ tri_count) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npoly; i += gridDim.x * blockDim.x) {
        const uint64_t n = first_point[i + 1] - first_point[i];
        tri_count[i] = n >= 2 ? n - 2 : 0;
    }
}

// with holes: N + 2H - sub, H = rings - 1 when 1 <= rings <= N (else 0), clamped at 0
__global__ void polygon_ring_counts_k(const uint64_t* __restrict__ first_point, const uint64_t* __restrict__ first_ring,
                                      uint32_t npoly, uint32_t sub, uint64_t* __restrict__ count) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npoly; i += gridDim.x * blockDim.x) {
        const uint64_t n = first_point[i + 1] - first_point[i], r = first_ring[i + 1] - first_ring[i];
        const uint64_t t = n + (r >= 1 && r <= n ? 2 * (r - 1) : 0);
        count[i] = t >= sub ? t - sub : 0;
    }
}

// single-block exclusive scan of u64 counts (npoly up to a few million: chunked loop)
__global__ void __launch_bounds__(1024) exclusive_scan_u64_k(const uint64_t* __restrict__ in, uint32_t count,
                                                            uint64_t* __restrict__ out) {
    __shared__ uint64_t warp_sums[32];
    __shared__ uint64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    for (uint32_t base = 0; base < count; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const uint64_t v = i < count ? in[i] : 0;
        uint64_t inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint64_t t = __shfl_up_sync(0xFFFFFFFFu, inc, d);
            if ((int)lane >= d) inc += t;
        }
        if (lane == 31) warp_sums[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            uint64_t w = warp_sums[lane];
            uint64_t winc = w;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint64_t t = __shfl_up_sync(0xFFFFFFFFu, winc, d);
                if ((int)lane >= d) winc += t;
            }
            warp_sums[lane] = winc - w;
        }
        __syncthreads();
        const uint64_t c = carry;
        if (i < count) out[i] = c + warp_sums[warp] + inc - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = c + warp_sums[warp] + inc;
        __syncthreads();
    }
    if (threadIdx.x == 0) out[count] = carry;
}

__global__ void unirand_seed_batch_k(const uint64_t* __restrict__ first_point, uint32_t npoly, uint64_t seed,
                                     uint64_t poly_index0, uint32_t* __restrict__ out) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t i = warp; i < npoly; i += nwarps) {
        const uint64_t n64 = first_point[i + 1] - first_point[i];
        const uint32_t n = (uint32_t)(n64 > 0xFFFFFFFFull ? 0xFFFFFFFFull : n64);
        uint32_t off, prime;
        unirand_seed_warp(n, seed, poly_index0 + i, lane, &off, &prime);
        if (lane == 0) {
            out[2 * (size_t)i] = off;
            out[2 * (size_t)i + 1] = prime;
        }
    }
}

}  // namespace

// ---- host side -------------------------------------------------------------------------------
// header of the work-list memory (words)
enum { HDR_CLASS_BEGIN = 0, HDR_CLASS_END = CLASS_SLOTS, HDR_QUEUE_HEAD = 2 * CLASS_SLOTS, HDR_SPEC_COUNT = 5 * CLASS_SLOTS,
       HDR_GENERAL_COUNT = 6 * CLASS_SLOTS, HEADER_WORDS = 8 * CLASS_SLOTS };
static_assert(NUM_CLASSES <= CLASS_SLOTS && 2 * NUM_CLASSES + 2 <= 3 * CLASS_SLOTS, "work-list header too small");

int mr_polygon_size_sort(mr_context* ctx, const uint64_t* first_point, uint32_t npoly, uint32_t* hist, uint32_t* cursor,
                         uint32_t* class_begin, uint32_t* class_end, uint32_t* order) {
    static_assert(NBINS == MR_SIZE_BINS, "size bins");
    const unsigned cblocks = (unsigned)std::min<uint64_t>(((uint64_t)npoly + 255) / 256, (uint64_t)ctx->sm_count * 2);
    size_hist_k<<<cblocks, 256, 0, ctx->stream>>>(first_point, npoly, hist);
    MR_LAUNCH_CHECK(ctx, "size_hist_k");
    size_scan_k<<<1, 1024, 0, ctx->stream>>>(hist, cursor, class_begin, class_end);
    MR_LAUNCH_CHECK(ctx, "size_scan_k");
    size_scatter_k<<<cblocks, 256, 0, ctx->stream>>>(first_point, npoly, cursor, order);
    MR_LAUNCH_CHECK(ctx, "size_scatter_k");
    return MR_OK;
}

int mr_polygon_offsets_impl(mr_context* ctx, const uint64_t* first_point_dev, uint32_t npoly,
                            uint64_t* first_tri_dev) {
    // counts are written into first_tri_dev[0..npoly) then scanned in place via a temp
    void* tmp = nullptr;
    int rc = mr_scratch(ctx, MR_SLOT_MISC, (size_t)(npoly + 1) * 8, &tmp);
    if (rc) return rc;
    const unsigned blocks = (unsigned)std::min<uint64_t>(((uint64_t)npoly + 255) / 256 + 1, 1024);
    polygon_offsets_k<<<blocks, 256, 0, ctx->stream>>>(first_point_dev, npoly, static_cast<uint64_t*>(tmp));
    MR_LAUNCH_CHECK(ctx, "polygon_offsets_k");
    exclusive_scan_u64_k<<<1, 1024, 0, ctx->stream>>>(static_cast<uint64_t*>(tmp), npoly, first_tri_dev);
    MR_LAUNCH_CHECK(ctx, "exclusive_scan_u64_k");
    return MR_OK;
}

int mr_polygon_ring_counts(mr_context* ctx, const uint64_t* first_point, const uint64_t* first_ring, uint32_t npoly,
                           uint32_t sub, uint64_t* out) {
    void* tmp = nullptr;
    int rc = mr_scratch(ctx, MR_SLOT_MISC, (size_t)(npoly + 1) * 8, &tmp);
    if (rc) return rc;
    const unsigned blocks = (unsigned)std::min<uint64_t>(((uint64_t)npoly + 255) / 256 + 1, 1024);
    polygon_ring_counts_k<<<blocks, 256, 0, ctx->stream>>>(first_point, first_ring, npoly, sub, static_cast<uint64_t*>(tmp));
    MR_LAUNCH_CHECK(ctx, "polygon_ring_counts_k");
    exclusive_scan_u64_k<<<1, 1024, 0, ctx->stream>>>(static_cast<uint64_t*>(tmp), npoly, out);
    MR_LAUNCH_CHECK(ctx, "exclusive_scan_u64_k");
    return MR_OK;
}

int mr_unirand_seed_batch_impl(mr_context* ctx, const uint64_t* first_point_dev, uint32_t npoly, uint64_t seed,
                               uint64_t poly_index0, uint32_t* out_dev) {
    if (npoly == 0) return MR_OK;
    const unsigned blocks = (unsigned)std::min<uint64_t>(((uint64_t)npoly + 3) / 4, (uint64_t)ctx->sm_count * 8);
    unirand_seed_batch_k<<<blocks, 128, 0, ctx->stream>>>(first_point_dev, npoly, seed, poly_index0, out_dev);
    MR_LAUNCH_CHECK(ctx, "unirand_seed_batch_k");
    return MR_OK;
}

int mr_triangulate_tier_counts_impl(mr_context* ctx, uint32_t out[8]) {
    memset(out, 0, 8 * sizeof(uint32_t));
    if (!ctx->last_header_dev) return MR_OK;
    uint32_t hdr[HEADER_WORDS];
    MR_CUDA(ctx, cudaMemcpyAsync(hdr, ctx->last_header_dev, sizeof(hdr), cudaMemcpyDeviceToHost, ctx->stream));
    MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    // spec_count per internal class, folded into the documented size tiers <=64, <=128, <=256, <=512, <=1024
    for (int c = 0; c < NUM_CLASSES - 1; ++c) {
        const uint32_t nmax = class_nmax(c);
        const int tier = nmax <= 64u ? 0 : nmax <= 128u ? 1 : nmax <= 256u ? 2 : nmax <= 512u ? 3 : nmax <= 1024u ? 4 : 5;
        out[tier] += hdr[HDR_SPEC_COUNT + c];  // (tier 5, 1025..3072 points: handed to the general path, there is no retry tier)
    }
    out[6] = hdr[HDR_GENERAL_COUNT];
    out[7] = hdr[HDR_CLASS_END + NUM_CLASSES - 1] - hdr[HDR_CLASS_BEGIN + NUM_CLASSES - 1];  // the > 3072 class
    return MR_OK;
}

// ---- launch plan --------------------------------------------------------------------------------------------
// Kernel, block shape, blocks per SM and shared memory of every (size class, tier).  The function attributes and
// occupancy queries behind it cost ~50 driver calls; they are made once per context, not once per batch.
namespace {
struct ClassLaunch {
    const void* kern;  // triangulate_team_k<W> (args: BatchArgs, int) when team > 1, else triangulate_fast_k<..> (BatchArgs, int, int)
    int team;          // warps cooperating on one polygon (1 = independent warps)
    int wpb;           // warps per block
    int per_sm;        // resident blocks per SM
    size_t smem;       // dynamic shared memory per block
};
struct PolyPlan {
    ClassLaunch first[NUM_CLASSES - 1], spec[NUM_CLASSES - 1];
};

int build_plan(mr_context* ctx, PolyPlan* plan) {
    for (int spec = 0; spec < 2; ++spec) {
        for (int c = 0; c < NUM_CLASSES - 1; ++c) {
            ClassLaunch& out = spec ? plan->spec[c] : plan->first[c];
            const FCaps caps = fast_caps(c, spec != 0);
            const FLayout L = fast_layout(caps);
            if (spec && c == XL_CLASS) {  // contract-cap arenas of a 3072-point polygon do not fit shared memory
                out = {nullptr, 1, 1, 0, 0};
                continue;
            }
            if (!fast_layout_ok(caps, L)) return mr_fail(ctx, MR_E_CUDA, "fast-path workspace layout is inconsistent");
            if (L.total > ctx->smem_optin) return mr_fail(ctx, MR_E_CUDA, "fast-path workspace exceeds shared memory");
            const int team = spec ? 1 : team_warps(c);
            if (team > 1) {  // one polygon per block, `team` warps per polygon
                void (*kern)(const BatchArgs, int) = nullptr;  // one instantiation per team width: see team_warps
                switch (team) {
                    case 3: kern = triangulate_team_k<3>; break;
                    case 4: kern = triangulate_team_k<4>; break;
                    case 6: kern = triangulate_team_k<6>; break;
                    case 8: kern = triangulate_team_k<8>; break;
                }
                if (!kern) return mr_fail(ctx, MR_E_CUDA, "no team kernel of this width");
                MR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
                int per_sm = 0;
                MR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, team * 32, L.total));
                out = {reinterpret_cast<const void*>(kern), team, team, per_sm < 1 ? 1 : per_sm, L.total};
            } else {
                // independent warps, 4, 2 or 1 per block: whichever puts the most polygons on an SM (ties: larger blocks)
                void (*kern)(const BatchArgs, int, int) = triangulate_fast_k<false, -1>;  // retry tiers
                if (!spec) {
                    switch (c) {
                        case 0: kern = triangulate_fast_k<false, 0>; break;
                        // (compile-time class constants were measured for the other kernels too: no gain for the
                        // single-warp conflict-list classes, 8 % slower for the team kernels)
                        case 1: case 2: case 3: case 4: case 5: kern = triangulate_fast_k<true, -1>; break;
                        default: return mr_fail(ctx, MR_E_CUDA, "no single-warp kernel for this class");
                    }
                }
                // one attribute per kernel function: the largest block any class launches it with
                int wpb = 1, per_sm = 1;
                for (int w = MAX_WARPS_PER_BLOCK; w >= 1; w >>= 1) {
                    if (L.total * w > ctx->smem_optin) continue;
                    cudaFuncAttributes fa;
                    MR_CUDA(ctx, cudaFuncGetAttributes(&fa, kern));
                    if ((size_t)fa.maxDynamicSharedSizeBytes < L.total * w)
                        MR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(L.total * w)));
                    int b = 0;
                    MR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kern, w * 32, L.total * w));
                    if (b * w > per_sm * wpb || (w == MAX_WARPS_PER_BLOCK && b >= 1)) {
                        wpb = w;
                        per_sm = b;
                    }
                }
                out = {reinterpret_cast<const void*>(kern), 1, wpb, per_sm, L.total * wpb};
            }
        }
    }
    return MR_OK;
}

int get_plan(mr_context* ctx, PolyPlan** plan_out) {
    if (!ctx->poly_plan) {
        PolyPlan* p = new (std::nothrow) PolyPlan();
        if (!p) return mr_fail(ctx, MR_E_NOMEM, "polygon launch plan");
        const int rc = build_plan(ctx, p);
        if (rc) {
            delete p;
            return rc;
        }
        ctx->poly_plan = p;
    }
    *plan_out = static_cast<PolyPlan*>(ctx->poly_plan);
    return MR_OK;
}

// launches class c's kernel of the given tier; `units` = polygons it can possibly find in its queue (bounds the grid)
int launch_class(mr_context* ctx, const ClassLaunch& L, BatchArgs& a, int c, int spec, cudaStream_t st, uint32_t units) {
    uint64_t grid = (uint64_t)ctx->sm_count * L.per_sm;
    const uint64_t need = L.team > 1 ? units : ((uint64_t)units + L.wpb - 1) / L.wpb;
    if (need < grid) grid = need ? need : 1;
    if (L.team > 1) {
        void* args[] = {&a, &c};
        MR_CUDA(ctx, cudaLaunchKernel(L.kern, dim3((unsigned)grid), dim3(L.wpb * 32), args, L.smem, st));
    } else {
        void* args[] = {&a, &c, &spec};
        MR_CUDA(ctx, cudaLaunchKernel(L.kern, dim3((unsigned)grid), dim3(L.wpb * 32), args, L.smem, st));
    }
    MR_LAUNCH_CHECK(ctx, L.team > 1 ? "triangulate_team_k" : "triangulate_fast_k");
    return MR_OK;
}

void fill_batch_args(BatchArgs& a, const mr_polygon_job* j, uint32_t* header, uint32_t* order, uint32_t* spec_list,
                     uint32_t* general_list) {
    a.xy = j->xy;
    a.first_point = j->first_point;
    a.point_base = j->point_base;
    a.npoly = j->npoly;
    a.offset_prime = j->offset_prime;
    a.seed = j->seed;
    a.poly_index0 = j->poly_index0;
    a.vtx_out = static_cast<unsigned char*>(j->vtx_out);
    a.first_tri = j->first_tri;
    a.tri_base = j->tri_base;
    a.bbox_out = j->bbox_out;
    a.status_out = j->status_out;
    a.ntri_out = j->ntri_out;
    sink_layout(a, j->layout, a.vtx_out);
    a.order = order;
    a.class_begin = header + HDR_CLASS_BEGIN;
    a.class_end = header + HDR_CLASS_END;
    a.queue_head = header + HDR_QUEUE_HEAD;
    a.spec_list = spec_list;
    a.spec_count = header + HDR_SPEC_COUNT;
    a.general_list = general_list;
    a.general_count = header + HDR_GENERAL_COUNT;
    a.tier1_ws = nullptr;
    a.tier1_ws_stride = 0;
    a.par_ws = nullptr;
}

// global scratch of the n <= 64 kernel's parallel search: one slice per warp of its full grid
int class0_scratch(mr_context* ctx, const PolyPlan& plan, BatchArgs& a) {
    void* pw = nullptr;
    const ClassLaunch& L0 = plan.first[0];
    const int rc = mr_scratch(ctx, MR_SLOT_PAR, (size_t)ctx->sm_count * L0.per_sm * L0.wpb * PAR_GL_BYTES, &pw);
    if (rc) return rc;
    a.par_ws = static_cast<unsigned char*>(pw);
    return MR_OK;
}

// general path: global-memory workspaces, one per warp of the grid.  which == 0: polygons handed over by the fast
// path; which == 1: the 1025..MR_MAX_POLYGON_POINTS class.
int launch_general(mr_context* ctx, BatchArgs& a, int which, uint32_t units) {
    const uint32_t nmax = which == 0 ? class_nmax(XL_CLASS - 1) : MR_MAX_POLYGON_POINTS;
    const Caps c1 = tier1_caps(nmax);
    const WsLayout L1 = ws_layout(c1, false);
    const int wpb = which == 0 ? 4 : 1;
    uint64_t blocks = (uint64_t)ctx->sm_count;
    const uint64_t need = ((uint64_t)units + wpb - 1) / wpb;
    if (need < blocks) blocks = need ? need : 1;
    void* t1 = nullptr;
    const int rc = mr_scratch(ctx, which == 0 ? MR_SLOT_TIER1 : MR_SLOT_TIER1B, (size_t)blocks * wpb * L1.total, &t1);
    if (rc) return rc;
    a.tier1_ws = static_cast<unsigned char*>(t1);
    a.tier1_ws_stride = L1.total;
    triangulate_general_k<<<(unsigned)blocks, wpb * 32, 0, ctx->stream>>>(a, nmax, which);
    MR_LAUNCH_CHECK(ctx, "triangulate_general_k");
    return MR_OK;
}
}  // namespace

void mr_polygon_plan_free(mr_context* ctx) {
    delete static_cast<PolyPlan*>(ctx->poly_plan);
    ctx->poly_plan = nullptr;
}

int mr_triangulate_impl(mr_context* ctx, const mr_polygon_job* j, const uint64_t* first_point_host) {
    // all pointers in *j are device pointers here (staging happened in api.cu)
    const uint32_t npoly = j->npoly;
    if (npoly == 0) return MR_OK;
    PolyPlan* plan = nullptr;
    int rc = get_plan(ctx, &plan);
    if (rc) return rc;

    // work-list memory: header | hist[NBINS] | cursor[NBINS] | order[npoly] | spec_list[npoly] | general_list[npoly]
    const size_t header_words = HEADER_WORDS;
    void* work = nullptr;
    rc = mr_scratch(ctx, MR_SLOT_WORK, (header_words + 2 * (size_t)NBINS + 3 * (size_t)npoly) * 4, &work);
    if (rc) return rc;
    uint32_t* w = static_cast<uint32_t*>(work);
    uint32_t* hist = w + header_words;
    uint32_t* cursor = hist + NBINS;
    uint32_t* order = cursor + NBINS;
    uint32_t* spec_list = order + npoly;
    uint32_t* general_list = spec_list + npoly;
    ctx->last_header_dev = w;
    MR_CUDA(ctx, cudaMemsetAsync(w, 0, (header_words + 2 * (size_t)NBINS) * 4, ctx->stream));

    rc = mr_polygon_size_sort(ctx, j->first_point, npoly, hist, cursor, w + HDR_CLASS_BEGIN, w + HDR_CLASS_END, order);
    if (rc) return rc;

    // Polygons per class: known exactly when the caller's first_point lives on the host (then empty classes cost no
    // launch at all); otherwise every class may hold up to npoly polygons and its kernel finds out on the device.
    uint32_t count[NUM_CLASSES];
    for (int c = 0; c < NUM_CLASSES; ++c) count[c] = first_point_host ? 0u : npoly;
    if (first_point_host)
        for (uint32_t i = 0; i < npoly; ++i) {
            const uint64_t n = first_point_host[i + 1] - first_point_host[i];
            ++count[class_of(n > MR_MAX_POLYGON_POINTS ? 0u : (uint32_t)n)];  // invalid sizes ride in bin 0 (size_bin)
        }

    BatchArgs a;
    fill_batch_args(a, j, w, order, spec_list, general_list);
    if (count[0]) {
        rc = class0_scratch(ctx, *plan, a);
        if (rc) return rc;
    }

    // fast path: per class, first with typical-case arenas, then the overflow with contract-cap arenas.  The first pass
    // runs class after class on the caller's stream (measured: running the classes concurrently costs the 1M-polygon
    // batch 4 %, the large classes lose SM residency to the small ones; splitting off only the n <= 64 class gains
    // nothing).  The second pass is up to ten mostly empty kernels: each goes to its own side stream, so their launch
    // latencies overlap; the caller's stream forks and joins around it.
    static_assert(NUM_CLASSES - 1 <= MR_NUM_AUX, "one side stream per shared-memory class");
    for (int c = 0; c < NUM_CLASSES - 1; ++c) {
        if (!count[c]) continue;
        rc = launch_class(ctx, plan->first[c], a, c, 0, ctx->stream, count[c]);
        if (rc) return rc;
    }
    if (mr_aux_streams(ctx)) return mr_fail(ctx, MR_E_CUDA, "side streams");
    MR_CUDA(ctx, cudaEventRecord(ctx->fork_ev, ctx->stream));
    int first_error = MR_OK;
    bool forked[NUM_CLASSES - 1] = {false};
    for (int c = 0; c < NUM_CLASSES - 1 && !first_error; ++c) {
        if (!count[c] || !plan->spec[c].kern) continue;
        cudaStream_t st = ctx->aux[c];
        if (cudaStreamWaitEvent(st, ctx->fork_ev, 0) != cudaSuccess) { first_error = mr_fail(ctx, MR_E_CUDA, "cudaStreamWaitEvent"); break; }
        forked[c] = true;
        first_error = launch_class(ctx, plan->spec[c], a, c, 1, st, count[c]);
    }
    for (int c = 0; c < NUM_CLASSES - 1; ++c) {  // join every stream that was forked, also on the error path
        if (!forked[c]) continue;
        if (cudaEventRecord(ctx->join_ev[c], ctx->aux[c]) != cudaSuccess || cudaStreamWaitEvent(ctx->stream, ctx->join_ev[c], 0) != cudaSuccess)
            if (!first_error) first_error = mr_fail(ctx, MR_E_CUDA, "side-stream join");
    }
    if (first_error) return first_error;
    // general path
    uint32_t shared_total = 0;
    for (int c = 0; c < XL_CLASS; ++c) shared_total += count[c];
    if (shared_total) {
        rc = launch_general(ctx, a, 0, first_point_host ? shared_total : npoly);
        if (rc) return rc;
    }
    if (count[NUM_CLASSES - 1] || count[XL_CLASS]) {
        rc = launch_general(ctx, a, 1, first_point_host ? count[NUM_CLASSES - 1] + count[XL_CLASS] : npoly);
        if (rc) return rc;
    }
    return MR_OK;
}

// ---- small-batch path -----------------------------------------------------------------------------------------
// The reference's own call (Polygon.create_polygon, Polygon.zig:81-107; App.zig:68-83) triangulates ONE small polygon
// whose points, vertex buffer and bounding box all live in host memory.  For such jobs the batch machinery above is
// almost pure overhead (work-list kernels, a dozen staging copies, twenty launches).  Here the whole call is
//     one host->device copy   [xy | first_point | first_tri | offset_prime | order | header]      (work list built on the host)
//     one kernel per non-empty size class (one for App.zig's polygons)
//     one device->host copy   [header | status | ntri | bbox | vertices]
//     one stream synchronisation
// through a pinned block owned by the context.  The header comes back with the outputs; only if it reports polygons
// that outgrew their first-pass arenas (rare) are the retry tiers launched and the outputs copied again.
namespace {
constexpr uint32_t SMALL_MAX_POLYS = 2048;
constexpr size_t SMALL_MAX_BYTES = 8u << 20;
inline size_t up16(size_t x) { return (x + 15) & ~(size_t)15; }
}  // namespace

int mr_triangulate_small(mr_context* ctx, const mr_polygon_job* jp, int* rc_out) {
    const mr_polygon_job& j = *jp;
    *rc_out = MR_OK;
    const uint32_t npoly = j.npoly;
    if (npoly == 0 || npoly > SMALL_MAX_POLYS) return 0;
    // every buffer in plain host memory (a pinned vertex buffer takes the zero-copy route of the batch path)
    const void* ptrs[] = {j.xy, j.first_point, j.first_tri, j.vtx_out, j.offset_prime, j.bbox_out, j.status_out, j.ntri_out};
    for (const void* p : ptrs) {
        if (!p) continue;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
            cudaGetLastError();
            continue;  // unregistered host memory
        }
        if (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) return 0;
        if (p == j.vtx_out && at.type == cudaMemoryTypeHost) return 0;
    }
    if (j.first_point[0] < j.point_base || j.first_tri[0] < j.tri_base) return 0;  // the batch path reports it
    const uint64_t pts0 = j.first_point[0] - j.point_base, npts = j.first_point[npoly] - j.first_point[0];
    const uint64_t tri0 = j.first_tri[0] - j.tri_base, ntri = j.first_tri[npoly] - j.first_tri[0];
    const size_t vbytes = (size_t)ntri * 3u * j.layout.stride;
    // block layout
    size_t o = 0;
    const size_t o_xy = o;    o += up16((size_t)npts * 8);
    const size_t o_fp = o;    o += up16((size_t)(npoly + 1) * 8);
    const size_t o_ft = o;    o += up16((size_t)(npoly + 1) * 8);
    const size_t o_op = o;    o += j.offset_prime ? up16((size_t)npoly * 8) : 0;
    const size_t o_order = o; o += up16((size_t)npoly * 4);
    const size_t o_hdr = o;   o += up16((size_t)HEADER_WORDS * 4);
    const size_t in_end = o;
    const size_t o_stat = o;  o += up16((size_t)npoly * 4);
    const size_t o_ntri = o;  o += up16((size_t)npoly * 4);
    const size_t o_bbox = o;  o += up16((size_t)npoly * 16);
    const size_t o_vtx = (o + 31) & ~(size_t)31;
    o = o_vtx + up16(vbytes);
    const size_t out_end = o;
    const size_t o_spec = o;  o += up16((size_t)npoly * 4);   // device only
    const size_t o_gen = o;   o += up16((size_t)npoly * 4);   // device only
    if (npts > (1u << 20) || ntri > (1u << 20) || o > SMALL_MAX_BYTES) return 0;  // (also catches non-monotonic offsets)

    auto fail = [&](int rc) { *rc_out = rc; return 1; };
    PolyPlan* plan = nullptr;
    int rc = get_plan(ctx, &plan);
    if (rc) return fail(rc);
    if (ctx->small_bytes < o) {
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return fail(mr_fail(ctx, MR_E_CUDA, "sync"));
        if (ctx->small_pinned) cudaFreeHost(ctx->small_pinned);
        if (ctx->small_dev) cudaFree(ctx->small_dev);
        ctx->small_pinned = ctx->small_dev = nullptr;
        ctx->small_bytes = 0;
        const size_t want = std::max<size_t>(o * 2, 64u << 10);
        if (cudaMallocHost(&ctx->small_pinned, want) != cudaSuccess || cudaMalloc(&ctx->small_dev, want) != cudaSuccess) {
            cudaGetLastError();
            return fail(mr_fail(ctx, MR_E_NOMEM, "small-batch block"));
        }
        ctx->small_bytes = want;
    }
    unsigned char* hb = static_cast<unsigned char*>(ctx->small_pinned);
    unsigned char* db = static_cast<unsigned char*>(ctx->small_dev);

    // ---- inputs and the work list, built on the host ------------------------------------------------------
    memcpy(hb + o_xy, j.xy + 2 * pts0, (size_t)npts * 8);
    uint64_t* fp = reinterpret_cast<uint64_t*>(hb + o_fp);
    uint64_t* ft = reinterpret_cast<uint64_t*>(hb + o_ft);
    for (uint32_t i = 0; i <= npoly; ++i) {  // rebased: the block's xy / vertex arrays start at this job's first entries
        fp[i] = j.first_point[i] - j.first_point[0];
        ft[i] = j.first_tri[i] - j.first_tri[0];
    }
    if (j.offset_prime) memcpy(hb + o_op, j.offset_prime, (size_t)npoly * 8);
    uint32_t* hdr = reinterpret_cast<uint32_t*>(hb + o_hdr);
    uint32_t* order = reinterpret_cast<uint32_t*>(hb + o_order);
    memset(hdr, 0, (size_t)HEADER_WORDS * 4);
    uint32_t count[NUM_CLASSES] = {0};
    auto cls = [&](uint32_t i) {
        const uint64_t n = fp[i + 1] - fp[i];
        return class_of(n > MR_MAX_POLYGON_POINTS ? 0u : (uint32_t)n);
    };
    for (uint32_t i = 0; i < npoly; ++i) ++count[cls(i)];
    {   // queue order: class by class; inside a class largest first (stable counting sort on the size, like size_scatter_k
        // up to the order among equal sizes, which does not affect results)
        uint32_t begin[NUM_CLASSES], run = 0;
        for (int c = NUM_CLASSES - 1; c >= 0; --c) {  // descending sizes overall: the last class first, like the device sort
            begin[c] = run;
            hdr[HDR_CLASS_BEGIN + c] = run;
            run += count[c];
            hdr[HDR_CLASS_END + c] = run;
        }
        std::vector<std::pair<uint32_t, uint32_t>> keyed(npoly);
        for (uint32_t i = 0; i < npoly; ++i) keyed[i] = {(uint32_t)std::min<uint64_t>(fp[i + 1] - fp[i], 0xFFFFFFFFull), i};
        std::stable_sort(keyed.begin(), keyed.end(), [](const auto& x, const auto& y) { return x.first > y.first; });
        uint32_t cur[NUM_CLASSES];
        for (int c = 0; c < NUM_CLASSES; ++c) cur[c] = begin[c];
        for (uint32_t k = 0; k < npoly; ++k) order[cur[cls(keyed[k].second)]++] = keyed[k].second;
    }
    MR_CUDA(ctx, cudaMemcpyAsync(db, hb, in_end, cudaMemcpyHostToDevice, ctx->stream));

    mr_polygon_job d = j;
    d.xy = reinterpret_cast<const float*>(db + o_xy);
    d.first_point = reinterpret_cast<const uint64_t*>(db + o_fp);
    d.point_base = 0;
    d.first_tri = reinterpret_cast<const uint64_t*>(db + o_ft);
    d.tri_base = 0;
    d.offset_prime = j.offset_prime ? reinterpret_cast<const uint32_t*>(db + o_op) : nullptr;
    d.vtx_out = db + o_vtx;
    d.bbox_out = reinterpret_cast<float*>(db + o_bbox);
    d.status_out = reinterpret_cast<uint32_t*>(db + o_stat);
    d.ntri_out = reinterpret_cast<uint32_t*>(db + o_ntri);
    BatchArgs a;
    fill_batch_args(a, &d, reinterpret_cast<uint32_t*>(db + o_hdr), reinterpret_cast<uint32_t*>(db + o_order),
                    reinterpret_cast<uint32_t*>(db + o_spec), reinterpret_cast<uint32_t*>(db + o_gen));
    ctx->last_header_dev = reinterpret_cast<const uint32_t*>(db + o_hdr);
    if (count[0]) {
        rc = class0_scratch(ctx, *plan, a);
        if (rc) return fail(rc);
    }
    for (int c = 0; c < NUM_CLASSES - 1; ++c) {
        if (!count[c]) continue;
        rc = launch_class(ctx, plan->first[c], a, c, 0, ctx->stream, count[c]);
        if (rc) return fail(rc);
    }
    if (count[NUM_CLASSES - 1] || count[XL_CLASS]) {  // (the XL class's hand-overs are consumed by the same kernel)
        rc = launch_general(ctx, a, 1, count[NUM_CLASSES - 1] + count[XL_CLASS]);
        if (rc) return fail(rc);
    }
    auto fetch = [&]() -> int {
        MR_CUDA(ctx, cudaMemcpyAsync(hb + o_hdr, db + o_hdr, out_end - o_hdr, cudaMemcpyDeviceToHost, ctx->stream));
        MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return MR_OK;
    };
    rc = fetch();
    if (rc) return fail(rc);
    // ---- rare: polygons that outgrew the first-pass arenas ---------------------------------------------------
    uint32_t respec = 0;
    for (int c = 0; c < XL_CLASS; ++c) respec += hdr[HDR_SPEC_COUNT + c];
    if (respec || hdr[HDR_GENERAL_COUNT]) {
        for (int c = 0; c < XL_CLASS; ++c) {
            if (!hdr[HDR_SPEC_COUNT + c]) continue;
            rc = launch_class(ctx, plan->spec[c], a, c, 1, ctx->stream, hdr[HDR_SPEC_COUNT + c]);
            if (rc) return fail(rc);
        }
        // the spec tier may hand polygons on to the general path: its count is only known on the device
        rc = launch_general(ctx, a, 0, respec + hdr[HDR_GENERAL_COUNT]);
        if (rc) return fail(rc);
        rc = fetch();
        if (rc) return fail(rc);
    }
    // ---- outputs --------------------------------------------------------------------------------------------
    memcpy(static_cast<unsigned char*>(j.vtx_out) + (size_t)tri0 * 3u * j.layout.stride, hb + o_vtx, vbytes);
    if (j.status_out) memcpy(j.status_out, hb + o_stat, (size_t)npoly * 4);
    if (j.ntri_out) memcpy(j.ntri_out, hb + o_ntri, (size_t)npoly * 4);
    if (j.bbox_out) memcpy(j.bbox_out, hb + o_bbox, (size_t)npoly * 16);
    ctx->host_io = false;
    return 1;
}
