// triangulate_fast.cuh -- the fast path of the Seidel kernel (included inside triangulate.cu's
// anonymous namespace).  Same algorithm, same emit sequence as the general path; it applies when
// no two points of the polygon have identical coordinates (checked per polygon), which allows:
//
//   * rank space.  Points are renamed by their position in the (y, x) order, so
//     point_is_above(a, b) (Triangulation.zig:128-136) is the integer compare a < b on values that
//     are already in registers; coordinates are only loaded for is_left_of.  Original ids come
//     back at emission (the emit order of :405-422 is defined on original ids).
//   * 8-byte nodes: {child1:16 | child2:16, pa:13 | crumb-is-right:1 | type:2 | pb:16} fetched with one
//     LDS.64.  A segment node's crumb is always one of its two children (:351-358), so one bit holds
//     it; point and trapezoid nodes always have a null crumb.  The
//     breadcrumb chain of the segment search (:253-257,:306-310) is an explicit stack -- the
//     reference restores every crumb to null before the search returns, so this is unobservable.
//   * no null checks on inner nodes: point and segment nodes always have both children and their
//     points set (they are written non-null at :183-192 and :347-360); the unwraps that CAN fail
//     (:330 trapezoid.point2, :524-527, :58) are kept.
//   * lane-parallel point location.  Inner nodes never change once written (only trapezoid leaves
//     are converted in place), so a node that was on a point's search path stays on it.  loc[p]
//     caches the deepest node reached so far for every not-yet-inserted point; all lanes advance
//     the caches between insertions and add_point continues from the cache instead of the root.
//     Result: identical descents, but the bulk of them run 32 wide.
//   * lane-parallel segment search (items tier).  The search of add_segment (:231-314) is a
//     pre-order walk whose decisions depend only on immutable inner nodes, so for every edge that
//     has not been inserted yet the walk can be kept *in progress*: an ordered linked list of
//     "items", each the deepest node reached on one branch.  When a leaf is converted by a later
//     insertion, the item simply continues from it (a straddled point node appends a sibling item
//     right after, which is exactly the order in which the reference would push the leaves).  All
//     lanes advance all pending items between insertions; at its own insertion an edge only
//     finishes the last step or two and copies its list into node_stack.  Duplicates (the same
//     trapezoid reached over two paths, which the reference pushes twice) are kept as they are.
//   * pass 2 picks the next trapezoid with a warp arg-min (REDUX) over the stack instead of the
//     O(k) scan of :329-337: same winner, because ties go to the lowest stack index in both.
#pragma once

__device__ __forceinline__ uint32_t mr_lds_u16(uint32_t shared_addr) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(shared_addr));
    return v;
}

constexpr uint32_t FNIL14 = 0x1FFFu;  // null in the 13-bit pa field (ranks are < 1024 on this path)
constexpr uint32_t CRUMB_RIGHT = 0x2000u;  // segment node: crumb == child2 (the inside is on the right)
constexpr uint32_t FNIL = 0xFFFFu;

struct FCaps {
    uint32_t nmax, node_cap, stack_cap, add_cap;
    uint32_t item_cap;  // 0: no conflict lists (the segment search runs from the root at insertion)
    bool par_separate_out;  // parallel search writes its list straight into node_stack (retry tier)
};
// tight: sized for the typical polygon of the class; spec: the contract caps (second chance in shared memory)
__host__ __device__ inline FCaps fast_caps(int c, bool spec) {
    FCaps k;
    k.nmax = class_nmax(c);
    k.par_separate_out = spec;
    if (!spec) {
        if (c == 0) {
            // 7n nodes and 2.75n adds (the contract caps are 8n+64 and unbounded): no polygon of the benchmark's star
            // batch outgrows them, and the 6.1 KB workspace lets the register file, not shared memory, set the
            // occupancy (32 warps per SM at 64 registers; measured +3.5 % over contract-cap arenas at 28 warps)
            k.node_cap = 7u * k.nmax;
            k.stack_cap = 64u;  // the serial search hands over to the parallel one at 48 leaves (own output list)
            k.add_cap = 2u * k.nmax + (3u * k.nmax) / 4u;
        } else {
            // measured on convex input (n = 65..1024): nodes <= 4.82 n, items ever created <= 1.82 n (= the sum of the
            // stack lengths: n initial items plus one per straddled point node), adds <= 1.4 n
            k.node_cap = 5u * k.nmax + k.nmax / 4u + 16u;
            k.stack_cap = k.nmax + 32u;
            k.add_cap = 2u * k.nmax + 16u;
        }
        // conflict lists pay for themselves on larger polygons only (measured: 1.35-1.55x for n up to 1024,
        // a small loss for n <= 64 where the per-edge polling overhead exceeds the search it saves).
        // Items are not recycled, so the pool must hold every item ever created.
        k.item_cap = c >= 1 ? 2u * k.nmax + k.nmax / 2u + 64u : 0u;  // the pool is reused by the mountain-phase arrays later
    } else {
        k.item_cap = 0;  // measured: conflict lists slow the retry tier down (8.1 vs 6.1 ms on the 100k star batch)
        k.node_cap = MR_NODE_CAP(k.nmax);
        k.stack_cap = MR_STACK_CAP(k.nmax);
        k.add_cap = 3u * k.nmax + 16u;  // sort arrays (20 B per add) alias the node arena (8 B per node)
    }
    return k;
}

struct FLayout {
    size_t sxy, orig, rk, loc, cstack, stack, nodes, add_pp, add_key, add_m, mcount, mstart, efirst, total;
    size_t it_node, it_next, it_edge, ehead, ctr;  // items tier only
};
__host__ __device__ inline FLayout fast_layout(const FCaps& k) {
    FLayout L;
    size_t o = 0;
    L.sxy = o;     o += align16((size_t)k.nmax * 8);
    L.orig = o;    o += k.item_cap ? 0 : align16((size_t)k.nmax * 2);  // conflict-list classes: see below
    L.rk = o;      o += align16((size_t)k.nmax * 2);
    L.loc = o;     o += align16((size_t)k.nmax * 2);
    L.cstack = o;  o += k.item_cap ? 0 : align16((size_t)k.nmax * 4);  // 2n entries; only the search from the root uses it
    L.stack = o;   o += align16((size_t)k.stack_cap * 2);
    L.nodes = o;   o += align16((size_t)k.node_cap * 8);
    // mountain-phase arrays reuse what is dead once part 1 is done: the item pool (with the per-edge
    // tables) and, for efirst, the point-location cache
    const size_t pool = o;
    L.add_pp = o;  o += align16((size_t)k.add_cap * 4);
    L.add_key = o; o += align16((size_t)k.add_cap * 4);
    L.it_node = L.it_next = L.it_edge = L.ehead = L.ctr = 0;
    if (k.item_cap) {
        // Conflict-list classes are bound by the polygons that fit an SM, so every array that can live in dead
        // space does.  After the part-2 scan the node arena is dead; the finish phase lays its five u16 sort arrays
        // (Gpos, cum, Gid, Gm, S; 2*add_cap entries each) over it.  add_m is last read while Gpos/Gid/Gm are
        // written and S is not yet: it sits in S.  mcount is last used there too and cum is written after: it sits
        // in cum.  mstart lives until the end; it takes rk+loc (+ a few bytes of stack; all dead once the mountains
        // are ranked -- efirst, which aliases loc, is last read before mstart is first written).
        L.mcount = L.nodes + (size_t)k.add_cap * 4;   // = cum
        L.add_m = L.nodes + (size_t)k.add_cap * 16;   // = S
        L.mstart = L.rk;
        // orig (rank -> original id) is only read in part 2: it is rebuilt from rk after the trapezoidation, into the
        // node_stack's space behind mstart
        L.orig = L.rk + align16((size_t)(k.add_cap + 1) * 2);
        const size_t mountain_end = o;
        o = pool;
        L.it_node = o; o += align16((size_t)k.item_cap * 2);
        L.it_next = o; o += align16((size_t)k.item_cap * 2);
        L.it_edge = o; o += align16((size_t)k.item_cap * 2);
        L.ehead = o;   o += align16((size_t)k.nmax * 2);
        L.ctr = o;     o += 16;
        if (o < mountain_end) o = mountain_end;
    } else if (!k.par_separate_out) {
        // n <= 64 class: the same overlays (there mstart takes rk+loc+cstack+stack = 10n bytes >= 2*(add_cap+1))
        L.mcount = L.nodes + (size_t)k.add_cap * 4;   // = cum
        L.add_m = L.nodes + (size_t)k.add_cap * 16;   // = S
        L.mstart = L.rk;
    } else {
        L.add_m = o;   o += align16((size_t)k.add_cap * 2);
        L.mcount = o;  o += align16((size_t)k.add_cap * 4);
        L.mstart = o;  o += align16((size_t)(k.add_cap + 1) * 2);
        // retry tier: room for the parallel search's items up to the contract stack cap
        const size_t need = pool + 16 + align16((size_t)(k.stack_cap + 2u) * 4);
        if (o < need) o = need;
    }
    L.efirst = L.loc;
    L.total = o;
    return L;
}

// host-side check of the overlay assumptions above (called once per launch configuration)
inline bool fast_layout_ok(const FCaps& k, const FLayout& L) {
    if (k.par_separate_out) return true;  // retry tier: no overlays
    const bool sort_fits = (size_t)k.add_cap * 20 <= (size_t)k.node_cap * 8;              // Gpos, cum, Gid, Gm, S over the node arena
    const bool mstart_fits = k.item_cap ? (L.orig + (size_t)k.nmax * 2 <= L.nodes)          // mstart, then orig, over rk .. stack
                                        : (L.rk + align16((size_t)(k.add_cap + 1) * 2) <= L.nodes);
    const bool rank_fits = (size_t)k.nmax * 8 + (size_t)k.nmax * 2 * 8 <= (size_t)k.node_cap * 8 &&  // raw + keys (n2 <= 2n)
                           (size_t)k.nmax * 2 * 2 <= (size_t)k.add_cap * 4;                // kidx over add_pp
    return sort_fits && mstart_fits && rank_fits;
}

// per-warp global-memory scratch of the n <= 64 kernel's parallel search: items (node, next) and the output list,
// PAR_GL_CAP entries each -- more than MR_STACK_CAP(64), so that overflowing it is the contract's MR_POLY_ARENA
constexpr uint32_t PAR_GL_CAP = MR_STACK_CAP(64u) + 8u;
constexpr size_t PAR_GL_BYTES = ((size_t)PAR_GL_CAP * 3u * 2u + 127u) & ~(size_t)127u;

// outcome of the fast path besides a Result
enum : int { F_DONE = 0, F_REQUEUE_SPEC = 1, F_REQUEUE_GENERAL = 2 };

struct FPoly {
    MR_SPAN(const float2) sxy;
    MR_SPAN(uint2) nd;
    MR_SPAN(uint16_t) stack;   // node_stack of the segment being inserted: always shared memory ...
    MR_SPAN(uint16_t) gstack;  // ... unless this is non-null: the (rare) list that only fitted the global-memory scratch.
                       // Two members so that the compiler keeps `stack` in the shared address space (LDS/STS, no
                       // generic-pointer arithmetic on the hot path).
    MR_SPAN(uint16_t) cstack;
    uint32_t nnodes, nstack, status;
    uint32_t tier_node_cap, tier_stack_cap, spec_node_cap, spec_stack_cap;
    bool requeue;

    __device__ __forceinline__ uint32_t alloc() {
        if (nnodes >= min(tier_node_cap, spec_node_cap)) {  // one compare on the hot path
            if (nnodes >= spec_node_cap) status |= MR_POLY_ARENA; else requeue = true;
            return FNIL;
        }
        return nnodes++;
    }
    // is_left_of(point P, segment a->b)  Triangulation.zig:117-126
    __device__ __forceinline__ bool left_of(float2 P, uint32_t a, uint32_t b) const {
        const float2 A = sxy[a], B = sxy[b];
        const float mul1 = __fmul_rn(__fsub_rn(B.x, A.x), __fsub_rn(P.y, A.y));
        const float mul2 = __fmul_rn(__fsub_rn(B.y, A.y), __fsub_rn(P.x, A.x));
        return __fsub_rn(mul1, mul2) > 0.0f;
    }
    __device__ __forceinline__ static uint32_t type_of(uint32_t w1) { return (w1 >> 14) & 3u; }

    // the descent of add_point (:144-167) from `base`; returns the trapezoid, or FNIL when the walk
    // meets the point's own node (already inserted)
    __device__ __forceinline__ uint32_t locate(uint32_t pid, float2 P, uint32_t base) const {
        // (the whole-word tests of search_from_root were tried here too: no gain for n <= 64, 2.6 % slower in the
        // conflict-list classes)
        for (;;) {
            const uint2 v = nd[base];
            const uint32_t t = type_of(v.y);
            if (t == T_TRAPEZOID) return base;
            const uint32_t pa = v.y & FNIL14;
            bool first;
            if (t == T_POINT) {
                if (pa == pid) return FNIL;
                first = pid < pa;  // point_is_above(pid, pa) in rank space
            } else {
                first = left_of(P, pa, v.y >> 16);
            }
            base = first ? (v.x & 0xFFFFu) : (v.x >> 16);
        }
    }

    // :169-192 split trapezoid `base` at point pid
    __device__ __forceinline__ bool split(uint32_t base, uint32_t pid) {
        const uint2 v = nd[base];
        if (nnodes + 2u > min(tier_node_cap, spec_node_cap)) {  // both clones at once (the failing alloc decides the flag)
            if (nnodes + 1u > min(tier_node_cap, spec_node_cap)) {
                alloc();
            } else {
                alloc();
                alloc();
            }
            return false;
        }
        const uint32_t lower = nnodes;      // :178 lower first
        const uint32_t upper = nnodes + 1u;  // :179
        nnodes += 2u;
        nd[lower] = make_uint2(v.x, (v.y & 0xFFFFC000u) | pid);        // point1 = pid
        nd[upper] = make_uint2(v.x, (v.y & 0x0000FFFFu) | (pid << 16));  // point2 = pid
        nd[base] = make_uint2(upper | (lower << 16), pid | (T_POINT << 14) | (FNIL << 16));
        return true;
    }

    __device__ __forceinline__ bool push(uint32_t id) {
        if (nstack >= min(tier_stack_cap, spec_stack_cap)) {
            if (nstack >= spec_stack_cap) status |= MR_POLY_ARENA; else requeue = true;
            return false;
        }
        stack[nstack++] = (uint16_t)id;
        return true;
    }

    // One step of the segment search (:234-296) at inner node v for segment (up, lo): returns the child
    // to continue with; *both is set when child2 has to be searched afterwards (breadcrumb case).
    __device__ __forceinline__ uint32_t dfs_step(const uint2 v, uint32_t up, uint32_t lo, const float2 Pu,
                                                  const float2 Pl, bool* both) const {
        const uint32_t pa = v.y & FNIL14;
        bool first;  // take child1
        if (type_of(v.y) == T_POINT) {
            // :234-259 collapsed.  As written: pa == up -> child2; pa == lo -> child1; pa above up -> child2;
            // lo above pa -> child1; otherwise (up above pa above lo) breadcrumb + child1.  In rank space
            // (up < lo, "above" is "<") that is exactly:
            first = pa > up;
            *both = first && (pa < lo);
        } else {
            // :260-296 with the five cases folded into operand selects (same tests, same operands)
            *both = false;
            const uint32_t o1 = pa, o2 = v.y >> 16;
            const bool share_up = (up == o1) | (up == o2);                           // :266
            const bool share_lo = (lo == o1) | (lo == o2);                           // :270
            const bool top_is_above = up < o1;                                       // :275
            const bool contained = !share_up & !share_lo & top_is_above & (lo < o2); // :277
            const bool use_lower = share_up | (!share_lo & top_is_above);            // :269,:284 test the lower point
            const float2 A = sxy[o1], B = sxy[o2];
            const float2 Q = use_lower ? Pl : Pu;
            // contained: !is_left_of(o1, up, lo) (:281); otherwise is_left_of(Q, o1, o2)
            const float ax = contained ? Pu.x : A.x, ay = contained ? Pu.y : A.y;
            const float bx = contained ? Pl.x : B.x, by = contained ? Pl.y : B.y;
            const float px = contained ? A.x : Q.x, py = contained ? A.y : Q.y;
            const float mul1 = __fmul_rn(__fsub_rn(bx, ax), __fsub_rn(py, ay));
            const float mul2 = __fmul_rn(__fsub_rn(by, ay), __fsub_rn(px, ax));
            first = (__fsub_rn(mul1, mul2) > 0.0f) != contained;
        }
        return first ? (v.x & 0xFFFFu) : (v.x >> 16);
    }

    // pass 1 of add_segment (:230-314), literally from the root.  Returns 1 when done, 0 on failure, and 2 when
    // the walk has produced `give_up` leaves without finishing (the caller then redoes it in parallel).
    __device__ int search_from_root(uint32_t up, uint32_t lo, uint32_t give_up) {
        const float2 Pu = sxy[up], Pl = sxy[lo];
        uint32_t base = 0;
        // The breadcrumb stack.  A pending breadcrumb is a point node on the path to the current node, and every call of
        // add_point creates at most one point node: at most 2n of them exist (on a consistent DAG n, of which n - 2 can
        // lie between the endpoints; the reference's failing cases can hold several nodes of one point).  The stack has
        // 2n entries, so it cannot overflow and the push is branch-free: the node is always stored into the next free
        // slot, and the slot is kept only for a breadcrumb.  A running shared-memory address in the product build (one
        // store and one predicated add per visit), an index into the bounds-checked span in the checked build.
#ifdef MR_CHECKED
        uint32_t ncr = 0;
#define MR_CR_PUSH_IF(c, x) (cstack[ncr] = (uint16_t)(x), ncr += (c) ? 1u : 0u)
#define MR_CR_EMPTY() (ncr == 0u)
#define MR_CR_POP() (cstack[--ncr])
#else
        // (a 32-bit shared-window address: as a C++ pointer the compiler carries the generic pointer beside it)
        const uint32_t cr0 = (uint32_t)__cvta_generic_to_shared(cstack);
        uint32_t cr = cr0;
#define MR_CR_PUSH_IF(c, x)                                                                      \
    do {                                                                                         \
        asm volatile("st.shared.u16 [%0], %1;" ::"r"(cr), "h"((unsigned short)(x)));             \
        if (c) cr += 2u;                                                                         \
    } while (0)
#define MR_CR_EMPTY() (cr == cr0)
#define MR_CR_POP() (cr -= 2u, mr_lds_u16(cr))
#endif
        nstack = 0;
        static_assert(T_POINT == 0 && T_SEGMENT == 1 && T_TRAPEZOID == 2 && FNIL == 0xFFFFu, "the word tests below read these bits");
        // A point node's second word is 0xFFFF0000 | rank (pb = FNIL, type 0, crumb 0, rank < 0x2000): as a signed
        // number it lies below every other node's (segment nodes and trapezoids with a lower point are positive,
        // trapezoids without one are 0xFFFF8000 | ...).  The run of point nodes -- a quarter of all instructions of
        // the n <= 64 kernel -- therefore tests the type and compares the rank on the whole word: no masks.
        const int up_w = (int)(0xFFFF0000u | up), lo_w = (int)(0xFFFF0000u | lo), point_end = (int)0xFFFF2000u;
        for (;;) {      // loop1 :231
            uint2 v = nd[base];
            for (;;) {  // loop :232, with runs of point nodes in a loop of their own
                int y = (int)v.y;
                while (y < point_end) {
                    const bool first = y > up_w;  // :234-259 collapsed, see dfs_step
                    MR_CR_PUSH_IF(first & (y < lo_w), base);  // up above pa above lo: breadcrumb, child2 comes later
                    base = first ? (v.x & 0xFFFFu) : (v.x >> 16);
                    v = nd[base];
                    y = (int)v.y;
                }
                if ((v.y & 0xFFFFu) >= 0x8000u) break;  // a trapezoid
                bool both;
                base = dfs_step(v, up, lo, Pu, Pl, &both);  // a segment node: never a breadcrumb
                v = nd[base];
            }
            if (!push(base)) return 0;  // :302
            if (MR_CR_EMPTY()) break;   // :306-313
            if (nstack >= give_up) return 2;
            base = nd[MR_CR_POP()].x >> 16;
        }
        return 1;
#undef MR_CR_PUSH_IF
#undef MR_CR_EMPTY
#undef MR_CR_POP
    }

    // The same search as a lane-parallel frontier expansion, for the searches that explode (the same
    // trapezoid reached over many DAG paths is pushed once per path).  Every branch of the walk is an
    // item in a linked list; a straddled point node links a sibling item right behind the current one,
    // so the list order is the order in which the serial walk pushes its leaves.  All lanes advance all
    // items until every item sits on a trapezoid; the list is then copied into node_stack.
    //   it_node/it_next: item arrays (cap entries), out: node_stack to fill (out_cap entries), ctr: shared
    //   word.  Returns 1 done, 0 failure (status/requeue set).
    template <bool GLOBAL>
    __device__ int search_parallel(uint32_t up, uint32_t lo, MR_SPAN(uint16_t) it_node, MR_SPAN(uint16_t) it_next, uint32_t cap,
                                   MR_SPAN(uint16_t) out, uint32_t out_cap, MR_SPAN(uint32_t) ctr, uint32_t lane) {
        const float2 Pu = sxy[up], Pl = sxy[lo];
        __syncwarp();
        if (lane == 0) {
            it_node[0] = 0;
            it_next[0] = (uint16_t)FNIL;
            ctr[0] = 1;
            ctr[1] = 0;
        }
        __syncwarp();
        for (;;) {
            const uint32_t cnt = min(ctr[0], cap);
            __syncwarp();  // every lane has read the count before any lane's atomicAdd moves it (lanes need not run in lock-step)
            bool advanced = false;
            for (uint32_t it = lane; it < cnt; it += 32) {
                uint32_t node = it_node[it];
                uint2 v = nd[node];
                if (type_of(v.y) == T_TRAPEZOID) continue;
                advanced = true;
                do {
                    bool both;
                    const uint32_t next = dfs_step(v, up, lo, Pu, Pl, &both);
                    if (both) {
                        const uint32_t nw = atomicAdd(&ctr[0], 1u);
                        if (nw >= cap) {
                            ctr[1] = 1;
                            break;
                        }
                        it_node[nw] = (uint16_t)(v.x >> 16);  // child2: after everything under child1
                        it_next[nw] = it_next[it];
                        it_next[it] = (uint16_t)nw;
                    }
                    node = next;
                    v = nd[node];
                } while (type_of(v.y) != T_TRAPEZOID);
                it_node[it] = (uint16_t)node;
            }
            __syncwarp();
            if (ctr[1]) {  // more items than `cap`: at least that many leaves
                if (cap > spec_stack_cap) status |= MR_POLY_ARENA; else requeue = true;
                return 0;
            }
            if (!__any_sync(0xFFFFFFFFu, advanced) && ctr[0] == cnt) break;
        }
        // copy in list order; the contract cap applies to the number of pushes exactly as in the serial walk
        const uint32_t total = ctr[0];
        if (total > spec_stack_cap) {
            status |= MR_POLY_ARENA;
            return 0;
        }
        if (total > out_cap) {
            requeue = true;
            return 0;
        }
        uint32_t it = 0;
        for (uint32_t j = 0; j < total; ++j) {  // warp-uniform walk
            if (lane == 0) out[j] = it_node[it];
            it = it_next[it];
        }
        __syncwarp();
        if (GLOBAL) gstack = out; else stack = out;
        nstack = total;
        return 1;
    }

    // pass 2 of add_segment (:316-395) on node_stack; p1 is the rank id of the edge's first point
    __device__ bool pass2(uint32_t p1, uint32_t up, uint32_t lo, uint32_t lane, uint32_t serial_below) {
        return !MR_SPAN_IS_NULL(gstack) ? pass2_on<true>(p1, up, lo, lane, serial_below) : pass2_on<false>(p1, up, lo, lane, serial_below);
    }
    // Pass 2 for a stack of K <= 2 entries, written out straight (every lane runs the same code; no loop, no
    // selection scan).  The loop :325-395 takes the crossed trapezoids in the order of their lower points (highest
    // first) and ends with the one that holds the segment's lower point; each step converts its trapezoid into a
    // segment node and closes the open trapezoid on the side its lower point lies on (:375), opening a new one there.
    // With all lower points non-null, those above `lo` pairwise distinct and exactly one entry whose lower point is not
    // above `lo` -- the case of every consistent trapezoidation -- that order is a sort by lower point, and the node
    // ids are known up front (left = A, right = A + 1, step s allocates A + 2 + s).  All loads are issued together and
    // the side tests are independent, which is what the latency-bound main warp of a polygon needs.  Returns 1 done,
    // 0 failed (status / requeue set as the loop would), -1 when the conditions do not hold: the caller then runs the
    // loop as written.
    template <int K>
    __device__ __forceinline__ int pass2_small(uint32_t p1, uint32_t up, uint32_t lo) {
        static_assert(K <= 2, "three and four entries written out straight measured slower (DESIGN 5.3)");
        const uint32_t A = nnodes;
        const uint32_t cap = min(tier_node_cap, spec_node_cap);
        uint32_t e[K], x[K], np[K];
#pragma unroll
        for (int i = 0; i < K; ++i) e[i] = stack[i];
#pragma unroll
        for (int i = 0; i < K; ++i) {
            const uint2 w = nd[e[i]];
            x[i] = w.x;
            np[i] = w.y >> 16;
        }
        bool odd = false;
        int finals = 0;
#pragma unroll
        for (int i = 0; i < K; ++i) {
            odd = odd || np[i] == FNIL;
            finals += np[i] < lo ? 0 : 1;
#pragma unroll
            for (int j = i + 1; j < K; ++j) odd = odd || (np[i] == np[j]);  // (a duplicate of the last entry shows up in `finals`)
        }
        if (odd || finals != 1) return -1;
        if (A + (uint32_t)K + 1u > cap) {  // the loop's failing add_node sees nnodes == cap
            if (cap >= spec_node_cap) status |= MR_POLY_ARENA; else requeue = true;
            return 0;
        }
        nnodes = A + (uint32_t)K + 1u;
        // ascending lower point: the steps in the loop's order, then the entry that holds `lo`
        if constexpr (K == 2) {
            const bool sw = np[0] > np[1];
            const uint32_t n0 = sw ? np[1] : np[0];
            const uint32_t e0 = sw ? e[1] : e[0];
            const uint32_t x0 = sw ? x[1] : x[0];
            np[1] = sw ? np[0] : np[1];
            e[1] = sw ? e[0] : e[1];
            x[1] = sw ? x[0] : x[1];
            np[0] = n0;
            e[0] = e0;
            x[0] = x0;
        }
        bool is_left[K];  // :375, one independent test per step
#pragma unroll
        for (int i = 0; i + 1 < K; ++i) is_left[i] = left_of(sxy[np[i]], up, lo);
        const uint32_t seg_y = up | ((p1 == up) ? 0u : CRUMB_RIGHT) | (T_SEGMENT << 14) | (lo << 16);  // :351-360
        const uint32_t trap = T_TRAPEZOID << 14;
        uint32_t cur_l = A, cur_r = A + 1u, p_l = up, p_r = up;
        __syncwarp();
#pragma unroll
        for (int i = 0; i + 1 < K; ++i) {
            nd[e[i]] = make_uint2(cur_l | (cur_r << 16), seg_y);  // :347-360
            if (is_left[i]) {                                       // :375-382
                nd[cur_l] = make_uint2((x[i] & 0xFFFFu) | (e[i] << 16), p_l | trap | (np[i] << 16));
                cur_l = A + 2u + (uint32_t)i;
                p_l = np[i];
            } else {                                                // :383-391
                nd[cur_r] = make_uint2(e[i] | (x[i] & 0xFFFF0000u), p_r | trap | (np[i] << 16));
                cur_r = A + 2u + (uint32_t)i;
                p_r = np[i];
            }
        }
        nd[e[K - 1]] = make_uint2(cur_l | (cur_r << 16), seg_y);     // :366-373
        nd[cur_l] = make_uint2((x[K - 1] & 0xFFFFu) | (e[K - 1] << 16), p_l | trap | (lo << 16));
        nd[cur_r] = make_uint2(e[K - 1] | (x[K - 1] & 0xFFFF0000u), p_r | trap | (lo << 16));
        return 1;
    }

    template <bool GLOBAL>
    __device__ bool pass2_on(uint32_t p1, uint32_t up, uint32_t lo, uint32_t lane, uint32_t serial_below) {
        // Stacks of one and two entries written out straight (measured: up to two beats up to three and four, DESIGN
        // 5.3).  Each size returns on its own: one `r` for both sizes costs the team kernels 16 bytes of spill at their
        // 80-register cap.
        if (!GLOBAL && nstack <= 2u && nstack > 0u) {
            if (nstack == 1u) {
                const int r = pass2_small<1>(p1, up, lo);
                if (r >= 0) return r != 0;
            } else {
                const int r = pass2_small<2>(p1, up, lo);
                if (r >= 0) return r != 0;
            }
        }
        MR_SPAN(uint16_t) stk = GLOBAL ? gstack : stack;
        // The two open trapezoids live in registers until they are closed.
        uint32_t left = alloc();
        if (left == FNIL) return false;
        uint32_t right = alloc();
        if (right == FNIL) return false;
        const uint32_t fresh = FNIL | (FNIL << 16);
        uint32_t lx = fresh, ly = up | (T_TRAPEZOID << 14) | (FNIL << 16);
        uint32_t rx = fresh, ry = ly;
        const bool crumb_left = (p1 == up);  // :351
        while (nstack > 0) {                 // :325
            // :329-337: the entry with the highest point2 (lowest rank) strictly above `low`; ties and
            // "none" resolve to the lowest index -> arg-min over (rank << 16 | index)
            uint32_t base_index = 0, low = lo;
            if (nstack <= serial_below) {  // short stack: the scan as written
                for (uint32_t i = 0; i < nstack; ++i) {
                    const uint32_t np = nd[stk[i]].y >> 16;
                    if (np == FNIL) {  // :330 `.?`
                        status |= MR_POLY_NULL_UNWRAP;
                        return false;
                    }
                    if (np < low) {
                        low = np;
                        base_index = i;
                    }
                }
            } else {
                uint32_t best = 0xFFFFFFFFu;
                bool null_p2 = false;
                for (uint32_t i = lane; i < nstack; i += 32) {
                    const uint32_t np = nd[stk[i]].y >> 16;
                    null_p2 = null_p2 || (np == FNIL);
                    best = min(best, (np << 16) | i);
                }
                if (__any_sync(0xFFFFFFFFu, null_p2)) {  // :330 `.?`
                    status |= MR_POLY_NULL_UNWRAP;
                    return false;
                }
                best = __reduce_min_sync(0xFFFFFFFFu, best);
                if ((best >> 16) < lo) {
                    low = best >> 16;
                    base_index = best & 0xFFFFu;
                }
            }
            const uint32_t base_id = stk[base_index];
            const uint32_t bch = nd[base_id].x;  // :347-360
            lx = (lx & 0xFFFF0000u) | (bch & 0xFFFFu);
            rx = (rx & 0x0000FFFFu) | (bch & 0xFFFF0000u);
            __syncwarp();
            nd[base_id] = make_uint2(left | (right << 16), up | (crumb_left ? 0u : CRUMB_RIGHT) | (T_SEGMENT << 14) | (lo << 16));
            if (lo == low) {  // :366-373
                lx = (lx & 0xFFFFu) | (base_id << 16);
                ly = (ly & 0xFFFFu) | (low << 16);
                rx = (rx & 0xFFFF0000u) | base_id;
                ry = (ry & 0xFFFFu) | (low << 16);
                break;
            } else if (left_of(sxy[low], up, lo)) {  // :375-382
                lx = (lx & 0xFFFFu) | (base_id << 16);
                ly = (ly & 0xFFFFu) | (low << 16);
                nd[left] = make_uint2(lx, ly);
                left = alloc();
                if (left == FNIL) return false;
                lx = fresh;
                ly = low | (T_TRAPEZOID << 14) | (FNIL << 16);
            } else {  // :383-391
                rx = (rx & 0xFFFF0000u) | base_id;
                ry = (ry & 0xFFFFu) | (low << 16);
                nd[right] = make_uint2(rx, ry);
                right = alloc();
                if (right == FNIL) return false;
                rx = fresh;
                ry = low | (T_TRAPEZOID << 14) | (FNIL << 16);
            }
            stk[base_index] = stk[nstack - 1];  // :394
            --nstack;
            __syncwarp();
        }
        nd[left] = make_uint2(lx, ly);
        nd[right] = make_uint2(rx, ry);
        return true;
    }
};

// ---- warp teams (large classes) ----------------------------------------------------------------------
// In the classes above 128 points a polygon's workspace is so large that only a few polygons fit an SM, and
// a lone warp issues one instruction every ~6 cycles: most issue slots of the SM sit idle.  There a block of
// W warps works on ONE polygon: warp 0 (the main warp) runs the algorithm, the other warps join it for the
// lane-parallel phases -- loading and ranking the points, the refresh of the point-location caches and of the
// pending edges' conflict lists, and the final group/sort/emit -- which are loops over independent entries.  Protocol (all block-wide barriers, same count on every warp):
//   main: ts->cmd = phase (LOAD, REFRESH|flags, FINISH); barrier; its share of the phase  (per phase; the phase
//         functions contain their own barriers and are called by every warp with the same arguments)
// ("barrier" = named barrier 1 over the W*32 threads of the block, team_bar)
//   main: ts->cmd = TEAM_STOP; barrier                                                     (per polygon, by the kernel)
//   helpers: loop { barrier; read ts->cmd; STOP -> leave; their share of the phase }
// W == 1 compiles to the single-warp code (no block barriers).
enum : uint32_t { TEAM_STOP = 0u, TEAM_REFRESH = 1u, TEAM_ITEMS = 2u, TEAM_LOAD = 4u, TEAM_FINISH = 8u };
constexpr int TEAM_MAX_WARPS = 8;
// block-shared words of a team (one polygon per block in the team kernel)
struct TeamShared {
    uint32_t cmd;        // TEAM_* of the phase the main warp is entering
    uint32_t n;          // points of the current polygon
    uint32_t arg0, arg1; // REFRESH: item count at start; FINISH: adds A, mountains M
    uint32_t qidx;       // queue position of the current polygon
    uint32_t flag0, flag1;  // LOAD: non-finite seen, tie seen; FINISH: not-acute seen
    uint32_t T;          // FINISH: triangles
    float part[TEAM_MAX_WARPS][4];  // FINISH: per-warp bbox partials {min x, max x, last y, has last}
};

// Team barrier: named barrier 1 with an explicit thread count -- the main warp and the helper warps arrive from
// different code, which bar.sync allows as long as whole warps arrive (unlike __syncthreads()'s convergence rule).
template <int W>
__device__ __forceinline__ void team_bar() {
    asm volatile("bar.sync 1, %0;" ::"r"(W * 32) : "memory");
}
template <int W>
__device__ __forceinline__ void team_sync() {
    if (W > 1) team_bar<W>(); else __syncwarp();
}

struct FItems {
    MR_SPAN(uint16_t) it_node;
    MR_SPAN(uint16_t) it_next;
    MR_SPAN(uint16_t) it_edge;
    MR_SPAN(uint16_t) ehead;
    MR_SPAN(const uint16_t) rk;  // rank of original point i: edge e runs from rk[e] to rk[e+1 mod n]
    MR_SPAN(uint32_t) ctr;
    uint32_t cap;
};

// One pending item of the conflict lists: continue its walk until it sits on a trapezoid; a straddled point node
// links a sibling item right behind it (handled by a later round).
__device__ __forceinline__ void advance_item(const FPoly& P, const FItems& I, uint32_t it, uint32_t n) {
    const uint32_t e = I.it_edge[it];
    if (I.ehead[e] == FNIL) return;  // edge already inserted
    uint32_t node = I.it_node[it];
    uint2 v = P.nd[node];
    if (FPoly::type_of(v.y) == T_TRAPEZOID) return;
    const uint32_t pa = I.rk[e], pb = I.rk[e + 1u == n ? 0u : e + 1u];
    const uint32_t up = min(pa, pb), lo = max(pa, pb);  // (upper, lower)  :218-224
    const float2 Pu = P.sxy[up], Pl = P.sxy[lo];
    do {
        bool both;
        const uint32_t next = P.dfs_step(v, up, lo, Pu, Pl, &both);
        if (both) {
            const uint32_t nw = atomicAdd(&I.ctr[0], 1u);
            if (nw >= I.cap) {
                I.ctr[1] = 1;
                break;
            }
            I.it_node[nw] = (uint16_t)(v.x >> 16);  // child2, searched after everything under child1
            I.it_edge[nw] = (uint16_t)e;
            I.it_next[nw] = I.it_next[it];
            I.it_next[it] = (uint16_t)nw;
        }
        node = next;
        v = P.nd[node];
    } while (FPoly::type_of(v.y) != T_TRAPEZOID);
    I.it_node[it] = (uint16_t)node;
}

// Lane-parallel advance of every pending point's cached location and (do_items) of every pending edge's search.
// Called by all W*32 threads of the team with the same arguments; tid = 0 .. W*32-1.
template <int W>
__device__ __forceinline__ void team_refresh(MR_SPAN(const float2) sxy, MR_SPAN(uint2) nd, MR_SPAN(uint16_t) loc, uint32_t n, bool do_items,
                                             const FItems I, uint32_t items_end, uint32_t tid) {
    constexpr uint32_t T = (uint32_t)W * 32u;
    FPoly P;  // only the immutable views are used here (locate, dfs_step)
    P.sxy = sxy;
    P.nd = nd;
    for (uint32_t r = tid; r < n; r += T) {  // loc is in rank space
        const uint32_t cur = loc[r];
        if (cur != FNIL) loc[r] = (uint16_t)P.locate(r, sxy[r], cur);  // never FNIL: r is not inserted yet
    }
    if (do_items) {
        // new sibling items are handled in the next round; items_end = the item count when the refresh began
        // (read by the main warp before the team started, so every warp runs the same rounds)
        uint32_t start = 0, end = items_end;
        while (start < end) {
            for (uint32_t it = start + tid; it < end; it += T) advance_item(P, I, it, n);
            team_sync<W>();  // every append of this round is done
            start = end;
            end = min(I.ctr[0], I.cap);
            team_sync<W>();  // everyone has read the counter before the next round moves it
        }
    }
}


// Load, validate and rank a polygon's points; all W*32 threads of the team call it (tid = 0 .. W*32-1).
// Returns 0 ok, 1 non-finite coordinate, 2 coincident points (same value on every thread).
template <int W>
__device__ __forceinline__ int team_load_rank(const float2* src, unsigned char* ws, const FCaps& caps, const FLayout& L, uint32_t n,
                                              uint32_t tid, TeamShared* ts) {
    constexpr uint32_t T = (uint32_t)W * 32u;
    MR_SPAN(float2) sxy = MR_MAKE_SPAN(float2, reinterpret_cast<float2*>(ws + L.sxy), caps.nmax);
    MR_SPAN(uint16_t) orig = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.orig), caps.nmax);
    MR_SPAN(uint16_t) rk = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.rk), caps.nmax);
    MR_SPAN(uint16_t) loc = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.loc), caps.nmax);
    // Original coordinates are staged in the node arena (free until the trapezoidation starts).
    MR_SPAN(float2) raw = MR_MAKE_SPAN(float2, reinterpret_cast<float2*>(ws + L.nodes), n);
    bool finite = true;
    for (uint32_t i = tid; i < n; i += T) {
        const float2 v = __ldg(src + i);
        raw[i] = v;
        finite = finite && isfinite(v.x) && isfinite(v.y);
    }
    if (W > 1) {
        if (!finite) ts->flag0 = 1u;
        team_bar<W>();
        if (ts->flag0) return 1;
    } else {
        __syncwarp();
        if (!__all_sync(0xFFFFFFFFu, finite)) return 1;
    }
    // rank = position in the (y, x) order (point_is_above, Triangulation.zig:128-136): bitonic sort of
    // order-preserving 64-bit keys, staged behind the raw coordinates in the node arena (O(n log^2 n);
    // the O(n^2) count it replaces was 29 % of the instructions at n = 1024).  -0 and +0 compare equal
    // as floats, so the key maps both to +0; the emitted coordinates still come from `raw`.
    uint32_t n2 = 32;
    while (n2 < n) n2 <<= 1;
    // 8n + 8*n2 <= 8*node_cap and 2*n2 <= 4n <= 4*add_cap (fast_layout_ok)
    MR_SPAN(unsigned long long) keys = MR_MAKE_SPAN(unsigned long long, reinterpret_cast<unsigned long long*>(ws + L.nodes) + n,
                                                    min(n2, caps.node_cap - n));
    MR_SPAN(uint16_t) kidx = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.add_pp), min(n2, 2u * caps.add_cap));
    for (uint32_t i = tid; i < n2; i += T) {
        unsigned long long k = ~0ull;  // padding sorts last
        if (i < n) {
            const float2 v = raw[i];
            uint32_t by = __float_as_uint(v.y == 0.0f ? 0.0f : v.y), bx = __float_as_uint(v.x == 0.0f ? 0.0f : v.x);
            by ^= (by >> 31) ? 0xFFFFFFFFu : 0x80000000u;
            bx ^= (bx >> 31) ? 0xFFFFFFFFu : 0x80000000u;
            k = ((unsigned long long)by << 32) | bx;
        }
        keys[i] = k;
        kidx[i] = (uint16_t)i;
    }
    team_sync<W>();
    for (uint32_t size = 2; size <= n2; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t t = tid; t < (n2 >> 1); t += T) {
                const uint32_t lo_i = ((t & ~(stride - 1u)) << 1) | (t & (stride - 1u));
                const uint32_t hi_i = lo_i | stride;
                const bool up_dir = (lo_i & size) == 0u;
                const unsigned long long ka = keys[lo_i], kb = keys[hi_i];
                if ((ka > kb) == up_dir) {
                    keys[lo_i] = kb;
                    keys[hi_i] = ka;
                    const uint16_t ia = kidx[lo_i];
                    kidx[lo_i] = kidx[hi_i];
                    kidx[hi_i] = ia;
                }
            }
            team_sync<W>();
        }
    }
    bool tie = false;
    for (uint32_t r = tid; r < n; r += T) {
        if (r + 1u < n && keys[r] == keys[r + 1u]) tie = true;
        rk[kidx[r]] = (uint16_t)r;
    }
    if (W > 1) {
        if (tie) ts->flag1 = 1u;
        team_bar<W>();
        if (ts->flag1) return 2;
    } else {
        if (__any_sync(0xFFFFFFFFu, tie)) return 2;
        __syncwarp();
    }
    for (uint32_t i = tid; i < n; i += T) {
        const uint32_t r = rk[i];
        sxy[r] = raw[i];
        orig[r] = (uint16_t)i;
        loc[i] = 0;  // every point starts at the root
    }
    team_sync<W>();
    return 0;
}

__device__ __forceinline__ Sink fast_sink(const BatchArgs& a, uint32_t pi, uint32_t* cap_tri) {
    const uint64_t t0 = a.first_tri[pi] - a.tri_base;
    *cap_tri = (uint32_t)(a.first_tri[pi + 1] - a.first_tri[pi]);
    Sink sink;
    sink.base = a.vtx_out + t0 * 3u * a.stride;
    sink.cap_vtx = *cap_tri * 3u;
    sink.stride = a.stride;
    sink.off_x = a.off_x;
    sink.off_c = a.off_c;
    sink.fast32 = a.fast32;
    return sink;
}

// Last phase: the A adds (add_pp, add_m, mstart, zeroed mcount are in place) are grouped by mountain, every
// mountain is sorted (:555), and the emission loop :558-586 runs in closed form.  All W*32 threads of the team
// call it; only the main warp's *res is filled.  Returns F_DONE or F_REQUEUE_GENERAL (same on every thread).
template <int W>
__device__ __forceinline__ int team_finish(const Sink& sink, uint32_t cap_tri, unsigned char* ws, const FCaps& caps,
                                           const FLayout& L, uint32_t A, uint32_t tid, TeamShared* ts, Result* res) {
    constexpr uint32_t TT = (uint32_t)W * 32u;
    const uint32_t lane = tid & 31u, warp = tid >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    MR_SPAN(const float2) sxy = MR_MAKE_SPAN(const float2, reinterpret_cast<const float2*>(ws + L.sxy), caps.nmax);
    MR_SPAN(const uint16_t) orig = MR_MAKE_SPAN(const uint16_t, reinterpret_cast<const uint16_t*>(ws + L.orig), caps.nmax);
    MR_SPAN(const uint32_t) add_pp = MR_MAKE_SPAN(const uint32_t, reinterpret_cast<const uint32_t*>(ws + L.add_pp), caps.add_cap);
    MR_SPAN(const uint16_t) add_m = MR_MAKE_SPAN(const uint16_t, reinterpret_cast<const uint16_t*>(ws + L.add_m), caps.add_cap);
    MR_SPAN(uint32_t) mcount = MR_MAKE_SPAN(uint32_t, reinterpret_cast<uint32_t*>(ws + L.mcount), caps.add_cap);
    MR_SPAN(const uint16_t) mstart = MR_MAKE_SPAN(const uint16_t, reinterpret_cast<const uint16_t*>(ws + L.mstart), caps.add_cap + 1u);

    // ---- group entries by mountain, stable sort by (rank, append position)  (:555) ----------------
    // sort arrays alias the node arena: Gpos, cum, Gid, Gm, S -- u16 each, E = 2A entries
    const uint32_t E = 2u * A;
    const size_t ecap = (size_t)caps.add_cap * 2;
    uint16_t* const sort0 = reinterpret_cast<uint16_t*>(ws + L.nodes);
    MR_SPAN(uint16_t) Gpos = MR_MAKE_SPAN(uint16_t, sort0, ecap);
    MR_SPAN(uint16_t) cum = MR_MAKE_SPAN(uint16_t, sort0 + ecap, ecap);
    MR_SPAN(uint16_t) Gid = MR_MAKE_SPAN(uint16_t, sort0 + 2 * ecap, ecap);
    MR_SPAN(uint16_t) Gm = MR_MAKE_SPAN(uint16_t, sort0 + 3 * ecap, ecap);
    MR_SPAN(uint16_t) S = MR_MAKE_SPAN(uint16_t, sort0 + 4 * ecap, ecap);
    for (uint32_t ai = tid; ai < A; ai += TT) {
        const uint32_t m = add_m[ai];
        const uint32_t pp = add_pp[ai];
        const uint32_t slot = mstart[m] + atomicAdd(&mcount[m], 2u);
        Gpos[slot] = (uint16_t)(2u * ai);  // p1 appended first (:60)
        Gid[slot] = (uint16_t)(pp & FNIL14);
        Gpos[slot + 1] = (uint16_t)(2u * ai + 1u);  // then p2 (:61)
        Gid[slot + 1] = (uint16_t)(pp >> 16);
        Gm[slot] = (uint16_t)m;
        Gm[slot + 1] = (uint16_t)m;
    }
    team_sync<W>();
    for (uint32_t g = tid; g < E; g += TT) {
        const uint32_t m = Gm[g];
        const uint32_t s = mstart[m], t = mstart[m + 1];
        const uint32_t mykey = ((uint32_t)Gid[g] << 16) | Gpos[g];  // (rank, append position)
        uint32_t rank = 0;
        for (uint32_t h = s; h < t; ++h) rank += ((((uint32_t)Gid[h] << 16) | Gpos[h]) < mykey) ? 1u : 0u;
        S[s + rank] = Gid[g];
    }
    team_sync<W>();

    // ---- triangles: valid j, acute check, slots  (:558-586 in closed form) -------------------------
    uint32_t T = 0;
    if (W == 1) {
        uint32_t running = 0;
        bool all_acute = true;
        for (uint32_t b = 0; b < E; b += 32) {
            const uint32_t g = b + lane;
            bool valid = false;
            if (g < E) {
                const uint32_t s = mstart[Gm[g]];
                if (g >= s + 2u) {
                    const uint32_t c = S[g], a1 = S[g - 1], a2 = S[s];
                    valid = (c != a1) && (c != a2);
                    if (valid && !is_acute_shortcut(MR_SPAN_RAW(sxy), c, a1, a2)) all_acute = false;
                }
            }
            const uint32_t vm = __ballot_sync(0xFFFFFFFFu, valid);
            if (g < E) cum[g] = (uint16_t)(running + __popc(vm & (lt_mask | (1u << lane))));
            running += __popc(vm);
        }
        all_acute = __all_sync(0xFFFFFFFFu, all_acute);
        __syncwarp();
        // a push_triangle_if_acute returned false somewhere: the literal loop of the general path decides
        if (!all_acute) return F_REQUEUE_GENERAL;
        T = running;
    } else {
        // the flags (with the acute checks) by everyone, then the ordered prefix sum by the main warp
        bool all_acute = true;
        for (uint32_t g = tid; g < E; g += TT) {
            bool valid = false;
            const uint32_t s = mstart[Gm[g]];
            if (g >= s + 2u) {
                const uint32_t c = S[g], a1 = S[g - 1], a2 = S[s];
                valid = (c != a1) && (c != a2);
                if (valid && !is_acute_shortcut(MR_SPAN_RAW(sxy), c, a1, a2)) all_acute = false;
            }
            cum[g] = valid ? 1u : 0u;
        }
        if (!all_acute) ts->flag0 = 1u;
        team_bar<W>();
        if (ts->flag0) return F_REQUEUE_GENERAL;
        if (warp == 0) {
            uint32_t running = 0;
            for (uint32_t b = 0; b < E; b += 32) {
                const uint32_t g = b + lane;
                const bool valid = g < E && cum[g] != 0u;
                const uint32_t vm = __ballot_sync(0xFFFFFFFFu, valid);
                if (g < E) cum[g] = (uint16_t)(running + __popc(vm & (lt_mask | (1u << lane))));
                running += __popc(vm);
            }
            if (lane == 0) ts->T = running;
        }
        team_bar<W>();
        T = ts->T;
    }

    float mn = 0.0f, mx = 0.0f, lasty = 0.0f;
    bool has_last = false;
    MR_SPAN(uint16_t) tri = Gpos;  // Gpos is dead after the sort; 2*add_cap entries >= 3*cap_tri
    for (uint32_t g = tid; g < E; g += TT) {
        const uint32_t m = Gm[g];
        const uint32_t s = mstart[m], t = mstart[m + 1];
        if (g < s + 2u) continue;
        const uint32_t c = S[g], a1 = S[g - 1], a2 = S[s];
        if (c == a1 || c == a2) continue;
        const uint32_t before = s ? cum[s - 1] : 0u;
        const uint32_t slot = before + (cum[t - 1] - cum[g]);
        // the emit order (:405-422) is defined on the original point ids
        const uint32_t oc = orig[c], o1 = orig[a1], o2 = orig[a2];
        uint32_t second, third;
        if ((o1 > oc && o2 > oc) || (o1 < oc && o2 < oc)) {
            second = o1 > o2 ? a2 : a1;
            third = o1 > o2 ? a1 : a2;
        } else if (o2 > oc) {
            second = a2;
            third = a1;
        } else {
            second = a1;
            third = a2;
        }
        const float2 q0 = sxy[c], q1 = sxy[second], q2 = sxy[third];
        mn = fmin_acc(fmin_acc(fmin_acc(mn, q0.x), q1.x), q2.x);
        mx = fmax_acc(fmax_acc(fmax_acc(mx, q0.x), q1.x), q2.x);
        if (slot == T - 1u) {
            lasty = q2.y;
            has_last = true;
        }
        if (slot < cap_tri) {  // the triangle's points in emit order; the vertices go out in a second, linear pass
            tri[3u * slot] = (uint16_t)c;
            tri[3u * slot + 1u] = (uint16_t)second;
            tri[3u * slot + 2u] = (uint16_t)third;
        }
    }
    // The polygon's vertex range is contiguous: written linearly, every warp store covers 32 consecutive vertices
    // (1 KB) instead of 32 vertices 96 bytes apart -- whole lines for L2, and full-size PCIe writes when the
    // range is pinned host memory (measured: 100k star batch 4.77 -> 4.63 ms on the device, 9.5 -> 7.3 ms end to end).
    team_sync<W>();
    {
        const uint32_t nv = 3u * (T < cap_tri ? T : cap_tri);
        for (uint32_t v = tid; v < nv; v += TT) sink.write(v, sxy[tri[v]]);
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        mn = fmin_acc(mn, __shfl_xor_sync(0xFFFFFFFFu, mn, d));
        mx = fmax_acc(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, d));
    }
    {
        const uint32_t lm = __ballot_sync(0xFFFFFFFFu, has_last);
        has_last = lm != 0u;
        lasty = lm ? __shfl_sync(0xFFFFFFFFu, lasty, __ffs(lm) - 1) : 0.0f;
    }
    if (T < cap_tri) sink.zero(3u * T, sink.cap_vtx, tid, TT);
    if (W > 1) {
        if (lane == 0) {
            ts->part[warp][0] = mn;
            ts->part[warp][1] = mx;
            ts->part[warp][2] = lasty;
            ts->part[warp][3] = has_last ? 1.0f : 0.0f;
        }
        team_bar<W>();
        if (warp != 0) return F_DONE;
        mn = mx = lasty = 0.0f;  // exactly one warp holds the last triangle (slot T-1), if there is one
#pragma unroll
        for (int w = 0; w < W; ++w) {
            mn = fmin_acc(mn, ts->part[w][0]);
            mx = fmax_acc(mx, ts->part[w][1]);
            if (ts->part[w][3] != 0.0f) lasty = ts->part[w][2];
        }
    }
    uint32_t status = MR_POLY_OK;
    if (T > cap_tri) status |= MR_POLY_OVERFLOW;
    if (T < cap_tri) status |= MR_POLY_UNDERFILL;
    res->b1x = mn;
    res->b2x = mx;
    res->b1y = T ? fmin_acc(mn, lasty) : 0.0f;
    res->b2y = T ? fmax_acc(mx, lasty) : 0.0f;
    res->status = status;
    res->ntri = T < cap_tri ? T : cap_tri;
    return F_DONE;
}

__device__ __forceinline__ FItems fast_items(unsigned char* ws, const FLayout& L, const FCaps& caps) {
    FItems I;
    I.it_node = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.it_node), caps.item_cap);
    I.it_next = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.it_next), caps.item_cap);
    I.it_edge = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.it_edge), caps.item_cap);
    I.ehead = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.ehead), caps.item_cap ? caps.nmax : 0u);
    I.rk = MR_MAKE_SPAN(const uint16_t, reinterpret_cast<const uint16_t*>(ws + L.rk), caps.nmax);
    I.ctr = MR_MAKE_SPAN(uint32_t, reinterpret_cast<uint32_t*>(ws + L.ctr), caps.item_cap ? 4u : 0u);  // [0] items allocated, [1] pool overflow flag
    I.cap = caps.item_cap;
    return I;
}

// The helper warps of a team: join the main warp in the phase it announces, until it says stop.
template <int W>
__device__ void team_helper(const BatchArgs& a, uint32_t pi, unsigned char* ws, const FCaps caps, const FLayout L,
                            TeamShared* ts) {
    FPoly P;
    P.sxy = MR_MAKE_SPAN(const float2, reinterpret_cast<const float2*>(ws + L.sxy), caps.nmax);
    P.nd = MR_MAKE_SPAN(uint2, reinterpret_cast<uint2*>(ws + L.nodes), caps.node_cap);
    MR_SPAN(uint16_t) loc = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.loc), caps.nmax);
    const FItems I = fast_items(ws, L, caps);
    for (;;) {
        team_bar<W>();
        const uint32_t cmd = ts->cmd;
        if (cmd == TEAM_STOP) break;
        if (cmd & TEAM_REFRESH) {
            team_refresh<W>(P.sxy, P.nd, loc, ts->n, (cmd & TEAM_ITEMS) != 0u, I, ts->arg0, threadIdx.x);
            team_bar<W>();
        } else if (cmd == TEAM_LOAD) {
            const uint64_t p0 = a.first_point[pi] - a.point_base;
            team_load_rank<W>(reinterpret_cast<const float2*>(a.xy) + p0, ws, caps, L, ts->n, threadIdx.x, ts);
        } else {  // TEAM_FINISH
            uint32_t cap_tri;
            const Sink sink = fast_sink(a, pi, &cap_tri);
            team_finish<W>(sink, cap_tri, ws, caps, L, ts->arg0, threadIdx.x, ts, nullptr);
        }
    }
}

// All 32 lanes of the main warp call this.  Returns F_DONE with *res filled, or a requeue code.
// ITEMS: the class keeps conflict lists (caps.item_cap != 0); a compile-time switch so that the n <= 64 kernel and
// the retry tiers do not carry the conflict-list code, nor the conflict-list classes the search from the root.
template <int W, bool ITEMS>
__device__ int process_polygon_fast(const BatchArgs& a, uint32_t pi, unsigned char* ws, const FCaps caps,
                                    const FLayout L, Result* res, TeamShared* ts, unsigned char* par_gl = nullptr) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const uint64_t p0 = a.first_point[pi] - a.point_base;
    const uint64_t np64 = a.first_point[pi + 1] - a.first_point[pi];
    const uint32_t n = (uint32_t)(np64 > 0xFFFFFFFFull ? 0xFFFFFFFFull : np64);
    uint32_t cap_tri;
    const Sink sink = fast_sink(a, pi, &cap_tri);

    res->status = MR_POLY_OK;
    res->ntri = 0;
    res->b1x = res->b1y = res->b2x = res->b2y = 0.0f;
    res->requeue = false;

    if (n < 3u) {
        res->status = MR_POLY_DEGENERATE;
        sink.zero(0, sink.cap_vtx, lane);
        return F_DONE;
    }
    if (n > MR_MAX_POLYGON_POINTS) {
        res->status = MR_POLY_TOO_LARGE;
        sink.zero(0, sink.cap_vtx, lane);
        return F_DONE;
    }
    if (n > caps.nmax) return F_REQUEUE_GENERAL;

    MR_SPAN(float2) sxy = MR_MAKE_SPAN(float2, reinterpret_cast<float2*>(ws + L.sxy), caps.nmax);
    MR_SPAN(uint16_t) orig = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.orig), caps.nmax);
    MR_SPAN(uint16_t) rk = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.rk), caps.nmax);
    MR_SPAN(uint16_t) loc = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.loc), caps.nmax);

    // ---- load, validate, rank (all warps of the team) ------------------------------------------------
    if (W > 1) {
        if (lane == 0) {
            ts->cmd = TEAM_LOAD;
            ts->n = n;
            ts->flag0 = ts->flag1 = 0u;
        }
        team_bar<W>();
    }
    {
        const int lr = team_load_rank<W>(reinterpret_cast<const float2*>(a.xy) + p0, ws, caps, L, n, lane, ts);
        if (lr == 1) {
            res->status = MR_POLY_NONFINITE;
            sink.zero(0, sink.cap_vtx, lane);
            return F_DONE;
        }
        if (lr == 2) return F_REQUEUE_GENERAL;  // coincident points: general path
    }

    // ---- unirand (unirand.zig:12-50) -------------------------------------------------------------
    uint32_t ur_offset, ur_prime;
    if (a.offset_prime) {
        ur_offset = __ldg(a.offset_prime + 2 * (size_t)pi);
        ur_prime = __ldg(a.offset_prime + 2 * (size_t)pi + 1);
    } else {
        unirand_seed_warp(n, a.seed, a.poly_index0 + pi, lane, &ur_offset, &ur_prime);
    }

    if (ITEMS && a.offset_prime) {
        // An explicit (offset, prime) pair can come back to an edge it has inserted already (unirand.zig:16 is a plain
        // multiply-add-modulo; unirand_seed only hands out primes that do not divide n), and the reference then searches
        // and splits again (:493).  An edge's conflict list is consumed by its first insertion, so such polygons take the
        // literal search from the root: the next tier.  The order repeats iff gcd(prime, n) > 1 when both values are
        // below n; with larger values the u32 product wraps and the order is not an arithmetic progression mod n at all.
        bool repeats = ur_offset >= n || ur_prime >= n;
        if (!repeats) {
            uint32_t g = n, h = ur_prime;
            while (h) {
                const uint32_t t = g % h;
                g = h;
                h = t;
            }
            repeats = g != 1u;
        }
        if (repeats) return F_REQUEUE_SPEC;
    }

    // ---- part 1: trapezoidation ---------------------------------------------------------------------
    FPoly P;
    P.sxy = sxy;
    P.nd = MR_MAKE_SPAN(uint2, reinterpret_cast<uint2*>(ws + L.nodes), caps.node_cap);
    P.stack = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.stack), caps.stack_cap);
    P.cstack = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.cstack), caps.item_cap ? 0u : 2u * caps.nmax);
    P.gstack = MR_SPAN_NULL(uint16_t);
    P.nnodes = 1;  // :479 root trapezoid
    P.nstack = 0;
    P.status = MR_POLY_OK;
    P.spec_node_cap = MR_NODE_CAP(n);
    P.spec_stack_cap = MR_STACK_CAP(n);
    P.tier_node_cap = caps.node_cap;
    P.tier_stack_cap = caps.stack_cap;
    P.requeue = false;
    P.nd[0] = make_uint2(FNIL | (FNIL << 16), FNIL14 | (T_TRAPEZOID << 14) | (FNIL << 16));
    __syncwarp();

    // ---- conflict lists of the pending edges (items tier) ---------------------------------------------
    constexpr bool use_items = ITEMS;
    // the caches are refreshed every refresh_every edges, the conflict lists every item_mult-th refresh (single warp:
    // measured best of 1/2/4/8 on n <= 1024); countdowns instead of `at % period` (a run-time modulo per edge)
    // (without conflict lists -- n <= 64 and the retry tiers -- every 4th edge measured best of 1/2/3/4/6/8/16)
    // (teams: caches every n/64 edges measured best of n/32..n/128, lists every 3rd refresh best of 2/3/4/8, DESIGN 5.3)
    const uint32_t refresh_every = W > 1 ? (n + 63u) / 64u : (!ITEMS ? 4u * ((n + 63u) / 64u) : (n + 63u) / 64u);
    const uint32_t item_mult = W > 1 ? 3u : 4u;
    uint32_t refresh_wait = 0, item_wait = 0;
    const FItems I = fast_items(ws, L, caps);
    MR_SPAN(uint16_t) it_node = I.it_node;
    MR_SPAN(uint16_t) it_next = I.it_next;
    MR_SPAN(uint16_t) it_edge = I.it_edge;
    MR_SPAN(uint16_t) ehead = I.ehead;
    MR_SPAN(uint32_t) ctr = I.ctr;
    if (use_items) {
        for (uint32_t e = lane; e < n; e += 32) {  // every edge starts with one item at the root
            it_node[e] = 0;
            it_next[e] = (uint16_t)FNIL;
            it_edge[e] = (uint16_t)e;
            ehead[e] = (uint16_t)e;
        }
        if (lane == 0) {
            ctr[0] = n;
            ctr[1] = 0;
        }
    }
    __syncwarp();

    // scratch of the parallel search (tiers without conflict lists): the mountain-phase arrays, free in part 1
    MR_SPAN(uint16_t) stack_home = P.stack;
    MR_SPAN(uint16_t) par_node = MR_SPAN_NULL(uint16_t);
    MR_SPAN(uint16_t) par_next = MR_SPAN_NULL(uint16_t);
    MR_SPAN(uint16_t) par_out = MR_SPAN_NULL(uint16_t);
    MR_SPAN(uint32_t) par_ctr = MR_SPAN_NULL(uint32_t);
    uint32_t par_cap = 0, par_out_cap = 0;
    if (!use_items) {
        const size_t bytes = (L.efirst == L.loc ? L.total : L.efirst) - L.add_pp - 16;  // pool region minus the counter
        par_ctr = MR_MAKE_SPAN(uint32_t, reinterpret_cast<uint32_t*>(ws + L.add_pp), 4u);
        unsigned char* base = ws + L.add_pp + 16;
        if (caps.par_separate_out) {  // retry tier: the list goes to the (contract-cap) node_stack itself
            par_cap = (uint32_t)(bytes / 4);
            par_out = stack_home;
            par_out_cap = caps.stack_cap;
        } else {  // typical-case tier: items and the output list share the region 2:1
            par_cap = (uint32_t)(bytes / 6);
            par_out = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(base + (size_t)par_cap * 4), par_cap);
            par_out_cap = par_cap;
        }
        par_node = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(base), par_cap);
        par_next = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(base) + par_cap, par_cap);
    }

    const bool ur_simple = ur_offset < n && ur_prime < n;
    uint32_t ur_edge = ur_offset;
    bool ok = true;
    for (uint32_t at = 0; at < n && ok; ++at) {  // :484-494
        const bool refresh_now = refresh_wait == 0u;
        refresh_wait = refresh_now ? refresh_every - 1u : refresh_wait - 1u;
        const bool items_now = use_items && refresh_now && item_wait == 0u;
        if (refresh_now) item_wait = item_wait == 0u ? item_mult - 1u : item_wait - 1u;
        if (W == 1) {
            // Single warp: the refresh written out in place.  (Same loops as team_refresh<1>, but the n <= 64 kernel is
            // measurably faster -- 3 % -- with this exact form; the compiler's register allocation differs.)
            if (refresh_now) {
                // lane-parallel advance of every pending point's cached location (loc is in rank space)
                for (uint32_t r = lane; r < n; r += 32) {
                    const uint32_t cur = loc[r];
                    if (cur != FNIL) loc[r] = (uint16_t)P.locate(r, sxy[r], cur);  // never FNIL: r is not inserted yet
                }
                if (items_now) {
                    // lane-parallel advance of every pending edge's search; new sibling items are handled in
                    // the next round
                    uint32_t start = 0, end = ctr[0];
                    while (start < end) {
                        for (uint32_t it = start + lane; it < end; it += 32) {
                            const uint32_t e = it_edge[it];
                            if (ehead[e] == FNIL) continue;  // edge already inserted
                            uint32_t node = it_node[it];
                            uint2 v = P.nd[node];
                            if (FPoly::type_of(v.y) == T_TRAPEZOID) continue;
                            const uint32_t ra = rk[e], rb = rk[e + 1u == n ? 0u : e + 1u];
                            const uint32_t up = min(ra, rb), lo = max(ra, rb);  // (upper, lower)  :218-224
                            const float2 Pu = sxy[up], Pl = sxy[lo];
                            do {
                                bool both;
                                const uint32_t next = P.dfs_step(v, up, lo, Pu, Pl, &both);
                                if (both) {
                                    const uint32_t nw = atomicAdd(&ctr[0], 1u);
                                    if (nw >= caps.item_cap) {
                                        ctr[1] = 1;
                                        break;
                                    }
                                    it_node[nw] = (uint16_t)(v.x >> 16);  // child2, searched after everything under child1
                                    it_edge[nw] = (uint16_t)e;
                                    it_next[nw] = it_next[it];
                                    it_next[it] = (uint16_t)nw;
                                }
                                node = next;
                                v = P.nd[node];
                            } while (FPoly::type_of(v.y) != T_TRAPEZOID);
                            it_node[it] = (uint16_t)node;
                        }
                        __syncwarp();
                        start = end;
                        end = min(ctr[0], caps.item_cap);
                        __syncwarp();  // every lane has read the counter before the next round moves it
                    }
                    if (ctr[1]) {  // pool exhausted: the next tier redoes this polygon with the literal search
                        P.requeue = true;
                        break;
                    }
                }
                __syncwarp();
            }
        } else if (refresh_now) {
            const bool do_items = items_now;
            const uint32_t items_end = do_items ? ctr[0] : 0u;
            if (lane == 0) {
                ts->cmd = TEAM_REFRESH | (do_items ? TEAM_ITEMS : 0u);
                ts->arg0 = items_end;
            }
            team_bar<W>();
            team_refresh<W>(sxy, P.nd, loc, n, do_items, I, items_end, lane);
            team_bar<W>();
            if (do_items && ctr[1]) {  // pool exhausted: the next tier redoes this polygon with the literal search
                P.requeue = true;
                break;
            }
        }
        // unirand.zig:16: (at * prime + offset) % top in u32 arithmetic.  With offset, prime < n (always so for
        // unirand_seed's own output) the sequence is an add-and-wrap; explicit pairs outside that keep the formula.
        uint32_t edge;
        if (ur_simple) {
            edge = ur_edge;
            ur_edge += ur_prime;
            if (ur_edge >= n) ur_edge -= n;
        } else {
            edge = (uint32_t)(at * ur_prime + ur_offset) % n;
        }
        const uint32_t p1 = rk[edge];
        const uint32_t p2 = rk[edge + 1u == n ? 0u : edge + 1u];
        const uint32_t up = min(p1, p2), lo = max(p1, p2);  // :218-224 in rank space
        // Everything the insertion of this edge reads that is immutable (rank-space coordinates) or untouched until it is
        // used (the two location caches, the head of the edge's conflict list) is loaded here, together: the loads
        // overlap instead of sitting one behind the other on the polygon's dependent chain.
        // (Conflict-list classes only -- their polygons are latency-bound; the n <= 64 kernel is issue-bound and measured
        // 2 % slower with the hoisted form.)
        float2 Pu = make_float2(0.0f, 0.0f), Pl = Pu;
        uint32_t cur_p1 = FNIL, cur_p2 = FNIL;
        if (ITEMS) {
            Pu = sxy[up];
            Pl = sxy[lo];
            cur_p1 = loc[p1];
            cur_p2 = loc[p2];
        }
        uint32_t it = FNIL, it_node0 = 0, it_next0 = FNIL;
        if (use_items) {
            it = ehead[edge];
            if (it != FNIL) {  // always: orders that come back to an edge were sent to the next tier above
                it_node0 = it_node[it];
                it_next0 = it_next[it];
            }
        }
        // add_point(p1), add_point(p2)  :489-490
#pragma unroll
        for (int which = 0; which < 2 && ok; ++which) {
            const uint32_t pid = which ? p2 : p1;
            const uint32_t cur = ITEMS ? (which ? cur_p2 : cur_p1) : (uint32_t)loc[pid];
            if (cur != FNIL) {  // not inserted yet (an inserted point's walk ends at its own node, :149-152)
                const uint32_t leaf = P.locate(pid, ITEMS ? (pid == up ? Pu : Pl) : sxy[pid], cur);
                ok = P.split(leaf, pid);
                loc[pid] = (uint16_t)FNIL;
            }
        }
        if (!ok) break;
        // add_segment(p1, p2)  :493 -- pass 1
        if (use_items) {
            // finish this edge's search (its own two points were inserted a moment ago) and copy the
            // leaves, in list order, into node_stack
            P.nstack = 0;
            bool first_item = true;
            while (it != FNIL && ok) {
                uint32_t node = first_item ? it_node0 : it_node[it];
                uint32_t nxt = first_item ? it_next0 : it_next[it];
                first_item = false;
                for (;;) {
                    const uint2 v = P.nd[node];
                    if (FPoly::type_of(v.y) == T_TRAPEZOID) break;
                    bool both;
                    const uint32_t next = P.dfs_step(v, up, lo, Pu, Pl, &both);
                    if (both) {
                        const uint32_t nw = ctr[0];
                        if (nw >= caps.item_cap) {
                            P.requeue = true;
                            ok = false;
                            break;
                        }
                        __syncwarp();
                        if (lane == 0) ctr[0] = nw + 1u;
                        it_node[nw] = (uint16_t)(v.x >> 16);
                        it_edge[nw] = (uint16_t)edge;
                        it_next[nw] = (uint16_t)nxt;
                        nxt = nw;
                        __syncwarp();
                    }
                    node = next;
                }
                if (!ok) break;
                ok = P.push(node);  // :302
                it = nxt;
            }
            ehead[edge] = (uint16_t)FNIL;
            if (!ok) break;
        } else {
            // serial walk; a search that has already produced 48 leaves is one of the exploding ones and is
            // redone as a parallel frontier expansion (items + output list live in the mountain arrays,
            // unused during part 1)
            P.stack = stack_home;
            P.gstack = MR_SPAN_NULL(uint16_t);
            const int sr = P.search_from_root(up, lo, par_cap ? 48u : 0xFFFFFFFFu);
            if (sr == 2) {
                if (!P.search_parallel<false>(up, lo, par_node, par_next, par_cap, par_out, par_out_cap, par_ctr, lane)) {
                    ok = false;
                    if (par_gl && P.requeue) {
                        // The shared-memory scratch is sized for occupancy, not for the worst case: the (rare) search
                        // that outgrows it is redone in this warp's global-memory scratch, which holds the contract cap
                        // -- cheaper than sending the polygon to the retry launch, whose few polygons run alone on the GPU.
                        P.requeue = false;
                        uint16_t* g = reinterpret_cast<uint16_t*>(par_gl);
                        ok = P.search_parallel<true>(up, lo, MR_MAKE_SPAN(uint16_t, g, PAR_GL_CAP), MR_MAKE_SPAN(uint16_t, g + PAR_GL_CAP, PAR_GL_CAP),
                                                     PAR_GL_CAP, MR_MAKE_SPAN(uint16_t, g + 2u * PAR_GL_CAP, PAR_GL_CAP), PAR_GL_CAP, par_ctr, lane) != 0;
                    }
                }
            } else if (sr == 0) {
                ok = false;
            }
            if (!ok) break;
        }
        ok = P.pass2(p1, up, lo, lane, 16u);  // pass 2: scan as written below 16 entries, REDUX arg-min above
        __syncwarp();
    }
    if (P.requeue) return F_REQUEUE_SPEC;
    if (!ok) {
        res->status = P.status | (sink.cap_vtx ? MR_POLY_UNDERFILL : 0u);
        sink.zero(0, sink.cap_vtx, lane);
        return F_DONE;
    }

    if (ITEMS) {
        // rank -> original id, needed from here on: rebuilt behind mstart's place in the dead node_stack (fast_layout)
        for (uint32_t i = lane; i < n; i += 32) orig[rk[i]] = (uint16_t)i;
        __syncwarp();
    }

    // ---- part 2: inside trapezoids -> adds, in node id order (:510-540) ---------------------------
    MR_SPAN(uint32_t) add_pp = MR_MAKE_SPAN(uint32_t, reinterpret_cast<uint32_t*>(ws + L.add_pp), caps.add_cap);
    MR_SPAN(uint32_t) add_key = MR_MAKE_SPAN(uint32_t, reinterpret_cast<uint32_t*>(ws + L.add_key), caps.add_cap);
    MR_SPAN(uint16_t) add_m = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.add_m), caps.add_cap);
    MR_SPAN(uint32_t) mcount = MR_MAKE_SPAN(uint32_t, reinterpret_cast<uint32_t*>(ws + L.mcount), caps.add_cap);
    MR_SPAN(uint16_t) mstart = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.mstart), caps.add_cap + 1u);
    MR_SPAN(uint16_t) efirst = MR_MAKE_SPAN(uint16_t, reinterpret_cast<uint16_t*>(ws + L.efirst), caps.nmax);
    const uint32_t PMASK = 0xFFFF1FFFu;  // (pa, pb) without the type and crumb bits

    uint32_t A = 0;
    bool bad = false, over = false;
    for (uint32_t b = 0; b < P.nnodes; b += 32) {
        const uint32_t id = b + lane;
        uint32_t cnt = 0, k0 = 0, k1 = 0, mypp = 0;
        bool lane_bad = false;
        if (id < P.nnodes) {
            const uint2 v = P.nd[id];
            if (FPoly::type_of(v.y) == T_TRAPEZOID) {
                const uint32_t c1 = v.x & 0xFFFFu, c2 = v.x >> 16;
                if (c1 != FNIL) {                                    // :516
                    // :517 crumb == child2.  Segment node: the stored bit; any other node has a null crumb,
                    // which equals child2 only when child2 is null too.
                    const uint2 c1n = P.nd[c1];
                    const bool inside = FPoly::type_of(c1n.y) == T_SEGMENT ? (c1n.y & CRUMB_RIGHT) != 0u : (c1n.x >> 16) == FNIL;
                    if (inside) {
                        mypp = v.y & PMASK;
                        if ((mypp & FNIL14) == FNIL14 || (mypp >> 16) == FNIL || c2 == FNIL) {
                            lane_bad = true;  // :524-527
                        } else {
                            const uint32_t c2pp = P.nd[c2].y & PMASK, c1pp = P.nd[c1].y & PMASK;
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
                            if ((k0 & FNIL14) == FNIL14 || (k0 >> 16) == FNIL) lane_bad = true;  // :58
                            if (cnt == 2 && ((k1 & FNIL14) == FNIL14 || (k1 >> 16) == FNIL)) lane_bad = true;
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
            add_key[off] = k0;
            add_pp[off] = mypp;
        }
        if (cnt == 2) {
            add_key[off + 1] = k1;
            add_pp[off + 1] = mypp;
        }
        A += total;
    }
    if (over) return F_REQUEUE_SPEC;  // more adds than this tier holds (the kernel maps this to the next tier up)
    if (bad) {
        res->status = MR_POLY_NULL_UNWRAP | (sink.cap_vtx ? MR_POLY_UNDERFILL : 0u);
        sink.zero(0, sink.cap_vtx, lane);
        return F_DONE;
    }
    __syncwarp();

    // ---- mountains: rank by first appearance (keys are (upper, lower) rank pairs) ----------------
    for (uint32_t i = lane; i < n; i += 32) efirst[i] = (uint16_t)FNIL;
    __syncwarp();
    uint32_t M = 0;
    for (uint32_t b = 0; b < A; b += 32) {
        const uint32_t ai = b + lane;
        const bool valid = ai < A;
        const uint32_t key = valid ? add_key[ai] : 0u;
        const uint32_t ku = key & FNIL14, kl = key >> 16;
        uint32_t e = FNIL;
        if (valid && ku < n && kl < n && ku < kl) {  // (upper, lower) of a polygon edge?
            const uint32_t ou = orig[ku], ol = orig[kl];
            if ((ou + 1u == n ? 0u : ou + 1u) == ol) e = ou;
            else if ((ol + 1u == n ? 0u : ol + 1u) == ou) e = ol;
        }
        const uint32_t same = __match_any_sync(0xFFFFFFFFu, valid ? key : (0xC0000000u + lane));
        const bool leader = valid && ((same & lt_mask) == 0u);
        uint32_t first = ai;
        if (leader) {
            if (e != FNIL) {
                const uint32_t f = efirst[e];
                if (f != FNIL) first = f; else efirst[e] = (uint16_t)ai;
            } else {
                for (uint32_t h = 0; h < b; ++h)  // rare: the key node is not a segment of the polygon
                    if (add_key[h] == key) {
                        first = h;
                        break;
                    }
            }
        }
        first = __shfl_sync(0xFFFFFFFFu, first, __ffs(same) - 1);
        const bool isfirst = valid && first == ai;
        const uint32_t fm = __ballot_sync(0xFFFFFFFFu, isfirst);
        // first adds store their mountain rank with bit 15 set; the others the index of the first add
        if (valid) add_m[ai] = (uint16_t)(isfirst ? (0x8000u | (M + __popc(fm & lt_mask))) : first);
        M += __popc(fm);
        __syncwarp();
    }
    for (uint32_t ai = lane; ai < A; ai += 32) {
        const uint32_t v = add_m[ai];
        if (!(v & 0x8000u)) add_m[ai] = (uint16_t)(add_m[v] & 0x7FFFu);  // add_m[v] is a first add, never rewritten here
    }
    __syncwarp();
    for (uint32_t ai = lane; ai < A; ai += 32) add_m[ai] &= 0x7FFFu;
    for (uint32_t i = lane; i < M; i += 32) mcount[i] = 0u;
    __syncwarp();
    for (uint32_t ai = lane; ai < A; ai += 32) atomicAdd(&mcount[add_m[ai]], 2u);
    __syncwarp();
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
            if (i < M) mstart[i] = (uint16_t)(run + inc - v);
            run += __shfl_sync(0xFFFFFFFFu, inc, 31);
        }
        if (lane == 0) mstart[M] = (uint16_t)run;
    }
    __syncwarp();
    for (uint32_t i = lane; i < M; i += 32) mcount[i] = 0u;
    __syncwarp();

    // ---- group, sort, emit (all warps of the team) ---------------------------------------------------
    if (W > 1) {
        if (lane == 0) {
            ts->cmd = TEAM_FINISH;
            ts->arg0 = A;
            ts->flag0 = 0u;
        }
        team_bar<W>();
    }
    return team_finish<W>(sink, cap_tri, ws, caps, L, A, lane, ts, res);
}

