/*
 * o_triangulation.c -- oracle restatement of Polygon/Triangulation.zig.
 * TEST INFRASTRUCTURE ONLY (see mr_oracle.h).
 *
 * Seidel-style trapezoidation in a flat node arena, grouping of the inside
 * trapezoids into monotone mountains, and the emission loop -- statement for
 * statement, with these representation changes only:
 *   - `?u32` null is the sentinel MR_O_NULL (null==null and null!=value keep
 *     their meaning; a forced unwrap `.?` of null aborts the polygon with
 *     MR_POLY_NULL_UNWRAP instead of panicking / being UB)
 *   - std.debug.print calls (Triangulation.zig:142,181,194,195,226,346,371,372,
 *     380,388,513) are removed; they do not affect results
 *   - the edge order comes from an explicit mr_o_unirand instead of
 *     unirand_seed's std.crypto.random draws (:483)
 *   - a full pass of the emission loop (:558-586) without progress ends the
 *     mountain with MR_POLY_STUCK (the reference would loop forever)
 *   - the contract's resource caps MR_NODE_CAP(n) / MR_STACK_CAP(n) abandon the polygon
 *     with MR_POLY_ARENA (the reference would keep allocating)
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include "mr_oracle.h"

enum { T_POINT = 0, T_SEGMENT = 1, T_TRAPEZOID = 2 }; /* Triangulation.zig:40 */

typedef struct mountain { /* Triangulation.zig:46 */
    uint32_t p1, p2;
    uint32_t* list;
    uint32_t len, cap;
} mountain;

struct mr_o_tri {
    uint32_t root_node; /* :4 */
    mr_o_node* nodes;   /* :6 */
    uint32_t nnodes, cap_nodes;
    const float* points; /* :9, xy pairs */
    uint32_t* node_stack; /* :12 */
    uint32_t nstack, cap_stack;
    mountain* mountains; /* MountainList.backend :44 */
    uint32_t nmount, cap_mount;
    uint32_t status;
    uint32_t node_cap, stack_cap; /* MR_NODE_CAP(n), MR_STACK_CAP(n) */
    mr_o_stats* stats;
};

/* Test-only switch (tests/test_oracle_cpu.py::test_arena_caps_are_not_a_divergence): multiplies the contract
 * caps (safety valve at 2^27 entries; the reference has no bound at all, but its DFS re-pushes a
 * merged trapezoid once per DAG path and pass 2 is quadratic in the stack, so an unbounded run of
 * an exploding polygon does not end in practical time -- measured: 3,203 such polygons, 8 threads,
 * > 15 minutes and 5 GB without finishing).  The test shows that every polygon the contract caps
 * abandon is still not finished correctly with caps many times larger. */
static uint32_t g_caps_mult = 1;
void mr_o_test_lift_caps(uint32_t multiplier) { g_caps_mult = multiplier ? multiplier : 1u; }
static uint32_t lifted(uint32_t cap) {
    const uint64_t v = (uint64_t)cap * g_caps_mult;
    return v > (1u << 27) ? (1u << 27) : (uint32_t)v;
}

/* Test-only switch (tests/_poly_float_edges.py): one float rule replaced by a wrong restatement; 0 = the reference. */
static uint32_t g_mutant = MR_O_MUT_NONE;
void mr_o_test_mutant(uint32_t id) { g_mutant = id < MR_O_MUT_COUNT ? id : MR_O_MUT_NONE; }
uint32_t mr_o_mutant(void) { return g_mutant; }

static float ftz(float v) { return fpclassify(v) == FP_SUBNORMAL ? copysignf(0.0f, v) : v; }

mr_o_tri* mr_o_tri_new(void) { /* :427-435 */
    return (mr_o_tri*)calloc(1, sizeof(mr_o_tri));
}

void mr_o_tri_destroy(mr_o_tri* t) { /* :437-440 */
    uint32_t i;
    if (!t) return;
    for (i = 0; i < t->cap_mount; ++i) free(t->mountains[i].list);
    free(t->mountains);
    free(t->nodes);
    free(t->node_stack);
    free(t);
}

uint32_t mr_o_tri_node_count(const mr_o_tri* t) { return t->nnodes; }
const mr_o_node* mr_o_tri_nodes(const mr_o_tri* t) { return t->nodes; }

/* :102-107 and :109-115 share the arena growth.  Contract cap: MR_NODE_CAP(n). */
static uint32_t arena_push(mr_o_tri* t) {
    if (t->nnodes >= t->node_cap) {
        t->status |= MR_POLY_ARENA;
        return MR_O_NULL;
    }
    if (t->nnodes == t->cap_nodes) {
        t->cap_nodes = t->cap_nodes ? t->cap_nodes * 2u : 256u;
        t->nodes = (mr_o_node*)realloc(t->nodes, (size_t)t->cap_nodes * sizeof(mr_o_node));
    }
    return t->nnodes++;
}

static uint32_t add_node(mr_o_tri* t, uint32_t type) { /* :102-107 */
    uint32_t id = arena_push(t);
    mr_o_node* nd;
    if (id == MR_O_NULL) return id;
    nd = &t->nodes[id];
    nd->type = type;
    nd->crumb = nd->child1 = nd->child2 = nd->point1 = nd->point2 = MR_O_NULL;
    return id;
}

static uint32_t clone_node(mr_o_tri* t, uint32_t node) { /* :109-115 */
    uint32_t id = arena_push(t);
    if (id == MR_O_NULL) return id;
    t->nodes[id] = t->nodes[node];
    return id;
}

static int is_left_of_mutant(const float* p, const float* a, const float* b) {
    switch (g_mutant) {
        case MR_O_MUT_SIDE_FMA:
            return fmaf(b[0] - a[0], p[1] - a[1], -((b[1] - a[1]) * (p[0] - a[0]))) > 0.0f;
        case MR_O_MUT_SIDE_F64:
            return ((double)b[0] - a[0]) * ((double)p[1] - a[1]) - ((double)b[1] - a[1]) * ((double)p[0] - a[0]) > 0.0;
        case MR_O_MUT_SIDE_EXACTDIFF: /* a product of two floats is exact in double; the difference keeps its sign */
            return (double)(b[0] - a[0]) * (double)(p[1] - a[1]) - (double)(b[1] - a[1]) * (double)(p[0] - a[0]) > 0.0;
        case MR_O_MUT_SIDE_REFORM:
            return (a[0] - p[0]) * (b[1] - p[1]) - (a[1] - p[1]) * (b[0] - p[0]) > 0.0f;
        case MR_O_MUT_SIDE_FTZ: {
            const float m1 = ftz(ftz(ftz(b[0]) - ftz(a[0])) * ftz(ftz(p[1]) - ftz(a[1])));
            const float m2 = ftz(ftz(ftz(b[1]) - ftz(a[1])) * ftz(ftz(p[0]) - ftz(a[0])));
            return ftz(m1 - m2) > 0.0f;
        }
        default: /* MR_O_MUT_SIDE_GE */
            return (b[0] - a[0]) * (p[1] - a[1]) - (b[1] - a[1]) * (p[0] - a[0]) >= 0.0f;
    }
}

/* sort key of one coordinate: order-preserving u32, -0 mapped to +0 unless `rawzero`; `signflip` flips the sign bit only */
static uint32_t order_key(float v, int rawzero, int signflip) {
    uint32_t u;
    if (!rawzero && v == 0.0f) v = 0.0f;
    memcpy(&u, &v, 4);
    if (signflip) return u ^ 0x80000000u;
    return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}

static int point_is_above_mutant(float lx, float ly, float rx, float ry) {
    switch (g_mutant) {
        case MR_O_MUT_ORDER_RAWZERO:
        case MR_O_MUT_ORDER_SIGNFLIP: {
            const int raw = g_mutant == MR_O_MUT_ORDER_RAWZERO, flip = g_mutant == MR_O_MUT_ORDER_SIGNFLIP;
            const uint32_t kly = order_key(ly, raw, flip), kry = order_key(ry, raw, flip);
            return kly < kry || (kly == kry && order_key(lx, raw, flip) < order_key(rx, raw, flip));
        }
        case MR_O_MUT_ORDER_DAZ:
            lx = ftz(lx), ly = ftz(ly), rx = ftz(rx), ry = ftz(ry);
            return ly < ry || (ly == ry && lx < rx);
        default: /* MR_O_MUT_ORDER_TIE_LE */
            return ly < ry || (ly == ry && lx <= rx);
    }
}

/* :117-126 -- two separately rounded products, one rounded difference (compile with
 * -ffp-contract=off; the volatile-free form is safe on x86-64 SSE2, FLT_EVAL_METHOD 0) */
static int is_left_of(const mr_o_tri* t, uint32_t pid, uint32_t s1, uint32_t s2) {
    const float* p = &t->points[2u * pid];
    const float* a = &t->points[2u * s1];
    const float* b = &t->points[2u * s2];
    float mul1, mul2, d;
    if (g_mutant >= MR_O_MUT_SIDE_FMA && g_mutant <= MR_O_MUT_SIDE_GE) return is_left_of_mutant(p, a, b);
    mul1 = (b[0] - a[0]) * (p[1] - a[1]);
    mul2 = (b[1] - a[1]) * (p[0] - a[0]);
    d = mul1 - mul2;
    return d > 0.0f;
}

/* :128-136 -- lexicographic (y, x); smaller y is "above" */
static int point_is_above(const mr_o_tri* t, uint32_t lhs, uint32_t rhs) {
    float ly = t->points[2u * lhs + 1u], ry = t->points[2u * rhs + 1u];
    if (g_mutant >= MR_O_MUT_ORDER_RAWZERO && g_mutant <= MR_O_MUT_ORDER_TIE_LE)
        return point_is_above_mutant(t->points[2u * lhs], ly, t->points[2u * rhs], ry);
    if (ly < ry) return 1;
    if (ly == ry) return t->points[2u * lhs] < t->points[2u * rhs];
    return 0;
}

/* `.?` : returns 0 and flags the polygon when the optional is null */
#define UNWRAP(dst, expr)                      \
    do {                                       \
        uint32_t v_ = (expr);                  \
        if (v_ == MR_O_NULL) {                 \
            t->status |= MR_POLY_NULL_UNWRAP;  \
            return 0;                          \
        }                                      \
        (dst) = v_;                            \
    } while (0)

/* :139-196 */
static int add_point(mr_o_tri* t, uint32_t point_id) {
    uint32_t base = t->root_node;
    uint32_t lower, upper;
    for (;;) { /* :144-167 */
        mr_o_node* nd = &t->nodes[base];
        uint32_t next, p;
        if (t->stats) {
            t->stats->descent_steps++;
            t->stats->point_steps++;
        }
        if (nd->type == T_TRAPEZOID) break;
        if (nd->type == T_POINT) {
            if (nd->point1 == point_id) return 1; /* :149-152 already added */
            UNWRAP(p, nd->point1);
            if (point_is_above(t, point_id, p))
                UNWRAP(next, nd->child1);
            else
                UNWRAP(next, nd->child2);
        } else {
            uint32_t s1, s2;
            UNWRAP(s1, nd->point1);
            UNWRAP(s2, nd->point2);
            if (is_left_of(t, point_id, s1, s2))
                UNWRAP(next, nd->child1);
            else
                UNWRAP(next, nd->child2);
        }
        base = next;
    }
    lower = clone_node(t, base); /* :178 -- lower first */
    upper = clone_node(t, base); /* :179 */
    if (lower == MR_O_NULL || upper == MR_O_NULL) return 0;
    { /* :183-188 -- the found trapezoid becomes the point node in place */
        mr_o_node* nd = &t->nodes[base];
        nd->type = T_POINT;
        nd->point1 = point_id;
        nd->point2 = MR_O_NULL;
        nd->crumb = MR_O_NULL;
        nd->child1 = upper;
        nd->child2 = lower;
    }
    t->nodes[upper].point2 = point_id; /* :191 */
    t->nodes[lower].point1 = point_id; /* :192 */
    return 1;
}

static int stack_push(mr_o_tri* t, uint32_t v) {
    if (t->nstack >= t->stack_cap) { /* contract cap MR_STACK_CAP(n) */
        t->status |= MR_POLY_ARENA;
        return 0;
    }
    if (t->nstack == t->cap_stack) {
        t->cap_stack = t->cap_stack ? t->cap_stack * 2u : 64u;
        t->node_stack = (uint32_t*)realloc(t->node_stack, (size_t)t->cap_stack * 4u);
    }
    t->node_stack[t->nstack++] = v;
    return 1;
}

/* :215-396 */
static int add_segment(mr_o_tri* t, uint32_t point1, uint32_t point2) {
    uint32_t up, lo; /* upper_segment_point, lower_segment_point */
    uint32_t base, breadcrumb = MR_O_NULL;
    uint32_t left_trap, right_trap;
    if (point_is_above(t, point1, point2)) { /* :218-224 */
        up = point1;
        lo = point2;
    } else {
        up = point2;
        lo = point1;
    }
    base = t->root_node;
    t->nstack = 0; /* :230 */
    for (;;) {     /* loop1 :231 */
        for (;;) { /* loop :232 */
            mr_o_node* nd = &t->nodes[base];
            if (t->stats) t->stats->descent_steps++;
            if (nd->type == T_POINT) { /* :234-259 */
                uint32_t pc;
                UNWRAP(pc, nd->point1);
                if (up == pc) {
                    UNWRAP(base, nd->child2);
                } else if (lo == pc) {
                    UNWRAP(base, nd->child1);
                } else {
                    int bottom_point_is_above = point_is_above(t, lo, pc);
                    int top_point_is_below = point_is_above(t, pc, up);
                    if (top_point_is_below) {
                        UNWRAP(base, nd->child2);
                    } else if (bottom_point_is_above) {
                        UNWRAP(base, nd->child1);
                    } else { /* :252-257 straddles: leave a breadcrumb, take child1 */
                        nd->crumb = breadcrumb;
                        breadcrumb = base;
                        UNWRAP(base, nd->child1);
                    }
                }
            } else if (nd->type == T_SEGMENT) { /* :260-296 */
                uint32_t o1, o2;
                int is_left;
                UNWRAP(o1, nd->point1);
                UNWRAP(o2, nd->point2);
                if (up == o2 || up == o1) {
                    is_left = is_left_of(t, lo, o1, o2);
                } else if (lo == o1 || lo == o2) {
                    is_left = is_left_of(t, up, o1, o2);
                } else {
                    int top_is_above = point_is_above(t, up, o1);
                    int bottom_is_below = point_is_above(t, lo, o2);
                    if (top_is_above && bottom_is_below) {
                        is_left = !is_left_of(t, o1, up, lo);
                    } else if (top_is_above && !bottom_is_below) {
                        is_left = is_left_of(t, lo, o1, o2);
                    } else {
                        is_left = is_left_of(t, up, o1, o2);
                    }
                }
                if (is_left)
                    UNWRAP(base, nd->child1);
                else
                    UNWRAP(base, nd->child2);
            } else {
                break; /* :297 */
            }
        }
        if (!stack_push(t, base)) return 0; /* :302 */
        if (breadcrumb != MR_O_NULL) { /* :306-313 */
            uint32_t crumb = breadcrumb;
            breadcrumb = t->nodes[crumb].crumb;
            t->nodes[crumb].crumb = MR_O_NULL;
            UNWRAP(base, t->nodes[crumb].child2);
        } else {
            break;
        }
    }
    if (t->stats) {
        t->stats->sum_stack += t->nstack;
        if (t->nstack > t->stats->max_stack) t->stats->max_stack = t->nstack;
    }

    /* pass 2 :316-395 */
    left_trap = add_node(t, T_TRAPEZOID); /* :319-320 */
    if (left_trap == MR_O_NULL) return 0;
    t->nodes[left_trap].point1 = up;
    right_trap = add_node(t, T_TRAPEZOID); /* :322-323 */
    if (right_trap == MR_O_NULL) return 0;
    t->nodes[right_trap].point1 = up;

    while (t->nstack > 0) { /* :325 */
        uint32_t base_index = 0;
        uint32_t base_id = t->node_stack[0];
        uint32_t low_point = lo;
        uint32_t i;
        for (i = 0; i < t->nstack; ++i) { /* :329-337 first strictly-higher wins */
            uint32_t node = t->node_stack[i];
            uint32_t np;
            UNWRAP(np, t->nodes[node].point2);
            if (t->stats) t->stats->select_steps++;
            if (point_is_above(t, np, low_point)) {
                low_point = np;
                base_index = i;
                base_id = node;
            }
        }
        /* :347-360 the trapezoid becomes a segment node in place */
        t->nodes[base_id].type = T_SEGMENT;
        t->nodes[left_trap].child1 = t->nodes[base_id].child1;
        t->nodes[base_id].child1 = left_trap;
        t->nodes[base_id].crumb = (point1 == up) ? left_trap : right_trap; /* :351-355 */
        t->nodes[right_trap].child2 = t->nodes[base_id].child2;
        t->nodes[base_id].child2 = right_trap;
        t->nodes[base_id].point1 = up;
        t->nodes[base_id].point2 = lo;

        if (lo == low_point) { /* :366-373 */
            t->nodes[left_trap].child2 = base_id;
            t->nodes[left_trap].point2 = low_point;
            t->nodes[right_trap].child1 = base_id;
            t->nodes[right_trap].point2 = low_point;
            break;
        } else if (is_left_of(t, low_point, up, lo)) { /* :375-382 */
            t->nodes[left_trap].child2 = base_id;
            t->nodes[left_trap].point2 = low_point;
            left_trap = add_node(t, T_TRAPEZOID);
            if (left_trap == MR_O_NULL) return 0;
            t->nodes[left_trap].point1 = low_point;
        } else { /* :383-391 */
            t->nodes[right_trap].child1 = base_id;
            t->nodes[right_trap].point2 = low_point;
            right_trap = add_node(t, T_TRAPEZOID);
            if (right_trap == MR_O_NULL) return 0;
            t->nodes[right_trap].point1 = low_point;
        }
        /* :394 swapRemove */
        t->node_stack[base_index] = t->node_stack[t->nstack - 1u];
        t->nstack--;
    }
    return 1;
}

/* MountainList.add_point :49-62 */
static int mountain_add(mr_o_tri* t, uint32_t key, uint32_t p1, uint32_t p2) {
    mountain* found = NULL;
    uint32_t i;
    uint32_t k1 = t->nodes[key].point1, k2 = t->nodes[key].point2;
    for (i = 0; i < t->nmount; ++i) { /* :51-55 keeps the last match */
        mountain* m = &t->mountains[i];
        if (m->p1 == k1 && m->p2 == k2) found = m;
    }
    if (!found) { /* :56-59 */
        uint32_t a, b;
        UNWRAP(a, k1);
        UNWRAP(b, k2);
        if (t->nmount == t->cap_mount) {
            uint32_t nc = t->cap_mount ? t->cap_mount * 2u : 32u;
            t->mountains = (mountain*)realloc(t->mountains, (size_t)nc * sizeof(mountain));
            memset(&t->mountains[t->cap_mount], 0, (size_t)(nc - t->cap_mount) * sizeof(mountain));
            t->cap_mount = nc;
        }
        found = &t->mountains[t->nmount++];
        found->p1 = a;
        found->p2 = b;
        found->len = 0; /* keeps its allocation from earlier polygons */
    }
    if (found->len + 2u > found->cap) {
        found->cap = found->cap ? found->cap * 2u : 16u;
        found->list = (uint32_t*)realloc(found->list, (size_t)found->cap * 4u);
    }
    found->list[found->len++] = p1; /* :60 */
    found->list[found->len++] = p2; /* :61 */
    return 1;
}

static void ordered_remove(mountain* m, uint32_t idx) {
    memmove(&m->list[idx], &m->list[idx + 1u], (size_t)(m->len - idx - 1u) * 4u);
    m->len--;
}

/* :398-425 */
static int push_triangle_if_acute(mr_o_tri* t, uint32_t point, uint32_t axis1, uint32_t axis2,
                                  void* ctx, mr_o_emit_fn emit) {
    const float* P = t->points;
    float nx1 = P[2u * point] - P[2u * axis1];
    float ny1 = P[2u * point + 1u] - P[2u * axis1 + 1u];
    float nx2 = P[2u * point] - P[2u * axis2];
    float ny2 = P[2u * point + 1u] - P[2u * axis2 + 1u];
    float diff;
    const float pi_f32 = 3.14159274101257324f; /* std.math.pi coerced to f32 */
    int is_acute;
    if (g_mutant == MR_O_MUT_ACUTE_CR_ATAN2)
        diff = (float)atan2((double)ny1, (double)nx1) - (float)atan2((double)ny2, (double)nx2);
    else if (g_mutant == MR_O_MUT_ACUTE_DAZ_ATAN2)
        diff = ftz(mr_o_atan2f(ftz(ny1), ftz(nx1))) - ftz(mr_o_atan2f(ftz(ny2), ftz(nx2)));
    else
        diff = mr_o_atan2f(ny1, nx1) - mr_o_atan2f(ny2, nx2);
    if (diff < 0.0f) diff = -diff; /* @abs; NaN stays NaN and compares false */
    is_acute = diff < pi_f32;
    if (g_mutant == MR_O_MUT_ACUTE_PI_DOWN) is_acute = diff < 3.14159250259399414f; /* 0x40490fda */
    if (g_mutant == MR_O_MUT_ACUTE_LE) is_acute = diff <= pi_f32;
    if (g_mutant == MR_O_MUT_ACUTE_ALWAYS) is_acute = 1;
#define EMIT(id) emit(ctx, (id), P[2u * (id)], P[2u * (id) + 1u])
    if (is_acute) {
        EMIT(point);
        if ((axis1 > point && axis2 > point) || (axis1 < point && axis2 < point)) {
            if (axis1 > axis2) {
                EMIT(axis2);
                EMIT(axis1);
            } else {
                EMIT(axis1);
                EMIT(axis2);
            }
        } else if (axis2 > point) {
            EMIT(axis2);
            EMIT(axis1);
        } else if (axis1 > point) {
            EMIT(axis1);
            EMIT(axis2);
        }
        /* remaining case (an axis equals `point`) emits only the centre, as written */
        if (t->stats) t->stats->triangles++;
    } else if (t->stats) {
        t->stats->not_acute++;
    }
#undef EMIT
    return is_acute;
}

/* :446-589 */
uint32_t mr_o_tri_create_polygon(mr_o_tri* t, const float* xy, uint32_t n, mr_o_unirand rng,
                                 void* ctx, mr_o_emit_fn emit, mr_o_stats* stats) {
    uint32_t edge, item, mi;
    t->nstack = 0; /* :453-455 */
    t->nnodes = 0;
    t->points = xy;
    t->status = MR_POLY_OK;
    t->stats = stats;
    t->nmount = 0;
    t->node_cap = lifted(MR_NODE_CAP(n));
    t->stack_cap = lifted(MR_STACK_CAP(n));

    t->root_node = add_node(t, T_TRAPEZOID); /* :479 */

    while (mr_o_unirand_next(&rng, &edge)) { /* :484-494 */
        uint32_t p1 = edge;
        uint32_t p2 = (uint32_t)(((uint64_t)edge + 1u) % n);
        if (!add_point(t, p1)) goto done;
        if (!add_point(t, p2)) goto done;
        if (!add_segment(t, p1, p2)) goto done;
    }

    /* part 2 :510-540 */
    for (item = 0; item < t->nnodes; ++item) {
        mr_o_node* nd = &t->nodes[item];
        uint32_t point1, point2, child1, child2;
        if (nd->type != T_TRAPEZOID) continue;
        if (nd->child1 == MR_O_NULL) continue; /* :516,:521 */
        if (t->nodes[nd->child1].crumb != t->nodes[nd->child1].child2) continue; /* :517-520 */
        if (nd->point1 == MR_O_NULL || nd->point2 == MR_O_NULL || nd->child2 == MR_O_NULL) {
            t->status |= MR_POLY_NULL_UNWRAP; /* :524-527 */
            goto done;
        }
        point1 = nd->point1;
        point2 = nd->point2;
        child1 = nd->child1;
        child2 = nd->child2;
        if (point1 == t->nodes[child2].point1 && point2 == t->nodes[child2].point2) { /* :528 */
            if (!mountain_add(t, child1, point1, point2)) goto done;
        } else if (point1 == t->nodes[child1].point1 && point2 == t->nodes[child1].point2) { /* :531 */
            if (!mountain_add(t, child2, point1, point2)) goto done;
        } else { /* :534-538 */
            if (!mountain_add(t, child1, point1, point2)) goto done;
            if (!mountain_add(t, child2, point1, point2)) goto done;
        }
    }

    /* part 3 :553-587 */
    for (mi = 0; mi < t->nmount; ++mi) {
        mountain* m = &t->mountains[mi];
        uint32_t i;
        if (stats) {
            stats->mountains++;
            if (m->len > stats->max_mountain) stats->max_mountain = m->len;
        }
        /* :555 std.sort.insertion -- stable */
        for (i = 1; i < m->len; ++i) {
            uint32_t j = i;
            while (j > 0 && point_is_above(t, m->list[j], m->list[j - 1u])) {
                uint32_t tmp = m->list[j];
                m->list[j] = m->list[j - 1u];
                m->list[j - 1u] = tmp;
                --j;
            }
        }
        while (m->len > 2u) { /* loop :558 */
            uint32_t p1 = m->len - 2u, p2 = m->len - 1u, p3 = 0;
            uint32_t len0 = m->len;
            int progressed = 0;
            for (item = 1; item < len0; ++item) { /* :562 */
                if (m->list[p1] == m->list[p2]) { /* :563-566 */
                    ordered_remove(m, p1);
                    progressed = 1;
                    break;
                }
                if (m->list[p2] == m->list[p3]) { /* :567-570 */
                    ordered_remove(m, p2);
                    progressed = 1;
                    break;
                }
                if (push_triangle_if_acute(t, m->list[p2], m->list[p1], m->list[p3], ctx, emit)) {
                    ordered_remove(m, p2); /* :579 */
                    progressed = 1;
                    break;
                }
                p1 = p2; /* :582-584 */
                p2 = p3;
                p3 = item;
            }
            if (!progressed) { /* the reference would repeat the same pass forever */
                t->status |= MR_POLY_STUCK;
                break;
            }
        }
    }
done:
    if (stats) stats->nodes += t->nnodes;
    return t->status;
}
