/*
 * mr_oracle.h -- CPU parity oracle for the myrenderer geometry hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under myrenderer_b200/ (the product) may
 * include, link, import or execute anything in oracle/.  Only tests/,
 * __graft_entry__.smoke() and bench.py's CPU-baseline legs use it.
 *
 * What it is: a plain-C restatement of the reference's Zig code for the path
 * (Polygon/Triangulation.zig, Polygon/unirand.zig, Polygon/Polygon.zig:50-79,
 * Terrain/Terrain.zig:21-50,114-124), each function citing the lines it
 * follows.  The reference cannot be compiled here (no Zig toolchain; `mach`
 * and `zigimg` are un-vendored URL dependencies, build.zig.zon:27-34), so there
 * is no oracle/_ref build.
 *
 * PARITY PINNING STATUS (see DESIGN.md "Oracle"):
 *   - the reference has no tests, golden vectors or fixtures with expected
 *     outputs (SURVEY 4, 8-c).  The oracle is pinned against (1) the
 *     hand-derived known answer for App.zig's polygon2 traced from the Zig
 *     source (SURVEY 8-a: 18 nodes, triangles (2,3,1),(3,0,1)), (2) structural
 *     invariants of the reference algorithm, (3) the reference-authored inputs
 *     (HEIGHTMAP.png, polygon1, polygon2).  Beyond that: PARITY UNPINNED for
 *       * std.crypto.random (unirand.zig:31)  -- replaced by an explicit stream
 *       * std.math.atan2 f32 (Triangulation.zig:403) -- restated from the musl
 *         algorithm Zig's std ports; cannot change the output for finite input
 *         except in the corner documented at mr_o_atan2f
 *       * terrain normals and index buffer -- NEW SPEC, no reference code exists
 */
#ifndef MR_ORACLE_H
#define MR_ORACLE_H

#include <stdint.h>
#include "../include/myrenderer_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define MR_O_NULL 0xFFFFFFFFu /* Zig `null` of a ?u32 */

/* --- unirand.zig ---------------------------------------------------------- */
typedef struct mr_o_unirand {
    uint32_t at, top, offset, prime;
} mr_o_unirand;

uint64_t mr_o_rng_state0(uint64_t seed, uint64_t index);
uint32_t mr_o_rng_u32(uint64_t* state);
void mr_o_unirand_seed(mr_o_unirand* r, uint32_t top, uint64_t* rng_state);
void mr_o_unirand_explicit(mr_o_unirand* r, uint32_t top, uint32_t offset, uint32_t prime);
int mr_o_unirand_next(mr_o_unirand* r, uint32_t* out); /* 1 = value, 0 = null */

/* --- std.math.atan2 (f32) -------------------------------------------------- */
float mr_o_atanf(float x);
float mr_o_atan2f(float y, float x);

/* --- Triangulation.zig ----------------------------------------------------- */
typedef struct mr_o_node {
    uint32_t type; /* 0 point, 1 segment, 2 trapezoid */
    uint32_t crumb, child1, child2, point1, point2;
} mr_o_node;

typedef struct mr_o_stats {
    uint64_t nodes;          /* nodes allocated                                   */
    uint64_t max_stack;      /* largest node_stack (k) in add_segment             */
    uint64_t sum_stack;      /* sum of k over edges                               */
    uint64_t descent_steps;  /* DAG nodes visited by add_point + add_segment      */
    uint64_t mountains;      /* monotone mountains created                        */
    uint64_t max_mountain;   /* longest mountain list (with duplicates)           */
    uint64_t triangles;      /* triangles emitted                                 */
    uint64_t not_acute;      /* push_triangle_if_acute calls that returned false  */
    uint64_t point_steps;    /* descent_steps spent in add_point                  */
    uint64_t select_steps;   /* iterations of the pass-2 selection loop (:329-337) */
} mr_o_stats;

typedef struct mr_o_tri mr_o_tri; /* reusable arenas, like the Zig struct */
typedef void (*mr_o_emit_fn)(void* ctx, uint32_t point_id, float x, float y);

mr_o_tri* mr_o_tri_new(void);
void mr_o_tri_destroy(mr_o_tri* t);
/* Returns a MR_POLY_* status word.  stats may be NULL. */
uint32_t mr_o_tri_create_polygon(mr_o_tri* t, const float* xy, uint32_t n, mr_o_unirand rng,
                                 void* ctx, mr_o_emit_fn emit, mr_o_stats* stats);
/* Test-only: multiply the contract caps MR_NODE_CAP / MR_STACK_CAP (1 = contract; safety valve 2^27). */
void mr_o_test_lift_caps(uint32_t multiplier);
/* Test-only: replace one float rule of the reference by a plausible wrong restatement of it (a "mutant"), so that the
 * tests can show that their inputs tell the two apart (tests/_poly_float_edges.py).  0 restores the reference rules.
 * Set it only while no oracle call is running; it applies to every thread. */
enum {
    MR_O_MUT_NONE = 0,
    /* is_left_of, Triangulation.zig:117-126 */
    MR_O_MUT_SIDE_FMA,       /* fmaf(bx-ax, py-ay, -mul2): mul1 unrounded */
    MR_O_MUT_SIDE_F64,       /* every operation in double */
    MR_O_MUT_SIDE_EXACTDIFF, /* f32 differences, exact products and a correctly signed difference in double */
    MR_O_MUT_SIDE_REFORM,    /* (ax-px)*(by-py) - (ay-py)*(bx-px): same exact sign, other roundings */
    MR_O_MUT_SIDE_FTZ,       /* inputs, differences, products and result flushed to +-0 when subnormal */
    MR_O_MUT_SIDE_GE,        /* d >= 0 */
    /* point_is_above, Triangulation.zig:128-136 */
    MR_O_MUT_ORDER_RAWZERO,  /* -0 before +0 (the sort key without its zero normalisation) */
    MR_O_MUT_ORDER_SIGNFLIP, /* key = bits ^ sign bit only: negative coordinates sort backwards */
    MR_O_MUT_ORDER_DAZ,      /* subnormal coordinates compare as zero */
    MR_O_MUT_ORDER_TIE_LE,   /* ly == ry && lx <= rx */
    /* push_triangle_if_acute, Triangulation.zig:398-425 */
    MR_O_MUT_ACUTE_CR_ATAN2, /* correctly rounded atan2 (double atan2 rounded to f32) */
    MR_O_MUT_ACUTE_PI_DOWN,  /* compare with 0x40490fda */
    MR_O_MUT_ACUTE_LE,       /* diff <= pi */
    MR_O_MUT_ACUTE_ALWAYS,   /* every corner acute */
    MR_O_MUT_ACUTE_DAZ_ATAN2,/* atan2 arguments and result flushed to +-0 when subnormal */
    /* render_point bbox, Polygon.zig:73-76 */
    MR_O_MUT_BBOX_TIE_REPLACES, /* v <= acc ? v : acc (a hardware fminf/fmaxf on +-0) */
    MR_O_MUT_BBOX_OWN_Y,        /* p1.y / p2.y accumulate their own min / max */
    /* non-finite rejection */
    MR_O_MUT_NONFINITE_X_ONLY,  /* only x coordinates are checked */
    MR_O_MUT_NONFINITE_NAN_ONLY,/* infinities pass */
    MR_O_MUT_COUNT
};
void mr_o_test_mutant(uint32_t id);
uint32_t mr_o_mutant(void);
/* Introspection for tests: node arena after the last create_polygon. */
uint32_t mr_o_tri_node_count(const mr_o_tri* t);
const mr_o_node* mr_o_tri_nodes(const mr_o_tri* t);

/* --- Polygon.zig ------------------------------------------------------------ */
/* Same contract as mr_triangulate_batch with host pointers; nthreads<=0 -> all cores.
 * ids_out (optional) receives the emitted PointIDs, 3 per triangle slot, 0xFFFFFFFF when unused. */
int mr_o_polygon_batch(const mr_polygon_job* job, uint32_t* ids_out, int nthreads,
                       mr_o_stats* stats_total);
void mr_o_palette(float rgb_out[12]);
/* bench.py only: mean seconds per Polygon.create_polygon-shaped call (reusable arenas, one polygon), timed in C */
double mr_o_time_create_polygon(const float* xy, uint32_t n, uint32_t offset, uint32_t prime, uint32_t reps);

/* --- Terrain.zig ------------------------------------------------------------ */
int mr_o_terrain_build(const mr_terrain_job* job, int nthreads);
void mr_o_heightmap_normalize(const uint16_t* in, uint64_t count, float* out);
/* Expanded non-indexed stream exactly as the WGSL shader computes it for shader vertex `vi`
 * of an n x n terrain (Terrain.zig:24-48); h is the f32 heightmap. Returns 0 if the lookup
 * index is outside [0,n*n) (the reference reads out of bounds there, SURVEY 8-a2'). */
int mr_o_terrain_shader_vertex(const float* h, uint32_t n, uint64_t vi,
                               const mr_terrain_params* p, float out4[4]);

/* tiles + culling: same contracts as mr_terrain_tile_bounds / mr_terrain_cull with host pointers; the visibility
 * test is SceneNode.zig:96-110 (mr_o_scene_node_should_render is the per-box form) */
int mr_o_terrain_tile_bounds(const void* height, uint32_t fmt, uint32_t n, uint32_t tile_rows, uint32_t tile_cols,
                             const mr_terrain_params* p, float* bbox_out);
int mr_o_scene_node_should_render(const float xform[16], const float p0[4], const float p1[4]);
int mr_o_terrain_cull(const float* bbox, uint32_t n, uint32_t tile_rows, uint32_t tile_cols, const float xform[16],
                      uint32_t* visible_out, uint32_t* visible_ids_out, uint32_t* idx_out, uint64_t counts_out[2]);

/* --- synthetic inputs (same definitions as the library's generators) -------- */
void mr_o_synth_heightmap_u16(uint64_t seed, uint32_t n, uint32_t row0, uint32_t rows,
                              uint16_t* out);
void mr_o_synth_polygon_sizes(uint64_t seed, uint64_t poly_index0, uint32_t npoly, uint32_t nmin,
                              uint32_t nmax, int dist, uint64_t* first_point_out);
void mr_o_synth_polygons(uint64_t seed, uint64_t poly_index0, const uint64_t* first_point,
                         uint32_t npoly, float* xy_out);
void mr_o_synth_polygons_family(int family, uint64_t seed, uint64_t poly_index0,
                                const uint64_t* first_point, uint32_t npoly, float* xy_out);

int mr_o_hardware_threads(void);

#ifdef __cplusplus
}
#endif
#endif
