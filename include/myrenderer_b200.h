/*
 * myrenderer_b200.h -- C ABI of the B200-native geometry-generation library.
 *
 * This is the drop-in boundary for ONE hot path of platypro/myrenderer: the
 * heightmap -> grid mesh build and the batched Seidel polygon triangulation.
 * The reference has no FFI today (its seam is three Zig functions); each entry
 * point below names the reference interface whose *body* it replaces.  All
 * citations are relative to the reference tree.
 *
 *   Terrain.create_terrain            Terrain/Terrain.zig:88-129   -> mr_terrain_build
 *   WGSL vertex formula               Terrain/Terrain.zig:21-50    -> mr_terrain_build (positions)
 *   Polygon.create_polygon            Polygon/Polygon.zig:81-107   -> mr_triangulate_batch (mr_triangulate_earclip)
 *   Triangulation.create_polygon      Polygon/Triangulation.zig:446-589 -> mr_triangulate_batch
 *   render_point (emit sink)          Polygon/Polygon.zig:65-79    -> mr_triangulate_batch (vtx_out, bbox_out)
 *   unirand_seed / Unirand.next       Polygon/unirand.zig:12-50    -> mr_unirand_seed_batch (+ inside the kernel)
 *   Triangulation.new / destroy       Polygon/Triangulation.zig:427-440 -> mr_context_create / mr_context_destroy
 *   VertexLayout.native               Renderer/VertexLayout.zig:12-30 -> mr_layout
 *   VertexBuffer{vertex_count,first_vertex}  Renderer/VertexBuffer.zig:5-24 -> mr_draw_range
 *   SceneNode.render visibility test  Renderer/SceneNode.zig:96-110 -> mr_terrain_cull (per terrain tile)
 *   Terrain bounding box              Terrain/Terrain.zig:103-110   -> mr_terrain_describe, mr_terrain_tile_bounds
 *
 * Conventions
 *   - plain C types only; no exceptions cross this boundary; every function
 *     returns MR_OK (0) or a negative MR_E_* code.
 *   - data pointers in job structs may be device pointers or host pointers.
 *     Host pointers are staged through context-owned device scratch (the copy
 *     is part of the call); device pointers are used in place.
 *   - all work is ordered on the context's stream and is asynchronous for
 *     device pointers until mr_sync().  A call that was given ANY host pointer
 *     (pageable or pinned, input or output) returns only after its inputs have
 *     been read and its results are in the caller's buffers.
 *   - there is no CPU fallback: without a CUDA device every compute entry
 *     point fails with MR_E_CUDA.
 */
#ifndef MYRENDERER_B200_H
#define MYRENDERER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MR_ABI_VERSION 1

/* ---- return codes -------------------------------------------------------- */
#define MR_OK 0
#define MR_E_BADARG (-1)  /* null pointer, bad size, bad layout                         */
#define MR_E_CUDA (-2)    /* a CUDA runtime call failed; see mr_last_error()            */
#define MR_E_NOMEM (-3)   /* scratch allocation failed                                  */
#define MR_E_ARENA (-4)   /* a polygon overflowed every arena tier (status_out says which) */

/* ---- per-polygon status word (bit set) ------------------------------------
 * The reference has undefined behaviour (ReleaseFast) or a safety panic
 * (Debug) in these situations; the library and the oracle define them
 * identically instead.                                                       */
#define MR_POLY_OK 0u
#define MR_POLY_DEGENERATE 1u   /* n < 3: Polygon.zig:82 computes len-2 (underflow); nothing emitted     */
#define MR_POLY_NONFINITE 2u    /* NaN/Inf coordinate: point_is_above is no longer an order; nothing emitted */
#define MR_POLY_NULL_UNWRAP 4u  /* a `.?` in Triangulation.zig hit null; polygon abandoned, output zero-filled */
#define MR_POLY_OVERFLOW 8u     /* more than n-2 triangles produced (Polygon.zig:78 appendAssumeCapacity); extras dropped */
#define MR_POLY_STUCK 16u       /* Triangulation.zig:558-586 made a full pass without progress (reference would spin) */
#define MR_POLY_TOO_LARGE 32u   /* n above MR_MAX_POLYGON_POINTS; nothing emitted                        */
#define MR_POLY_ARENA 64u       /* resource cap hit: node id >= MR_NODE_CAP(n) or DFS stack >= MR_STACK_CAP(n); nothing emitted */
#define MR_POLY_UNDERFILL 128u  /* fewer than n-2 triangles produced; tail of the range is zero (WebGPU zero-init) */
#define MR_POLY_NO_EAR 256u     /* mr_triangulate_earclip only: a lap of the ring found no ear (never on a simple polygon) */

#define MR_MAX_POLYGON_POINTS 4096u
/* Resource caps (part of the contract; the oracle applies the same ones).  The reference's
 * segment search (Triangulation.zig:231-314) is a DFS over a DAG with merged trapezoids and can
 * push the same trapezoid many times; on non-convex input the stack and the node arena can grow
 * without useful bound (16.5M entries were observed for one 1024-gon).  A polygon that would
 * allocate node id >= MR_NODE_CAP(n) or push stack entry index >= MR_STACK_CAP(n) is abandoned
 * with MR_POLY_ARENA and emits nothing. */
#define MR_NODE_CAP(n) (8u * (uint32_t)(n) + 64u)
#define MR_STACK_CAP(n) (16u * (uint32_t)(n) + 64u)

/* ---- vertex layout: mirror of VertexLayout.native (VertexLayout.zig:12-30) -
 * stride = @sizeOf(T); attr[i] = {@offsetOf(T, field i), component count of
 * float32x2/x3/x4, shader_location = i}.  Offsets are run-time values because
 * Zig may reorder the fields of a non-extern struct.  Bytes of a vertex not
 * covered by an attribute are written as zero.                               */
#define MR_MAX_ATTR 4
typedef struct mr_attr {
    uint32_t offset;   /* bytes from the start of the vertex; multiple of 4 */
    uint32_t ncomp;    /* 2, 3 or 4 float32 components                      */
    uint32_t location; /* shader_location (informational)                   */
} mr_attr;

typedef struct mr_layout {
    uint32_t stride; /* array_stride in bytes; multiple of 4, 8..256 */
    uint32_t nattr;
    mr_attr attr[MR_MAX_ATTR];
} mr_layout;

/* Ready-made layouts.
 * GPUVertex{x: Vec2, color: Vec3} (Polygon.zig:26-29), Vec3 = 16-byte @Vector:
 *   _DECL   : fields in declaration order      x@0,  color@16, stride 32
 *   _ZIGAUTO: fields sorted by alignment       color@0, x@16,  stride 32
 * TerrainVertex{pos: Vec3, normal: Vec3} (new type; SURVEY 8-a4): pos@0, normal@16, stride 32. */
#define MR_LAYOUT_GPUVERTEX_DECL 0
#define MR_LAYOUT_GPUVERTEX_ZIGAUTO 1
#define MR_LAYOUT_TERRAINVERTEX 2
int mr_layout_preset(int which, mr_layout* out);

/* ---- draw descriptor: mirror of VertexBuffer (VertexBuffer.zig:5-9,20-24) - */
typedef struct mr_draw_range {
    uint32_t vertex_count;   /* primitive_count * 3 */
    uint32_t instance_count; /* 1                   */
    uint32_t first_vertex;   /* offset * 3          */
    uint32_t first_instance; /* 0                   */
} mr_draw_range;

/* ---- context: owns stream + device scratch (Triangulation.new/destroy) ---- */
typedef struct mr_context mr_context;

int mr_abi_version(void);
/* bit 0: bounds-checked build (-DMR_CHECKED, see myrenderer_b200/csrc/Makefile `checked`) */
int mr_build_flags(void);
int mr_device_count(int* count_out);
int mr_context_create(int device, mr_context** ctx_out);
int mr_context_destroy(mr_context* ctx);
/* Use an existing cudaStream_t (passed as void*) instead of the context's own. */
int mr_context_set_stream(mr_context* ctx, void* cuda_stream);
int mr_context_stream(mr_context* ctx, void** cuda_stream_out);
int mr_sync(mr_context* ctx);
/* Text of the last error on this context (never NULL). */
const char* mr_last_error(const mr_context* ctx);
/* Kernels launched by this context since creation (monotonic). */
uint64_t mr_launch_count(const mr_context* ctx);
/* Host-pointer calls stage through context-owned device scratch that grows to the largest call made
 * (one 16384^2 host-buffer terrain build holds ~15 GB).  mr_context_trim synchronises and frees all of
 * it; the next call re-allocates what it needs.  mr_context_scratch_bytes reports the current total. */
int mr_context_trim(mr_context* ctx);
int mr_context_scratch_bytes(const mr_context* ctx, uint64_t* bytes_out);

/* ---- plain device-memory helpers for hosts without a CUDA binding (Zig) --- */
int mr_device_alloc(mr_context* ctx, size_t bytes, void** dev_out);
int mr_device_free(mr_context* ctx, void* dev);
int mr_pinned_alloc(mr_context* ctx, size_t bytes, void** host_out);
int mr_pinned_free(mr_context* ctx, void* host);
int mr_copy(mr_context* ctx, void* dst, const void* src, size_t bytes); /* any direction, stream-ordered */
int mr_fill_zero(mr_context* ctx, void* dev, size_t bytes);

/* ---- terrain ---------------------------------------------------------------
 * Grid mesh of an n x n heightmap.
 *   height texel (r,c), row-major r*n+c:
 *       MR_HEIGHT_U16: raw PNG grayscale16 value v; h = 1.0f - (float)v / 65535.0f   (Terrain.zig:120)
 *       MR_HEIGHT_F32: h itself.  Any float: NaN, +-inf, +-0 and subnormals are computed with IEEE
 *                      semantics, with no flush to zero of inputs or results.
 *   position(r,c) = ( grid_step*(float)r - origin_scale*(float)n,
 *                     height_scale*h,
 *                     grid_step*(float)c - origin_scale*(float)n )                  (Terrain.zig:24-48, indexed form)
 *     each product and the difference separately rounded (no FMA).
 *   normal(r,c)  [NEW SPEC, none in the reference]: clamped central differences
 *       rm=max(r-1,0) rp=min(r+1,n-1) (same for c)
 *       gx = (height_scale*(h[rp][c]-h[rm][c])) / (grid_step*(float)(rp-rm))
 *       gz = (height_scale*(h[r][cp]-h[r][cm])) / (grid_step*(float)(cp-cm))
 *       len = sqrtf(((gx*gx)+1.0f)+(gz*gz));  inv = 1.0f/len;  normal = (-gx*inv, inv, -gz*inv)
 *     IEEE round-to-nearest for every operation, no FMA; n==1 gives gx=gz=0.  (One reciprocal and
 *     two products instead of three quotients: at most 1 ulp from the quotient form.)
 *   NaN outputs (of the mesh, the tile boxes and anything else this header calls bit-exact): where an
 *     output float is NaN, its sign and payload are unspecified (the GPU writes a canonical NaN, a CPU
 *     may carry an input's payload).  Every other output, signed zeros and infinities included, is
 *     bit-exact as specified.
 *   indices [NEW SPEC]: u32, 6 per quad, quads (r,c) r,c in [0,n-1) row-major, corner order of
 *       Terrain.zig:28-35 under cw front faces (Pipeline.zig:145-149):
 *       (r+1,c) (r,c) (r+1,c+1) (r+1,c+1) (r,c) (r,c+1)   with i(r,c)=r*n+c
 * Performance note: the quotients by grid_step and 2*grid_step use an exact reciprocal-and-correct
 * scheme that is enabled only for divisors it has been verified for over all 2^32 dividends
 * (mr_selftest_fastdiv): grid_step = 0.2f (the reference's constant, divisors 0.2f and 0.4f).  Any
 * other grid_step is computed with IEEE division -- same results by definition, but the vertex kernel
 * becomes issue-bound (about 0.6 instead of 0.9 of the HBM roofline).
 * vtx_out must be 4-byte aligned and idx_out 8-byte aligned (MR_E_BADARG otherwise).
 * The job describes a row band so that one call can be one rank's shard:
 *   vertex (r,c) is written at vtx_out + ((r - vtx_row0)*n + c)*stride for r in [row_begin,row_end)
 *   quad row q is written at idx_out + (q - idx_qrow0)*6*(n-1) for q in [qrow_begin,qrow_end)
 *   height points at texel row height_row0 and holds height_rows rows; it must cover
 *   [max(row_begin-1,0), min(row_end+1,n)).
 * vtx_out / idx_out may be NULL to skip that product.                         */
#define MR_HEIGHT_U16 0
#define MR_HEIGHT_F32 1

typedef struct mr_terrain_params {
    float grid_step;    /* 0.2 (Terrain.zig:36) */
    float origin_scale; /* 0.1 (Terrain.zig:36) */
    float height_scale; /* 5.0 (Terrain.zig:48) */
} mr_terrain_params;

typedef struct mr_terrain_job {
    uint32_t n;
    uint32_t height_fmt;
    const void* height;
    uint32_t height_row0, height_rows;
    uint32_t row_begin, row_end;
    void* vtx_out;
    uint32_t vtx_row0;
    uint32_t qrow_begin, qrow_end;
    uint32_t* idx_out;
    uint32_t idx_qrow0;
    mr_layout layout; /* attr[0] = position (ncomp>=3), attr[1] = normal (ncomp>=3, optional) */
    mr_terrain_params params;
} mr_terrain_job;

int mr_terrain_params_default(mr_terrain_params* out);
int mr_terrain_build(mr_context* ctx, const mr_terrain_job* job);
/* Whole mesh in one call: all rows, all quads. */
int mr_terrain_build_full(mr_context* ctx, const void* height, uint32_t height_fmt, uint32_t n,
                          const mr_layout* layout, const mr_terrain_params* params, void* vtx_out,
                          uint32_t* idx_out);
/* bounding box + draw descriptor (Terrain.zig:103-110,126 adapted to the indexed mesh) */
int mr_terrain_describe(uint32_t n, const mr_terrain_params* params, float bbox_min[3],
                        float bbox_max[3], uint64_t* vertex_count, uint64_t* index_count);
/* Self-test used by the test-suite: compares the kernels' constant-divisor quotient routine with IEEE
 * division for all 2^32 dividends and returns the number of mismatches (0 expected).  force_fast != 0
 * exercises the reciprocal-and-correct path even for a divisor the library would not enable it for. */
int mr_selftest_fastdiv(mr_context* ctx, float divisor, int force_fast, uint64_t* mismatches_out);
/* Standalone heightmap normalisation (Terrain.zig:114-124): u16 -> f32. */
int mr_heightmap_normalize(mr_context* ctx, const uint16_t* in, uint64_t count, float* out);

/* ---- terrain tiles and culling (SURVEY 8-f rank 4) -----------------------------
 * The mesh is cut into tiles of tile_rows x tile_cols QUADS (the last tile of a row / column may be
 * smaller); tile t = tr * tiles_c + tc covers quad rows [tr*tile_rows, ...) and quad columns
 * [tc*tile_cols, ...), i.e. vertex rows r0..r1 and columns c0..c1 INCLUSIVE with r1 = last quad row + 1.
 *
 * mr_terrain_tile_bounds writes one bounding box per tile in the form SceneNode keeps them
 * (SceneNode.zig:11-22, Terrain.zig:103-110 per tile instead of per terrain): 8 floats
 *     p0 = (min x, min y, min z, 1)   p1 = (max x, max y, max z, 1)
 * over the tile's vertices, positions as defined for mr_terrain_build (x from the row, z from the
 * column, y = height_scale * h).  min/max are exact (comparisons only), so the boxes are bit-exact;
 * a y bound that is zero is written as +0.0f (with height_scale == 0, or a float map holding both
 * zeros, the sign of a zero bound would otherwise depend on the order of the reduction).  NaN heights
 * are skipped by the min/max; a tile of NaNs only has min +inf and max -inf, so its y bounds are
 * height_scale*(+-inf) in order (-inf, +inf at height_scale 5; NaN at height_scale 0).
 *
 * mr_terrain_cull applies the reference's visibility test (SceneNode.zig:96-110) to every tile box:
 *     q0 = M * p0 unless some component of p0 is -inf;  q1 = M * p1 unless some component of p1 is +inf
 *     visible = all(q1 > 0) or all(q0 < 1)                                (all four components, no divide)
 * with M the composed transform as the memory image of mach.math.Mat4x4 (four column Vec4s:
 * xform[4*col + row]) and M * p evaluated like mach's Mat4x4.mulVec: result[i] starts at 0 and adds
 * xform[4*j + i] * p[j] for j = 0..3 in order, every operation separately rounded.  (mach is not
 * vendored in the reference tree: mulVec is restated from the mach source -- parity unpinned.)
 * bbox may hold any floats.  "Some component is -inf" is fminf over the four components == -inf (and
 * fmaxf == +inf for p1), so the skip rule ignores NaN components; a NaN that reaches a comparison makes
 * it false.  Subnormal inputs and products are not flushed to zero.
 * Outputs, each optional (NULL to skip), device or host pointers:
 *     visible_out[t]      1 / 0 per tile
 *     visible_ids_out[k]  the visible tiles in ascending order, k < counts_out[0]
 *     idx_out             compacted index buffer: the visible tiles in ascending order, each tile's quads
 *                         row-major, six indices per quad exactly as mr_terrain_build writes them --
 *                         one drawIndexed(counts_out[1]) draws what survives the cull
 *     counts_out[2]       {visible tiles, indices written} as uint64
 * Any tile size is accepted, up to and beyond the terrain (one tile may hold all (n-1)^2 quads); with idx_out
 * the tile count is at most 2^31-1 (only 1 x 1 tiles of an n > 46341 terrain exceed it).  The arguments are checked
 * before any kernel runs, so a rejected call writes no output.
 * Alignment (MR_E_BADARG otherwise): bbox_out of mr_terrain_tile_bounds 16 bytes (a box is two float4),
 * idx_out of mr_terrain_cull 8 bytes.
 *
 * mr_terrain_cull_frustum is mr_terrain_cull with the standard six-plane frustum test in place of the
 * reference's: the outputs, argument checks, alignment, device / host pointers, the checks before any kernel
 * runs and the 2^31-1 tile limit with idx_out are those above.  The reference's test does no perspective divide
 * and is kept for parity; this one is the cull to draw with under a perspective camera.  Bit for bit:
 *   view_proj is the memory image of mach's Mat4x4, as xform above: clip[i] = sum_j view_proj[4j+i] * v[j].  The
 *     clip volume is WebGPU's, -w <= x <= w, -w <= y <= w, 0 <= z <= w (math.zig's perspective maps near..far to
 *     depth 0..w).
 *   Row i is R_i = (view_proj[i], view_proj[4+i], view_proj[8+i], view_proj[12+i]).  The six planes are
 *     R3+R0, R3-R0, R3+R1, R3-R1, R2, R3-R2, each component one rounded f32 add or subtract; not normalised.
 *   Per plane (a, b, c, d) and box: lo = p0.xyz, hi = p1.xyz (the w components are not read);
 *     px = (a >= 0) ? hi.x : lo.x, py likewise from b, pz from c (so -0 picks hi and a NaN coefficient picks lo);
 *     s = ((a*px + b*py) + c*pz) + d, every product and sum rounded on its own (no FMA, no flush to zero).
 *   A tile is culled iff s < 0 for some plane; a NaN s never culls.  bbox may hold any floats.
 * Properties that follow: in exact arithmetic a box with any point inside the clip volume is never culled; a box
 * lying wholly on the outer side of one plane is culled; SceneNode's default box (-inf..+inf) is never culled, since
 * every p-vertex term is +inf or NaN; and, as usual for this test, a box near the frustum's edges and corners can
 * survive although it lies outside. */
int mr_terrain_tile_count(uint32_t n, uint32_t tile_rows, uint32_t tile_cols, uint32_t* tiles_r_out,
                          uint32_t* tiles_c_out);
int mr_terrain_tile_bounds(mr_context* ctx, const void* height, uint32_t height_fmt, uint32_t n,
                           uint32_t tile_rows, uint32_t tile_cols, const mr_terrain_params* params,
                           float* bbox_out /* tiles * 8 */);
int mr_terrain_cull(mr_context* ctx, const float* bbox /* tiles * 8 */, uint32_t n, uint32_t tile_rows,
                    uint32_t tile_cols, const float xform[16], uint32_t* visible_out,
                    uint32_t* visible_ids_out, uint32_t* idx_out, uint64_t* counts_out);
int mr_terrain_cull_frustum(mr_context* ctx, const float* bbox /* tiles * 8 */, uint32_t n, uint32_t tile_rows,
                            uint32_t tile_cols, const float view_proj[16], uint32_t* visible_out,
                            uint32_t* visible_ids_out, uint32_t* idx_out, uint64_t* counts_out);

/* ---- polygons --------------------------------------------------------------
 * Triangulates npoly polygons exactly as Triangulation.create_polygon would,
 * one after the other, with render_point as the emit sink.
 *   polygon i has points xy[2*(first_point[i]-point_base) ...], n_i = first_point[i+1]-first_point[i]
 *   its vertex range starts at vertex 3*(first_tri[i]-tri_base) of vtx_out and holds 3*(n_i-2) vertices
 *   (first_tri = exclusive prefix sum of max(n_i-2,0); see mr_polygon_offsets)
 *   colour of emitted vertex k of the polygon = palette[(k/3)%4]                 (Polygon.zig:50-57,78)
 *   bbox_out[4*i..] = {p1.x,p1.y,p2.x,p2.y} with the update rule as written      (Polygon.zig:73-76)
 * Edge insertion order (unirand.zig): either explicit per-polygon (offset,prime)
 * pairs, or drawn on the device by the port of unirand_seed from the documented
 * stream  R_k(i) = splitmix64 stream keyed by (seed, poly_index0+i)  -- see mr_rng_u32.
 * Output triangles are bit-identical to the reference's for the same (offset,prime).
 * Float semantics, on every path (all size classes, the small-batch path, the general path):
 *   - coordinates are compared and the side test is evaluated with IEEE f32 semantics, each operation rounded on
 *     its own, with no flush to zero: subnormal coordinates, differences and products keep their values
 *   - in the (y, x) order of point_is_above -0 equals +0; two points equal in both coordinates up to the sign of
 *     zero are coincident
 *   - finiteness is checked on both coordinates of every point: a NaN or +-inf anywhere gives MR_POLY_NONFINITE
 *   - a bbox component that is zero is always +0 (the accumulators start at +0 and a tie keeps the accumulator) */
typedef struct mr_polygon_job {
    const float* xy;
    const uint64_t* first_point; /* npoly+1 entries */
    uint64_t point_base;
    uint32_t npoly;
    const uint32_t* offset_prime; /* 2*npoly {offset,prime} or NULL -> seeded */
    uint64_t seed;
    uint64_t poly_index0;
    mr_layout layout; /* attr[0] = x (ncomp 2), attr[1] = color (ncomp 3) */
    void* vtx_out;
    const uint64_t* first_tri; /* npoly+1 entries */
    uint64_t tri_base;
    float* bbox_out;      /* 4*npoly or NULL */
    uint32_t* status_out; /* npoly   or NULL */
    uint32_t* ntri_out;   /* npoly   or NULL: triangles actually emitted */
} mr_polygon_job;

int mr_triangulate_batch(mr_context* ctx, const mr_polygon_job* job);
/* Introspection: how the last mr_triangulate_batch on this context spread its polygons over the
 * arena tiers.  out[0..4] = polygons re-run with contract-cap arenas, by size (<=64, <=128, <=256,
 * <=512, <=1024 points); out[5] = polygons of 1025..3072 points handed from their shared-memory
 * pass to the general path (there is no retry tier at that size); out[6] = polygons of up to 1024
 * points handed to the general path (coincident points, not-acute corner, ...); out[7] = polygons
 * of 3073..MR_MAX_POLYGON_POINTS points (always general path).  Synchronises the stream. */
int mr_triangulate_tier_counts(mr_context* ctx, uint32_t out[8]);
/* ---- ear clipping ------------------------------------------------------------
 * mr_triangulate_batch reproduces the reference's triangulator, which fails on many non-convex polygons (DESIGN.md
 * section 2).  mr_triangulate_earclip triangulates every simple polygon correctly, into the same output format: the
 * job, its checks, alignment, layouts, host / device pointers, point_base / tri_base and the optional outputs are those
 * of mr_triangulate_batch; offset_prime, seed and poly_index0 are ignored.  It stages host pointers like a large batch
 * (no small-batch path), and leaves mr_triangulate_tier_counts and the reference path's launch state as they were.
 *   n < 3, a NaN / +-inf coordinate on either axis, n > MR_MAX_POLYGON_POINTS: MR_POLY_DEGENERATE / NONFINITE /
 *     TOO_LARGE written exactly as mr_triangulate_batch writes them (range zeroed, ntri 0, bbox +0).
 *   Every other polygon emits exactly n-2 triangles, triangle k coloured palette[k % 4], bbox by the rule of
 *   mr_triangulate_batch over the emitted vertices in order.  A first_tri range of another size keeps the reference
 *   path's rule: triangles past it are dropped (MR_POLY_OVERFLOW, still counted in the bbox), a shorter polygon leaves a
 *   zeroed tail (MR_POLY_UNDERFILL); ntri = min(n-2, range).
 * Bit for bit.  P[i] is point i; a == b is float equality of both coordinates (-0 == +0).
 *   orient(a, b, c) = sign of the EXACT value of (bx-ax)(cy-ay) - (by-ay)(cx-ax) for the float inputs (nothing rounded
 *     or flushed; mr_selftest_orient exposes the device's predicate).
 *   Winding s: m = the first index smallest in (y, x); pm / nm = the nearest ring predecessor / successor of m whose
 *     point differs from P[m]; s = orient(P[pm], P[m], P[nm]), or +1 if that is 0 or all points coincide.
 *   Ring: doubly linked over 0..n-1.  Cursor c = 0, stop = c.  While the ring has k > 3 vertices, with p = prev(c),
 *     q = next(c), c is an ear if
 *       (a) P[c] == P[p] or P[c] == P[q] (a zero-length edge), or
 *       (b) s*orient(p, c, q) > 0 and no blocker lies in the closed triangle: a blocker is a ring vertex r not in
 *           {p, c, q} with s*orient(prev(r), r, next(r)) <= 0, P[r] different from P[p], P[c] and P[q], and
 *           s*orient(p, c, r) >= 0, s*orient(c, q, r) >= 0, s*orient(q, p, r) >= 0.
 *     Ear: emit (p, c, q) if s > 0 else (q, c, p), unlink c, c = next(q), stop = c.
 *     Not an ear: c = next(c); if c == stop, a whole lap found no ear: clip c anyway as above and set MR_POLY_NO_EAR.
 *   At k = 3: emit (prev(c), c, next(c)), ordered by the same rule.
 * Properties: a simple polygon (collinear and repeated vertices allowed) never sets MR_POLY_NO_EAR and its triangles
 * tile it exactly, every one with orientation >= 0 in raw (x, y) (two-ears theorem: a vertex that is not strictly
 * convex is the only kind that can lie in an ear's triangle).  Any other input still gets n-2 triangles and a defined,
 * bit-exact result.  Cost: O(n^2) candidate tests per polygon in the worst case, each scanning up to n blockers. */
int mr_triangulate_earclip(mr_context* ctx, const mr_polygon_job* job);
/* Self-test used by the test-suite: sign_out[i] = orient of the triple abc[6i..6i+5] = (ax, ay, bx, by, cx, cy), as
 * mr_triangulate_earclip evaluates it (-1, 0, +1). */
int mr_selftest_orient(mr_context* ctx, const float* abc /* 6 per triple */, uint64_t count, int8_t* sign_out);
/* ---- ear clipping of polygons with holes ---------------------------------------------------------------------
 * mr_triangulate_earclip_holes triangulates polygons whose point range holds several rings: an outer boundary and holes.
 * The job, its checks, alignment, layouts, host / device pointers, sub-ranges, optional outputs, palette, bbox rule and
 * OVERFLOW / UNDERFILL rule are those of mr_triangulate_earclip, with the triangle count T = N + 2H - 2 in place of
 * n - 2 (N points, H holes; see mr_polygon_offsets_rings).  The rings of polygon i are first_ring[i] ..
 * first_ring[i+1]-1; ring r starts at point ring_start[r - ring_base] and ends where the next ring starts (the last one
 * at first_point[i+1]).  first_ring and ring_start may be device or host pointers (host ones are staged like
 * first_point).  The ring arrays are read per polygon inside the kernel, so bad ring data is a polygon status, not an
 * MR_E_BADARG.  Checks, in this order, each written as mr_triangulate_earclip writes a reject (range zeroed, ntri 0,
 * bbox +0):
 *   R = first_ring[i+1] - first_ring[i] (as uint64) is 0 or larger than N:                     MR_POLY_DEGENERATE
 *   N + 2(R-1) > MR_MAX_POLYGON_POINTS:                                                          MR_POLY_TOO_LARGE
 *   the first ring start differs from first_point[i], ring starts do not increase, or a ring has fewer than 3 points:
 *                                                                                                MR_POLY_DEGENERATE
 *   a NaN / +-inf coordinate on either axis of any point:                                        MR_POLY_NONFINITE
 * Bit for bit (orient, a == b and the winding rule as for mr_triangulate_earclip):
 *   s = the winding of the outer ring; each hole has its own winding by the same rule.  M(h) = the first point of hole
 *   h largest in (x, y).  Holes are merged one at a time in decreasing (x, y) of M(h), equal M in hole order, into the
 *   current ring C (initially the outer ring, positions 0..L-1 in ring order).  For hole h with M = M(h), y = My:
 *   1. Crossing edges: ring edges (C[k], C[k+1]) = (a, b) with s*(b.y - a.y) > 0, min(a.y, b.y) <= My <= max(a.y, b.y)
 *      and s*orient(a, b, M) >= 0.  Edge 2 crosses nearer than edge 1 when
 *        cross(a1, b1, a2, b2, My) = sign of the EXACT (b2.y - My)*O(a1,b1,a2) + (My - a2.y)*O(a1,b1,b2) > 0
 *      (O the exact orient value; mr_selftest_crossing exposes the device's predicate).  The nearest edge k is the one
 *      with the smallest crossing x (the order cross() decides), the first in position order among equal crossings.
 *      No crossing edge: the hole is bridged to position 0 and MR_POLY_BAD_HOLE is set.
 *   2. Target t: if a.y == My then t = k; else if b.y == My then t = k+1; else t = k if a.x >= b.x else k+1, and with
 *      u = sign(P[t].y - My), every position r whose point differs from M, whose vertex is not strictly convex
 *      (s*orient(C[r-1], C[r], C[r+1]) <= 0) and which lies in the closed triangle (M, crossing point, P[t]) -- u*sign(P[r].y - My) >= 0, s*orient(a, b, r) >= 0,
 *      u*orient(M, P[t], r) <= 0 -- replaces t, in position order, if u*orient(M, r, t) > 0, or it is 0 and
 *      P[r].x < P[t].x (smallest angle to the ray, then nearest).
 *   3. Copy: the first position k' (in position order) whose point equals P[t] and whose wedge contains M:
 *      s*orient(C[k'-1], P[t], C[k'+1]) > 0 ? (s*orient(C[k'-1], P[t], M) > 0 and s*orient(P[t], C[k'+1], M) > 0)
 *                                           : (s*orient(C[k'-1], P[t], M) > 0 or  s*orient(P[t], C[k'+1], M) > 0);
 *      t itself when there is none.
 *   4. Splice after position k': C[0..k'], M and the rest of the hole from M on (in reverse ring order if the hole's
 *      winding equals s), M again, C[k'] again, C[k'+1..L-1].
 *   The merged ring of N + 2H points is then clipped exactly as mr_triangulate_earclip clips a ring of that many points:
 *   its own winding, ring walk, rules (a) and (b), emit order and NO_EAR fallback, unchanged.  (Rule (b)'s point-equality
 *   exclusion keeps the two copies of a bridge endpoint from blocking each other's ears.)  With H = 0 the result is
 *   mr_triangulate_earclip's, byte for byte.
 * Properties: for valid input -- outer ring and holes simple, holes strictly inside the outer ring and pairwise
 * disjoint -- neither MR_POLY_NO_EAR nor MR_POLY_BAD_HOLE is set and the N + 2H - 2 triangles tile the polygon with its
 * holes removed, every one with orientation >= 0 in raw (x, y).  Any other input still gets T triangles and a defined,
 * bit-exact result.  Cost: the merge is O(H * (N + 2H)) predicate evaluations per polygon, the clip that of a ring of
 * N + 2H points. */
#define MR_POLY_BAD_HOLE 512u /* mr_triangulate_earclip_holes only: no ring edge crossed a hole's ray (a hole outside the ring) */
typedef struct mr_polygon_rings {
    const uint64_t* first_ring; /* npoly+1 entries: polygon i owns rings first_ring[i] .. first_ring[i+1]-1 */
    uint64_t ring_base;         /* ring_start is indexed by (ring - ring_base), like point_base / tri_base */
    const uint64_t* ring_start; /* absolute point index of each ring's first point; a polygon's first ring starts at
                                   first_point[i] and is its outer boundary, the others are holes */
} mr_polygon_rings;
int mr_triangulate_earclip_holes(mr_context* ctx, const mr_polygon_job* job, const mr_polygon_rings* rings);
/* ---- indexed ear clipping ------------------------------------------------------------------------------------
 * mr_triangulate_earclip_indexed writes the triangles of mr_triangulate_earclip (rings == NULL) or of
 * mr_triangulate_earclip_holes (rings != NULL) as point indices: three u32 per triangle into idx_out, so that the
 * caller's own xy array, bound as a float32x2 vertex buffer, is drawn with drawIndexed (12 bytes per triangle instead
 * of three vertices).  Bit for bit:
 *   Same polygons, same rules: the status rules, checks, triangles, their corner order, the OVERFLOW / UNDERFILL rule,
 *     bbox_out, status_out and ntri_out are those of the entry point named above.  With vtx_out, everything the call
 *     writes besides idx_out is byte-identical to what that entry point writes for the same job.
 *   Indices: polygon i's index range is idx_out[3*(first_tri[i]-tri_base) .. 3*(first_tri[i+1]-tri_base)).  For
 *     triangle t < ntri_out[i], entries 3t, 3t+1, 3t+2 of the range are its three corners in the order its vertices are
 *     emitted, corner k (the polygon's k-th point, k < N) as the low 32 bits of first_point[i] + k - index_base.  With
 *     holes, k is the input point a merged-ring position was taken from, so both copies of a bridge endpoint carry the
 *     same index.  The value is always defined; it is unambiguous while the points indexed stay below 2^32 apart.
 *   index_base selects what the indices point into: point_base indexes the rows of xy; 0 gives absolute point numbers,
 *     so that a job over a sub-range (a rank's shard) writes the same indices as the whole batch does, straight into a
 *     global index buffer.
 *   Zeros: the rest of each range is 0 -- an UNDERFILL tail, and the whole range of a DEGENERATE / TOO_LARGE /
 *     NONFINITE polygon.  A (0, 0, 0) triangle rasterises nothing, as zeroed vertices draw nothing.
 *   vtx_out may be NULL here (in this entry point only): the layout is then not read, and bbox_out, status_out and
 *     ntri_out are still written.  NULL indices or idx_out, or an idx_out that is not 4-byte aligned: MR_E_BADARG.
 *     Every check runs before any kernel, so a rejected call writes nothing.
 *   idx_out may be a device or a host pointer like the other outputs: pinned host memory is stored into directly, a
 *     pageable one is staged and only the job's range, [3*(first_tri[0]-tri_base), 3*(first_tri[npoly]-tri_base)), is
 *     copied back.
 *   Like mr_triangulate_earclip, the call leaves mr_triangulate_tier_counts and the reference path's state as they were.
 * mr_polygon_draw_indexed_range is the indexed sibling of mr_polygon_draw_range (drawIndexed's arguments, IndexedDraw.zig's
 * IndexBuffer): index_count = 3*(first_tri_next - first_tri_i), first_index = 3*(first_tri_i - tri_base),
 * instance_count 1, base_vertex 0, first_instance 0; MR_E_BADARG when a range is negative or a field does not fit its
 * u32. */
typedef struct mr_polygon_indices {
    uint32_t* idx_out;   /* 3 per triangle of the first_tri ranges: idx_out[3*(first_tri[i]-tri_base) ...] */
    uint64_t index_base; /* index of point k of polygon i = (uint32_t)(first_point[i] + k - index_base)       */
} mr_polygon_indices;
int mr_triangulate_earclip_indexed(mr_context* ctx, const mr_polygon_job* job, const mr_polygon_rings* rings,
                                   const mr_polygon_indices* indices);
typedef struct mr_draw_indexed_range { /* mirror of drawIndexed's arguments / IndexedDraw.zig's IndexBuffer */
    uint32_t index_count, instance_count, first_index;
    int32_t base_vertex;
    uint32_t first_instance;
} mr_draw_indexed_range;
int mr_polygon_draw_indexed_range(uint64_t first_tri_i, uint64_t first_tri_next, uint64_t tri_base,
                                  mr_draw_indexed_range* out);
/* Self-test used by the test-suite: sign_out[i] = cross(a1, b1, a2, b2, My) above for q[9i..9i+8] =
 * (a1x, a1y, b1x, b1y, a2x, a2y, b2x, b2y, My), as mr_triangulate_earclip_holes evaluates it (-1, 0, +1). */
int mr_selftest_crossing(mr_context* ctx, const float* q /* 9 per case */, uint64_t count, int8_t* sign_out);
/* first_tri[0..npoly] for mr_triangulate_earclip_holes: the exclusive prefix sum of max(N + 2H - 2, 0) with
 * H = first_ring[i+1] - first_ring[i] - 1 when 1 <= first_ring[i+1] - first_ring[i] <= N, else H = 0 (device or host
 * pointers, like mr_polygon_offsets). */
int mr_polygon_offsets_rings(mr_context* ctx, const uint64_t* first_point, const uint64_t* first_ring, uint32_t npoly,
                             uint64_t* first_tri_out);
/* first_tri[0..npoly] from first_point[0..npoly] (device or host pointers). */
int mr_polygon_offsets(mr_context* ctx, const uint64_t* first_point, uint32_t npoly,
                       uint64_t* first_tri_out);
/* Draw descriptor of polygon i inside the packed buffer (VertexBuffer.new(offset, prims)). */
int mr_polygon_draw_range(uint64_t first_tri_i, uint64_t first_tri_next, uint64_t tri_base,
                          mr_draw_range* out);

/* ---- unirand (Polygon/unirand.zig) -----------------------------------------
 * The reference draws from std.crypto.random; this library replaces that with a
 * documented counter-based stream so results are reproducible:
 *   state0(i) = seed ^ (0x9E3779B97F4A7C15 * (i + 1))
 *   draw: state += 0x9E3779B97F4A7C15; z = state;
 *         z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9; z = (z ^ (z >> 27)) * 0x94D049BB133111EB;
 *         z ^= z >> 31; return (uint32_t)(z >> 32)
 * unirand_seed consumes one draw for the offset, then one draw per prime-table
 * entry that passes `prime < top and top % prime != 0` (short-circuit `and`,
 * unirand.zig:42).                                                            */
uint32_t mr_rng_u32(uint64_t* state);
uint64_t mr_rng_state0(uint64_t seed, uint64_t index);
/* Host restatement of the seeding rule, used by callers that want explicit pairs. */
int mr_unirand_seed_host(uint32_t top, uint64_t seed, uint64_t index, uint32_t* offset_out,
                         uint32_t* prime_out);
/* Device port: offset_prime_out[2*i..] for polygon sizes n_i. */
int mr_unirand_seed_batch(mr_context* ctx, const uint64_t* first_point, uint32_t npoly,
                          uint64_t seed, uint64_t poly_index0, uint32_t* offset_prime_out);

/* ---- synthetic inputs (benchmark workloads, SURVEY 8-d) --------------------- */
/* u16[r][c] = splitmix64(seed ^ (r*n+c)) >> 48 for rows [row0,row0+rows). */
int mr_synth_heightmap_u16(mr_context* ctx, uint64_t seed, uint32_t n, uint32_t row0,
                           uint32_t rows, uint16_t* out);
/* Polygon sizes: MR_SIZES_UNIFORM n = nmin + hash % (nmax-nmin+1);
 *                MR_SIZES_LOGUNIFORM n = floor(nmin * (nmax/nmin)^u).
 * Writes first_point_out[0..npoly] (absolute, starting at 0) -- host-side helper. */
#define MR_SIZES_UNIFORM 0
#define MR_SIZES_LOGUNIFORM 1
int mr_synth_polygon_sizes(uint64_t seed, uint64_t poly_index0, uint32_t npoly, uint32_t nmin,
                           uint32_t nmax, int dist, uint64_t* first_point_out);
/* Star-shaped simple polygons with positive shoelace area in raw (x,y), centre (100,100),
 * radius 20..90.  xy_out holds first_point[npoly]-first_point[0] points. */
int mr_synth_polygons(mr_context* ctx, uint64_t seed, uint64_t poly_index0,
                      const uint64_t* first_point, uint32_t npoly, float* xy_out);
/* The same with a choice of family.  All families are simple polygons with positive shoelace area in
 * raw (x,y) inside [0,200]^2, vertex k of polygon i drawn from the counter hash keyed by (seed, i, k):
 *   MR_FAMILY_STAR     star-shaped about (100,100), radius 20..90 (= mr_synth_polygons).  Strongly
 *                      non-convex; the reference algorithm fails on most of them above ~30 points.
 *   MR_FAMILY_ELLIPSE  convex: jittered points of a randomly rotated ellipse (semi-axes 40..90).
 *   MR_FAMILY_ZIPPER   non-convex, y-monotone: the right chain walks down the even levels and the
 *                      left chain back up the odd levels of n strictly increasing jittered y levels,
 *                      x free inside each chain's half -- jagged on both sides, but no edge contains
 *                      a non-adjacent edge vertically, which is the precondition of the reference's
 *                      segment-search defect (Triangulation.zig:275-286, see DESIGN.md section 2):
 *                      the reference triangulates every member correctly for every edge order. */
#define MR_FAMILY_STAR 0
#define MR_FAMILY_ELLIPSE 1
#define MR_FAMILY_ZIPPER 2
int mr_synth_polygons_family(mr_context* ctx, int family, uint64_t seed, uint64_t poly_index0,
                             const uint64_t* first_point, uint32_t npoly, float* xy_out);

/* ---- multi-GPU plumbing (one process per GPU) ------------------------------ */
#define MR_IPC_HANDLE_BYTES 64
int mr_ipc_export(mr_context* ctx, void* dev, unsigned char handle_out[MR_IPC_HANDLE_BYTES]);
int mr_ipc_open(mr_context* ctx, const unsigned char handle[MR_IPC_HANDLE_BYTES], void** dev_out);
int mr_ipc_close(mr_context* ctx, void* dev);
/* Contiguous cost-balanced split of npoly polygons over nranks: range_out[0..nranks]. Host helper. */
int mr_polygon_partition(const uint64_t* first_point, uint32_t npoly, uint32_t nranks,
                         uint32_t* range_out);
/* Row-band split of an n-row terrain: rows_out[0..nranks], quad rows qrows_out[0..nranks]. */
int mr_terrain_partition(uint32_t n, uint32_t nranks, uint32_t* rows_out, uint32_t* qrows_out);

#ifdef __cplusplus
}
#endif
#endif /* MYRENDERER_B200_H */
