//! myrenderer_b200.zig -- Zig declarations for the C ABI of libmyrenderer_b200.a
//! (include/myrenderer_b200.h).  Drop this file next to Polygon/ and Terrain/ in the renderer.
//!
//! NOT COMPILED IN THIS REPOSITORY: the build image has no Zig toolchain (and the reference's
//! `mach` / `zigimg` dependencies are un-vendored URLs), so this file is the documented binding,
//! checked by eye against the header; the same calls are exercised from C++ (examples/app_scene.cpp)
//! and Python (tests/).  Written for the Zig version the reference pins (0.14.0-dev, build.zig.zon:18).
const std = @import("std");

pub const Context = opaque {};

pub const MAX_ATTR = 4;
pub const Attr = extern struct { offset: u32, ncomp: u32, location: u32 };
pub const Layout = extern struct { stride: u32, nattr: u32, attr: [MAX_ATTR]Attr };
pub const DrawRange = extern struct { vertex_count: u32, instance_count: u32, first_vertex: u32, first_instance: u32 };
pub const TerrainParams = extern struct { grid_step: f32, origin_scale: f32, height_scale: f32 };

pub const HEIGHT_U16: u32 = 0;
pub const HEIGHT_F32: u32 = 1;

pub const TerrainJob = extern struct {
    n: u32,
    height_fmt: u32,
    height: ?*const anyopaque,
    height_row0: u32,
    height_rows: u32,
    row_begin: u32,
    row_end: u32,
    vtx_out: ?*anyopaque,
    vtx_row0: u32,
    qrow_begin: u32,
    qrow_end: u32,
    idx_out: ?[*]u32,
    idx_qrow0: u32,
    layout: Layout,
    params: TerrainParams,
};

pub const PolygonJob = extern struct {
    xy: [*]const f32,
    first_point: [*]const u64,
    point_base: u64,
    npoly: u32,
    offset_prime: ?[*]const u32,
    seed: u64,
    poly_index0: u64,
    layout: Layout,
    vtx_out: ?*anyopaque,
    first_tri: [*]const u64,
    tri_base: u64,
    bbox_out: ?[*]f32,
    status_out: ?[*]u32,
    ntri_out: ?[*]u32,
};

// mr_polygon_rings: the rings (outer boundary, then holes) of each polygon of a PolygonJob
pub const PolygonRings = extern struct {
    first_ring: [*]const u64,
    ring_base: u64,
    ring_start: [*]const u64,
};

// mr_polygon_indices: where mr_triangulate_earclip_indexed writes three u32 point indices per triangle
pub const PolygonIndices = extern struct {
    idx_out: [*]u32,
    index_base: u64,
};

// mr_draw_indexed_range: drawIndexed's arguments for one polygon (IndexedDraw.zig's IndexBuffer)
pub const DrawIndexedRange = extern struct { index_count: u32, instance_count: u32, first_index: u32, base_vertex: i32, first_instance: u32 };

pub extern fn mr_context_create(device: c_int, ctx_out: *?*Context) c_int;
pub extern fn mr_context_destroy(ctx: ?*Context) c_int;
pub extern fn mr_sync(ctx: ?*Context) c_int;
pub extern fn mr_last_error(ctx: ?*const Context) [*:0]const u8;
pub extern fn mr_terrain_params_default(out: *TerrainParams) c_int;
pub extern fn mr_terrain_build(ctx: ?*Context, job: *const TerrainJob) c_int;
pub extern fn mr_terrain_build_full(ctx: ?*Context, height: *const anyopaque, height_fmt: u32, n: u32, layout: ?*const Layout, params: ?*const TerrainParams, vtx_out: ?*anyopaque, idx_out: ?[*]u32) c_int;
pub extern fn mr_terrain_describe(n: u32, params: ?*const TerrainParams, bbox_min: ?*[3]f32, bbox_max: ?*[3]f32, vertex_count: ?*u64, index_count: ?*u64) c_int;
pub extern fn mr_triangulate_batch(ctx: ?*Context, job: *const PolygonJob) c_int;
pub extern fn mr_triangulate_earclip(ctx: ?*Context, job: *const PolygonJob) c_int;
pub extern fn mr_triangulate_earclip_holes(ctx: ?*Context, job: *const PolygonJob, rings: *const PolygonRings) c_int;
pub extern fn mr_polygon_draw_range(first_tri_i: u64, first_tri_next: u64, tri_base: u64, out: *DrawRange) c_int;
pub extern fn mr_triangulate_earclip_indexed(ctx: ?*Context, job: *const PolygonJob, rings: ?*const PolygonRings, indices: *const PolygonIndices) c_int;
pub extern fn mr_polygon_draw_indexed_range(first_tri_i: u64, first_tri_next: u64, tri_base: u64, out: *DrawIndexedRange) c_int;
pub extern fn mr_unirand_seed_host(top: u32, seed: u64, index: u64, offset_out: *u32, prime_out: *u32) c_int;
pub extern fn mr_context_trim(ctx: ?*Context) c_int;
pub extern fn mr_pinned_alloc(ctx: ?*Context, bytes: usize, host_out: *?*anyopaque) c_int;
pub extern fn mr_pinned_free(ctx: ?*Context, host: ?*anyopaque) c_int;
// terrain tiles + culling (SceneNode.zig:96-110 per tile)
pub extern fn mr_terrain_tile_count(n: u32, tile_rows: u32, tile_cols: u32, tiles_r_out: ?*u32, tiles_c_out: ?*u32) c_int;
pub extern fn mr_terrain_tile_bounds(ctx: ?*Context, height: *const anyopaque, height_fmt: u32, n: u32, tile_rows: u32, tile_cols: u32, params: ?*const TerrainParams, bbox_out: [*]f32) c_int;
pub extern fn mr_terrain_cull(ctx: ?*Context, bbox: [*]const f32, n: u32, tile_rows: u32, tile_cols: u32, xform: *const [16]f32, visible_out: ?[*]u32, visible_ids_out: ?[*]u32, idx_out: ?[*]u32, counts_out: ?*[2]u64) c_int;
// the six-plane frustum test (WebGPU clip volume) in place of SceneNode's; same arguments and outputs
pub extern fn mr_terrain_cull_frustum(ctx: ?*Context, bbox: [*]const f32, n: u32, tile_rows: u32, tile_cols: u32, view_proj: *const [16]f32, visible_out: ?[*]u32, visible_ids_out: ?[*]u32, idx_out: ?[*]u32, counts_out: ?*[2]u64) c_int;

pub const Error = error{GeometryBackend};

pub fn check(rc: c_int) Error!void {
    if (rc != 0) return Error.GeometryBackend;
}

/// VertexLayout.create(T) -> Layout, from the same comptime reflection Renderer/VertexLayout.zig:12-30 uses,
/// so the offsets are the ones the Zig compiler actually chose for T.
pub fn layoutOf(comptime T: type, comptime Vec2: type, comptime Vec3: type, comptime Vec4: type) Layout {
    var l = std.mem.zeroes(Layout);
    l.stride = @sizeOf(T);
    inline for (0.., @typeInfo(T).@"struct".fields) |i, field| {
        l.attr[i] = .{
            .offset = @offsetOf(T, field.name),
            .ncomp = switch (field.type) {
                Vec2 => 2,
                Vec3 => 3,
                Vec4 => 4,
                else => @compileError("unsupported vertex field type"),
            },
            .location = i,
        };
        l.nattr = i + 1;
    }
    return l;
}
