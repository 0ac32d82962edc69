// mr_host.hpp -- C++17 host-side mirror of the reference's interface for the geometry hot path,
// over the C ABI of libmyrenderer_b200 (include/myrenderer_b200.h).
//
// The reference is Zig (compiled code) and no Zig toolchain exists in the build image, so the host
// layer above the C ABI is written in C++ with the reference's names, argument meaning and error
// behaviour; the Zig declarations a maintainer would use instead are in zig/myrenderer_b200.zig and
// INTEGRATION.md.
//
//   mr::VertexLayout::create<T>()      Renderer/VertexLayout.zig:9-31   (offsets via offsetof, like @offsetOf)
//   mr::VertexBuffer::create(...)      Renderer/VertexBuffer.zig:11-35  (draw descriptor + mapped host range)
//   mr::Terrain::create_terrain        Terrain/Terrain.zig:88-129
//   mr::Polygon::create_polygon        Polygon/Polygon.zig:81-107
//   mr::Triangulation::create_polygon  Polygon/Triangulation.zig:446-451 (emit callback form)
//   mr::unirand_seed / Unirand::next   Polygon/unirand.zig:12-50
//
// Errors: the Zig functions return error unions; here every failure throws mr::Error carrying the
// MR_E_* code (the Zig shim maps non-zero to error.GeometryBackend).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <functional>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/myrenderer_b200.h"

namespace mr {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& what) : std::runtime_error(what), code(c) {}
};

// mach.math.Vec2/3/4: Vec3 wraps @Vector(3, f32) => 16 bytes, align 16 (SURVEY D9)
struct alignas(8) Vec2 { float v[2]; };
struct alignas(16) Vec3 { float v[3]; float pad_; };
struct alignas(16) Vec4 { float v[4]; };
using Point = Vec2;  // Triangulation.zig:16

class Context {
   public:
    explicit Context(int device = 0) {
        const int rc = mr_context_create(device, &ctx_);
        if (rc != MR_OK) throw Error(rc, "mr_context_create: no usable CUDA device (there is no CPU fallback)");
    }
    ~Context() { mr_context_destroy(ctx_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    mr_context* get() const { return ctx_; }
    void check(int rc, const char* where) const {
        if (rc != MR_OK) throw Error(rc, std::string(where) + ": " + mr_last_error(ctx_));
    }
    void sync() const { check(mr_sync(ctx_), "mr_sync"); }

   private:
    mr_context* ctx_ = nullptr;
};

// ---- VertexLayout.create(T) ------------------------------------------------------------------
template <class F> struct format_of;
template <> struct format_of<Vec2> { static constexpr uint32_t ncomp = 2; };
template <> struct format_of<Vec3> { static constexpr uint32_t ncomp = 3; };
template <> struct format_of<Vec4> { static constexpr uint32_t ncomp = 4; };

struct VertexLayout {
    mr_layout native{};
    // fields: {offsetof(T, field), components} in declaration (shader_location) order
    static VertexLayout create(uint32_t size_of_t, std::initializer_list<std::pair<size_t, uint32_t>> fields) {
        VertexLayout L;
        L.native.stride = size_of_t;
        uint32_t i = 0;
        for (auto& f : fields) {
            L.native.attr[i] = {static_cast<uint32_t>(f.first), f.second, i};
            ++i;
        }
        L.native.nattr = i;
        return L;
    }
};
#define MR_FIELD(T, name) std::pair<size_t, uint32_t>{offsetof(T, name), ::mr::format_of<decltype(T::name)>::ncomp}

struct GPUVertex {  // Polygon.zig:26-29
    Vec2 x;
    Vec3 color;
};
struct TerrainVertex {  // new type (SURVEY 8-a4)
    Vec3 pos;
    Vec3 normal;
};
inline VertexLayout gpu_vertex_layout() { return VertexLayout::create(sizeof(GPUVertex), {MR_FIELD(GPUVertex, x), MR_FIELD(GPUVertex, color)}); }
inline VertexLayout terrain_vertex_layout() { return VertexLayout::create(sizeof(TerrainVertex), {MR_FIELD(TerrainVertex, pos), MR_FIELD(TerrainVertex, normal)}); }

// ---- VertexBuffer ----------------------------------------------------------------------------------
// The reference's buffer is a WebGPU buffer mapped at creation; here `mapped` plays the mapped range.
struct VertexBuffer {
    std::vector<unsigned char> mapped;  // vertex_buffer (zero-initialised like a mapped WebGPU buffer)
    uint32_t vertex_count = 3;
    uint32_t instance_count = 1;
    uint32_t first_vertex = 0;
    uint32_t first_instance = 0;
    // VertexBuffer.new(renderer, offset, primitive_count, T)  VertexBuffer.zig:11-31
    static VertexBuffer create(uint32_t offset, uint32_t primitive_count, uint32_t size_of_t) {
        VertexBuffer b;
        b.mapped.assign(static_cast<size_t>(primitive_count) * size_of_t * 3, 0);
        b.vertex_count = primitive_count * 3;
        b.first_vertex = offset * 3;
        return b;
    }
    template <class T> T* map() { return reinterpret_cast<T*>(mapped.data()); }  // VertexBuffer.zig:33-35
};

// ---- unirand ------------------------------------------------------------------------------------------
struct Unirand {  // unirand.zig:6-22
    uint32_t at = 0, top = 0, offset = 0, prime = 1;
    std::optional<uint32_t> next() {
        std::optional<uint32_t> r;
        if (top > 0 && at < top) r = static_cast<uint32_t>(at * prime + offset) % top;
        at += 1;
        return r;
    }
};
inline Unirand unirand_seed(uint32_t top, uint64_t seed, uint64_t index = 0) {  // unirand.zig:26-50
    Unirand u;
    u.top = top;
    const int rc = mr_unirand_seed_host(top, seed, index, &u.offset, &u.prime);
    if (rc != MR_OK) throw Error(rc, "mr_unirand_seed_host");
    return u;
}

// ---- Terrain ---------------------------------------------------------------------------------------------
struct TerrainMesh {
    uint32_t size = 0;
    VertexBuffer vertex_buffer;
    std::vector<uint32_t> index_buffer;
    float bounding_box_p0[3]{}, bounding_box_p1[3]{};
};

class Terrain {
   public:
    explicit Terrain(Context& ctx) : ctx_(ctx) { mr_terrain_params_default(&params_); }
    // create_terrain over decoded PNG pixels (image.pixels.grayscale16, Terrain.zig:95,116): n x n u16
    TerrainMesh create_terrain(const uint16_t* grayscale16, uint32_t n) {
        TerrainMesh m;
        m.size = n;
        const VertexLayout L = terrain_vertex_layout();
        m.vertex_buffer.mapped.assign(static_cast<size_t>(n) * n * L.native.stride, 0);
        m.vertex_buffer.vertex_count = n * n;
        m.index_buffer.assign(n > 1 ? 6ull * (n - 1) * (n - 1) : 0, 0);
        ctx_.check(mr_terrain_build_full(ctx_.get(), grayscale16, MR_HEIGHT_U16, n, &L.native, &params_,
                                         m.vertex_buffer.mapped.data(), m.index_buffer.empty() ? nullptr : m.index_buffer.data()),
                   "mr_terrain_build_full");
        mr_terrain_describe(n, &params_, m.bounding_box_p0, m.bounding_box_p1, nullptr, nullptr);
        return m;
    }

   private:
    Context& ctx_;
    mr_terrain_params params_{};
};

// ---- Polygon / Triangulation ---------------------------------------------------------------------------------
struct PolygonObj {
    VertexBuffer vertex_buffer;
    float bounding_box_p0[3]{}, bounding_box_p1[3]{};
    uint32_t status = 0, ntri = 0;
};

// A polygon as points plus an index buffer (mr_triangulate_earclip_indexed): bind `points` as a float32x2 vertex buffer
// and draw `indices` with drawIndexed.
struct IndexedPolygonObj {
    std::vector<Point> points;      // the outer ring, then each hole
    std::vector<uint32_t> indices;  // three per triangle, into points
    float bounding_box_p0[3]{}, bounding_box_p1[3]{};
    uint32_t status = 0, ntri = 0;
};

class Polygon {
   public:
    explicit Polygon(Context& ctx) : ctx_(ctx), layout_(gpu_vertex_layout()) {}
    // Polygon.create_polygon(vertices); the edge order is unirand_seed(n) drawn from (seed, index), or the
    // explicit (offset, prime) pair when given.
    PolygonObj create_polygon(const std::vector<Point>& vertices, uint64_t seed = 0, uint64_t index = 0,
                              const uint32_t* offset_prime = nullptr) {
        if (vertices.size() < 2) throw Error(MR_E_BADARG, "create_polygon: vertices.len - 2 underflows (Polygon.zig:82)");
        PolygonObj o;
        const uint32_t n = static_cast<uint32_t>(vertices.size());
        o.vertex_buffer = VertexBuffer::create(0, n - 2, layout_.native.stride);
        const uint64_t first_point[2] = {0, n};
        const uint64_t first_tri[2] = {0, n - 2};
        float bbox[4];
        mr_polygon_job j{};
        j.xy = reinterpret_cast<const float*>(vertices.data());
        j.first_point = first_point;
        j.npoly = 1;
        j.offset_prime = offset_prime;
        j.seed = seed;
        j.poly_index0 = index;
        j.layout = layout_.native;
        j.vtx_out = o.vertex_buffer.mapped.data();
        j.first_tri = first_tri;
        j.bbox_out = bbox;
        j.status_out = &o.status;
        j.ntri_out = &o.ntri;
        ctx_.check(mr_triangulate_batch(ctx_.get(), &j), "mr_triangulate_batch");
        o.bounding_box_p0[0] = bbox[0];  // Polygon.zig:96-97
        o.bounding_box_p0[1] = bbox[1];
        o.bounding_box_p1[0] = bbox[2];
        o.bounding_box_p1[1] = bbox[3];
        return o;
    }
    // The same polygon triangulated by ear clipping (mr_triangulate_earclip): correct on every simple polygon, no edge order.
    PolygonObj create_polygon_earclip(const std::vector<Point>& vertices) {
        if (vertices.size() < 2) throw Error(MR_E_BADARG, "create_polygon: vertices.len - 2 underflows (Polygon.zig:82)");
        PolygonObj o;
        const uint32_t n = static_cast<uint32_t>(vertices.size());
        o.vertex_buffer = VertexBuffer::create(0, n - 2, layout_.native.stride);
        const uint64_t first_point[2] = {0, n};
        const uint64_t first_tri[2] = {0, n - 2};
        float bbox[4];
        mr_polygon_job j{};
        j.xy = reinterpret_cast<const float*>(vertices.data());
        j.first_point = first_point;
        j.npoly = 1;
        j.layout = layout_.native;
        j.vtx_out = o.vertex_buffer.mapped.data();
        j.first_tri = first_tri;
        j.bbox_out = bbox;
        j.status_out = &o.status;
        j.ntri_out = &o.ntri;
        ctx_.check(mr_triangulate_earclip(ctx_.get(), &j), "mr_triangulate_earclip");
        o.bounding_box_p0[0] = bbox[0];
        o.bounding_box_p0[1] = bbox[1];
        o.bounding_box_p1[0] = bbox[2];
        o.bounding_box_p1[1] = bbox[3];
        return o;
    }
    // A polygon with holes (mr_triangulate_earclip_holes): N + 2H - 2 triangles, N the points of all rings.
    PolygonObj create_polygon_earclip(const std::vector<Point>& outer, const std::vector<std::vector<Point>>& holes) {
        std::vector<Point> pts(outer);
        std::vector<uint64_t> ring_start{0};
        for (const auto& h : holes) {
            ring_start.push_back(pts.size());
            pts.insert(pts.end(), h.begin(), h.end());
        }
        if (pts.size() < 2) throw Error(MR_E_BADARG, "create_polygon: vertices.len - 2 underflows (Polygon.zig:82)");
        PolygonObj o;
        const uint64_t n = pts.size(), ntri = n + 2 * holes.size() - 2;
        o.vertex_buffer = VertexBuffer::create(0, static_cast<uint32_t>(ntri), layout_.native.stride);
        const uint64_t first_point[2] = {0, n};
        const uint64_t first_tri[2] = {0, ntri};
        const uint64_t first_ring[2] = {0, ring_start.size()};
        float bbox[4];
        mr_polygon_job j{};
        j.xy = reinterpret_cast<const float*>(pts.data());
        j.first_point = first_point;
        j.npoly = 1;
        j.layout = layout_.native;
        j.vtx_out = o.vertex_buffer.mapped.data();
        j.first_tri = first_tri;
        j.bbox_out = bbox;
        j.status_out = &o.status;
        j.ntri_out = &o.ntri;
        const mr_polygon_rings rings{first_ring, 0, ring_start.data()};
        ctx_.check(mr_triangulate_earclip_holes(ctx_.get(), &j, &rings), "mr_triangulate_earclip_holes");
        o.bounding_box_p0[0] = bbox[0];
        o.bounding_box_p0[1] = bbox[1];
        o.bounding_box_p1[0] = bbox[2];
        o.bounding_box_p1[1] = bbox[3];
        return o;
    }
    // The same polygon with holes as points plus indices (mr_triangulate_earclip_indexed, no vertex buffer).
    IndexedPolygonObj create_polygon_earclip_indexed(const std::vector<Point>& outer, const std::vector<std::vector<Point>>& holes) {
        IndexedPolygonObj o;
        o.points = outer;
        std::vector<uint64_t> ring_start{0};
        for (const auto& h : holes) {
            ring_start.push_back(o.points.size());
            o.points.insert(o.points.end(), h.begin(), h.end());
        }
        if (o.points.size() < 2) throw Error(MR_E_BADARG, "create_polygon: vertices.len - 2 underflows (Polygon.zig:82)");
        const uint64_t n = o.points.size(), ntri = n + 2 * holes.size() - 2;
        o.indices.assign(3 * ntri, 0);
        const uint64_t first_point[2] = {0, n};
        const uint64_t first_tri[2] = {0, ntri};
        const uint64_t first_ring[2] = {0, ring_start.size()};
        float bbox[4];
        mr_polygon_job j{};
        j.xy = reinterpret_cast<const float*>(o.points.data());
        j.first_point = first_point;
        j.npoly = 1;
        j.first_tri = first_tri;
        j.bbox_out = bbox;
        j.status_out = &o.status;
        j.ntri_out = &o.ntri;
        const mr_polygon_rings rings{first_ring, 0, ring_start.data()};
        const mr_polygon_indices indices{o.indices.data(), 0};
        ctx_.check(mr_triangulate_earclip_indexed(ctx_.get(), &j, &rings, &indices), "mr_triangulate_earclip_indexed");
        o.bounding_box_p0[0] = bbox[0];
        o.bounding_box_p0[1] = bbox[1];
        o.bounding_box_p1[0] = bbox[2];
        o.bounding_box_p1[1] = bbox[3];
        return o;
    }
    const VertexLayout& layout() const { return layout_; }

   private:
    Context& ctx_;
    VertexLayout layout_;
};

class Triangulation {
   public:
    explicit Triangulation(Context& ctx) : poly_(ctx) {}
    // create_polygon(points, context, emit): a callback cannot cross the C ABI, so the filled vertex range
    // is replayed through `emit` in the reference's emit order.  Returns the MR_POLY_* status.
    template <class Ctx>
    uint32_t create_polygon(const std::vector<Point>& points, Ctx& context, const std::function<void(Ctx&, Point)>& emit,
                            uint64_t seed = 0, uint64_t index = 0, const uint32_t* offset_prime = nullptr) {
        PolygonObj o = poly_.create_polygon(points, seed, index, offset_prime);
        const mr_layout& L = poly_.layout().native;
        for (uint32_t k = 0; k < o.ntri * 3; ++k) {
            Point p;
            std::memcpy(&p, o.vertex_buffer.mapped.data() + static_cast<size_t>(k) * L.stride + L.attr[0].offset, sizeof(p));
            emit(context, p);
        }
        return o.status;
    }

   private:
    Polygon poly_;
};

}  // namespace mr
