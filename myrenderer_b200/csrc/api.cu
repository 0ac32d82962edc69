// api.cu -- the extern "C" surface of libmyrenderer_b200: context, memory helpers, argument
// validation, host<->device staging, and the host-side helpers (layout presets, partitions,
// unirand host restatement).  Kernels live in terrain.cu / triangulate.cu / synth.cu.
#include <algorithm>
#include <new>
#include "common.cuh"
#include "unirand.cuh"

int mr_heightmap_normalize_impl(mr_context* ctx, const uint16_t* in, uint64_t count, float* out);
int mr_terrain_tile_bounds_impl(mr_context* ctx, const void* height_dev, uint32_t height_fmt, uint32_t n, uint32_t tile_rows,
                                uint32_t tile_cols, const mr_terrain_params* p, float* bbox_dev);
int mr_terrain_cull_impl(mr_context* ctx, const float* bbox_dev, uint32_t n, uint32_t tile_rows, uint32_t tile_cols,
                         const float xform[16], bool frustum, uint32_t* visible_dev, uint32_t* ids_dev,
                         unsigned long long* first_index_dev, uint32_t* idx_dev, unsigned long long* counts_dev);
int mr_selftest_fastdiv_impl(mr_context* ctx, float b, int force_fast, unsigned long long* mismatches_dev);
int mr_polygon_offsets_impl(mr_context* ctx, const uint64_t* first_point_dev, uint32_t npoly, uint64_t* first_tri_dev);
int mr_triangulate_tier_counts_impl(mr_context* ctx, uint32_t out[8]);
int mr_unirand_seed_batch_impl(mr_context* ctx, const uint64_t* first_point_dev, uint32_t npoly, uint64_t seed,
                               uint64_t poly_index0, uint32_t* out_dev);
int mr_synth_heightmap_u16_impl(mr_context* ctx, uint64_t seed, uint32_t n, uint32_t row0, uint32_t rows,
                                uint16_t* out_dev);
int mr_synth_polygons_impl(mr_context* ctx, int family, uint64_t seed, uint64_t poly_index0, const uint64_t* first_point_dev,
                           uint32_t npoly, float* xy_dev);

namespace {
// unirand.zig:24: host view of the table defined once in unirand.cuh (mr_unirand_seed_host)
const uint32_t k_primes_host[MR_NPRIMES] = {MR_PRIME_LIST};

bool layout_ok(const mr_layout* L, uint32_t need_attrs, uint32_t ncomp0) {
    if (!L || L->nattr < need_attrs || L->nattr > MR_MAX_ATTR) return false;
    if (L->stride < 8 || L->stride > 256 || (L->stride & 3u)) return false;
    for (uint32_t i = 0; i < L->nattr; ++i) {
        if (L->attr[i].offset & 3u) return false;
        if (L->attr[i].ncomp < 2 || L->attr[i].ncomp > 4) return false;
        if (L->attr[i].offset + 4u * L->attr[i].ncomp > L->stride) return false;
    }
    if (L->attr[0].ncomp < ncomp0) return false;
    return true;
}
}  // namespace

extern "C" {

int mr_abi_version(void) { return MR_ABI_VERSION; }

int mr_build_flags(void) {
#ifdef MR_CHECKED
    return 1;
#else
    return 0;
#endif
}

int mr_device_count(int* count_out) {
    if (!count_out) return MR_E_BADARG;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *count_out = 0;
        return MR_E_CUDA;
    }
    *count_out = n;
    return MR_OK;
}

int mr_context_create(int device, mr_context** ctx_out) {
    if (!ctx_out) return MR_E_BADARG;
    *ctx_out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return MR_E_CUDA;  // no CPU fallback
    }
    if (device < 0 || device >= n) return MR_E_BADARG;
    if (cudaSetDevice(device) != cudaSuccess) return MR_E_CUDA;
    mr_context* ctx = new (std::nothrow) mr_context();
    if (!ctx) return MR_E_NOMEM;
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        delete ctx;
        return MR_E_CUDA;
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return MR_E_CUDA;
    }
    ctx->own_stream = true;
    *ctx_out = ctx;
    return MR_OK;
}

int mr_context_destroy(mr_context* ctx) {
    if (!ctx) return MR_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < MR_NUM_SCRATCH; ++i)
        if (ctx->scratch[i]) cudaFree(ctx->scratch[i]);
    if (ctx->pinned_mailbox) cudaFreeHost(ctx->pinned_mailbox);
    if (ctx->small_pinned) cudaFreeHost(ctx->small_pinned);
    if (ctx->small_dev) cudaFree(ctx->small_dev);
    mr_polygon_plan_free(ctx);
    for (int i = 0; i < MR_NUM_AUX; ++i) {
        if (ctx->aux[i]) cudaStreamDestroy(ctx->aux[i]);
        if (ctx->join_ev[i]) cudaEventDestroy(ctx->join_ev[i]);
    }
    if (ctx->fork_ev) cudaEventDestroy(ctx->fork_ev);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return MR_OK;
}

int mr_context_trim(mr_context* ctx) {
    if (!ctx) return MR_E_BADARG;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < MR_NUM_SCRATCH; ++i) {
        if (ctx->scratch[i]) MR_CUDA(ctx, cudaFree(ctx->scratch[i]));
        ctx->scratch[i] = nullptr;
        ctx->scratch_bytes[i] = 0;
    }
    ctx->last_header_dev = nullptr;
    return MR_OK;
}

int mr_context_scratch_bytes(const mr_context* ctx, uint64_t* bytes_out) {
    if (!ctx || !bytes_out) return MR_E_BADARG;
    uint64_t t = 0;
    for (int i = 0; i < MR_NUM_SCRATCH; ++i) t += ctx->scratch_bytes[i];
    *bytes_out = t;
    return MR_OK;
}

int mr_context_set_stream(mr_context* ctx, void* cuda_stream) {
    if (!ctx) return MR_E_BADARG;
    MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = static_cast<cudaStream_t>(cuda_stream);
    ctx->own_stream = false;
    return MR_OK;
}

int mr_context_stream(mr_context* ctx, void** cuda_stream_out) {
    if (!ctx || !cuda_stream_out) return MR_E_BADARG;
    *cuda_stream_out = ctx->stream;
    return MR_OK;
}

int mr_sync(mr_context* ctx) {
    if (!ctx) return MR_E_BADARG;
    MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MR_OK;
}

const char* mr_last_error(const mr_context* ctx) { return ctx ? ctx->err : "null context"; }
uint64_t mr_launch_count(const mr_context* ctx) { return ctx ? ctx->launches : 0; }

int mr_device_alloc(mr_context* ctx, size_t bytes, void** dev_out) {
    if (!ctx || !dev_out) return MR_E_BADARG;
    cudaSetDevice(ctx->device);
    cudaError_t e = cudaMalloc(dev_out, bytes ? bytes : 16);
    if (e != cudaSuccess) return mr_fail(ctx, MR_E_NOMEM, "cudaMalloc", e);
    return MR_OK;
}
int mr_device_free(mr_context* ctx, void* dev) {
    if (!ctx) return MR_E_BADARG;
    MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    MR_CUDA(ctx, cudaFree(dev));
    return MR_OK;
}
int mr_pinned_alloc(mr_context* ctx, size_t bytes, void** host_out) {
    if (!ctx || !host_out) return MR_E_BADARG;
    cudaError_t e = cudaMallocHost(host_out, bytes ? bytes : 16);
    if (e != cudaSuccess) return mr_fail(ctx, MR_E_NOMEM, "cudaMallocHost", e);
    return MR_OK;
}
int mr_pinned_free(mr_context* ctx, void* host) {
    if (!ctx) return MR_E_BADARG;
    MR_CUDA(ctx, cudaFreeHost(host));
    return MR_OK;
}
int mr_copy(mr_context* ctx, void* dst, const void* src, size_t bytes) {
    if (!ctx || (!dst && bytes) || (!src && bytes)) return MR_E_BADARG;
    MR_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, ctx->stream));
    return MR_OK;
}
int mr_fill_zero(mr_context* ctx, void* dev, size_t bytes) {
    if (!ctx || (!dev && bytes)) return MR_E_BADARG;
    MR_CUDA(ctx, cudaMemsetAsync(dev, 0, bytes, ctx->stream));
    return MR_OK;
}

int mr_layout_preset(int which, mr_layout* out) {
    if (!out) return MR_E_BADARG;
    memset(out, 0, sizeof(*out));
    out->stride = 32;
    out->nattr = 2;
    out->attr[0].location = 0;
    out->attr[1].location = 1;
    switch (which) {
        case MR_LAYOUT_GPUVERTEX_DECL:
            out->attr[0] = {0, 2, 0};
            out->attr[1] = {16, 3, 1};
            return MR_OK;
        case MR_LAYOUT_GPUVERTEX_ZIGAUTO:
            out->attr[0] = {16, 2, 0};
            out->attr[1] = {0, 3, 1};
            return MR_OK;
        case MR_LAYOUT_TERRAINVERTEX:
            out->attr[0] = {0, 3, 0};
            out->attr[1] = {16, 3, 1};
            return MR_OK;
        default: return MR_E_BADARG;
    }
}

int mr_terrain_params_default(mr_terrain_params* out) {
    if (!out) return MR_E_BADARG;
    out->grid_step = 0.2f;     // Terrain.zig:36
    out->origin_scale = 0.1f;  // Terrain.zig:36
    out->height_scale = 5.0f;  // Terrain.zig:48
    return MR_OK;
}

int mr_terrain_describe(uint32_t n, const mr_terrain_params* params, float bbox_min[3], float bbox_max[3],
                        uint64_t* vertex_count, uint64_t* index_count) {
    mr_terrain_params p;
    if (params) p = *params; else mr_terrain_params_default(&p);
    if (n == 0) return MR_E_BADARG;
    const float bound = (float)n * p.origin_scale;  // Terrain.zig:103-104
    if (bbox_min) {
        bbox_min[0] = -bound;
        bbox_min[1] = 0.0f;
        bbox_min[2] = -bound;
    }
    if (bbox_max) {  // Terrain.zig:109: (bound, 5.0, bound); 5.0 is height_scale * 1.0
        bbox_max[0] = bound;
        bbox_max[1] = p.height_scale;
        bbox_max[2] = bound;
    }
    if (vertex_count) *vertex_count = (uint64_t)n * n;
    if (index_count) *index_count = 6ull * (uint64_t)(n - 1) * (uint64_t)(n - 1);
    return MR_OK;
}

int mr_terrain_build(mr_context* ctx, const mr_terrain_job* job) {
    if (!ctx || !job) return MR_E_BADARG;
    const mr_terrain_job& j = *job;
    if (j.n == 0 || j.n > 65535u || !j.height) return mr_fail(ctx, MR_E_BADARG, "terrain: n must be 1..65535 and height non-null");
    if (j.height_fmt != MR_HEIGHT_U16 && j.height_fmt != MR_HEIGHT_F32) return mr_fail(ctx, MR_E_BADARG, "terrain: bad height_fmt");
    if (j.row_begin > j.row_end || j.row_end > j.n) return mr_fail(ctx, MR_E_BADARG, "terrain: bad row range");
    if (j.qrow_begin > j.qrow_end || j.qrow_end > j.n - 1u) return mr_fail(ctx, MR_E_BADARG, "terrain: bad quad-row range");
    const bool want_v = j.vtx_out && j.row_end > j.row_begin;
    const bool want_i = j.idx_out && j.n > 1 && j.qrow_end > j.qrow_begin;
    if (j.vtx_out && !layout_ok(&j.layout, 1, 3)) return mr_fail(ctx, MR_E_BADARG, "terrain: bad vertex layout");
    if (j.vtx_out && j.layout.nattr > 1 && j.layout.attr[1].ncomp < 3) return mr_fail(ctx, MR_E_BADARG, "terrain: normal needs 3 components");
    if (j.vtx_out && j.vtx_row0 > j.row_begin) return mr_fail(ctx, MR_E_BADARG, "terrain: vtx_row0 > row_begin");
    if (j.idx_out && j.idx_qrow0 > j.qrow_begin) return mr_fail(ctx, MR_E_BADARG, "terrain: idx_qrow0 > qrow_begin");
    if (j.vtx_out && (reinterpret_cast<uintptr_t>(j.vtx_out) & 3u)) return mr_fail(ctx, MR_E_BADARG, "terrain: vtx_out must be 4-byte aligned");
    if (j.idx_out && (reinterpret_cast<uintptr_t>(j.idx_out) & 7u)) return mr_fail(ctx, MR_E_BADARG, "terrain: idx_out must be 8-byte aligned");
    if (want_v) {
        const uint32_t need_lo = j.row_begin > 0 ? j.row_begin - 1 : 0;
        const uint32_t need_hi = std::min(j.row_end + 1, j.n);
        if (j.height_row0 > need_lo || (uint64_t)j.height_row0 + j.height_rows < need_hi)
            return mr_fail(ctx, MR_E_BADARG, "terrain: height rows do not cover the band plus halo");
    }
    if (!want_v && !want_i) return MR_OK;  // empty band: nothing to produce
    MR_CUDA(ctx, cudaSetDevice(ctx->device));

    mr_terrain_job d = j;
    if (!want_v) d.vtx_out = nullptr;
    if (!want_i) d.idx_out = nullptr;
    mr_staging io(ctx);
    bool vs = false, is = false;
    void* vdev = nullptr;
    uint32_t* idev = nullptr;
    const size_t row_bytes = (size_t)j.n * j.layout.stride;
    const size_t qrow_bytes = 6u * (size_t)(j.n - 1u) * 4u;
    // a staged output holds its band only: rows [row_begin, row_end), quad rows [qrow_begin, qrow_end)
    const size_t vbytes = (size_t)(j.row_end - j.row_begin) * row_bytes;
    const size_t ibytes = (size_t)(j.qrow_end - j.qrow_begin) * qrow_bytes;
    unsigned char* idst = nullptr;  // where a staged band goes in the caller's buffer
    // The index buffer does not depend on the heightmap.  When it has to travel to a host buffer, it is built and copied
    // on a side stream first, so that its device-to-host copy overlaps the heightmap's host-to-device copy (PCIe is full
    // duplex) and the vertex kernel, instead of both copies queueing behind both kernels.
    cudaStream_t idx_stream = ctx->stream;
    if (want_i) {
        // (device outputs keep the caller's idx_qrow0 origin)
        idev = io.out(MR_SLOT_BBOX, j.idx_out, ibytes, &is);
        if (io.rc) return io.rc;
        if (is) {
            d.idx_out = idev;
            d.idx_qrow0 = j.qrow_begin;
            idst = reinterpret_cast<unsigned char*>(j.idx_out) + (size_t)(j.qrow_begin - j.idx_qrow0) * qrow_bytes;
            if (want_v && !io.where(j.vtx_out).device) {
                if (mr_aux_streams(ctx)) return mr_fail(ctx, MR_E_CUDA, "side streams");
                MR_CUDA(ctx, cudaEventRecord(ctx->fork_ev, ctx->stream));  // order after earlier work on the context
                MR_CUDA(ctx, cudaStreamWaitEvent(ctx->aux[0], ctx->fork_ev, 0));
                idx_stream = ctx->aux[0];
            }
        }
    }
    int rc;
    if (idx_stream != ctx->stream) {
        mr_terrain_job di = d;
        di.vtx_out = nullptr;
        rc = mr_terrain_build_impl(ctx, &di, idx_stream);
        if (rc) return rc;
        MR_CUDA(ctx, cudaMemcpyAsync(idst, idev, ibytes, cudaMemcpyDeviceToHost, idx_stream));
        MR_CUDA(ctx, cudaEventRecord(ctx->join_ev[0], idx_stream));
        d.idx_out = nullptr;
    }
    if (want_v) {
        const size_t texel = j.height_fmt == MR_HEIGHT_U16 ? 2 : 4;
        d.height = io.in(MR_SLOT_XY, j.height, (size_t)j.height_rows * j.n * texel);
        vdev = io.out(MR_SLOT_VTX, j.vtx_out, vbytes, &vs);
        if (io.rc) return io.rc;
        if (vs) {
            d.vtx_out = vdev;
            d.vtx_row0 = j.row_begin;
        }
    }
    rc = mr_terrain_build_impl(ctx, &d, ctx->stream);
    if (rc) return rc;
    if (vs) {
        unsigned char* vdst = static_cast<unsigned char*>(j.vtx_out) + (size_t)(j.row_begin - j.vtx_row0) * row_bytes;
        MR_CUDA(ctx, cudaMemcpyAsync(vdst, vdev, vbytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (is && idx_stream == ctx->stream) MR_CUDA(ctx, cudaMemcpyAsync(idst, idev, ibytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (idx_stream != ctx->stream) MR_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->join_ev[0], 0));
    return io.finish(MR_OK);
}

int mr_terrain_build_full(mr_context* ctx, const void* height, uint32_t height_fmt, uint32_t n, const mr_layout* layout,
                          const mr_terrain_params* params, void* vtx_out, uint32_t* idx_out) {
    if (!ctx) return MR_E_BADARG;
    mr_terrain_job j;
    memset(&j, 0, sizeof(j));
    j.n = n;
    j.height_fmt = height_fmt;
    j.height = height;
    j.height_row0 = 0;
    j.height_rows = n;
    j.row_begin = 0;
    j.row_end = n;
    j.vtx_out = vtx_out;
    j.vtx_row0 = 0;
    j.qrow_begin = 0;
    j.qrow_end = n ? n - 1 : 0;
    j.idx_out = idx_out;
    j.idx_qrow0 = 0;
    if (layout) j.layout = *layout; else mr_layout_preset(MR_LAYOUT_TERRAINVERTEX, &j.layout);
    if (params) j.params = *params; else mr_terrain_params_default(&j.params);
    return mr_terrain_build(ctx, &j);
}

int mr_terrain_tile_count(uint32_t n, uint32_t tile_rows, uint32_t tile_cols, uint32_t* tiles_r_out, uint32_t* tiles_c_out) {
    if (n < 2 || tile_rows == 0 || tile_cols == 0) return MR_E_BADARG;
    if (tiles_r_out) *tiles_r_out = (n - 1u + tile_rows - 1u) / tile_rows;
    if (tiles_c_out) *tiles_c_out = (n - 1u + tile_cols - 1u) / tile_cols;
    return MR_OK;
}

int mr_terrain_tile_bounds(mr_context* ctx, const void* height, uint32_t height_fmt, uint32_t n, uint32_t tile_rows,
                           uint32_t tile_cols, const mr_terrain_params* params, float* bbox_out) {
    if (!ctx || !height || !bbox_out) return MR_E_BADARG;
    uint32_t tr = 0, tc = 0;
    if (n > 65535u || mr_terrain_tile_count(n, tile_rows, tile_cols, &tr, &tc) != MR_OK) return mr_fail(ctx, MR_E_BADARG, "tiles: bad n or tile size");
    if (height_fmt != MR_HEIGHT_U16 && height_fmt != MR_HEIGHT_F32) return mr_fail(ctx, MR_E_BADARG, "tiles: bad height_fmt");
    if (reinterpret_cast<uintptr_t>(bbox_out) & 15u) return mr_fail(ctx, MR_E_BADARG, "tiles: bbox_out must be 16-byte aligned");
    mr_terrain_params p;
    if (params) p = *params; else mr_terrain_params_default(&p);
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    mr_staging io(ctx);
    const void* hdev = io.in(MR_SLOT_XY, height, (size_t)n * n * (height_fmt == MR_HEIGHT_U16 ? 2 : 4));
    float* bdev = io.out(MR_SLOT_VTX, bbox_out, (size_t)tr * tc * 32);
    if (io.rc) return io.rc;
    return io.finish(mr_terrain_tile_bounds_impl(ctx, hdev, height_fmt, n, tile_rows, tile_cols, &p, bdev));
}

namespace {
// mr_terrain_cull and mr_terrain_cull_frustum: the same checks, staging and copy-back; only the visibility test differs.
int terrain_cull_common(mr_context* ctx, const float* bbox, uint32_t n, uint32_t tile_rows, uint32_t tile_cols, const float xform[16],
                        bool frustum, uint32_t* visible_out, uint32_t* visible_ids_out, uint32_t* idx_out, uint64_t* counts_out) {
    if (!ctx || !bbox || !xform) return MR_E_BADARG;
    uint32_t tr = 0, tc = 0;
    if (n > 65535u || mr_terrain_tile_count(n, tile_rows, tile_cols, &tr, &tc) != MR_OK) return mr_fail(ctx, MR_E_BADARG, "cull: bad n or tile size");
    if (idx_out && (reinterpret_cast<uintptr_t>(idx_out) & 7u)) return mr_fail(ctx, MR_E_BADARG, "cull: idx_out must be 8-byte aligned");
    const size_t ntiles = (size_t)tr * tc;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    mr_staging io(ctx);
    const float* bdev = io.in(MR_SLOT_XY, bbox, ntiles * 32);
    uint32_t* vdev = io.out(MR_SLOT_FP, visible_out, ntiles * 4);
    if (io.rc) return io.rc;
    // visible ids, per-slot first index and the counts are needed internally even when the caller does not ask for them
    void *work = nullptr, *cdev = nullptr;
    int rc = mr_scratch(ctx, MR_SLOT_MISC, ntiles * 12 + 16, &work);
    if (!rc && !counts_out) rc = mr_scratch(ctx, MR_SLOT_OP, 16, &cdev);
    if (rc) return rc;
    unsigned long long* first_index = static_cast<unsigned long long*>(work);
    uint32_t* ids_scratch = reinterpret_cast<uint32_t*>(first_index + ntiles);
    // host outputs of a length known after the kernel: only their filled prefixes travel back
    bool si = false, sx = false, sc = false;
    uint32_t* idev = visible_ids_out ? io.out(MR_SLOT_FT, visible_ids_out, ntiles * 4, &si) : ids_scratch;
    uint32_t* xdev = io.out(MR_SLOT_BBOX, idx_out, 24ull * (size_t)(n - 1u) * (n - 1u), &sx);
    if (counts_out) cdev = io.out(MR_SLOT_OP, counts_out, 16, &sc);
    if (io.rc) return io.rc;
    rc = mr_terrain_cull_impl(ctx, bdev, n, tile_rows, tile_cols, xform, frustum, vdev, idev, first_index, xdev,
                              static_cast<unsigned long long*>(cdev));
    if (rc) return rc;
    uint64_t counts[2] = {0, 0};
    if (si || sx || sc) {
        MR_CUDA(ctx, cudaMemcpyAsync(counts, cdev, 16, cudaMemcpyDeviceToHost, ctx->stream));
        MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (sc) memcpy(counts_out, counts, 16);
        if (si && counts[0]) MR_CUDA(ctx, cudaMemcpyAsync(visible_ids_out, idev, (size_t)counts[0] * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (sx && counts[1]) MR_CUDA(ctx, cudaMemcpyAsync(idx_out, xdev, (size_t)counts[1] * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    return io.finish(MR_OK);
}
}  // namespace

int mr_terrain_cull(mr_context* ctx, const float* bbox, uint32_t n, uint32_t tile_rows, uint32_t tile_cols, const float xform[16],
                    uint32_t* visible_out, uint32_t* visible_ids_out, uint32_t* idx_out, uint64_t* counts_out) {
    return terrain_cull_common(ctx, bbox, n, tile_rows, tile_cols, xform, false, visible_out, visible_ids_out, idx_out, counts_out);
}

int mr_terrain_cull_frustum(mr_context* ctx, const float* bbox, uint32_t n, uint32_t tile_rows, uint32_t tile_cols,
                            const float view_proj[16], uint32_t* visible_out, uint32_t* visible_ids_out, uint32_t* idx_out,
                            uint64_t* counts_out) {
    return terrain_cull_common(ctx, bbox, n, tile_rows, tile_cols, view_proj, true, visible_out, visible_ids_out, idx_out, counts_out);
}

int mr_selftest_fastdiv(mr_context* ctx, float divisor, int force_fast, uint64_t* mismatches_out) {
    if (!ctx || !mismatches_out) return MR_E_BADARG;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    void* d = nullptr;
    int rc = mr_scratch(ctx, MR_SLOT_MISC, 8, &d);
    if (rc) return rc;
    MR_CUDA(ctx, cudaMemsetAsync(d, 0, 8, ctx->stream));
    rc = mr_selftest_fastdiv_impl(ctx, divisor, force_fast, static_cast<unsigned long long*>(d));
    if (rc) return rc;
    MR_CUDA(ctx, cudaMemcpyAsync(mismatches_out, d, 8, cudaMemcpyDeviceToHost, ctx->stream));
    MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->host_io = false;
    return MR_OK;
}

int mr_heightmap_normalize(mr_context* ctx, const uint16_t* in, uint64_t count, float* out) {
    if (!ctx || (count && (!in || !out))) return MR_E_BADARG;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    mr_staging io(ctx);
    const uint16_t* din = io.in(MR_SLOT_XY, in, (size_t)count * 2);
    float* dout = io.out(MR_SLOT_VTX, out, (size_t)count * 4);
    if (io.rc) return io.rc;
    return io.finish(mr_heightmap_normalize_impl(ctx, din, count, dout));
}

int mr_polygon_offsets(mr_context* ctx, const uint64_t* first_point, uint32_t npoly, uint64_t* first_tri_out) {
    if (!ctx || !first_point || !first_tri_out) return MR_E_BADARG;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    mr_staging io(ctx);
    const uint64_t* dfp = io.in(MR_SLOT_FP, first_point, (size_t)(npoly + 1) * 8);
    uint64_t* dft = io.out(MR_SLOT_FT, first_tri_out, (size_t)(npoly + 1) * 8);
    if (io.rc) return io.rc;
    return io.finish(mr_polygon_offsets_impl(ctx, dfp, npoly, dft));
}

int mr_polygon_offsets_rings(mr_context* ctx, const uint64_t* first_point, const uint64_t* first_ring, uint32_t npoly,
                             uint64_t* first_tri_out) {
    if (!ctx || !first_point || !first_ring || !first_tri_out) return MR_E_BADARG;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    mr_staging io(ctx);
    const uint64_t* dfp = io.in(MR_SLOT_FP, first_point, (size_t)(npoly + 1) * 8);
    const uint64_t* dfr = io.in(MR_SLOT_FR, first_ring, (size_t)(npoly + 1) * 8);
    uint64_t* dft = io.out(MR_SLOT_FT, first_tri_out, (size_t)(npoly + 1) * 8);
    if (io.rc) return io.rc;
    return io.finish(mr_polygon_ring_counts(ctx, dfp, dfr, npoly, 2, dft));
}

int mr_polygon_draw_range(uint64_t first_tri_i, uint64_t first_tri_next, uint64_t tri_base, mr_draw_range* out) {
    if (!out || first_tri_next < first_tri_i || first_tri_i < tri_base) return MR_E_BADARG;
    const uint64_t prims = first_tri_next - first_tri_i, off = first_tri_i - tri_base;
    if (prims * 3 > 0xFFFFFFFFull || off * 3 > 0xFFFFFFFFull) return MR_E_BADARG;  // VertexBuffer fields are u32
    out->vertex_count = (uint32_t)(prims * 3);  // VertexBuffer.zig:21
    out->instance_count = 1;
    out->first_vertex = (uint32_t)(off * 3);  // VertexBuffer.zig:22
    out->first_instance = 0;
    return MR_OK;
}

int mr_polygon_draw_indexed_range(uint64_t first_tri_i, uint64_t first_tri_next, uint64_t tri_base, mr_draw_indexed_range* out) {
    if (!out || first_tri_next < first_tri_i || first_tri_i < tri_base) return MR_E_BADARG;
    const uint64_t prims = first_tri_next - first_tri_i, off = first_tri_i - tri_base;
    if (prims > 0xFFFFFFFFull / 3 || off > 0xFFFFFFFFull / 3) return MR_E_BADARG;  // drawIndexed's fields are u32
    out->index_count = (uint32_t)(prims * 3);
    out->instance_count = 1;
    out->first_index = (uint32_t)(off * 3);
    out->base_vertex = 0;
    out->first_instance = 0;
    return MR_OK;
}

namespace {
// mr_triangulate_batch, mr_triangulate_earclip, mr_triangulate_earclip_holes (rings != nullptr) and
// mr_triangulate_earclip_indexed (indices != nullptr, checked by the caller; vtx_out may then be null): the same checks,
// staging and copy-back; ear clipping takes no edge order and has no small-batch path.
int triangulate_common(mr_context* ctx, const mr_polygon_job* job, bool earclip, const mr_polygon_rings* rings = nullptr,
                       const mr_polygon_indices* indices = nullptr) {
    if (!ctx || !job) return MR_E_BADARG;
    if (rings && (!rings->first_ring || !rings->ring_start) && job->npoly) return mr_fail(ctx, MR_E_BADARG, "polygons: null ring pointer");
    const mr_polygon_job& j = *job;
    if (j.npoly == 0) return MR_OK;
    if (!j.xy || !j.first_point || !j.first_tri || (!j.vtx_out && !indices)) return mr_fail(ctx, MR_E_BADARG, "polygons: null pointer");
    if (j.vtx_out) {
        if (!layout_ok(&j.layout, 1, 2)) return mr_fail(ctx, MR_E_BADARG, "polygons: bad vertex layout");
        if (j.layout.nattr > 1 && j.layout.attr[1].ncomp < 3) return mr_fail(ctx, MR_E_BADARG, "polygons: colour needs 3 components");
        if (reinterpret_cast<uintptr_t>(j.vtx_out) & 3u) return mr_fail(ctx, MR_E_BADARG, "polygons: vtx_out must be 4-byte aligned");
    }
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!earclip) {  // the reference's own call shape (Polygon.create_polygon: one small polygon, everything in host memory)
        int rc_small = MR_OK;
        if (mr_triangulate_small(ctx, &j, &rc_small)) return rc_small;
    }

    mr_staging io(ctx);
    // Host buffers need the sizes of their arrays: xy covers [point_base, first_point[npoly]), the vertex and index
    // buffers [tri_base, first_tri[npoly]) and ring_start [ring_base, first_ring[npoly]).  Offsets that live on the device
    // are read with one synchronisation, and all of them are checked before any data moves.
    const bool need_sizes = !io.where(j.xy).device || !io.where(j.vtx_out).device || (indices && !io.where(indices->idx_out).device);
    const bool need_nrings = rings && !io.where(rings->ring_start).device;
    uint64_t fp_ends[2] = {0, 0}, ft_ends[2] = {0, 0}, fr_end = 0;
    bool enqueued = false;
    cudaError_t e = cudaSuccess;
    auto read = [&](const uint64_t* a, uint32_t i, uint64_t* v) {
        if (!io.where(a).device) {
            *v = a[i];
        } else {
            enqueued = true;
            if (e == cudaSuccess) e = cudaMemcpyAsync(v, a + i, 8, cudaMemcpyDeviceToHost, ctx->stream);
        }
    };
    if (need_sizes) {
        read(j.first_point, 0, &fp_ends[0]);
        read(j.first_point, j.npoly, &fp_ends[1]);
        read(j.first_tri, 0, &ft_ends[0]);
        read(j.first_tri, j.npoly, &ft_ends[1]);
    }
    if (need_nrings) read(rings->first_ring, j.npoly, &fr_end);
    if (e != cudaSuccess) return mr_fail(ctx, MR_E_CUDA, "cudaMemcpyAsync", e);
    if (enqueued) MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (need_sizes && (fp_ends[0] < j.point_base || ft_ends[0] < j.tri_base))
        return mr_fail(ctx, MR_E_BADARG, "polygons: base beyond first offset");
    if (need_nrings && fr_end < rings->ring_base) return mr_fail(ctx, MR_E_BADARG, "polygons: ring_base beyond the last ring");
    const uint64_t npts = need_sizes ? fp_ends[1] - j.point_base : 0;
    const uint64_t ntri = need_sizes ? ft_ends[1] - j.tri_base : 0;
    const uint64_t nrings = need_nrings ? fr_end - rings->ring_base : 0;

    mr_polygon_job d = j;
    d.xy = io.in(MR_SLOT_XY, j.xy, (size_t)npts * 8);
    d.first_point = io.in(MR_SLOT_FP, j.first_point, (size_t)(j.npoly + 1) * 8);
    d.first_tri = io.in(MR_SLOT_FT, j.first_tri, (size_t)(j.npoly + 1) * 8);
    d.offset_prime = earclip ? nullptr : io.in(MR_SLOT_OP, j.offset_prime, (size_t)j.npoly * 8);
    mr_polygon_rings dr{};
    if (rings) {
        dr.first_ring = io.in(MR_SLOT_FR, rings->first_ring, (size_t)(j.npoly + 1) * 8);
        dr.ring_base = rings->ring_base;
        dr.ring_start = io.in(MR_SLOT_RS, rings->ring_start, (size_t)nrings * 8);
    }
    bool sv = false;
    const size_t vbytes = j.vtx_out ? (size_t)ntri * 3u * j.layout.stride : 0;
    // The vertex range is written over the whole kernel run: into pinned host memory the kernels store
    // directly (zero-copy over PCIe, overlapping the transfer with the triangulation; measured 10.3 vs
    // 12.3 ms for the 100k batch); pageable host memory is staged and copied back.
    if (void* alias = io.where(j.vtx_out).alias) {
        d.vtx_out = alias;
        ctx->host_io = true;  // the kernels store into the caller's host buffer: the call returns after they finish
    } else {
        d.vtx_out = io.out(MR_SLOT_VTX, j.vtx_out, vbytes, &sv);
    }
    d.bbox_out = io.out(MR_SLOT_BBOX, j.bbox_out, (size_t)j.npoly * 16);
    d.status_out = io.out(MR_SLOT_STATUS, j.status_out, (size_t)j.npoly * 4);
    d.ntri_out = io.out(MR_SLOT_NTRI, j.ntri_out, (size_t)j.npoly * 4);
    // the index range like the vertex range: pinned memory stored into directly, pageable memory staged
    mr_polygon_indices di{};
    bool si = false;
    if (indices) {
        di.index_base = indices->index_base;
        if (void* alias = io.where(indices->idx_out).alias) {
            di.idx_out = static_cast<uint32_t*>(alias);
            ctx->host_io = true;
        } else {
            di.idx_out = io.out(MR_SLOT_IDX, indices->idx_out, (size_t)ntri * 12u, &si);
        }
    }
    if (io.rc) return io.rc;
    const int rc = indices   ? mr_triangulate_earclip_indexed_impl(ctx, &d, rings ? &dr : nullptr, &di)
                   : rings   ? mr_triangulate_earclip_holes_impl(ctx, &d, &dr)
                   : earclip ? mr_triangulate_earclip_impl(ctx, &d)
                             : mr_triangulate_impl(ctx, &d, io.where(j.first_point).device ? nullptr : j.first_point);
    if (rc) return rc;
    if (sv) {  // the polygons of this job own [first_tri[0], first_tri[npoly]) only
        const size_t off = (size_t)(ft_ends[0] - j.tri_base) * 3u * j.layout.stride;
        MR_CUDA(ctx, cudaMemcpyAsync(static_cast<unsigned char*>(j.vtx_out) + off, static_cast<unsigned char*>(d.vtx_out) + off,
                                     vbytes - off, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (si) {
        const size_t off = (size_t)(ft_ends[0] - j.tri_base) * 3u;
        MR_CUDA(ctx, cudaMemcpyAsync(indices->idx_out + off, di.idx_out + off, ((size_t)ntri * 3u - off) * 4u,
                                     cudaMemcpyDeviceToHost, ctx->stream));
    }
    return io.finish(MR_OK);
}
}  // namespace

int mr_triangulate_batch(mr_context* ctx, const mr_polygon_job* job) { return triangulate_common(ctx, job, false); }

int mr_triangulate_earclip(mr_context* ctx, const mr_polygon_job* job) { return triangulate_common(ctx, job, true); }

int mr_triangulate_earclip_holes(mr_context* ctx, const mr_polygon_job* job, const mr_polygon_rings* rings) {
    if (!rings) return MR_E_BADARG;
    return triangulate_common(ctx, job, true, rings);
}

int mr_triangulate_earclip_indexed(mr_context* ctx, const mr_polygon_job* job, const mr_polygon_rings* rings,
                                   const mr_polygon_indices* indices) {
    if (!ctx || !job || !indices || !indices->idx_out) return MR_E_BADARG;
    if (reinterpret_cast<uintptr_t>(indices->idx_out) & 3u) return mr_fail(ctx, MR_E_BADARG, "polygons: idx_out must be 4-byte aligned");
    return triangulate_common(ctx, job, true, rings, indices);
}

int mr_selftest_crossing(mr_context* ctx, const float* q, uint64_t count, int8_t* sign_out) {
    if (!ctx || (count && (!q || !sign_out))) return MR_E_BADARG;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    mr_staging io(ctx);
    const float* din = io.in(MR_SLOT_XY, q, (size_t)count * 36);
    int8_t* dout = io.out(MR_SLOT_VTX, sign_out, (size_t)count);
    if (io.rc) return io.rc;
    return io.finish(mr_selftest_crossing_impl(ctx, din, count, dout));
}

int mr_selftest_orient(mr_context* ctx, const float* abc, uint64_t count, int8_t* sign_out) {
    if (!ctx || (count && (!abc || !sign_out))) return MR_E_BADARG;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    mr_staging io(ctx);
    const float* din = io.in(MR_SLOT_XY, abc, (size_t)count * 24);
    int8_t* dout = io.out(MR_SLOT_VTX, sign_out, (size_t)count);
    if (io.rc) return io.rc;
    return io.finish(mr_selftest_orient_impl(ctx, din, count, dout));
}

int mr_triangulate_tier_counts(mr_context* ctx, uint32_t out[8]) {
    if (!ctx || !out) return MR_E_BADARG;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    return mr_triangulate_tier_counts_impl(ctx, out);
}

uint64_t mr_rng_state0(uint64_t seed, uint64_t index) { return mr_rng_state0_hd(seed, index); }

uint32_t mr_rng_u32(uint64_t* state) {
    // sequential form of the same stream: draw k of state0 == k-th call starting from state0
    const uint32_t v = mr_rng_draw(*state, 0u);
    *state += MR_GOLDEN;
    return v;
}

// unirand.zig:26-50, host restatement (same draws as the device port)
int mr_unirand_seed_host(uint32_t top, uint64_t seed, uint64_t index, uint32_t* offset_out, uint32_t* prime_out) {
    if (!offset_out || !prime_out) return MR_E_BADARG;
    if (top == 1u) {
        *offset_out = 0;
        *prime_out = 1;
        return MR_OK;
    }
    uint64_t st = mr_rng_state0_hd(seed, index);
    *offset_out = mr_rng_u32(&st) % (uint32_t)(top - 1u) + 1u;
    uint32_t best = 1;
    for (int i = 0; i < MR_NPRIMES; ++i) {
        const uint32_t p = k_primes_host[i];
        if (p < top && top % p != 0u) {
            if (mr_rng_u32(&st) % 3u > 0u) best = p;
        }
    }
    *prime_out = best;
    return MR_OK;
}

int mr_unirand_seed_batch(mr_context* ctx, const uint64_t* first_point, uint32_t npoly, uint64_t seed,
                          uint64_t poly_index0, uint32_t* offset_prime_out) {
    if (!ctx || !first_point || !offset_prime_out) return MR_E_BADARG;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    mr_staging io(ctx);
    const uint64_t* dfp = io.in(MR_SLOT_FP, first_point, (size_t)(npoly + 1) * 8);
    uint32_t* dout = io.out(MR_SLOT_OP, offset_prime_out, (size_t)npoly * 8);
    if (io.rc) return io.rc;
    return io.finish(mr_unirand_seed_batch_impl(ctx, dfp, npoly, seed, poly_index0, dout));
}

int mr_synth_heightmap_u16(mr_context* ctx, uint64_t seed, uint32_t n, uint32_t row0, uint32_t rows, uint16_t* out) {
    if (!ctx || !out) return MR_E_BADARG;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    mr_staging io(ctx);
    uint16_t* dout = io.out(MR_SLOT_VTX, out, (size_t)rows * n * 2);
    if (io.rc) return io.rc;
    return io.finish(mr_synth_heightmap_u16_impl(ctx, seed, n, row0, rows, dout));
}

int mr_synth_polygons(mr_context* ctx, uint64_t seed, uint64_t poly_index0, const uint64_t* first_point,
                      uint32_t npoly, float* xy_out) {
    return mr_synth_polygons_family(ctx, MR_FAMILY_STAR, seed, poly_index0, first_point, npoly, xy_out);
}

int mr_synth_polygons_family(mr_context* ctx, int family, uint64_t seed, uint64_t poly_index0, const uint64_t* first_point,
                             uint32_t npoly, float* xy_out) {
    if (!ctx || !first_point || !xy_out) return MR_E_BADARG;
    if (family != MR_FAMILY_STAR && family != MR_FAMILY_ELLIPSE && family != MR_FAMILY_ZIPPER)
        return mr_fail(ctx, MR_E_BADARG, "synth_polygons: unknown family");
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    mr_staging io(ctx);
    size_t bytes = 0;
    if (!io.where(xy_out).device) {
        if (io.where(first_point).device) return mr_fail(ctx, MR_E_BADARG, "synth_polygons: host xy_out needs host first_point");
        bytes = (size_t)(first_point[npoly] - first_point[0]) * 8;
    }
    const uint64_t* dfp = io.in(MR_SLOT_FP, first_point, (size_t)(npoly + 1) * 8);
    float* dout = io.out(MR_SLOT_XY, xy_out, bytes);
    if (io.rc) return io.rc;
    return io.finish(mr_synth_polygons_impl(ctx, family, seed, poly_index0, dfp, npoly, dout));
}

int mr_ipc_export(mr_context* ctx, void* dev, unsigned char handle_out[MR_IPC_HANDLE_BYTES]) {
    if (!ctx || !dev || !handle_out) return MR_E_BADARG;
    static_assert(sizeof(cudaIpcMemHandle_t) <= MR_IPC_HANDLE_BYTES, "ipc handle size");
    cudaIpcMemHandle_t h;
    MR_CUDA(ctx, cudaIpcGetMemHandle(&h, dev));
    memset(handle_out, 0, MR_IPC_HANDLE_BYTES);
    memcpy(handle_out, &h, sizeof(h));
    return MR_OK;
}
int mr_ipc_open(mr_context* ctx, const unsigned char handle[MR_IPC_HANDLE_BYTES], void** dev_out) {
    if (!ctx || !handle || !dev_out) return MR_E_BADARG;
    MR_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    MR_CUDA(ctx, cudaIpcOpenMemHandle(dev_out, h, cudaIpcMemLazyEnablePeerAccess));
    return MR_OK;
}
int mr_ipc_close(mr_context* ctx, void* dev) {
    if (!ctx || !dev) return MR_E_BADARG;
    MR_CUDA(ctx, cudaIpcCloseMemHandle(dev));
    return MR_OK;
}

// Contiguous split of polygons over ranks, balanced by the cost model w(n) = n*log2(n) + n
// (descent work of the trapezoidation) -- SURVEY 8-e.
int mr_polygon_partition(const uint64_t* first_point, uint32_t npoly, uint32_t nranks, uint32_t* range_out) {
    if (!first_point || !range_out || nranks == 0) return MR_E_BADARG;
    std::vector<double> acc((size_t)npoly + 1, 0.0);
    for (uint32_t i = 0; i < npoly; ++i) {
        const double n = (double)(first_point[i + 1] - first_point[i]);
        const double w = n > 1.0 ? n * std::log2(n) + n : 1.0;
        acc[i + 1] = acc[i] + w;
    }
    const double total = acc[npoly];
    range_out[0] = 0;
    uint32_t cur = 0;
    for (uint32_t r = 1; r < nranks; ++r) {
        const double target = total * (double)r / (double)nranks;
        while (cur < npoly && acc[cur + 1] <= target) ++cur;
        range_out[r] = cur;
    }
    range_out[nranks] = npoly;
    return MR_OK;
}

int mr_terrain_partition(uint32_t n, uint32_t nranks, uint32_t* rows_out, uint32_t* qrows_out) {
    if (n == 0 || nranks == 0) return MR_E_BADARG;
    for (uint32_t r = 0; r <= nranks; ++r) {
        if (rows_out) rows_out[r] = (uint32_t)((uint64_t)n * r / nranks);
        if (qrows_out) qrows_out[r] = (uint32_t)((uint64_t)(n - 1) * r / nranks);
    }
    return MR_OK;
}

}  // extern "C"
