// common.cuh -- context, error plumbing and host/device pointer staging shared by the
// translation units of libmyrenderer_b200.  Product code: never includes anything from oracle/.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include "../../include/myrenderer_b200.h"

// ---- scratch slots -----------------------------------------------------------------------------------------
// The growing device buffers of mr_context (mr_scratch), by what they hold.  Rule: within one call, no two live buffers
// share a slot; a slot that several entry points use holds one buffer of whichever call is running.
enum mr_slot {
    MR_SLOT_XY,      // polygon points (triangulation in, mr_synth_polygons_family out); the heightmap (terrain build, tile
                     // bounds, mr_heightmap_normalize); the tile boxes (cull); the self-test inputs
    MR_SLOT_FP,      // first_point (triangulation, offsets, unirand seeds, polygon synthesis); the cull's visible flags
    MR_SLOT_FT,      // first_tri (triangulation in, offsets out); the cull's visible tile ids
    MR_SLOT_OP,      // offset_prime (triangulation in, mr_unirand_seed_batch out); the cull's two counts
    MR_SLOT_VTX,     // vertex buffers (triangulation, terrain build); tile bounds; normalised heights; self-test signs;
                     // the synthetic heightmap
    MR_SLOT_BBOX,    // polygon bounding boxes; terrain index buffers (build, cull)
    MR_SLOT_STATUS,  // polygon status
    MR_SLOT_NTRI,    // polygon triangle counts
    MR_SLOT_WORK,    // reference-path work list; its header outlives the call (mr_triangulate_tier_counts)
    MR_SLOT_TIER1,   // general-path workspaces of polygons handed over by the fast path
    MR_SLOT_MISC,    // prefix-sum temporary (mr_polygon_offsets_impl, mr_polygon_ring_counts); the cull's work list;
                     // the fast-division self-test's counter
    MR_SLOT_TIER1B,  // general-path workspaces of the 1025..MR_MAX_POLYGON_POINTS class
    MR_SLOT_PAR,     // parallel-search scratch of the n <= 64 kernel
    MR_SLOT_EC_WORK, // ear-clip work list (apart from MR_SLOT_WORK, so the tier counts survive an ear-clip call)
    MR_SLOT_FR,      // first_ring
    MR_SLOT_RS,      // ring_start
    MR_SLOT_IDX,     // polygon index buffers (mr_triangulate_earclip_indexed)
    MR_NUM_SCRATCH
};
static_assert(MR_NUM_SCRATCH == 17, "scratch slot count");

constexpr int MR_NUM_AUX = 12;

struct mr_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 148;
    size_t smem_optin = 0;
    uint64_t launches = 0;
    char err[512] = {0};
    // growing device scratch slots used to stage host pointers and hold work lists
    void* scratch[MR_NUM_SCRATCH] = {nullptr};
    size_t scratch_bytes[MR_NUM_SCRATCH] = {0};
    // small pinned mailbox for device->host scalars
    void* pinned_mailbox = nullptr;
    // side streams for the polygon size classes' retry pass (independent, mostly empty kernels whose launch
    // latencies then overlap); created on first use
    cudaStream_t aux[MR_NUM_AUX] = {nullptr};
    cudaEvent_t fork_ev = nullptr;
    cudaEvent_t join_ev[MR_NUM_AUX] = {nullptr};
    // set whenever a call consumed or produced caller HOST memory (staged copy, pinned source, zero-copy alias):
    // such a call synchronises before it returns (mr_finish_host_io)
    bool host_io = false;
    // polygon launch plan (kernel, block, blocks per SM, shared memory per size class), built once per context
    void* poly_plan = nullptr;
    // small-batch path: one pinned block + its device mirror (inputs, work list, outputs of a call in one copy each way)
    void* small_pinned = nullptr;
    void* small_dev = nullptr;
    size_t small_bytes = 0;
    // work-list header of the last mr_triangulate_batch (mr_triangulate_tier_counts)
    const uint32_t* last_header_dev = nullptr;
};

inline int mr_aux_streams(mr_context* ctx) {
    if (ctx->fork_ev) return 0;
    for (int i = 0; i < MR_NUM_AUX; ++i) {
        if (cudaStreamCreateWithFlags(&ctx->aux[i], cudaStreamNonBlocking) != cudaSuccess) return -2;
        if (cudaEventCreateWithFlags(&ctx->join_ev[i], cudaEventDisableTiming) != cudaSuccess) return -2;
    }
    if (cudaEventCreateWithFlags(&ctx->fork_ev, cudaEventDisableTiming) != cudaSuccess) return -2;
    return 0;
}

inline int mr_fail(mr_context* ctx, int code, const char* what, cudaError_t e = cudaSuccess) {
    if (ctx) {
        if (e != cudaSuccess)
            snprintf(ctx->err, sizeof(ctx->err), "%s: %s", what, cudaGetErrorString(e));
        else
            snprintf(ctx->err, sizeof(ctx->err), "%s", what);
    }
    return code;
}

#define MR_CUDA(ctx, call)                                              \
    do {                                                                \
        cudaError_t e_ = (call);                                        \
        if (e_ != cudaSuccess) return mr_fail((ctx), MR_E_CUDA, #call, e_); \
    } while (0)

#define MR_LAUNCH_CHECK(ctx, name)                                      \
    do {                                                                \
        cudaError_t e_ = cudaGetLastError();                            \
        if (e_ != cudaSuccess) return mr_fail((ctx), MR_E_CUDA, name, e_); \
        (ctx)->launches++;                                              \
    } while (0)

inline int mr_scratch(mr_context* ctx, mr_slot slot, size_t bytes, void** out) {
    if (bytes == 0) bytes = 16;
    if (ctx->scratch_bytes[slot] < bytes) {
        if (ctx->scratch[slot]) {
            MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            MR_CUDA(ctx, cudaFree(ctx->scratch[slot]));
            ctx->scratch[slot] = nullptr;
            ctx->scratch_bytes[slot] = 0;
        }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&ctx->scratch[slot], want);
        if (e != cudaSuccess) return mr_fail(ctx, MR_E_NOMEM, "scratch cudaMalloc", e);
        ctx->scratch_bytes[slot] = want;
    }
    *out = ctx->scratch[slot];
    return MR_OK;
}

// End of an entry point: if the call touched caller host memory in any way, wait for the stream, so that inputs may
// be reused and outputs read as soon as the call returns (the header's contract for host pointers).
inline int mr_finish_host_io(mr_context* ctx) {
    if (!ctx->host_io) return MR_OK;
    ctx->host_io = false;
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return mr_fail(ctx, MR_E_CUDA, "cudaStreamSynchronize", e);
    return MR_OK;
}

// Where a caller buffer lives: device (or managed) memory that kernels use as it is, pinned host memory, which kernels
// reach through its device alias under UVA, or pageable host memory.  A null pointer counts as device memory.
struct mr_loc {
    bool device;
    void* alias;  // pinned host memory: its device alias
};

// The caller buffers of one entry point: validate the arguments first, then stage inputs and outputs, run the work on
// ctx->stream, and end with finish().  Each caller pointer is classified once (one cudaPointerGetAttributes).  Host
// inputs are copied into scratch slot `slot`; host outputs are produced in it and copied back over the whole range by
// finish(), or by the caller when it asks for `staged` (a part of the buffer, or on another stream).  The first failure
// is kept in rc and turns every later step into a no-op returning null, so a caller checks rc once before its work.
struct mr_staging {
    mr_context* ctx;
    int rc = MR_OK;

    explicit mr_staging(mr_context* c) : ctx(c) {}

    mr_loc where(const void* p) {
        if (!p) return {true, nullptr};
        for (int i = 0; i < nseen; ++i)
            if (seen[i].p == p) return seen[i].loc;
        mr_loc l{false, nullptr};
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
            cudaGetLastError();  // not known to CUDA: pageable host memory
        } else {
            l.device = a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
            l.alias = a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
        }
        if (nseen < MR_NUM_SCRATCH) seen[nseen++] = {p, l};
        return l;
    }

    // a device pointer holding `bytes` of src (src itself when kernels can read it)
    template <class T>
    const T* in(mr_slot slot, const T* src, size_t bytes) {
        if (rc) return nullptr;
        if (bytes == 0 || where(src).device) return src;
        ctx->host_io = true;  // a pinned source is copied asynchronously: the call must not return before it is read
        void* d = nullptr;
        if ((rc = mr_scratch(ctx, slot, bytes, &d))) return nullptr;
        const cudaError_t e = cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) rc = mr_fail(ctx, MR_E_CUDA, "cudaMemcpyAsync", e);
        return rc ? nullptr : static_cast<const T*>(d);
    }

    // the device buffer to produce output dst in (dst itself when kernels can write it)
    template <class T>
    T* out(mr_slot slot, T* dst, size_t bytes, bool* staged = nullptr) {
        if (staged) *staged = false;
        if (rc) return nullptr;
        if (bytes == 0 || where(dst).device) return dst;
        ctx->host_io = true;
        void* d = nullptr;
        if ((rc = mr_scratch(ctx, slot, bytes, &d))) return nullptr;
        if (staged) *staged = true;
        else back[nback++] = {dst, d, bytes};  // one per slot at most, by the slot rule
        return static_cast<T*>(d);
    }

    // the end of a call whose work returned work_rc: the whole-range copy-backs in the order of their out() calls, then
    // the synchronisation of mr_finish_host_io
    int finish(int work_rc) {
        if (work_rc) return work_rc;
        for (int i = 0; i < nback; ++i)
            MR_CUDA(ctx, cudaMemcpyAsync(back[i].dst, back[i].dev, back[i].bytes, cudaMemcpyDeviceToHost, ctx->stream));
        return mr_finish_host_io(ctx);
    }

private:
    struct { const void* p; mr_loc loc; } seen[MR_NUM_SCRATCH];  // (pointers past the last entry are asked again)
    int nseen = 0;
    struct { void* dst; const void* dev; size_t bytes; } back[MR_NUM_SCRATCH];
    int nback = 0;
};

// ---- shared device helpers ------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t mr_mix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// internal entry points implemented in the other translation units
// vertices on ctx->stream; the index kernel on idx_stream
int mr_terrain_build_impl(mr_context* ctx, const mr_terrain_job* job, cudaStream_t idx_stream);
// first_point_host: the caller's host copy of first_point when it has one (lets the scheduler skip empty size classes)
int mr_triangulate_impl(mr_context* ctx, const mr_polygon_job* job, const uint64_t* first_point_host);
// all-host-pointer jobs small enough for the one-block path; returns 1 when it handled the job, 0 when it does not apply
int mr_triangulate_small(mr_context* ctx, const mr_polygon_job* job, int* rc_out);
void mr_polygon_plan_free(mr_context* ctx);
// Stable counting sort of polygon ids by size, largest first (triangulate.cu; sizes above MR_MAX_POLYGON_POINTS ride in
// bin 0).  hist and cursor hold MR_SIZE_BINS words each and must be zero; afterwards order[0..npoly) holds the ids and
// cursor[b] is the number of polygons of size >= b, so the sizes lo..hi occupy order[cursor[hi + 1] .. cursor[lo]).
// class_begin / class_end receive the reference path's size-class ranges (NUM_CLASSES words each).
constexpr uint32_t MR_SIZE_BINS = MR_MAX_POLYGON_POINTS + 1;
int mr_polygon_size_sort(mr_context* ctx, const uint64_t* first_point, uint32_t npoly, uint32_t* hist, uint32_t* cursor,
                         uint32_t* class_begin, uint32_t* class_end, uint32_t* order);
// ear clipping (earclip.cu); pointers as for mr_triangulate_impl
int mr_triangulate_earclip_impl(mr_context* ctx, const mr_polygon_job* job);
int mr_selftest_orient_impl(mr_context* ctx, const float* abc, uint64_t count, int8_t* sign_out);
int mr_triangulate_earclip_holes_impl(mr_context* ctx, const mr_polygon_job* job, const mr_polygon_rings* rings);
int mr_selftest_crossing_impl(mr_context* ctx, const float* q, uint64_t count, int8_t* sign_out);
// rings == nullptr: the polygons of mr_triangulate_earclip; job->vtx_out may be null
int mr_triangulate_earclip_indexed_impl(mr_context* ctx, const mr_polygon_job* job, const mr_polygon_rings* rings,
                                        const mr_polygon_indices* indices);
// out[0..npoly]: exclusive prefix sum of max(N + 2H - sub, 0) with H as for mr_polygon_offsets_rings (triangulate.cu;
// sub 2: first_tri, sub 0: the merged ring sizes the ear-clip size classes key on); device pointers
int mr_polygon_ring_counts(mr_context* ctx, const uint64_t* first_point, const uint64_t* first_ring, uint32_t npoly,
                           uint32_t sub, uint64_t* out);
