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

#define MR_NUM_SCRATCH 16

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

// true when the pointer can be dereferenced by a kernel on ctx->device
inline bool mr_is_device_ptr(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Pinned (page-locked) host memory is reachable from kernels under UVA: returns its device alias, or
// nullptr when `p` is not pinned host memory.  Used for outputs that are produced over a long kernel,
// where storing straight over PCIe overlaps the transfer with the compute.
inline void* mr_pinned_device_alias(void* p) {
    if (!p) return nullptr;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}

inline int mr_scratch(mr_context* ctx, int slot, size_t bytes, void** out) {
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

// Input staging: returns a device pointer holding `bytes` of src (src itself when already device).
inline int mr_stage_in(mr_context* ctx, int slot, const void* src, size_t bytes, const void** dev) {
    if (!src || bytes == 0 || mr_is_device_ptr(src)) {
        *dev = src;
        return MR_OK;
    }
    ctx->host_io = true;  // a pinned source is copied asynchronously: the call must not return before it is read
    void* d = nullptr;
    int rc = mr_scratch(ctx, slot, bytes, &d);
    if (rc) return rc;
    MR_CUDA(ctx, cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    *dev = d;
    return MR_OK;
}

// Output staging: device buffer to produce into; *staged says a copy-back is needed.
inline int mr_stage_out(mr_context* ctx, int slot, void* dst, size_t bytes, void** dev, bool* staged) {
    *staged = false;
    if (!dst || bytes == 0 || mr_is_device_ptr(dst)) {
        *dev = dst;
        return MR_OK;
    }
    ctx->host_io = true;
    void* d = nullptr;
    int rc = mr_scratch(ctx, slot, bytes, &d);
    if (rc) return rc;
    *dev = d;
    *staged = true;
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

inline int mr_copy_back(mr_context* ctx, void* dst, const void* dev, size_t bytes) {
    MR_CUDA(ctx, cudaMemcpyAsync(dst, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return MR_OK;
}

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
// out[0..npoly]: exclusive prefix sum of max(N + 2H - sub, 0) with H as for mr_polygon_offsets_rings (triangulate.cu;
// sub 2: first_tri, sub 0: the merged ring sizes the ear-clip size classes key on); device pointers
int mr_polygon_ring_counts(mr_context* ctx, const uint64_t* first_point, const uint64_t* first_ring, uint32_t npoly,
                           uint32_t sub, uint64_t* out);
