// terrain.cu -- heightmap -> grid mesh kernels for sm_100a.
//
// Replaces the body of Terrain.create_terrain (Terrain/Terrain.zig:88-129) plus the per-frame WGSL
// vertex formula (Terrain/Terrain.zig:21-50) with a one-off mesh build:
//   terrain_vertices_k   streaming stencil.  A (8+2) x (256+2) height tile is staged in shared memory
//                        as f32 (the u16 -> f32 of Terrain.zig:120 fused into the load), then one
//                        thread per column walks down the tile with a rolling 3-row window and emits
//                        ONE 32-byte store (STG.E.ENL2.256: position slot + normal slot) per vertex,
//                        i.e. 1 KB contiguous per warp instruction.  HBM-bound by design: 2 B read +
//                        32 B written per vertex.
//   terrain_indices_k    closed-form, write-only.  Quads are a linear stream (24 B each); a CTA builds
//                        1024 quads in shared memory and ships them with one TMA bulk store
//                        (cp.async.bulk.global.shared::cta -> UBLKCP), so no per-thread store math.
//   heightmap_normalize_k  standalone Terrain.zig:120.
// Float rules: every product/difference/quotient is its own IEEE round-to-nearest operation.  The
// quotients by the kernel-wide constants 65535, grid_step and 2*grid_step use the exact
// reciprocal-and-correct scheme  q = a*y; r = fma(-q,b,a); q' = fma(r,y,q)  with y = RN(1/b): for the
// constants enabled here it returns RN(a/b) for every a in the guarded exponent range (checked
// exhaustively on the GPU by mr_selftest_fastdiv, tests/test_gpu_parity.py); outside the range, or
// for other constants, __fdiv_rn is used.  So positions are bit-identical to the reference formula
// evaluated without FMA contraction and normals follow the spec in the header bit for bit.
#include "common.cuh"

namespace {

constexpr int TV_THREADS = 256;  // columns per tile
constexpr int TV_ROWS = 8;  // rows per tile; measured: 8 beats 4, 16 and 32 at n = 4096 and n = 16384

struct DivConst {
    float b;  // divisor
    float y;  // RN(1/b)
    int fast; // 1: the reciprocal-and-correct scheme is enabled for this divisor
};

struct TerrainArgs {
    const void* height;
    uint32_t n;
    uint32_t height_row0, height_rows;  // rows of the heightmap present at `height`
    uint32_t row_begin, row_end;
    unsigned char* vtx_out;
    uint32_t vtx_row0;
    float grid_step, origin_scale, height_scale;
    uint32_t stride, pos_off, nrm_off;  // nrm_off == 0xFFFFFFFF -> no normal attribute
    DivConst d1, d2;                    // grid_step*1, grid_step*2
};

// a / c.b, correctly rounded.
__device__ __forceinline__ float div_const(float a, const DivConst c) {
    const uint32_t e = (__float_as_uint(a) >> 23) & 0xFFu;
    if (c.fast && (e - 64u) <= 126u) {  // |a| in [2^-63, 2^64): no overflow/underflow anywhere below
        const float q = __fmul_rn(a, c.y);
        const float r = __fmaf_rn(-q, c.b, a);
        return __fmaf_rn(r, c.y, q);
    }
    return __fdiv_rn(a, c.b);
}

// Terrain.zig:120: 1.0 - f32(u16) / 65535.0   (the quotient via the exact scheme, all 65536 inputs verified)
__device__ __forceinline__ float height_from_u16(uint32_t v) {
    const float a = (float)v;
    const float y = 1.0f / 65535.0f;  // RN(1/65535), folded at compile time
    const float q = __fmul_rn(a, y);
    const float r = __fmaf_rn(-q, 65535.0f, a);
    return __fsub_rn(1.0f, __fmaf_rn(r, y, q));
}

template <bool U16>
__device__ __forceinline__ float load_height(const void* base, size_t idx) {
    if (U16) return height_from_u16(__ldg(reinterpret_cast<const uint16_t*>(base) + idx));
    return __ldg(reinterpret_cast<const float*>(base) + idx);
}

__device__ __forceinline__ void store_vertex32(unsigned char* p, float a0, float a1, float a2, float b0,
                                               float b1, float b2) {
    // one 256-bit store: [a0 a1 a2 0 | b0 b1 b2 0]
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(a0), "f"(a1), "f"(a2),
                 "f"(0.0f), "f"(b0), "f"(b1), "f"(b2), "f"(0.0f)
                 : "memory");
}

// FAST32: stride 32, {pos,normal} at {0,16} or {16,0}: one STG.256 per vertex.
template <bool U16, bool FAST32>
__global__ void __launch_bounds__(TV_THREADS) terrain_vertices_k(const TerrainArgs a) {
    __shared__ float tile[TV_ROWS + 2][TV_THREADS + 2];
    const uint32_t n = a.n;
    const uint32_t c0 = blockIdx.x * TV_THREADS;
    const uint32_t r0 = a.row_begin + blockIdx.y * TV_ROWS;
    const uint32_t tid = threadIdx.x;

    // ---- stage the (TV_ROWS+2) x (TV_THREADS+2) height tile, clamped at the borders ----
    // Rows are clamped to the terrain (central differences are one-sided at the border) and to the
    // rows the caller provided (a band-local buffer holds only the band plus its halo; rows beyond
    // it belong to tile rows past row_end, which are never emitted).
    {
        const int r_lo = (int)a.height_row0;
        const int r_hi = (int)min(n, a.height_row0 + a.height_rows) - 1;
        const uint32_t c = min(c0 + tid, n - 1);
        const char* base = static_cast<const char*>(a.height);
        const size_t tex = U16 ? 2 : 4;
#pragma unroll
        for (int rr = 0; rr < TV_ROWS + 2; ++rr) {
            int r = (int)r0 + rr - 1;
            r = max(r_lo, min(r, r_hi));
            tile[rr][tid + 1] = load_height<U16>(base, (size_t)(uint32_t)(r - r_lo) * n + c);
        }
        if (tid < 2 * (TV_ROWS + 2)) {
            const int rr = tid >> 1;
            const int side = tid & 1;
            int r = (int)r0 + rr - 1;
            r = max(r_lo, min(r, r_hi));
            int cc = side ? (int)c0 + TV_THREADS : (int)c0 - 1;
            cc = max(0, min(cc, (int)n - 1));
            tile[rr][side ? TV_THREADS + 1 : 0] = load_height<U16>(base, (size_t)(uint32_t)(r - r_lo) * n + (uint32_t)cc);
        }
        (void)tex;
    }
    __syncthreads();

    const uint32_t c = c0 + tid;
    if (c >= n) return;
    const float gs = a.grid_step, hs = a.height_scale;
    const float org = __fmul_rn(a.origin_scale, (float)n);
    const float z = __fsub_rn(__fmul_rn(gs, (float)c), org);
    const bool has_normal = a.nrm_off != 0xFFFFFFFFu;
    const bool col_border = (c == 0) || (c + 1 == n);
    const DivConst dc = col_border ? a.d1 : a.d2;  // grid_step * (cp - cm)
    const bool col_flat = n == 1;                 // cp == cm
    const uint32_t rows = min((uint32_t)TV_ROWS, a.row_end - r0);
    const size_t row_pitch = (size_t)n * a.stride;
    unsigned char* v = a.vtx_out + ((size_t)(r0 - a.vtx_row0) * n + c) * a.stride;

    float up = tile[0][tid + 1];
    float mid = tile[1][tid + 1];
#pragma unroll
    for (int rr = 0; rr < TV_ROWS; ++rr) {
        const float down = tile[rr + 2][tid + 1];
        if ((uint32_t)rr < rows) {
            const uint32_t r = r0 + rr;
            const float x = __fsub_rn(__fmul_rn(gs, (float)r), org);
            const float y = __fmul_rn(hs, mid);
            float nx = 0.0f, ny = 1.0f, nz = 0.0f;
            if (has_normal) {
                const float left = tile[rr + 1][tid];
                const float right = tile[rr + 1][tid + 2];
                const bool row_border = (r == 0) || (r + 1 == n);
                float gx = 0.0f, gz = 0.0f;
                if (!col_flat) {  // n > 1: rp != rm and cp != cm
                    gx = div_const(__fmul_rn(hs, __fsub_rn(down, up)), row_border ? a.d1 : a.d2);
                    gz = div_const(__fmul_rn(hs, __fsub_rn(right, left)), dc);
                }
                const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(gx, gx), 1.0f), __fmul_rn(gz, gz)));
                const float inv = __frcp_rn(len);
                nx = __fmul_rn(-gx, inv);
                ny = inv;
                nz = __fmul_rn(-gz, inv);
            }
            if (FAST32) {
                if (a.pos_off == 0)
                    store_vertex32(v, x, y, z, nx, ny, nz);
                else
                    store_vertex32(v, nx, ny, nz, x, y, z);
            } else {
                // generic layout: zero the vertex, then the attributes (4-byte granularity)
                float* f = reinterpret_cast<float*>(v);
                for (uint32_t k = 0; k < a.stride / 4; ++k) f[k] = 0.0f;
                float* p = reinterpret_cast<float*>(v + a.pos_off);
                p[0] = x;
                p[1] = y;
                p[2] = z;
                if (has_normal) {
                    float* q = reinterpret_cast<float*>(v + a.nrm_off);
                    q[0] = nx;
                    q[1] = ny;
                    q[2] = nz;
                }
            }
            v += row_pitch;
        }
        up = mid;
        mid = down;
    }
}

// ---- index buffer ------------------------------------------------------------------------
// Quad Q = q*(n-1) + c of quad row q owns words [6Q, 6Q+6) of the index stream:
//     i00+n, i00, i00+n+1, i00+n+1, i00, i00+1      with i00 = q*n + c = Q + q
// (corner order of Terrain.zig:28-35 / lookups :38-45).  A CTA fills TI_QUADS quads in shared memory
// and writes them with one bulk async copy; the shared buffer is offset so that it has the same
// alignment modulo 16 as the destination, and the (at most 8-byte) unaligned head/tail go out as
// plain stores.
constexpr int TI_THREADS = 256;
constexpr int TI_QPT = 4;  // quads per thread
constexpr int TI_QUADS = TI_THREADS * TI_QPT;

struct IndexArgs {
    uint32_t* out;        // first word of quad `quad_begin`
    uint32_t n;
    uint64_t quad_begin;  // global quad number of the first quad of this launch
    uint64_t quad_count;
    uint64_t div_magic;   // floor(2^48/(n-1)) + 1: q = (Q * magic) >> 48 for Q < 2^32
};

__global__ void __launch_bounds__(TI_THREADS) terrain_indices_k(const IndexArgs a) {
    __shared__ __align__(16) uint32_t buf[TI_QUADS * 6 + 4];
    const uint64_t q0 = (uint64_t)blockIdx.x * TI_QUADS;  // first quad of this CTA, relative to quad_begin
    const uint32_t nq = (uint32_t)min((uint64_t)TI_QUADS, a.quad_count - q0);
    uint32_t* dst = a.out + q0 * 6;  // 8-byte aligned
    const uint32_t mis = (uint32_t)((reinterpret_cast<uintptr_t>(dst) >> 2) & 3u);  // 0 or 2 words past 16 B
    uint32_t* sbuf = buf + mis;
    const uint32_t n = a.n;
#pragma unroll
    for (int k = 0; k < TI_QPT; ++k) {
        const uint32_t ql = k * TI_THREADS + threadIdx.x;
        if (ql < nq) {
            const uint32_t Q = (uint32_t)(a.quad_begin + q0 + ql);
            const uint32_t qrow = (uint32_t)(((uint64_t)Q * a.div_magic) >> 48);
            const uint32_t i00 = Q + qrow;
            uint2* s = reinterpret_cast<uint2*>(sbuf + ql * 6);
            s[0] = make_uint2(i00 + n, i00);
            s[1] = make_uint2(i00 + n + 1, i00 + n + 1);
            s[2] = make_uint2(i00, i00 + 1);
        }
    }
    // make the generic-proxy shared writes visible to the async proxy, then one thread issues the copy
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    const uint32_t words = nq * 6;
    const uint32_t head = mis ? 2u : 0u;                  // words before the first 16 B boundary
    const uint32_t body = ((words - head) / 4u) * 4u;     // words in whole 16 B groups
    if (threadIdx.x == 0 && body) {
        const uint32_t saddr = (uint32_t)__cvta_generic_to_shared(sbuf + head);
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst + head), "r"(saddr),
                     "r"(body * 4u)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    if (threadIdx.x == 32) {
        if (head) *reinterpret_cast<uint2*>(dst) = *reinterpret_cast<uint2*>(sbuf);
        if (words - head - body) *reinterpret_cast<uint2*>(dst + head + body) = *reinterpret_cast<uint2*>(sbuf + head + body);
    }
    if (threadIdx.x == 0 && body) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

__global__ void __launch_bounds__(256) heightmap_normalize_k(const uint16_t* __restrict__ in,
                                                             float* __restrict__ out, uint64_t count) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (; i < count; i += step) out[i] = height_from_u16(__ldg(in + i));
}

// ---- tiles and culling (SURVEY 8-f rank 4) --------------------------------------------------------
// Tile bounding boxes: one CTA per tile reduces the heights of the tile's (rows+1) x (cols+1) vertices to their
// minimum and maximum (comparisons only: exact) and writes p0 / p1 as SceneNode keeps them.  Read-only, 2 B per
// texel for a u16 map.
struct TileArgs {
    const void* height;
    uint32_t n, tile_rows, tile_cols, tiles_c;
    float grid_step, origin_scale, height_scale;
    float* bbox_out;
};

// One tile's box from its height extremes, as SceneNode keeps them (p0, p1, w = 1).  Selection by explicit compares
// (the first operand wins ties) and a zero y bound written as +0: with height_scale == 0 or a map holding both zeros
// the sign of a zero bound would otherwise depend on the order of the reduction.
__device__ __forceinline__ void write_tile_box(const TileArgs& a, uint32_t tr, uint32_t tc, uint32_t r0, uint32_t r1, uint32_t c0,
                                               uint32_t c1, float lo, float hi) {
    const float org = __fmul_rn(a.origin_scale, (float)a.n);
    const float xa = __fsub_rn(__fmul_rn(a.grid_step, (float)r0), org), xb = __fsub_rn(__fmul_rn(a.grid_step, (float)r1), org);
    const float za = __fsub_rn(__fmul_rn(a.grid_step, (float)c0), org), zb = __fsub_rn(__fmul_rn(a.grid_step, (float)c1), org);
    const float ya = __fmul_rn(a.height_scale, lo), yb = __fmul_rn(a.height_scale, hi);
    float y0 = yb < ya ? yb : ya, y1 = yb > ya ? yb : ya;
    y0 = y0 == 0.0f ? 0.0f : y0;
    y1 = y1 == 0.0f ? 0.0f : y1;
    float4* o = reinterpret_cast<float4*>(a.bbox_out + 8 * ((size_t)tr * a.tiles_c + tc));
    o[0] = make_float4(xb < xa ? xb : xa, y0, zb < za ? zb : za, 1.0f);
    o[1] = make_float4(xb > xa ? xb : xa, y1, zb > za ? zb : za, 1.0f);
}

template <bool U16>
__global__ void __launch_bounds__(256) terrain_tile_bounds_k(const TileArgs a) {
    const uint32_t t = blockIdx.x;
    const uint32_t tr = t / a.tiles_c, tc = t - tr * a.tiles_c;
    const uint32_t r0 = tr * a.tile_rows, c0 = tc * a.tile_cols;
    const uint32_t r1 = min(r0 + a.tile_rows, a.n - 1u), c1 = min(c0 + a.tile_cols, a.n - 1u);  // inclusive vertex range
    const uint32_t w = c1 - c0 + 1u, h = r1 - r0 + 1u;
    float lo = __uint_as_float(0x7F800000u), hi = __uint_as_float(0xFF800000u);
    for (uint32_t i = threadIdx.x; i < w * h; i += blockDim.x) {
        const uint32_t rr = i / w, cc = i - rr * w;
        const float v = load_height<U16>(a.height, (size_t)(r0 + rr) * a.n + c0 + cc);
        lo = v < lo ? v : lo;
        hi = v > hi ? v : hi;
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const float ol = __shfl_xor_sync(0xFFFFFFFFu, lo, d), oh = __shfl_xor_sync(0xFFFFFFFFu, hi, d);
        lo = ol < lo ? ol : lo;
        hi = oh > hi ? oh : hi;
    }
    __shared__ float slo[8], shi[8];
    if ((threadIdx.x & 31u) == 0) {
        slo[threadIdx.x >> 5] = lo;
        shi[threadIdx.x >> 5] = hi;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 8; ++k) {
            lo = slo[k] < lo ? slo[k] : lo;
            hi = shi[k] > hi ? shi[k] : hi;
        }
        write_tile_box(a, tr, tc, r0, r1, c0, c1, lo, hi);
    }
}

// The same for tiles of at most 512 columns, coalesced: a CTA takes a strip of whole tiles (<= 512 columns + the shared
// boundary column) of one tile row; thread t walks down columns t, t + 256, ... so that every warp load is contiguous,
// the per-column minima / maxima meet in shared memory and one thread per tile combines its columns.
constexpr int TB_COLS = 512;
// PAIR (u16 map, n and tile_cols even, 4-byte aligned base): a thread owns two adjacent columns and loads both texels
// with one 32-bit load (128 contiguous bytes per warp instruction); the odd boundary column is read on its own.
template <bool U16, bool PAIR>
__global__ void __launch_bounds__(256) terrain_tile_bounds_strip_k(const TileArgs a, uint32_t tiles_per_cta) {
    __shared__ float cmin[TB_COLS + 2], cmax[TB_COLS + 2];
    const uint32_t tr = blockIdx.y, tc0 = blockIdx.x * tiles_per_cta;
    const uint32_t r0 = tr * a.tile_rows, r1 = min(r0 + a.tile_rows, a.n - 1u);
    const uint32_t c_begin = tc0 * a.tile_cols;
    const uint32_t c_end = min(c_begin + tiles_per_cta * a.tile_cols, a.n - 1u);  // inclusive
    const float pinf = __uint_as_float(0x7F800000u), ninf = __uint_as_float(0xFF800000u);
    if (PAIR) {
        const uint32_t ncols = c_end - c_begin + 1u;
        const uint16_t* h16 = static_cast<const uint16_t*>(a.height);
        for (uint32_t p = threadIdx.x; 2u * p + 1u < ncols; p += blockDim.x) {
            float lo0 = pinf, hi0 = ninf, lo1 = pinf, hi1 = ninf;
#pragma unroll 8
            for (uint32_t r = r0; r <= r1; ++r) {
                const uint32_t two = __ldg(reinterpret_cast<const uint32_t*>(h16 + (size_t)r * a.n + c_begin + 2u * p));
                const float v0 = height_from_u16(two & 0xFFFFu), v1 = height_from_u16(two >> 16);
                lo0 = v0 < lo0 ? v0 : lo0;
                hi0 = v0 > hi0 ? v0 : hi0;
                lo1 = v1 < lo1 ? v1 : lo1;
                hi1 = v1 > hi1 ? v1 : hi1;
            }
            cmin[2u * p] = lo0;
            cmax[2u * p] = hi0;
            cmin[2u * p + 1u] = lo1;
            cmax[2u * p + 1u] = hi1;
        }
        if ((ncols & 1u) && threadIdx.x == blockDim.x - 1u) {  // the boundary column shared with the next strip
            float lo = pinf, hi = ninf;
            for (uint32_t r = r0; r <= r1; ++r) {
                const float v = load_height<true>(a.height, (size_t)r * a.n + c_end);
                lo = v < lo ? v : lo;
                hi = v > hi ? v : hi;
            }
            cmin[ncols - 1u] = lo;
            cmax[ncols - 1u] = hi;
        }
    } else {
        for (uint32_t c = c_begin + threadIdx.x; c <= c_end; c += blockDim.x) {
            float lo = pinf, hi = ninf;
#pragma unroll 8
            for (uint32_t r = r0; r <= r1; ++r) {
                const float v = load_height<U16>(a.height, (size_t)r * a.n + c);
                lo = v < lo ? v : lo;
                hi = v > hi ? v : hi;
            }
            cmin[c - c_begin] = lo;
            cmax[c - c_begin] = hi;
        }
    }
    __syncthreads();
    for (uint32_t t = threadIdx.x; t < tiles_per_cta; t += blockDim.x) {  // up to 512 tiles per strip (one-column tiles)
        const uint32_t tc = tc0 + t;
        if (tc >= a.tiles_c) break;
        const uint32_t c0 = tc * a.tile_cols, c1 = min(c0 + a.tile_cols, a.n - 1u);
        float lo = __uint_as_float(0x7F800000u), hi = __uint_as_float(0xFF800000u);
        for (uint32_t c = c0; c <= c1; ++c) {
            const float l = cmin[c - c_begin], h = cmax[c - c_begin];
            lo = l < lo ? l : lo;
            hi = h > hi ? h : hi;
        }
        write_tile_box(a, tr, tc, r0, r1, c0, c1, lo, hi);
    }
}

// The bandwidth form of the strip kernel (u16 map, n and the strip width multiples of 8, 16-byte aligned base).  The
// height 1 - v/65535 (Terrain.zig:120) is monotone non-increasing in the texel v, so the minimum height of a tile is the
// height of its LARGEST texel and vice versa: the reduction runs on the packed u16 pairs (vmaxu2 / vminu2, exact) and
// only the two results per tile go through the conversion.  A thread takes eight columns with one 128-bit load; four
// threads share a column group, each taking every fourth row, TB_LOADS independent loads in flight per thread (rows
// past the tile repeat its last row, harmless for min / max).
constexpr int TB_LOADS = 8;
__global__ void __launch_bounds__(256) terrain_tile_bounds_wide_k(const TileArgs a, uint32_t tiles_per_cta) {
    __shared__ __align__(16) uint16_t cmin[4][TB_COLS + 8], cmax[4][TB_COLS + 8];
    const uint32_t tr = blockIdx.y, tc0 = blockIdx.x * tiles_per_cta;
    const uint32_t r0 = tr * a.tile_rows, r1 = min(r0 + a.tile_rows, a.n - 1u);
    const uint32_t c_begin = tc0 * a.tile_cols;
    const uint32_t c_end = min(c_begin + tiles_per_cta * a.tile_cols, a.n - 1u);  // inclusive
    const uint32_t ncols = c_end - c_begin + 1u, groups = ncols >> 3;            // ncols % 8 is 0 (right edge) or 1
    const uint16_t* h16 = static_cast<const uint16_t*>(a.height);
    const uint32_t tx = threadIdx.x & 63u, ty = threadIdx.x >> 6, lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    for (uint32_t g = tx; g < groups; g += 64u) {
        const uint16_t* col = h16 + c_begin + 8u * g;
        uint4 lo = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu), hi = make_uint4(0u, 0u, 0u, 0u);
        for (uint32_t r = r0 + ty; r <= r1; r += 4u * TB_LOADS) {
            uint4 q[TB_LOADS];
#pragma unroll
            for (int j = 0; j < TB_LOADS; ++j)
                q[j] = __ldg(reinterpret_cast<const uint4*>(col + (size_t)min(r + 4u * j, r1) * a.n));
#pragma unroll
            for (int j = 0; j < TB_LOADS; ++j) {
                lo.x = __vminu2(lo.x, q[j].x), hi.x = __vmaxu2(hi.x, q[j].x);
                lo.y = __vminu2(lo.y, q[j].y), hi.y = __vmaxu2(hi.y, q[j].y);
                lo.z = __vminu2(lo.z, q[j].z), hi.z = __vmaxu2(hi.z, q[j].z);
                lo.w = __vminu2(lo.w, q[j].w), hi.w = __vmaxu2(hi.w, q[j].w);
            }
        }
        *reinterpret_cast<uint4*>(&cmin[ty][8u * g]) = lo;
        *reinterpret_cast<uint4*>(&cmax[ty][8u * g]) = hi;
    }
    if ((ncols & 7u) && warp == 7u) {  // the boundary column shared with the next strip
        uint32_t lo = 0xFFFFu, hi = 0u;
        for (uint32_t r = r0 + lane; r <= r1; r += 32u) {
            const uint32_t v = __ldg(h16 + (size_t)r * a.n + c_end);
            lo = min(lo, v);
            hi = max(hi, v);
        }
        lo = __reduce_min_sync(0xFFFFFFFFu, lo);
        hi = __reduce_max_sync(0xFFFFFFFFu, hi);
        if (lane < 4u) {
            cmin[lane][ncols - 1u] = (uint16_t)lo;
            cmax[lane][ncols - 1u] = (uint16_t)hi;
        }
    }
    __syncthreads();
    for (uint32_t t = warp; t < tiles_per_cta; t += 8u) {
        const uint32_t tc = tc0 + t;
        if (tc >= a.tiles_c) break;
        const uint32_t c0 = tc * a.tile_cols, c1 = min(c0 + a.tile_cols, a.n - 1u);
        uint32_t lo = 0xFFFFu, hi = 0u;
        for (uint32_t c = c0 - c_begin + lane; c <= c1 - c_begin; c += 32u) {
#pragma unroll
            for (int y = 0; y < 4; ++y) {
                lo = min(lo, (uint32_t)cmin[y][c]);
                hi = max(hi, (uint32_t)cmax[y][c]);
            }
        }
        lo = __reduce_min_sync(0xFFFFFFFFu, lo);
        hi = __reduce_max_sync(0xFFFFFFFFu, hi);
        if (lane == 0u) {
            write_tile_box(a, tr, tc, r0, r1, c0, c1, height_from_u16(hi), height_from_u16(lo));
        }
    }
}

// mach.math Mat4x4.mulVec: result[i] = 0; for j in 0..3: result[i] += m[j][i] * v[j]   (every operation rounded)
__device__ __forceinline__ float4 mach_mul_vec(const float* m, const float4 v) {
    const float vv[4] = {v.x, v.y, v.z, v.w};
    float r[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float acc = 0.0f;
#pragma unroll
        for (int j = 0; j < 4; ++j) acc = __fadd_rn(acc, __fmul_rn(m[4 * j + i], vv[j]));
        r[i] = acc;
    }
    return make_float4(r[0], r[1], r[2], r[3]);
}

struct CullArgs {
    const float* bbox;
    uint32_t ntiles, n, tile_rows, tile_cols, tiles_c;
    float m[16];
    uint32_t* visible_out;      // optional
    uint32_t* visible_ids;      // ntiles (scratch or the caller's)
    unsigned long long* first_index;  // ntiles: first index-buffer word of visible slot k (scratch)
    unsigned long long* counts;       // [0] visible tiles, [1] indices
};

// The six clip planes of the frustum test, (a, b, c, d) each, in the order of the header: R3+R0, R3-R0, R3+R1, R3-R1, R2,
// R3-R2 with R_i row i of the view-projection.  A parameter of its own rather than a tail of CullArgs, so that
// terrain_cull_indices_k, which takes CullArgs and then idx_out, keeps its parameter layout.
struct CullPlanes {
    float p[24];
};

// The frustum test for one box: culled iff s < 0 for some plane, s = ((a*px + b*py) + c*pz) + d at the p-vertex
// (hi where the coefficient is >= 0, else lo; -0 picks hi, NaN picks lo); every operation rounded on its own, so a NaN
// s never culls.  The w components of the box are not read.
__device__ __forceinline__ bool frustum_visible(const CullPlanes& pl, const float4 lo, const float4 hi) {
    bool culled = false;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const float pa = pl.p[4 * k], pb = pl.p[4 * k + 1], pc = pl.p[4 * k + 2], pd = pl.p[4 * k + 3];
        const float px = pa >= 0.0f ? hi.x : lo.x, py = pb >= 0.0f ? hi.y : lo.y, pz = pc >= 0.0f ? hi.z : lo.z;
        const float s = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(pa, px), __fmul_rn(pb, py)), __fmul_rn(pc, pz)), pd);
        culled |= s < 0.0f;
    }
    return !culled;
}

// Per tile either SceneNode.zig:96-110 (FRUSTUM false) or the six-plane frustum test (FRUSTUM true), then an ordered
// compaction.  One CTA of 1024 threads walks the tiles in chunks (a terrain has at most a few 10^4 tiles); the order of
// the visible list is the tile order.
template <bool FRUSTUM>
__global__ void __launch_bounds__(1024) terrain_cull_k(const CullArgs a, const CullPlanes pl) {
    __shared__ uint32_t wsum_t[32];
    __shared__ unsigned long long wsum_q[32];
    __shared__ uint32_t base_t;
    __shared__ unsigned long long base_q;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        base_t = 0;
        base_q = 0;
    }
    __syncthreads();
    const float inf = __uint_as_float(0x7F800000u);
    for (uint32_t t0 = 0; t0 < a.ntiles; t0 += 1024) {
        const uint32_t t = t0 + threadIdx.x;
        bool vis = false;
        uint32_t quads = 0;
        if (t < a.ntiles) {
            float4 p0 = *reinterpret_cast<const float4*>(a.bbox + 8 * (size_t)t);
            float4 p1 = *reinterpret_cast<const float4*>(a.bbox + 8 * (size_t)t + 4);
            if (FRUSTUM) {
                vis = frustum_visible(pl, p0, p1);
            } else {
                if (fminf(fminf(p0.x, p0.y), fminf(p0.z, p0.w)) != -inf) p0 = mach_mul_vec(a.m, p0);  // :100-101
                if (fmaxf(fmaxf(p1.x, p1.y), fmaxf(p1.z, p1.w)) != inf) p1 = mach_mul_vec(a.m, p1);   // :103-105
                vis = (p1.x > 0.0f && p1.y > 0.0f && p1.z > 0.0f && p1.w > 0.0f) ||
                      (p0.x < 1.0f && p0.y < 1.0f && p0.z < 1.0f && p0.w < 1.0f);  // :111
            }
            const uint32_t tr = t / a.tiles_c, tc = t - tr * a.tiles_c;
            const uint32_t qr = min(a.tile_rows, a.n - 1u - tr * a.tile_rows), qc = min(a.tile_cols, a.n - 1u - tc * a.tile_cols);
            quads = vis ? qr * qc : 0u;
            if (a.visible_out) a.visible_out[t] = vis ? 1u : 0u;
        }
        // block-wide exclusive scan of (visible, quads) in thread order
        uint32_t it = vis ? 1u : 0u;
        unsigned long long iq = quads;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t ot = __shfl_up_sync(0xFFFFFFFFu, it, d);
            const unsigned long long oq = __shfl_up_sync(0xFFFFFFFFu, iq, d);
            if ((int)lane >= d) {
                it += ot;
                iq += oq;
            }
        }
        if (lane == 31) {
            wsum_t[warp] = it;
            wsum_q[warp] = iq;
        }
        __syncthreads();
        if (warp == 0) {
            uint32_t st = wsum_t[lane];
            unsigned long long sq = wsum_q[lane];
            const uint32_t st0 = st;
            const unsigned long long sq0 = sq;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t ot = __shfl_up_sync(0xFFFFFFFFu, st, d);
                const unsigned long long oq = __shfl_up_sync(0xFFFFFFFFu, sq, d);
                if ((int)lane >= d) {
                    st += ot;
                    sq += oq;
                }
            }
            wsum_t[lane] = st - st0;  // exclusive over warps
            wsum_q[lane] = sq - sq0;
        }
        __syncthreads();
        const uint32_t slot = base_t + wsum_t[warp] + it - (vis ? 1u : 0u);
        const unsigned long long firstq = base_q + wsum_q[warp] + iq - quads;
        if (vis) {
            a.visible_ids[slot] = t;
            a.first_index[slot] = firstq * 6ull;
        }
        __syncthreads();
        if (threadIdx.x == 1023) {
            base_t += wsum_t[31] + it;
            base_q += wsum_q[31] + iq;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        a.counts[0] = base_t;
        a.counts[1] = base_q * 6ull;
    }
}

// compacted index buffer: CTA (k, y) writes chunks y, y + gridDim.y, ... of TI_QUADS quads of visible tile k -- the tile's
// quads are one contiguous run of the output -- each built in shared memory and shipped with one bulk async copy, like
// terrain_indices_k (CTAs beyond the visible count leave at once).  A tile may hold up to (n-1)^2 < 2^32 quads, more chunks
// than gridDim.y can count, hence the stride; the chunk offset is 64-bit because it steps past 2^32 on the way out.
__global__ void __launch_bounds__(TI_THREADS) terrain_cull_indices_k(const CullArgs a, uint32_t* __restrict__ idx_out) {
    __shared__ __align__(16) uint32_t buf[TI_QUADS * 6 + 4];
    if (blockIdx.x >= a.counts[0]) return;
    const uint32_t t = a.visible_ids[blockIdx.x];
    const uint32_t tr = t / a.tiles_c, tc = t - tr * a.tiles_c;
    const uint32_t r0 = tr * a.tile_rows, c0 = tc * a.tile_cols;
    const uint32_t qr = min(a.tile_rows, a.n - 1u - r0), qc = min(a.tile_cols, a.n - 1u - c0);
    const uint64_t tile_quads = (uint64_t)qr * qc;
    const uint32_t n = a.n;
    for (uint64_t q0 = (uint64_t)blockIdx.y * TI_QUADS; q0 < tile_quads; q0 += (uint64_t)gridDim.y * TI_QUADS) {
        if (q0 != (uint64_t)blockIdx.y * TI_QUADS) {  // the previous chunk's bulk copy must have read buf before it is refilled
            if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            __syncthreads();
        }
        const uint32_t nq = (uint32_t)min((uint64_t)TI_QUADS, tile_quads - q0);
        uint32_t* dst = idx_out + a.first_index[blockIdx.x] + q0 * 6;  // 24-byte quads: 8-byte aligned
        const uint32_t mis = (uint32_t)((reinterpret_cast<uintptr_t>(dst) >> 2) & 3u);
        uint32_t* sbuf = buf + mis;
#pragma unroll
        for (int k = 0; k < TI_QPT; ++k) {
            const uint32_t ql = k * TI_THREADS + threadIdx.x;
            if (ql < nq) {
                const uint32_t q = (uint32_t)q0 + ql;  // < qr * qc < 2^32
                const uint32_t lr = q / qc, lc = q - lr * qc;
                const uint32_t i00 = (r0 + lr) * n + c0 + lc;
                uint2* sm = reinterpret_cast<uint2*>(sbuf + ql * 6);
                sm[0] = make_uint2(i00 + n, i00);
                sm[1] = make_uint2(i00 + n + 1, i00 + n + 1);
                sm[2] = make_uint2(i00, i00 + 1);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        const uint32_t words = nq * 6;
        const uint32_t head = mis ? 2u : 0u;
        const uint32_t body = ((words - head) / 4u) * 4u;
        if (threadIdx.x == 0 && body) {
            const uint32_t saddr = (uint32_t)__cvta_generic_to_shared(sbuf + head);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst + head), "r"(saddr), "r"(body * 4u)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        if (threadIdx.x == 32) {
            if (head) *reinterpret_cast<uint2*>(dst) = *reinterpret_cast<uint2*>(sbuf);
            if (words - head - body) *reinterpret_cast<uint2*>(dst + head + body) = *reinterpret_cast<uint2*>(sbuf + head + body);
        }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// exhaustive check of div_const against __fdiv_rn over all 2^32 dividends
__global__ void __launch_bounds__(256) selftest_fastdiv_k(DivConst c, unsigned long long* mismatches) {
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    unsigned long long bad = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (1ull << 32); i += step) {
        const float av = __uint_as_float((uint32_t)i);
        const uint32_t g = __float_as_uint(div_const(av, c));
        const uint32_t w = __float_as_uint(__fdiv_rn(av, c.b));
        const bool both_nan = ((g & 0x7FFFFFFFu) > 0x7F800000u) && ((w & 0x7FFFFFFFu) > 0x7F800000u);
        if (g != w && !both_nan) ++bad;
    }
    if (bad) atomicAdd(mismatches, bad);
}

// The scheme is enabled only for divisors it has been verified for (see mr_selftest_fastdiv).
DivConst make_div_const(float b) {
    DivConst c;
    c.b = b;
    c.y = 1.0f / b;
    uint32_t bits;
    memcpy(&bits, &b, 4);
    // verified: 0.2f, 0.4f (default grid_step * 1, * 2)
    c.fast = (bits == 0x3E4CCCCDu || bits == 0x3ECCCCCDu) ? 1 : 0;
    return c;
}

}  // namespace

int mr_terrain_build_impl(mr_context* ctx, const mr_terrain_job* j, cudaStream_t idx_stream) {
    const uint32_t n = j->n;
    if (j->vtx_out && j->row_end > j->row_begin) {
        TerrainArgs a;
        a.height = j->height;
        a.n = n;
        a.height_row0 = j->height_row0;
        a.height_rows = j->height_rows;
        a.row_begin = j->row_begin;
        a.row_end = j->row_end;
        a.vtx_out = static_cast<unsigned char*>(j->vtx_out);
        a.vtx_row0 = j->vtx_row0;
        a.grid_step = j->params.grid_step;
        a.origin_scale = j->params.origin_scale;
        a.height_scale = j->params.height_scale;
        a.stride = j->layout.stride;
        a.pos_off = j->layout.attr[0].offset;
        a.nrm_off = j->layout.nattr > 1 ? j->layout.attr[1].offset : 0xFFFFFFFFu;
        a.d1 = make_div_const(j->params.grid_step * 1.0f);
        a.d2 = make_div_const(j->params.grid_step * 2.0f);
        const bool fast32 = a.stride == 32 && j->layout.nattr == 2 &&
                            ((a.pos_off == 0 && a.nrm_off == 16) || (a.pos_off == 16 && a.nrm_off == 0)) &&
                            (reinterpret_cast<uintptr_t>(a.vtx_out) % 32 == 0);
        const uint32_t rows = j->row_end - j->row_begin;
        dim3 grid((n + TV_THREADS - 1) / TV_THREADS, (rows + TV_ROWS - 1) / TV_ROWS);
        if (grid.y > 65535u) return mr_fail(ctx, MR_E_BADARG, "terrain band too tall for one launch");
        const bool u16 = j->height_fmt == MR_HEIGHT_U16;
        if (u16 && fast32)
            terrain_vertices_k<true, true><<<grid, TV_THREADS, 0, ctx->stream>>>(a);
        else if (u16)
            terrain_vertices_k<true, false><<<grid, TV_THREADS, 0, ctx->stream>>>(a);
        else if (fast32)
            terrain_vertices_k<false, true><<<grid, TV_THREADS, 0, ctx->stream>>>(a);
        else
            terrain_vertices_k<false, false><<<grid, TV_THREADS, 0, ctx->stream>>>(a);
        MR_LAUNCH_CHECK(ctx, "terrain_vertices_k");
    }
    if (j->idx_out && n > 1 && j->qrow_end > j->qrow_begin) {
        IndexArgs a;
        const uint64_t L = 6ull * (n - 1u);
        a.out = j->idx_out + (uint64_t)(j->qrow_begin - j->idx_qrow0) * L;
        a.n = n;
        a.quad_begin = (uint64_t)j->qrow_begin * (n - 1u);
        a.quad_count = (uint64_t)(j->qrow_end - j->qrow_begin) * (n - 1u);
        a.div_magic = ((1ull << 48) / (n - 1u)) + 1ull;
        const uint64_t blocks = (a.quad_count + TI_QUADS - 1) / TI_QUADS;
        if (blocks > 0x7FFFFFFFull) return mr_fail(ctx, MR_E_BADARG, "terrain index range too large for one launch");
        terrain_indices_k<<<(unsigned)blocks, TI_THREADS, 0, idx_stream>>>(a);
        MR_LAUNCH_CHECK(ctx, "terrain_indices_k");
    }
    return MR_OK;
}

int mr_heightmap_normalize_impl(mr_context* ctx, const uint16_t* in, uint64_t count, float* out) {
    if (count == 0) return MR_OK;
    uint64_t blocks = (count + 255) / 256;
    const uint64_t cap = (uint64_t)ctx->sm_count * 32;
    if (blocks > cap) blocks = cap;
    heightmap_normalize_k<<<(unsigned)blocks, 256, 0, ctx->stream>>>(in, out, count);
    MR_LAUNCH_CHECK(ctx, "heightmap_normalize_k");
    return MR_OK;
}

int mr_selftest_fastdiv_impl(mr_context* ctx, float b, int force_fast, unsigned long long* mismatches_dev) {
    DivConst c = make_div_const(b);
    if (force_fast) c.fast = 1;
    selftest_fastdiv_k<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(c, mismatches_dev);
    MR_LAUNCH_CHECK(ctx, "selftest_fastdiv_k");
    return MR_OK;
}

int mr_terrain_tile_bounds_impl(mr_context* ctx, const void* height_dev, uint32_t height_fmt, uint32_t n, uint32_t tile_rows,
                                uint32_t tile_cols, const mr_terrain_params* p, float* bbox_dev) {
    TileArgs a;
    a.height = height_dev;
    a.n = n;
    a.tile_rows = tile_rows;
    a.tile_cols = tile_cols;
    const uint32_t tiles_r = (n - 1u + tile_rows - 1u) / tile_rows;
    a.tiles_c = (n - 1u + tile_cols - 1u) / tile_cols;
    a.grid_step = p->grid_step;
    a.origin_scale = p->origin_scale;
    a.height_scale = p->height_scale;
    a.bbox_out = bbox_dev;
    if (tile_cols <= (uint32_t)TB_COLS && tiles_r <= 65535u) {  // coalesced strips of whole tiles
        const uint32_t per = std::max(1u, (uint32_t)TB_COLS / tile_cols);
        const dim3 grid((a.tiles_c + per - 1u) / per, tiles_r);
        const bool pair = height_fmt == MR_HEIGHT_U16 && (n & 1u) == 0u && (tile_cols & 1u) == 0u &&
                          (reinterpret_cast<uintptr_t>(height_dev) & 3u) == 0u;
        const bool wide = height_fmt == MR_HEIGHT_U16 && (n & 7u) == 0u && ((per * tile_cols) & 7u) == 0u &&
                          (reinterpret_cast<uintptr_t>(height_dev) & 15u) == 0u;
        if (wide)
            terrain_tile_bounds_wide_k<<<grid, 256, 0, ctx->stream>>>(a, per);
        else if (pair)
            terrain_tile_bounds_strip_k<true, true><<<grid, 256, 0, ctx->stream>>>(a, per);
        else if (height_fmt == MR_HEIGHT_U16)
            terrain_tile_bounds_strip_k<true, false><<<grid, 256, 0, ctx->stream>>>(a, per);
        else
            terrain_tile_bounds_strip_k<false, false><<<grid, 256, 0, ctx->stream>>>(a, per);
    } else {
        const unsigned grid = tiles_r * a.tiles_c;
        if (height_fmt == MR_HEIGHT_U16)
            terrain_tile_bounds_k<true><<<grid, 256, 0, ctx->stream>>>(a);
        else
            terrain_tile_bounds_k<false><<<grid, 256, 0, ctx->stream>>>(a);
    }
    MR_LAUNCH_CHECK(ctx, "terrain_tile_bounds_k");
    return MR_OK;
}

int mr_terrain_cull_impl(mr_context* ctx, const float* bbox_dev, uint32_t n, uint32_t tile_rows, uint32_t tile_cols,
                         const float xform[16], bool frustum, uint32_t* visible_dev, uint32_t* ids_dev,
                         unsigned long long* first_index_dev, uint32_t* idx_dev, unsigned long long* counts_dev) {
    CullArgs a;
    CullPlanes pl;
    memset(&pl, 0, sizeof(pl));
    if (frustum) {  // rows R_i = (xform[i], xform[4+i], xform[8+i], xform[12+i]); one rounded add or subtract per component
        for (int j = 0; j < 4; ++j) {
            const float r0 = xform[4 * j], r1 = xform[4 * j + 1], r2 = xform[4 * j + 2], r3 = xform[4 * j + 3];
            pl.p[0 + j] = r3 + r0;   // left:   w + x >= 0
            pl.p[4 + j] = r3 - r0;   // right:  w - x >= 0
            pl.p[8 + j] = r3 + r1;   // bottom: w + y >= 0
            pl.p[12 + j] = r3 - r1;  // top:    w - y >= 0
            pl.p[16 + j] = r2;       // near:   z >= 0 (WebGPU depth range)
            pl.p[20 + j] = r3 - r2;  // far:    w - z >= 0
        }
    }
    a.bbox = bbox_dev;
    a.n = n;
    a.tile_rows = tile_rows;
    a.tile_cols = tile_cols;
    const uint32_t tiles_r = (n - 1u + tile_rows - 1u) / tile_rows;
    a.tiles_c = (n - 1u + tile_cols - 1u) / tile_cols;
    a.ntiles = tiles_r * a.tiles_c;
    memcpy(a.m, xform, sizeof(a.m));
    a.visible_out = visible_dev;
    a.visible_ids = ids_dev;
    a.first_index = first_index_dev;
    a.counts = counts_dev;
    // one CTA column per tile: checked before anything runs, so that an error leaves every output untouched
    if (idx_dev && a.ntiles > 0x7FFFFFFFu) return mr_fail(ctx, MR_E_BADARG, "cull: more than 2^31-1 tiles with idx_out");
    if (frustum)
        terrain_cull_k<true><<<1, 1024, 0, ctx->stream>>>(a, pl);
    else
        terrain_cull_k<false><<<1, 1024, 0, ctx->stream>>>(a, pl);
    MR_LAUNCH_CHECK(ctx, "terrain_cull_k");
    if (idx_dev) {
        const uint64_t tile_quads = (uint64_t)std::min(tile_rows, n - 1u) * std::min(tile_cols, n - 1u);
        const uint64_t chunks = (tile_quads + TI_QUADS - 1) / TI_QUADS;  // terrain_cull_indices_k strides over the rest
        terrain_cull_indices_k<<<dim3(a.ntiles, (unsigned)std::min<uint64_t>(chunks, 65535u)), TI_THREADS, 0, ctx->stream>>>(a, idx_dev);
        MR_LAUNCH_CHECK(ctx, "terrain_cull_indices_k");
    }
    return MR_OK;
}
