// polygon_sink.cuh -- what the two polygon paths (triangulate.cu, earclip.cu) share: the emit sink of
// Polygon/Polygon.zig:65-79 with its palette and bounding-box accumulators, and the bounds-checked workspace spans.
// Included inside each file's anonymous namespace.
#pragma once

// ---- checked build -----------------------------------------------------------------------------------
// compute-sanitizer is not available on the GPU pool this library was developed on, and the reference path's workspace is
// full of deliberate overlays (five arrays laid over dead space), which is where an out-of-bounds write hides.  Every
// workspace array of both polygon paths is therefore declared through MR_SPAN / MR_MAKE_SPAN: in the product build these are raw
// pointers (no cost); with -DMR_CHECKED (make -C myrenderer_b200/csrc checked) they carry their length and every
// access traps on an index out of range.  tests/test_gpu_checked.py and tests/test_gpu_earclip.py run their cases against that library.
#ifdef MR_CHECKED
template <class T>
struct mr_span {
    T* p;
    uint32_t n;
    int line;
    __device__ __forceinline__ T& operator[](size_t i) const {
        if (i >= n) {
            printf("MR_CHECKED: index %llu out of range %u (span declared at line %d; block %u thread %u)\n",
                   (unsigned long long)i, n, line, blockIdx.x, threadIdx.x);
            __trap();
        }
        return p[i];
    }
    __device__ __forceinline__ bool is_null() const { return p == nullptr; }
    template <class U>
    __device__ __forceinline__ operator mr_span<U>() const { return mr_span<U>{p, n, line}; }  // T* -> const T*
};
#define MR_SPAN(T) mr_span<T>
#define MR_MAKE_SPAN(T, ptr, len) (mr_span<T>{(ptr), (uint32_t)(len), __LINE__})
#define MR_SPAN_NULL(T) (mr_span<T>{nullptr, 0u, __LINE__})
#define MR_SPAN_IS_NULL(s) ((s).is_null())
#define MR_SPAN_RAW(s) ((s).p)
#else
#define MR_SPAN(T) T*
#define MR_MAKE_SPAN(T, ptr, len) (ptr)
#define MR_SPAN_NULL(T) (static_cast<T*>(nullptr))
#define MR_SPAN_IS_NULL(s) ((s) == nullptr)
#define MR_SPAN_RAW(s) (s)
#endif

// Polygon.zig:50-57,66-71: palette[(len/3)%4], channels (hex&0xff, hex>>8&0xff, hex>>16&0xff)/255.0 of
// 0x5e315b, 0xcfff70, 0x3ca370, 0x4b5bab.  The twelve quotients are constants; their bit patterns
// (IEEE f32 division) are the ones of SURVEY 8-a12 and are checked against the oracle's computed
// palette in tests/test_oracle_cpu.py::test_palette_bits and by every vertex-buffer comparison.
__device__ __forceinline__ float3 palette(uint32_t tri) {
    switch (tri & 3u) {
        case 0: return make_float3(__uint_as_float(0x3EB6B6B7u), __uint_as_float(0x3E44C4C5u), __uint_as_float(0x3EBCBCBDu));
        case 1: return make_float3(__uint_as_float(0x3EE0E0E1u), __uint_as_float(0x3F800000u), __uint_as_float(0x3F4FCFD0u));
        case 2: return make_float3(__uint_as_float(0x3EE0E0E1u), __uint_as_float(0x3F23A3A4u), __uint_as_float(0x3E70F0F1u));
        default: return make_float3(__uint_as_float(0x3F2BABACu), __uint_as_float(0x3EB6B6B7u), __uint_as_float(0x3E969697u));
    }
}

struct Sink {
    unsigned char* base;  // polygon's vertex range
    uint32_t cap_vtx;     // 3*(n-2)
    uint32_t stride, off_x, off_c;
    int fast32;

    // vertex `k` of the polygon: position P, colour of triangle k/3
    __device__ __forceinline__ void write(uint32_t k, float2 P) const {
        const float3 c = palette(k / 3u);
        unsigned char* v = base + (size_t)k * stride;
        if (fast32) {
            if (off_x == 0)
                asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(v), "f"(P.x), "f"(P.y),
                             "f"(0.0f), "f"(0.0f), "f"(c.x), "f"(c.y), "f"(c.z), "f"(0.0f)
                             : "memory");
            else
                asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(v), "f"(c.x), "f"(c.y),
                             "f"(c.z), "f"(0.0f), "f"(P.x), "f"(P.y), "f"(0.0f), "f"(0.0f)
                             : "memory");
        } else {
            float* f = reinterpret_cast<float*>(v);
            for (uint32_t i = 0; i < stride / 4; ++i) f[i] = 0.0f;
            float* px = reinterpret_cast<float*>(v + off_x);
            px[0] = P.x;
            px[1] = P.y;
            if (off_c != 0xFFFFFFFFu) {
                float* pc = reinterpret_cast<float*>(v + off_c);
                pc[0] = c.x;
                pc[1] = c.y;
                pc[2] = c.z;
            }
        }
    }
    // zero vertices [k0, k1) cooperatively
    __device__ void zero(uint32_t k0, uint32_t k1, uint32_t lane, uint32_t nthreads = 32u) const {
        if (k1 <= k0) return;
        if (fast32) {
            for (uint32_t k = k0 + lane; k < k1; k += nthreads)
                asm volatile("st.global.v8.f32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" ::"l"(base + (size_t)k * 32),
                             "f"(0.0f)
                             : "memory");
        } else {
            uint32_t* w = reinterpret_cast<uint32_t*>(base + (size_t)k0 * stride);
            const size_t words = (size_t)(k1 - k0) * stride / 4;
            for (size_t i = lane; i < words; i += nthreads) w[i] = 0u;
        }
    }
};

__device__ __forceinline__ float fmin_acc(float acc, float v) { return v < acc ? v : acc; }
__device__ __forceinline__ float fmax_acc(float acc, float v) { return v > acc ? v : acc; }

// host: the sink fields of a polygon path's kernel arguments from the job's vertex layout and (device) vertex buffer.
// fast32 selects the single 32-byte store, which needs stride 32, position and colour at offsets 0 and 16 in either
// order, and a 32-byte-aligned buffer.
template <class Args>
inline void sink_layout(Args& a, const mr_layout& L, const void* vtx_out) {
    a.stride = L.stride;
    a.off_x = L.attr[0].offset;
    a.off_c = L.nattr > 1 ? L.attr[1].offset : 0xFFFFFFFFu;
    a.fast32 = (a.stride == 32 && L.nattr == 2 && ((a.off_x == 0 && a.off_c == 16) || (a.off_x == 16 && a.off_c == 0)) &&
                reinterpret_cast<uintptr_t>(vtx_out) % 32 == 0)
                   ? 1
                   : 0;
}
