// b200va_stream.cuh -- the tuned 128-bit streaming skeleton of vadd_vec, generalised over
// element type and operation (SURVEY.md section 8(f) row 4: STREAM-style kernels).
//
//   COPY   c[i] = a[i]                      2 x sizeof(T) bytes / element
//   SCALE  c[i] = s * a[i]                  2 x sizeof(T)
//   ADD    c[i] = a[i] + b[i]               3 x sizeof(T)      (f32 ADD == the vectorAdd hot path)
//   TRIAD  c[i] = fma(s, b[i], a[i])        3 x sizeof(T)      (one rounding: a + s*b)
//
// Element types: f32, f64 (computed natively, round-to-nearest-even, no FTZ) and f16 / bf16
// (operands widened exactly to f32, computed in f32 with s rounded to f32, result rounded
// to nearest-even into the storage type).  Same tile-strided, load-batch-then-store shape
// as vadd_vec; every global access is a 16-byte vector, `head`/tail elements are scalar.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstddef>
#include <cstdint>

#include "b200va_ptx.cuh"

namespace b200va {

enum : int { OP_COPY = 0, OP_SCALE = 1, OP_ADD = 2, OP_TRIAD = 3, OP_COUNT = 4 };
enum : int { DT_F32 = 0, DT_F64 = 1, DT_F16 = 2, DT_BF16 = 3, DT_COUNT = 4 };

struct u32x4 { uint32_t x, y, z, w; };

template <int LD>
__device__ __forceinline__ u32x4 ldg128_bits(const void* p)
{
    u32x4 r;
    if constexpr (LD == LD_NA_EF)
        asm volatile("ld.global.L1::no_allocate.v4.b32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
    else
        asm volatile("ld.global.v4.b32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
    return r;
}

template <int ST>
__device__ __forceinline__ void stg128_bits(void* p, const u32x4& v)
{
    if constexpr (ST == ST_NA)
        asm volatile("st.global.L1::no_allocate.v4.b32 [%0], {%1,%2,%3,%4};"
                     :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
    else
        asm volatile("st.global.v4.b32 [%0], {%1,%2,%3,%4};"
                     :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---- one element -----------------------------------------------------------------
template <int OP>
__device__ __forceinline__ float op_f32(float a, float b, float s)
{
    if constexpr (OP == OP_COPY) return a;
    else if constexpr (OP == OP_SCALE) return __fmul_rn(s, a);
    else if constexpr (OP == OP_ADD) return __fadd_rn(a, b);
    else return __fmaf_rn(s, b, a);
}

template <int OP>
__device__ __forceinline__ double op_f64(double a, double b, double s)
{
    if constexpr (OP == OP_COPY) return a;
    else if constexpr (OP == OP_SCALE) return __dmul_rn(s, a);
    else if constexpr (OP == OP_ADD) return __dadd_rn(a, b);
    else return __fma_rn(s, b, a);
}

template <int DT> struct dt_traits;
template <> struct dt_traits<DT_F32>  { using scalar = float;  static constexpr int size = 4; };
template <> struct dt_traits<DT_F64>  { using scalar = double; static constexpr int size = 8; };
template <> struct dt_traits<DT_F16>  { using scalar = float;  static constexpr int size = 2; };
template <> struct dt_traits<DT_BF16> { using scalar = float;  static constexpr int size = 2; };

__device__ __forceinline__ float widen_f16(uint32_t h) { return __half2float(__ushort_as_half(static_cast<unsigned short>(h))); }
__device__ __forceinline__ uint32_t narrow_f16(float f) { return __half_as_ushort(__float2half_rn(f)); }
__device__ __forceinline__ float widen_bf16(uint32_t h) { return __uint_as_float(h << 16); }
__device__ __forceinline__ uint32_t narrow_bf16(float f) { return __bfloat16_as_ushort(__float2bfloat16_rn(f)); }

// COPY never touches the value (bit-preserving, NaN payloads included).
template <int DT, int OP>
__device__ __forceinline__ uint32_t op_word(uint32_t a, uint32_t b, typename dt_traits<DT>::scalar s)
{
    if constexpr (OP == OP_COPY) return a;
    else if constexpr (DT == DT_F32) return __float_as_uint(op_f32<OP>(__uint_as_float(a), __uint_as_float(b), s));
    else if constexpr (DT == DT_F16) {
        const uint32_t lo = narrow_f16(op_f32<OP>(widen_f16(a & 0xffffu), widen_f16(b & 0xffffu), s));
        const uint32_t hi = narrow_f16(op_f32<OP>(widen_f16(a >> 16), widen_f16(b >> 16), s));
        return lo | (hi << 16);
    } else {
        const uint32_t lo = narrow_bf16(op_f32<OP>(widen_bf16(a & 0xffffu), widen_bf16(b & 0xffffu), s));
        const uint32_t hi = narrow_bf16(op_f32<OP>(widen_bf16(a >> 16), widen_bf16(b >> 16), s));
        return lo | (hi << 16);
    }
}

template <int DT, int OP>
__device__ __forceinline__ u32x4 op_vec(const u32x4& a, const u32x4& b, typename dt_traits<DT>::scalar s)
{
    if constexpr (DT == DT_F64 && OP != OP_COPY) {
        const double a0 = __hiloint2double(static_cast<int>(a.y), static_cast<int>(a.x));
        const double a1 = __hiloint2double(static_cast<int>(a.w), static_cast<int>(a.z));
        const double b0 = __hiloint2double(static_cast<int>(b.y), static_cast<int>(b.x));
        const double b1 = __hiloint2double(static_cast<int>(b.w), static_cast<int>(b.z));
        const double r0 = op_f64<OP>(a0, b0, s), r1 = op_f64<OP>(a1, b1, s);
        return u32x4{static_cast<uint32_t>(__double2loint(r0)), static_cast<uint32_t>(__double2hiint(r0)),
                     static_cast<uint32_t>(__double2loint(r1)), static_cast<uint32_t>(__double2hiint(r1))};
    } else if constexpr (DT == DT_F64) {
        return a;
    } else {
        return u32x4{op_word<DT, OP>(a.x, b.x, s), op_word<DT, OP>(a.y, b.y, s), op_word<DT, OP>(a.z, b.z, s),
                     op_word<DT, OP>(a.w, b.w, s)};
    }
}

// One scalar element at index i (head / tail / misaligned fallback).
template <int DT, int OP>
__device__ __forceinline__ void op_elem(const void* A, const void* B, void* C, size_t i, typename dt_traits<DT>::scalar s)
{
    constexpr bool binary = (OP == OP_ADD || OP == OP_TRIAD);
    if constexpr (DT == DT_F32) {
        const float b = binary ? static_cast<const float*>(B)[i] : 0.f;
        static_cast<uint32_t*>(C)[i] = op_word<DT, OP>(static_cast<const uint32_t*>(A)[i], __float_as_uint(b), s);
    } else if constexpr (DT == DT_F64) {
        if constexpr (OP == OP_COPY) static_cast<unsigned long long*>(C)[i] = static_cast<const unsigned long long*>(A)[i];
        else static_cast<double*>(C)[i] = op_f64<OP>(static_cast<const double*>(A)[i], binary ? static_cast<const double*>(B)[i] : 0.0, s);
    } else {
        const uint32_t a = static_cast<const unsigned short*>(A)[i];
        const uint32_t b = binary ? static_cast<const unsigned short*>(B)[i] : 0u;
        static_cast<unsigned short*>(C)[i] = static_cast<unsigned short>(op_word<DT, OP>(a, b, s) & 0xffffu);
    }
}

// ---- the streaming kernel ----------------------------------------------------------
// `head` elements peeled in front, `nvec` 16-byte vectors, scalar tail; CTA 0 does the edges.
// prefetch_first != 0: thread 0 bulk-prefetches the CTA's first input tile(s) into L2 ahead of the
// programmatic dependency on the previous launch (always legal: L2 is the coherence point; see
// vadd_vec EARLY = 2) -- set by the dispatcher for arrays that cannot be L2-resident.
template <int DT, int OP, int UNROLL, int LD, int ST>
__global__ void stream_vec(const void* A, const void* B, void* C, size_t n, size_t head, size_t nvec, size_t ntiles,
                           typename dt_traits<DT>::scalar s, int prefetch_first)
{
    constexpr int ES = dt_traits<DT>::size;
    constexpr int EPV = 16 / ES;
    constexpr bool binary = (OP == OP_ADD || OP == OP_TRIAD);
    const unsigned char* a = static_cast<const unsigned char*>(A) + head * ES;
    const unsigned char* b = static_cast<const unsigned char*>(B) + head * ES;
    unsigned char* c = static_cast<unsigned char*>(C) + head * ES;
    const size_t tile_vecs = static_cast<size_t>(blockDim.x) * UNROLL;
    pdl_launch_dependents();
    if (prefetch_first && threadIdx.x == 0 && blockIdx.x * tile_vecs < nvec) {
        const size_t t0 = blockIdx.x * tile_vecs;
        const uint32_t bytes = static_cast<uint32_t>((nvec - t0 < tile_vecs ? nvec - t0 : tile_vecs) * 16);
        bulk_prefetch_l2(a + t0 * 16, bytes);
        if constexpr (binary) bulk_prefetch_l2(b + t0 * 16, bytes);
    }
    pdl_wait();

    for (size_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const size_t v0 = tile * tile_vecs + threadIdx.x;
        if ((tile + 1) * tile_vecs <= nvec) {
            u32x4 ra[UNROLL], rb[UNROLL];
#pragma unroll
            for (int j = 0; j < UNROLL; ++j) ra[j] = ldg128_bits<LD>(a + (v0 + static_cast<size_t>(j) * blockDim.x) * 16);
            if constexpr (binary) {
#pragma unroll
                for (int j = 0; j < UNROLL; ++j) rb[j] = ldg128_bits<LD>(b + (v0 + static_cast<size_t>(j) * blockDim.x) * 16);
            } else {
#pragma unroll
                for (int j = 0; j < UNROLL; ++j) rb[j] = u32x4{0, 0, 0, 0};
            }
#pragma unroll
            for (int j = 0; j < UNROLL; ++j)
                stg128_bits<ST>(c + (v0 + static_cast<size_t>(j) * blockDim.x) * 16, op_vec<DT, OP>(ra[j], rb[j], s));
        } else {
#pragma unroll
            for (int j = 0; j < UNROLL; ++j) {
                const size_t v = v0 + static_cast<size_t>(j) * blockDim.x;
                if (v < nvec) {
                    const u32x4 x = ldg128_bits<LD>(a + v * 16);
                    const u32x4 y = binary ? ldg128_bits<LD>(b + v * 16) : u32x4{0, 0, 0, 0};
                    stg128_bits<ST>(c + v * 16, op_vec<DT, OP>(x, y, s));
                }
            }
        }
    }
    if (blockIdx.x == 0) {
        const size_t tail0 = head + nvec * EPV;
        if (threadIdx.x < head) op_elem<DT, OP>(A, B, C, threadIdx.x, s);
        if (tail0 + threadIdx.x < n) op_elem<DT, OP>(A, B, C, tail0 + threadIdx.x, s);
    }
}

// Mixed-misalignment fallback: one element per thread.
template <int DT, int OP>
__global__ void stream_scalar(const void* A, const void* B, void* C, size_t n, typename dt_traits<DT>::scalar s)
{
    const size_t i = static_cast<size_t>(blockDim.x) * blockIdx.x + threadIdx.x;
    if (i < n) op_elem<DT, OP>(A, B, C, i, s);
}

// ---- the grouped form: one launch over many independent (A, B, C, n) items ----------------
// The item table and the exclusive prefix of per-item tile counts travel by value in the kernel
// parameter block (__grid_constant__, read through the constant cache): no device allocation,
// so a call is capturable into a CUDA graph as it stands.  One CTA per tile; a CTA finds its
// item by binary search over the prefix, so the item index is uniform across the CTA.
struct GroupedItem {
    const void* a;
    const void* b;
    void* c;
    size_t n;
};

template <int CAP>
struct GroupedParams {
    GroupedItem item[CAP];
    unsigned long long first_tile[CAP];   // exclusive prefix of the items' tile counts
    unsigned long long total_tiles;
    int count;
};

// How an item is cut into tiles of `tile_vecs` 16-byte vectors.  The host (tile prefix) and the
// device (tile body) derive it from the same pointers with this one function, exactly as the
// stream_vec dispatcher does: `head` scalar elements up to A's 16-byte boundary, `nvec` vectors,
// a scalar tail.  Items whose A, B and C do not share a 16-byte phase take the scalar path:
// `tile_vecs * 16 / ES` elements per tile, one element per thread per step.  A vector item too
// short for one vector still gets one tile: its CTA does the edge elements.
struct GroupedShape {
    size_t head, nvec, ntiles;
    bool vec;
};

template <int ES, bool BINARY>
__host__ __device__ __forceinline__ GroupedShape grouped_shape(const void* A, const void* B, const void* C, size_t n,
                                                               size_t tile_vecs)
{
    const uintptr_t a = reinterpret_cast<uintptr_t>(A), b = reinterpret_cast<uintptr_t>(B), c = reinterpret_cast<uintptr_t>(C);
    GroupedShape sh;
    sh.vec = (a & 15u) == (c & 15u) && (!BINARY || (b & 15u) == (a & 15u));
    if (sh.vec) {
        sh.head = ((16u - (a & 15u)) & 15u) / ES;
        if (sh.head > n) sh.head = n;
        sh.nvec = (n - sh.head) * ES / 16;
        sh.ntiles = (sh.nvec + tile_vecs - 1) / tile_vecs;
        if (sh.ntiles == 0) sh.ntiles = 1;
    } else {
        const size_t tile_elems = tile_vecs * (16 / ES);
        sh.head = 0;
        sh.nvec = 0;
        sh.ntiles = (n + tile_elems - 1) / tile_elems;
    }
    return sh;
}

// Last item whose first tile is <= tile.
template <int CAP>
__device__ __forceinline__ int grouped_find(const GroupedParams<CAP>& p, unsigned long long tile)
{
    int lo = 0, hi = p.count - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (p.first_tile[mid] <= tile) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// Per element the same op_vec / op_elem as stream_vec and stream_scalar, so each item's result is
// bit-identical to b200va_stream on it.  prefetch_first: as in stream_vec, thread 0 bulk-prefetches
// the CTA's first tile into L2 ahead of the programmatic dependency (set for launches whose items
// sum to >= 128 MiB per array, which cannot be L2-resident).  Every global load and store comes
// after griddepcontrol.wait.
template <int DT, int OP, int UNROLL, int CAP>
__global__ void stream_grouped(const __grid_constant__ GroupedParams<CAP> p, typename dt_traits<DT>::scalar s,
                               int prefetch_first)
{
    constexpr int ES = dt_traits<DT>::size;
    constexpr int EPV = 16 / ES;
    constexpr bool binary = (OP == OP_ADD || OP == OP_TRIAD);
    const size_t tile_vecs = static_cast<size_t>(blockDim.x) * UNROLL;
    pdl_launch_dependents();
    if (prefetch_first && threadIdx.x == 0) {
        const int i = grouped_find(p, blockIdx.x);
        const GroupedItem& it = p.item[i];
        const GroupedShape sh = grouped_shape<ES, binary>(it.a, it.b, it.c, it.n, tile_vecs);
        const size_t v0 = (blockIdx.x - p.first_tile[i]) * tile_vecs;
        if (sh.vec && v0 < sh.nvec) {
            const uint32_t bytes = static_cast<uint32_t>((sh.nvec - v0 < tile_vecs ? sh.nvec - v0 : tile_vecs) * 16);
            bulk_prefetch_l2(static_cast<const unsigned char*>(it.a) + sh.head * ES + v0 * 16, bytes);
            if constexpr (binary) bulk_prefetch_l2(static_cast<const unsigned char*>(it.b) + sh.head * ES + v0 * 16, bytes);
        }
    }
    pdl_wait();

    for (unsigned long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const int i = grouped_find(p, tile);
        const GroupedItem& it = p.item[i];
        const size_t t = tile - p.first_tile[i];
        const GroupedShape sh = grouped_shape<ES, binary>(it.a, it.b, it.c, it.n, tile_vecs);
        if (!sh.vec) {
            const size_t tile_elems = tile_vecs * EPV;
            for (size_t e = t * tile_elems + threadIdx.x; e < (t + 1) * tile_elems && e < it.n; e += blockDim.x)
                op_elem<DT, OP>(it.a, it.b, it.c, e, s);
            continue;
        }
        const unsigned char* a = static_cast<const unsigned char*>(it.a) + sh.head * ES;
        const unsigned char* b = static_cast<const unsigned char*>(it.b) + sh.head * ES;
        unsigned char* c = static_cast<unsigned char*>(it.c) + sh.head * ES;
        const size_t v0 = t * tile_vecs + threadIdx.x;
        if ((t + 1) * tile_vecs <= sh.nvec) {
            u32x4 ra[UNROLL], rb[UNROLL];
#pragma unroll
            for (int j = 0; j < UNROLL; ++j) ra[j] = ldg128_bits<LD_PLAIN>(a + (v0 + static_cast<size_t>(j) * blockDim.x) * 16);
            if constexpr (binary) {
#pragma unroll
                for (int j = 0; j < UNROLL; ++j) rb[j] = ldg128_bits<LD_PLAIN>(b + (v0 + static_cast<size_t>(j) * blockDim.x) * 16);
            } else {
#pragma unroll
                for (int j = 0; j < UNROLL; ++j) rb[j] = u32x4{0, 0, 0, 0};
            }
#pragma unroll
            for (int j = 0; j < UNROLL; ++j)
                stg128_bits<ST_NA>(c + (v0 + static_cast<size_t>(j) * blockDim.x) * 16, op_vec<DT, OP>(ra[j], rb[j], s));
        } else {
#pragma unroll
            for (int j = 0; j < UNROLL; ++j) {
                const size_t v = v0 + static_cast<size_t>(j) * blockDim.x;
                if (v < sh.nvec) {
                    const u32x4 x = ldg128_bits<LD_PLAIN>(a + v * 16);
                    const u32x4 y = binary ? ldg128_bits<LD_PLAIN>(b + v * 16) : u32x4{0, 0, 0, 0};
                    stg128_bits<ST_NA>(c + v * 16, op_vec<DT, OP>(x, y, s));
                }
            }
        }
        if (t == 0) {
            const size_t tail0 = sh.head + sh.nvec * EPV;
            if (threadIdx.x < sh.head) op_elem<DT, OP>(it.a, it.b, it.c, threadIdx.x, s);
            if (tail0 + threadIdx.x < it.n) op_elem<DT, OP>(it.a, it.b, it.c, tail0 + threadIdx.x, s);
        }
    }
}

}  // namespace b200va
