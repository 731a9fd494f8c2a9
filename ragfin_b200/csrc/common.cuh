// Shared device helpers: candidate keys, storage traits, canonical fp64 reductions,
// warp-level sorted lists in shared memory, block bitonic sort.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace rfk {

typedef unsigned long long u64;

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xFFFFFFFFu;

// ---------------------------------------------------------------------------------
// Candidate key: (score, row) packed so that ONE unsigned 64-bit compare orders by
// (score descending, row ascending) when "larger key = better".  0 is "empty".
// ---------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t float_to_ordered(float f) {
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(f);
#else
    union { float f; uint32_t u; } c; c.f = f; uint32_t u = c.u;
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float ordered_to_float(uint32_t o) {
    uint32_t u = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}
__host__ __device__ __forceinline__ u64 make_key(float score, uint32_t row) {
    return ((u64)float_to_ordered(score) << 32) | (u64)(0xFFFFFFFFu - row);
}
__host__ __device__ __forceinline__ float key_score(u64 k) { return ordered_to_float((uint32_t)(k >> 32)); }
__host__ __device__ __forceinline__ uint32_t key_row(u64 k) { return 0xFFFFFFFFu - (uint32_t)k; }

// ---------------------------------------------------------------------------------
// Storage types.  DT: 0 = fp32, 1 = bf16, 2 = fp16.  Rows are [ld] elements, ld % 8 == 0.
// ---------------------------------------------------------------------------------
template <int DT> struct Store;
template <> struct Store<0> {
    typedef float T;
    static constexpr int kVec = 4;  // elements per 16-byte vector
    __device__ static __forceinline__ float to_f32(T v) { return v; }
    __device__ static __forceinline__ T from_f32(float v) { return v; }
    __device__ static __forceinline__ void unpack(const uint4& v, float* f) {
        f[0] = __uint_as_float(v.x); f[1] = __uint_as_float(v.y);
        f[2] = __uint_as_float(v.z); f[3] = __uint_as_float(v.w);
    }
};
template <> struct Store<1> {
    typedef __nv_bfloat16 T;
    static constexpr int kVec = 8;
    __device__ static __forceinline__ float to_f32(T v) { return __bfloat162float(v); }
    __device__ static __forceinline__ T from_f32(float v) { return __float2bfloat16_rn(v); }
    __device__ static __forceinline__ void unpack(const uint4& v, float* f) {
        f[0] = __uint_as_float(v.x << 16); f[1] = __uint_as_float(v.x & 0xFFFF0000u);
        f[2] = __uint_as_float(v.y << 16); f[3] = __uint_as_float(v.y & 0xFFFF0000u);
        f[4] = __uint_as_float(v.z << 16); f[5] = __uint_as_float(v.z & 0xFFFF0000u);
        f[6] = __uint_as_float(v.w << 16); f[7] = __uint_as_float(v.w & 0xFFFF0000u);
    }
};
template <> struct Store<2> {
    typedef __half T;
    static constexpr int kVec = 8;
    __device__ static __forceinline__ float to_f32(T v) { return __half2float(v); }
    __device__ static __forceinline__ T from_f32(float v) { return __float2half_rn(v); }
    __device__ static __forceinline__ void unpack(const uint4& v, float* f) {
        float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
        float2 b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
        float2 c = __half22float2(*reinterpret_cast<const __half2*>(&v.z));
        float2 d = __half22float2(*reinterpret_cast<const __half2*>(&v.w));
        f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
    }
};

// scalar filter: bit r of `allow` set <=> row r may be returned
__device__ __forceinline__ bool row_allowed(const uint32_t* __restrict__ allow, long long row) {
    return (__ldg(allow + (row >> 5)) >> (row & 31)) & 1u;
}

// streaming 128-bit load: read-only path, do not allocate in L1 (corpus is read once per scan)
__device__ __forceinline__ uint4 ldg_stream(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// ---------------------------------------------------------------------------------
// Canonical fp64 reduction (DESIGN.md "canonical arithmetic"; oracle/ragfin_oracle.py):
// lane p accumulates the terms i % 32 == p in increasing i, then a 16/8/4/2/1 xor
// butterfly.  Every lane returns the same value.  Must be called by a full warp.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ double warp_butterfly_f64(double v) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v = v + __shfl_xor_sync(kFull, v, off);
    return v;
}

// Normalisation of one stored row or query from its canonical sum of squares n2 (DESIGN.md 2): inv = 1 / sqrt(n2), and
// inv = 0 for a zero vector and for a non-finite one (any NaN or +-Inf component makes n2 NaN or +inf; a finite fp32 row
// cannot overflow n2 in fp64).  norm_elem maps the NaN that an Inf or NaN element times inv = 0 gives to +0, so a
// non-finite vector is stored as a zero vector and scores exactly 0 against everything.  Every normaliser uses these two.
__device__ __forceinline__ double inv_norm(double n2) {
    return n2 > 0.0 && n2 <= 1.7976931348623157e308 ? 1.0 / sqrt(n2) : 0.0;
}
__device__ __forceinline__ float norm_elem(float x, double inv) {
    const float y = (float)((double)x * inv);
    return y == y ? y : 0.0f;
}

template <int DT>
__device__ __forceinline__ double canonical_dot_row(const typename Store<DT>::T* __restrict__ row,
                                                    const float* __restrict__ q, int dim, int lane) {
    double acc = 0.0;
    int i = lane;
    for (; i + 23 * kWarp < dim; i += 24 * kWarp) {   // 24 loads in flight (one 768-wide row); adds stay in increasing-i order
        float a[24], b[24];
#pragma unroll
        for (int u = 0; u < 24; ++u) { a[u] = Store<DT>::to_f32(row[i + u * kWarp]); b[u] = q[i + u * kWarp]; }
#pragma unroll
        for (int u = 0; u < 24; ++u) acc = acc + (double)a[u] * (double)b[u];
    }
#pragma unroll 4
    for (; i < dim; i += kWarp) acc = acc + (double)Store<DT>::to_f32(row[i]) * (double)q[i];
    return warp_butterfly_f64(acc);
}

// ---------------------------------------------------------------------------------
// Sorted (descending) key list of `cap` entries (cap % 32 == 0) in shared memory, owned
// by one warp.  insert() requires nk > list[cap-1]; the smallest entry falls off.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void warp_list_insert(u64* list, int cap, u64 nk, int lane) {
    int pos = 0;
    for (int s = 0; s < cap; s += kWarp) pos += __popc(__ballot_sync(kFull, list[s + lane] > nk));
    for (int s = cap - kWarp; s >= 0; s -= kWarp) {
        if (s + kWarp <= pos) break;            // whole segment is above the insertion point
        const int idx = s + lane;
        u64 e = 0;
        if (idx > pos) e = list[idx - 1];
        __syncwarp();
        if (idx > pos) list[idx] = e;
        else if (idx == pos) list[idx] = nk;
        __syncwarp();
    }
}

// Block-wide bitonic sort, descending, n a power of two, data in shared memory.
__device__ __forceinline__ void block_bitonic_sort_desc(u64* a, int n, int tid, int nthreads) {
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < n; i += nthreads) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const u64 x = a[i], y = a[ixj];
                    const bool desc = (i & k) == 0;
                    if ((x < y) == desc) { a[i] = y; a[ixj] = x; }
                }
            }
            __syncthreads();
        }
    }
}

// synthetic data generator (SURVEY.md 8d); identical to oracle/ragfin_oracle.{py,c}
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ float synth_value(uint64_t key, uint64_t src_row, int dim, int col) {
    const uint64_t h = mix64((src_row * (uint64_t)dim + (uint64_t)col) ^ key);
    const int s = (int)((h & 0xFFFF) + ((h >> 16) & 0xFFFF) + ((h >> 32) & 0xFFFF) + (h >> 48));
    return (float)(s - 131070) * 1.52587890625e-05f;  // 2^-16
}

}  // namespace rfk
