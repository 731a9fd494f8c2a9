// Row deletion (ragfin_delete / ragfin_compact): the two kernels that tombstones need beyond the masks the search kernels
// already consume.
//   mask_and_popc_kernel   filtered search on a handle with tombstones: out = allow AND live, word by word, and the number
//                          of rows that survive both (the search's live allowed count)
//   compact_rows_kernel    physical compaction: live row r moves to off[r >> 5] + popc(word & ((1 << (r & 31)) - 1)),
//                          16-byte vector loads and stores, every old row read once and every survivor written once
#pragma once
#include "common.cuh"

namespace rfk {

// words = ceil(count / 32); bits of the last word at or past `count` are cleared in `out` (they are no rows).
// *popc must be zero on entry.
__global__ void __launch_bounds__(256) mask_and_popc_kernel(const uint32_t* __restrict__ allow, const uint32_t* __restrict__ live,
                                                            uint32_t* __restrict__ out, int64_t words, int64_t count,
                                                            unsigned long long* __restrict__ popc) {
    unsigned long long mine = 0;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < words; w += (int64_t)gridDim.x * blockDim.x) {
        uint32_t v = allow[w] & live[w];
        const int64_t tail = count - w * 32;
        if (tail < 32) v &= (1u << tail) - 1u;
        out[w] = v;
        mine += (unsigned long long)__popc(v);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) mine += __shfl_xor_sync(kFull, mine, off);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(popc, mine);
}

// One warp per row (grid-stride).  vec = 16-byte vectors per row (row bytes / 16; ld % 8 == 0 makes every row a whole number
// of them for every storage type).  off[w] = live rows before word w (exclusive prefix of the per-word popcounts).  dst and
// src are different allocations.
__global__ void __launch_bounds__(256) compact_rows_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int vec,
                                                           int64_t count, const uint32_t* __restrict__ live,
                                                           const uint32_t* __restrict__ off) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < count; r += warps) {
        const uint32_t w = __ldg(live + (r >> 5));
        const uint32_t bit = (uint32_t)(r & 31);
        if (!((w >> bit) & 1u)) continue;   // warp-uniform
        const int64_t to = (int64_t)__ldg(off + (r >> 5)) + __popc(w & ((1u << bit) - 1u));
        const uint4* s = src + r * vec;
        uint4* d = dst + to * vec;
        for (int i0 = 0; i0 < vec; i0 += 4 * kWarp) {   // four loads in flight per lane before the stores (a 768-d bf16 row: 3)
            uint4 t[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (i0 + u * kWarp + lane < vec) t[u] = __ldcs(s + i0 + u * kWarp + lane);
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (i0 + u * kWarp + lane < vec) __stcs(d + i0 + u * kWarp + lane, t[u]);
        }
    }
}

}  // namespace rfk
