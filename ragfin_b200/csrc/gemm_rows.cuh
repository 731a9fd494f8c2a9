// K3r: tensor-core sweep for at most 16 queries with the operand roles SWAPPED (append mode only).
//
// gemm_topk_kernel makes the queries the MMA's M dimension, so one query still costs a full 128-row MMA per corpus
// tile: at batch 1 the tensor pipe is 49 % busy multiplying zero padding and the GPU draws 370-440 W for an
// HBM-bound job (profiles/r01).  Here the CORPUS rows are M (two 128-row halves per 256-row tile) and the queries
// are N = 16: an MMA is 128 x 16 x 16 instead of 128 x 256 x 16 - one sixteenth of the tensor cycles for the same
// bytes - and the epilogue thread (TMEM lane = corpus row) reads 16 scores per half tile instead of 256.
//
//   shared memory   query block [num_kblocks][16 rows x 128 B] resident for the whole sweep (one TMA burst)
//                   + ring of `stages` (up to 4) corpus stages [256 rows x 128 B]: nothing but corpus bytes stream
//   tensor memory   2 tiles x 2 halves x 4 partial accumulators x 16 fp32 columns (256 columns)
//   epilogue        v[j] >= thr[j]  ->  append (score, row) to query j's buffer (exactly MODE 3 of gemm.cuh)
// Both operands are K-major SWIZZLE_128B tiles, so the corpus stages are the same TMA boxes as in gemm.cuh.
//
// MEASURED (10M x 768 bf16, k = 10, one B200, batch 1): 2.161 ms per call = 462.8 queries/s, sweep at 7 328 GB/s with
// the SM clock at 1.965 GHz; the standard orientation on the same box: 2.19-2.26 ms, 7 050 GB/s, clock capped to
// 1.1-1.2 GHz.  Two things had to be found first: (1) ring depth - 4 stages of 32 KB; with 5-6 stages (160-192 KB in
// flight per SM) the sweep drops to 6.8 TB/s, with 2 to 6.46; (2) the four k-steps of a k-block accumulate into four
// separate TMEM accumulators per half tile (summed in the epilogue) so that no MMA waits on the previous one's result.
// Default for <= 16 queries in append mode (gemm variant 0 = automatic, 3 = forced; 1 = standard orientation).
// The bound pass and finalize_append_kernel are shared with the main path; approximate scores need not be
// bit-identical between the two orientations (DESIGN.md 2.4 only uses |approx - exact| <= eps).
#pragma once
#include "gemm_astat.cuh"   // make_idesc_n

namespace rfk {

constexpr int kRN = 16;                        // queries per sweep (UMMA N)
constexpr int kRQBytes = kRN * kGKBytes;       // 2 KB: one k-block of the query block
constexpr int kRMaxStages = 4;                 // measured: 3-4 stages 7.28-7.33 TB/s, 5-6 stages 6.8 TB/s, 2 stages 6.46 TB/s
constexpr int kRSplit = 4;                     // partial accumulators per half tile = k-steps per k-block
constexpr int kRAccCols = 2 * kRSplit * kRN;   // TMEM columns of one tile's accumulators (128)
static_assert(kRSplit == kGKBytes / 32, "one partial accumulator per k-step of a k-block");

__host__ __device__ constexpr int rows_stages(int num_kblocks) {
    const long avail = 227L * 1024 - 1024 - 256 - (long)num_kblocks * kRQBytes;
    const int s = (int)(avail / kBBytes);
    return s > kRMaxStages ? kRMaxStages : s;
}
__host__ __device__ constexpr size_t rows_smem_bytes(int num_kblocks, int stages) {
    return 1024 + (size_t)num_kblocks * kRQBytes + (size_t)stages * kBBytes + 256;
}

struct RowsArgs {
    uint32_t idesc;         // M = 128, N = 16
    int num_kblocks, k_elems;
    int nq;                 // <= 16
    long long n_rows;
    int S;                  // corpus slices
    long long rows_per_slice;   // multiple of kGN
    int stages;
    u64* cand;              // [nq][cap]
    const float* thr;       // [nq]
    uint32_t* cnt;          // [nq]
    int cap;
    const uint32_t* allow;  // row mask (tombstones; bit set = row may be appended), or null
    const float* whi;       // range search: [nq] a row above it never takes a slot (window_words_kernel), else null
};

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}

template <int KIND>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_rows_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmB, const RowsArgs a) {
    extern __shared__ uint8_t rsm_raw[];
    const uint32_t raw = smem_u32(rsm_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* rsm = rsm_raw + (base - raw);
    const int stages = a.stages, nkb = a.num_kblocks;
    const uint32_t smQ = base;                                         // [nkb][2 KB]
    const uint32_t smB = base + (uint32_t)nkb * kRQBytes;              // [stages][32 KB]  (2 KB multiples keep 1 KB alignment)
    uint64_t* bars = reinterpret_cast<uint64_t*>(rsm + (size_t)nkb * kRQBytes + (size_t)stages * kBBytes);
    const uint32_t bar0 = smem_u32(bars);
    // barrier slots: full[kRMaxStages] empty[kRMaxStages] qfull tmem_full[2] tmem_empty[2]; tmem base after them
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (kRMaxStages + s); };
    const uint32_t qfull_bar = bar0 + 8u * (2 * kRMaxStages);
    auto tfull_bar = [&](int s) { return bar0 + 8u * (2 * kRMaxStages + 1 + s); };
    auto tempty_bar = [&](int s) { return bar0 + 8u * (2 * kRMaxStages + 3 + s); };
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kRMaxStages + 5);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        mbar_init(qfull_bar, 1);
        for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 128); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {   // 2 tiles x 2 halves x 4 partial accumulators x 16 columns
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    auto slice_tiles = [&](int sl, long long& r0, long long& r1) -> int {
        r0 = (long long)sl * a.rows_per_slice;
        r1 = r0 + a.rows_per_slice;
        if (r1 > a.n_rows) r1 = a.n_rows;
        return r1 > r0 ? (int)((r1 - r0 + kGN - 1) / kGN) : 0;
    };

    if (warp == 0) {
        if (lane == 0) {   // ===== TMA producer =====
            mbar_expect_tx(qfull_bar, (uint32_t)nkb * kRQBytes);
            for (int kb = 0; kb < nkb; ++kb) tma_load_2d(smQ + (uint32_t)kb * kRQBytes, &tmQ, kb * a.k_elems, 0, qfull_bar);
            int stage = 0;
            uint32_t phase = 0;
            for (int sl = blockIdx.x; sl < a.S; sl += gridDim.x) {
                long long r0, r1;
                const int ntiles = slice_tiles(sl, r0, r1);
                for (int t = 0; t < ntiles; ++t)
                    for (int kb = 0; kb < nkb; ++kb) {
                        mbar_wait(empty_bar(stage), phase ^ 1u);
                        mbar_expect_tx(full_bar(stage), kBBytes);
                        tma_load_2d(smB + (uint32_t)stage * kBBytes, &tmB, kb * a.k_elems, (int)(r0 + (long long)t * kGN), full_bar(stage));
                        if (++stage == stages) { stage = 0; phase ^= 1u; }
                    }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {   // ===== MMA issuer =====
            mbar_wait(qfull_bar, 0u);
            tc_fence_after();
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (int sl = blockIdx.x; sl < a.S; sl += gridDim.x) {
                long long r0, r1;
                const int ntiles = slice_tiles(sl, r0, r1);
                for (int t = 0; t < ntiles; ++t) {
                    mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
                    tc_fence_after();
                    for (int kb = 0; kb < nkb; ++kb) {
                        mbar_wait(full_bar(stage), phase);
                        tc_fence_after();
                        const uint64_t qd = make_smem_desc(smQ + (uint32_t)kb * kRQBytes);
#pragma unroll
                        for (int k4 = 0; k4 < kGKBytes / 32; ++k4) {
                            // An N = 16 MMA is ~8 tensor cycles but an accumulate into the SAME TMEM columns waits for the
                            // previous one (~170 cycles measured): the four k-steps of a k-block go to four separate
                            // accumulators per half (summed in the epilogue), giving eight independent chains.
#pragma unroll
                            for (int h = 0; h < 2; ++h) {   // corpus rows [128 h, 128 h + 128) of the tile are the M operand
                                const uint64_t cd = make_smem_desc(smB + (uint32_t)stage * kBBytes + (uint32_t)h * (kBBytes / 2));
                                const uint32_t d_tmem = tmem_base + (uint32_t)acc * kRAccCols + (uint32_t)h * (kRSplit * kRN) + (uint32_t)k4 * kRN;
                                tc_mma<KIND>(d_tmem, cd + 2u * k4, qd + 2u * k4, a.idesc, (uint32_t)(kb != 0));
                            }
                        }
                        tc_commit(empty_bar(stage));
                        if (++stage == stages) { stage = 0; phase ^= 1u; }
                    }
                    tc_commit(tfull_bar(acc));
                    if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
                }
            }
        }
    } else {   // ===== epilogue: thread <-> TMEM lane <-> corpus row of a half tile =====
        const int quarter = warp & 3;
        const int m = quarter * 32 + lane;
        float thr[kRN];
#pragma unroll
        for (int j = 0; j < kRN; ++j) thr[j] = j < a.nq ? __ldg(a.thr + j) : INFINITY;   // padding queries never append
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int sl = blockIdx.x; sl < a.S; sl += gridDim.x) {
            long long r0, r1;
            const int ntiles = slice_tiles(sl, r0, r1);
            for (int t = 0; t < ntiles; ++t) {
                mbar_wait(tfull_bar(acc), acc_phase);
                tc_fence_after();
                const long long trow = r0 + (long long)t * kGN;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    uint32_t v[kRSplit][kRN];
#pragma unroll
                    for (int p = 0; p < kRSplit; ++p)
                        tmem_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)acc * kRAccCols + (uint32_t)h * (kRSplit * kRN) + (uint32_t)p * kRN, v[p]);
                    const long long row = trow + h * 128 + m;
                    if (row < r1) {   // rows past the slice / corpus (zero-filled by TMA) never qualify
#pragma unroll
                        for (int j = 0; j < kRN; ++j) {
                            const float sc = (__uint_as_float(v[0][j]) + __uint_as_float(v[1][j])) + (__uint_as_float(v[2][j]) + __uint_as_float(v[3][j]));
                            // tombstones, and rows above a range search's ceiling, never take a slot
                            if (sc >= thr[j] && (a.whi == nullptr || sc <= __ldg(a.whi + j)) && (a.allow == nullptr || row_allowed(a.allow, row))) {
                                const uint32_t pos = atomicAdd(a.cnt + j, 1u);
                                if (pos < (uint32_t)a.cap) a.cand[(size_t)j * a.cap + pos] = make_key(sc + 0.0f, (uint32_t)row);
                            }
                        }
                    }
                }
                tc_fence_before();
                mbar_arrive(tempty_bar(acc));
                if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base) : "memory");
    }
}

}  // namespace rfk
