// K3p (EXPERIMENTAL, opt-in gemm variant 4): the large-batch sweep as a 2-SM MMA (tcgen05 cta_group::2).
//
// STATUS: compiles for sm_100a (ptxas accepts every instruction form below) but HAS NOT RUN ON A GPU YET - it was
// written after the round's GPU budget was spent.  It is never selected automatically; scripts/pair_check.py is the
// first thing to run on a B200 (raw-score parity against gemm_topk_kernel's dump mode, search parity against the
// oracle, then timing), under a timeout.  Nothing in tests/ selects it until that script has passed.
//
// Why: gemm_topk_kernel with C = 2 gives each CTA of the cluster its own query tile and multicasts every corpus tile
// into BOTH shared memories, so each SM's tensor core still reads A (16 KB) + the whole B tile (32 KB) per k-block
// from its own shared memory, and TMA writes 48 KB per k-block into each SM.  Batch 4096 is power-capped (DESIGN.md 9:
// SM clock 1.41 of 1.965 GHz), so the way up is fewer joules per flop.  Here the two CTAs of a cluster form ONE MMA of
// M = 256 (two query tiles, one per CTA) x N = 256: each CTA holds its own A tile and only HALF of the corpus tile
// (128 rows, 16 KB); the hardware feeds both tensor cores from both halves.  Per SM and k-block: shared-memory reads
// 16 + 16 KB instead of 16 + 32, TMA writes 32 KB instead of 48, no multicast, and a stage shrinks from 48 to 32 KB so
// the ring holds 6 stages in the same 192 KB.
//
//   CTA rank 0 (leader)  TMA producer (own A tile + corpus rows [0, 128) of the tile), MMA issuer for the pair,
//                        epilogue for query tile 2g
//   CTA rank 1           TMA producer (own A tile + corpus rows [128, 256)), epilogue for query tile 2g + 1
//   full[s]    leader only: one arrive.expect_tx (bytes of BOTH CTAs); both producers' TMA loads complete_tx on it
//              (cp.async.bulk.tensor ... .cta_group::2 with the leader's barrier address)
//   empty[s]   one per CTA, count 1: the leader's tcgen05.commit.cta_group::2 multicasts the arrive to both
//   tfull[a]   one per CTA, count 1: same multicast commit after the last k-block of a tile
//   tempty[a]  leader only, count 256: the 128 epilogue threads of each CTA arrive (the peer's through mapa)
// The accumulator of CTA r holds queries [128 r, +128) of the pair in its own tensor memory (lane = query) x 256
// columns = the 256 corpus rows of the tile, exactly the layout gemm_topk_kernel's epilogue reads, so the epilogue
// (append mode = MODE 3, raw dump = MODE 1) is the same code.  The bound pass stays on gemm_topk_kernel<.., 2, 2>.
#pragma once
#include "gemm.cuh"

namespace rfk {

constexpr int kPBRows = kGN / 2;                     // corpus rows of a tile held by each CTA of the pair
constexpr int kPBBytes = kPBRows * kGKBytes;         // 16 KB
constexpr int kPStageBytes = kABytes + kPBBytes;     // 32 KB
constexpr int kPMaxStages = 6;

__host__ __device__ constexpr size_t pair_smem_bytes(int stages) {
    return 1024 /*alignment slack*/ + (size_t)stages * kPStageBytes + 256 /*barriers*/;
}

// instruction descriptor of the pair's MMA: as make_idesc, M = 256 (128 rows per CTA)
__host__ __device__ constexpr uint32_t make_idesc_pair(int ab_format) {
    return (1u << 4) | ((uint32_t)ab_format << 7) | ((uint32_t)ab_format << 10) | ((uint32_t)(kGN >> 3) << 17) |
           ((uint32_t)((2 * kGM) >> 4) << 24);
}

// shared::cluster address of `saddr` (a shared::cta address of this CTA) in the CTA of rank `rank`
__device__ __forceinline__ uint32_t mapa_rank(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
// TMA load into this CTA's shared memory whose bytes complete on the LEADER's barrier (`bar` is a shared::cluster address)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar) {   // `bar` is a shared::cluster address
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {        // arrives on `bar` in both CTAs of the pair
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"((uint16_t)3)
                 : "memory");
}
template <int KIND>
__device__ __forceinline__ void tc_mma_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (KIND == 0) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc),
            "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc),
            "r"(accumulate)
            : "memory");
    }
}

// MODE 1 = dump raw scores (test hook), MODE 3 = append (see gemm_topk_kernel).  Launched with cluster dimension 2;
// GemmArgs as for gemm_topk_kernel with C = 2 (work items = (pair of query tiles, corpus slice)), a.idesc from
// make_idesc_pair, a.stages <= kPMaxStages; tmB boxes are 128 rows (kGN / 2), tmA boxes 128 rows.
template <int KIND, int MODE>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmArgs a) {
    static_assert(MODE == 1 || MODE == 3, "the pair kernel serves the dump hook and append mode");
    extern __shared__ uint8_t psm_raw[];
    const uint32_t raw = smem_u32(psm_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;                 // same offset in both CTAs: the MMA's descriptors
    uint8_t* psm = psm_raw + (base - raw);                        // address the peer's tiles by the leader's offsets
    const int stages = a.stages;
    const uint32_t smA = base;                                    // [stages][16 KB]  own query tile
    const uint32_t smB = base + (uint32_t)stages * kABytes;       // [stages][16 KB]  own half of the corpus tile
    uint64_t* bars = reinterpret_cast<uint64_t*>(psm + (size_t)stages * kPStageBytes);
    const uint32_t bar0 = smem_u32(bars);
    // barrier slots: full[0..6) empty[6..12) tmem_full[12..14) tmem_empty[14..16); tmem base at slot 16
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (kPMaxStages + s); };
    auto tfull_bar = [&](int s) { return bar0 + 8u * (2 * kPMaxStages + s); };
    auto tempty_bar = [&](int s) { return bar0 + 8u * (2 * kPMaxStages + 2 + s); };
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kPMaxStages + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = cluster_ctarank();
    const bool leader = crank == 0;
    const int cluster_id = blockIdx.x / 2, n_clusters = gridDim.x / 2;
    const int n_groups = (a.QT + 1) / 2;            // pairs of query tiles
    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 256); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    cluster_sync_all();   // both CTAs are running and their barriers exist before the paired allocation
    if (warp == 1) {   // both CTAs: all 512 columns of each SM's tensor memory (two 256-column accumulators)
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();   // the peer's tensor memory is allocated before the leader's MMAs write into it
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int n_items = n_groups * a.S;
    const int nkb = a.num_kblocks;
    auto item_geom = [&](int sl, long long& r0, long long& r1) -> int {
        r0 = (long long)sl * a.rows_per_slice;
        r1 = r0 + a.rows_per_slice;
        if (r1 > a.n_rows) r1 = a.n_rows;
        return r1 > r0 ? (int)((r1 - r0 + kGN - 1) / kGN) : 0;
    };

    if (warp == 0) {
        if (lane == 0) {   // ===== TMA producer (both CTAs) =====
            int stage = 0;
            uint32_t phase = 0;
            for (int item = cluster_id; item < n_items; item += n_clusters) {
                const int qt = (item % n_groups) * 2 + (int)crank, sl = item / n_groups;
                long long r0, r1;
                const int ntiles = item_geom(sl, r0, r1);
                for (int t = 0; t < ntiles; ++t) {
                    const int brow = (int)(r0 + (long long)t * kGN) + (int)crank * kPBRows;
                    for (int kb = 0; kb < nkb; ++kb) {
                        mbar_wait(empty_bar(stage), phase ^ 1u);          // own slot: the pair's MMAs are done with it
                        const uint32_t lfull = mapa_rank(full_bar(stage), 0u);
                        if (leader) mbar_expect_tx(full_bar(stage), 2u * kPStageBytes);   // both CTAs' A tile + B half
                        tma_load_2d_pair(smA + (uint32_t)stage * kABytes, &tmA, kb * a.k_elems, qt * kGM, lfull);
                        tma_load_2d_pair(smB + (uint32_t)stage * kPBBytes, &tmB, kb * a.k_elems, brow, lfull);
                        if (++stage == stages) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && leader) {   // ===== MMA issuer for the pair =====
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (int item = cluster_id; item < n_items; item += n_clusters) {
                const int sl = item / n_groups;
                long long r0, r1;
                const int ntiles = item_geom(sl, r0, r1);
                for (int t = 0; t < ntiles; ++t) {
                    mbar_wait(tempty_bar(acc), acc_phase ^ 1u);   // 256 arrivals: both CTAs' epilogues drained it
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + (uint32_t)acc * kGN;
                    for (int kb = 0; kb < nkb; ++kb) {
                        mbar_wait(full_bar(stage), phase);
                        tc_fence_after();
                        const uint64_t ad = make_smem_desc(smA + (uint32_t)stage * kABytes);
                        const uint64_t bd = make_smem_desc(smB + (uint32_t)stage * kPBBytes);
#pragma unroll
                        for (int k4 = 0; k4 < kGKBytes / 32; ++k4)
                            tc_mma_pair<KIND>(d_tmem, ad + 2u * k4, bd + 2u * k4, a.idesc, (uint32_t)((kb | k4) != 0));
                        tc_commit_pair(empty_bar(stage));
                        if (++stage == stages) { stage = 0; phase ^= 1u; }
                    }
                    tc_commit_pair(tfull_bar(acc));
                    if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
                }
            }
        }
    } else {   // ===== epilogue (both CTAs): thread <-> TMEM lane <-> query of this CTA's tile =====
        const int quarter = warp & 3;
        const int m = quarter * 32 + lane;
        int acc = 0;
        uint32_t acc_phase = 0;
        const uint32_t ltempty0 = mapa_rank(tempty_bar(0), 0u), ltempty1 = mapa_rank(tempty_bar(1), 0u);   // the leader's barriers
        for (int item = cluster_id; item < n_items; item += n_clusters) {
            const int qt = (item % n_groups) * 2 + (int)crank, sl = item / n_groups;
            long long r0, r1;
            const int ntiles = item_geom(sl, r0, r1);
            const int q = qt * kGM + m;
            const int qc = q < a.nq ? q : a.nq - 1;
            const float thr3 = (MODE == 3 && q < a.nq) ? __ldg(a.thr + qc) : INFINITY;   // padding lanes never append
            const float hi3 = (MODE == 3 && a.whi != nullptr) ? __ldg(a.whi + qc) : INFINITY;
            uint32_t* const cnt3 = MODE == 3 ? a.cnt + qc : nullptr;
            u64* const buf3 = MODE == 3 ? a.cand + (size_t)qc * a.cap : nullptr;
            for (int t = 0; t < ntiles; ++t) {
                mbar_wait(tfull_bar(acc), acc_phase);
                tc_fence_after();
                const long long trow = r0 + (long long)t * kGN;
                const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)acc * kGN;
                const int valid = r1 - trow < kGN ? (int)(r1 - trow) : kGN;   // rows of this tile inside the corpus
                uint32_t vb[2][32];
                tmem_ld32_async(taddr, vb[0]);
#pragma unroll 2
                for (int c = 0; c < kGN / 32; ++c) {
                    uint32_t(&v)[32] = vb[c & 1];
                    tmem_wait32(v);
                    if (c + 1 < kGN / 32) tmem_ld32_async(taddr + (uint32_t)(c + 1) * 32, vb[(c + 1) & 1]);
                    if (MODE == 1) {
                        if (q < a.nq) {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (c * 32 + j < valid) a.dump[(size_t)q * a.n_rows + trow + c * 32 + j] = __uint_as_float(v[j]);
                        }
                        continue;
                    }
                    if (valid < c * 32 + 32) {   // last tile of a slice only: rows past the corpus must never qualify
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (c * 32 + j >= valid) v[j] = 0x7FC00000u;
                    }
                    float gmx[4];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        float x = fmaxf(__uint_as_float(v[g * 8]), __uint_as_float(v[g * 8 + 1]));
#pragma unroll
                        for (int j = 2; j < 8; ++j) x = fmaxf(x, __uint_as_float(v[g * 8 + j]));
                        gmx[g] = x;
                    }
                    const float mx = fmaxf(fmaxf(gmx[0], gmx[1]), fmaxf(gmx[2], gmx[3]));
                    if (mx >= thr3) {
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            if (gmx[g] >= thr3) {
#pragma unroll
                                for (int j = 0; j < 8; ++j) {
                                    const float sc = __uint_as_float(v[g * 8 + j]);
                                    const long long row = trow + c * 32 + g * 8 + j;
                                    // tombstones, and rows above a range search's ceiling, never take a slot
                                    if (sc >= thr3 && sc <= hi3 && (a.allow == nullptr || row_allowed(a.allow, row))) {
                                        const uint32_t pos = atomicAdd(cnt3, 1u);
                                        if (pos < (uint32_t)a.cap) buf3[pos] = make_key(sc + 0.0f, (uint32_t)row);
                                    }
                                }
                            }
                        }
                    }
                }
                tc_fence_before();
                mbar_arrive_cluster(acc ? ltempty1 : ltempty0);   // the accumulator belongs to the pair: both epilogues release it to the leader
                if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();   // nobody leaves (or frees tensor memory) while the peer may still read its half or arrive here
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

}  // namespace rfk
