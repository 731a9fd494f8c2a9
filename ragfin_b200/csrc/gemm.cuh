// K3: large-batch scoring on the 5th-generation tensor cores (tcgen05 / TMEM / TMA), sm_100a only.
//
// Shape of the contraction: queries are the MMA M dimension (TMEM lane = query), corpus rows the N
// dimension, the embedding dimension is K.  One CTA owns a 128-query tile and sweeps a slice of the
// corpus in 256-row tiles; an epilogue thread therefore owns ONE query for the whole sweep and
// filters its accumulator columns against a private register threshold - the score matrix never
// leaves TMEM.
//
//   warp 0      TMA producer   cp.async.bulk.tensor.2d: A = query tile [128 x 128 B], B = corpus tile
//                              [256 x 128 B] per k-block, 128-byte swizzle, ring of `stages` slots
//   warp 1      MMA issuer     one thread issues tcgen05.mma (M=128, N=256, K=32 B) from shared-memory
//                              descriptors into one of two 256-column TMEM accumulators; tcgen05.commit
//                              releases the ring slot / publishes the accumulator
//   warps 2-5   epilogue       tcgen05.ld 32x32b.x32 (thread = TMEM lane = query), max-of-32 pre-filter,
//                              per-query candidate list (K' keys, unsorted, min-tracked) in shared memory
//
// Work items are (query tile, corpus slice) pairs, statically strided over the persistent grid; CTAs
// that run concurrently sweep the same slices with different query tiles so that the 126 MB L2
// absorbs the re-reads of the corpus.  Each item writes K' keys per query:
//   cand[(q * S + slice) * kp + j]   (unsorted, 0 = empty)  ->  finalize_kernel (sorted_lists = 0).
// Storage kinds: bf16 / fp16 through kind::f16 (queries rounded to the storage type; the rounding
// error is carried per query into the certificate), fp32 through kind::tf32.
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "kernels.cuh"   // block_kth_largest

namespace rfk {

constexpr int kGM = 128;            // queries per tile (UMMA M)
constexpr int kGN = 256;            // corpus rows per tile (UMMA N)
constexpr int kGKBytes = 128;       // bytes of K per k-block = one 128B swizzle row
constexpr int kGemmThreads = 192;   // 6 warps
constexpr int kABytes = kGM * kGKBytes;   // 16 KB
constexpr int kBBytes = kGN * kGKBytes;   // 32 KB
constexpr int kStageBytes = kABytes + kBBytes;
constexpr int kMaxStages = 4;

__host__ __device__ constexpr size_t gemm_smem_bytes(int stages, int kp) {
    return 1024 /*alignment slack*/ + (size_t)stages * kStageBytes + (size_t)kGM * kp * sizeof(u64) + 256 /*barriers*/;
}

// ---- PTX wrappers --------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar,
                                               uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster "
        "[%0], [%1, {%2, %3}], [%4], %5;" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar), "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_commit_mc(uint32_t bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"(cta_mask)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
template <int KIND>
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (KIND == 0) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc),
            "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc),
            "r"(accumulate)
            : "memory");
    }
}
// tcgen05.ld of 32 consecutive accumulator columns of this thread's TMEM lane.  The load is
// asynchronous: the registers are valid only after tmem_wait32(), which names them as in/out
// operands so that the compiler cannot move a use above the wait.
__device__ __forceinline__ void tmem_ld32_async(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_wait32(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                   "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                   "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
}

// K-major, 128-byte-swizzled operand tile: rows at 128 B pitch, 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);   // start address, 16-byte units
    d |= (uint64_t)1 << 16;                    // leading byte offset (unused for swizzled K-major) = 1
    d |= (uint64_t)(1024 >> 4) << 32;          // stride byte offset: 8 rows * 128 B
    d |= (uint64_t)1 << 46;                    // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                    // SWIZZLE_128B
    return d;
}

// instruction descriptor: D = fp32, A/B format (0 f16, 1 bf16, 2 tf32), both K-major, N = 256, M = 128
__host__ __device__ constexpr uint32_t make_idesc(int ab_format) {
    return (1u << 4) | ((uint32_t)ab_format << 7) | ((uint32_t)ab_format << 10) | ((uint32_t)(kGN >> 3) << 17) |
           ((uint32_t)(kGM >> 4) << 24);
}

// Stage switches of scripts/gemm_dbg_sweep.py (timing only, results invalid): compiled in only with
// -DRAGFIN_TIMING_EXPERIMENTS; in the default build RF_DBG(...) is the constant 0 and the branches vanish.
#ifdef RAGFIN_TIMING_EXPERIMENTS
#define RF_DBG(a, bit) ((a).dbg & (bit))
#else
#define RF_DBG(a, bit) 0
#endif

// ---- the kernel ------------------------------------------------------------------------------------
struct GemmArgs {
    uint32_t idesc;
    int num_kblocks;        // ceil(ld * esize / 128)
    int k_elems;            // elements of K per k-block (64 for 16-bit, 32 for fp32)
    int nq;
    long long n_rows;
    int QT;                 // query tiles
    int S;                  // corpus slices
    long long rows_per_slice;   // multiple of kGN
    int stages;
    int kp;
    u64* cand;              // [nq][S][kp]
    uint32_t* gtau;         // [nq] ordered-uint lower bound of the global K'-th approximate score (atomicMax)
    const uint32_t* allow;  // scalar filter bitmask over rows, or null
    float* dump;            // MODE 1: [nq][n_rows] raw scores.  MODE 2: [nq][S] block maxima (one block per "slice")
    int bound_tps;          // MODE 2: sample tiles per block ("slice" sl covers sample tiles [sl * bound_tps, +bound_tps))
    int bound_tiles;        // MODE 2: sample tiles in total
    long long bound_stride; // MODE 2: sample tile j is corpus tile j * bound_stride
    const float* thr;       // MODE 3: [nq] collection threshold (a row is appended when its score >= thr[q])
    uint32_t* cnt;          // MODE 3: [nq] rows appended so far (may exceed cap: overflow, the query goes to tier 2)
    int cap;                // MODE 3: capacity of one query's append buffer, cand = [nq][cap]
    const float* wcap;      // range search (window_words_kernel), else null.  MODE 2: [nq] sample rows above it are excluded
    const float* whi;       //   MODE 3: [nq] a row above it never takes a slot
    int dbg;                // timing experiments only (RAGFIN_GEMM_DEBUG): 1 skip epilogue filter, 2 skip MMAs, 4 skip A loads, 8 skip B loads
};

// Per-query candidate list of one epilogue thread: kp keys in shared memory (column layout
// lists[e * 128 + m]), unsorted; once full, `tau_key` is its minimum and a better key replaces it.
// `tau_s` is the score a row needs to be worth looking at: max(list minimum, global bound), where
// the global bound gtau[q] is the best list-minimum any CTA has published for this query - a valid
// lower bound of the global K'-th approximate score, so rows below it can never be candidates.
struct CandState {
    int cnt, minpos;
    u64 tau_key;
    float tau_s;
    uint32_t* gptr;   // &gtau[q], or null for padding lanes
    const uint32_t* allow;   // scalar filter bitmask, or null
};
__device__ __noinline__ void cand_insert(CandState& st, u64* lists, int m, int kp, float s, uint32_t row) {
    if (st.allow != nullptr && !row_allowed(st.allow, row)) return;   // filtered out (checked here, off the scan loop)
    const u64 key = make_key(s + 0.0f, row);
    if (st.cnt < kp) {
        lists[(size_t)st.cnt * kGM + m] = key;
        if (++st.cnt < kp) return;
    } else if (key > st.tau_key) {
        lists[(size_t)st.minpos * kGM + m] = key;
    } else {
        return;
    }
    u64 mn = ~0ull;
    int mp = 0;
#pragma unroll 8
    for (int e = 0; e < kp; ++e) {
        const u64 x = lists[(size_t)e * kGM + m];
        if (x < mn) { mn = x; mp = e; }
    }
    st.tau_key = mn;
    st.minpos = mp;
    const float t = key_score(mn);
    if (t > st.tau_s) {
        st.tau_s = t;
        if (st.gptr) atomicMax(st.gptr, float_to_ordered(t));   // publish: every CTA sweeping this query tightens
    }
}

// MODE: 0 = collect candidates in per-query lists (shared memory, K' best of the slice); 1 = dump raw scores (test
// hook); 2 = bound pass: score an evenly strided SAMPLE of corpus tiles and write each query's maximum per block of
// sample tiles.  The j-th largest of those block maxima is a valid lower bound of the j-th best score over the
// whole corpus (j distinct rows reach it), so the collecting pass starts with a tight threshold instead of warming
// up on its own slice.  3 = append: every row whose score reaches the query's fixed threshold thr[q] (bound pass:
// k-th largest block maximum minus twice the error bound) is appended to the query's buffer in global memory - no
// lists, no shared memory, nothing to maintain; finalize_append_kernel selects and rescans exactly.
// C = thread-block cluster size along the query-tile axis: the C CTAs of a cluster hold C different
// query tiles and sweep the same corpus slice in lockstep; each loads 1/C of every corpus tile and
// TMA-multicasts it into all C shared memories, so a corpus tile leaves L2 once per cluster.
template <int KIND, int MODE, int C>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_topk_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmArgs a) {
    extern __shared__ uint8_t gsm_raw[];
    const uint32_t raw = smem_u32(gsm_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;                 // SWIZZLE_128B tiles need 1024 B alignment
    uint8_t* gsm = gsm_raw + (base - raw);
    const int stages = a.stages, kp = a.kp;
    const uint32_t smA = base;                                    // [stages][16 KB]
    const uint32_t smB = base + (uint32_t)stages * kABytes;       // [stages][32 KB]
    u64* lists = reinterpret_cast<u64*>(gsm + (size_t)stages * kStageBytes);          // [kp][128]
    uint64_t* bars = reinterpret_cast<uint64_t*>(gsm + (size_t)stages * kStageBytes + (size_t)kGM * kp * sizeof(u64));
    const uint32_t bar0 = smem_u32(bars);
    // barrier slots: full[0..4) empty[4..8) tmem_full[8..10) tmem_empty[10..12); tmem base at slot 12
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (kMaxStages + s); };
    auto tfull_bar = [&](int s) { return bar0 + 8u * (2 * kMaxStages + s); };
    auto tempty_bar = [&](int s) { return bar0 + 8u * (2 * kMaxStages + 2 + s); };
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = C > 1 ? cluster_ctarank() : 0u;
    const uint16_t cmask = (uint16_t)((1u << C) - 1u);
    const int cluster_id = blockIdx.x / C, n_clusters = gridDim.x / C;
    const int n_groups = (a.QT + C - 1) / C;        // groups of C query tiles
    if (threadIdx.x == 0) {
        // empty[s] collects one tcgen05.commit from every CTA of the cluster: a slot may be refilled (by
        // multicast into all C CTAs) only when all C tensor cores are done reading it
        for (int s = 0; s < stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), C); }
        for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 128); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {   // allocate all 512 TMEM columns (two 256-column accumulators)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (C > 1) cluster_sync_all();   // peers' barriers must be initialised before any remote arrive / multicast
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int n_items = n_groups * a.S;
    const int nkb = a.num_kblocks;
    // rows of an item: first row of its tile 0, distance between consecutive tiles, end of the corpus part it may touch
    auto item_geom = [&](int sl, long long& r0, long long& r1, long long& step) -> int {
        if (MODE == 2) {
            const int j0 = sl * a.bound_tps;
            const int nt = a.bound_tiles - j0 < a.bound_tps ? a.bound_tiles - j0 : a.bound_tps;
            step = a.bound_stride * kGN;
            r0 = (long long)j0 * step;
            r1 = a.n_rows;
            return nt > 0 ? nt : 0;
        }
        step = kGN;
        r0 = (long long)sl * a.rows_per_slice;
        r1 = r0 + a.rows_per_slice;
        if (r1 > a.n_rows) r1 = a.n_rows;
        return r1 > r0 ? (int)((r1 - r0 + kGN - 1) / kGN) : 0;
    };

    if (warp == 0) {
        if (lane == 0) {   // ===== TMA producer =====
            int stage = 0;
            uint32_t phase = 0;
            constexpr int kSubRows = kGN / C;   // corpus rows this CTA fetches (and multicasts) per tile
            for (int item = cluster_id; item < n_items; item += n_clusters) {
                const int qt = (item % n_groups) * C + (int)crank, sl = item / n_groups;
                long long r0, r1, step;
                const int ntiles = item_geom(sl, r0, r1, step);
                for (int t = 0; t < ntiles; ++t) {
                    for (int kb = 0; kb < nkb; ++kb) {
                        mbar_wait(empty_bar(stage), phase ^ 1u);
                        mbar_expect_tx(full_bar(stage), (RF_DBG(a, 4) ? 0 : kABytes) + (RF_DBG(a, 8) ? 0 : kBBytes));   // own A tile + the whole B tile (C parts)
                        if (!RF_DBG(a, 4)) tma_load_2d(smA + (uint32_t)stage * kABytes, &tmA, kb * a.k_elems, qt * kGM, full_bar(stage));
                        const uint32_t bdst = smB + (uint32_t)stage * kBBytes + crank * (uint32_t)(kSubRows * kGKBytes);
                        const int brow = (int)(r0 + (long long)t * step) + (int)crank * kSubRows;
                        if (RF_DBG(a, 8)) {}
                        else if (C > 1) tma_load_2d_mc(bdst, &tmB, kb * a.k_elems, brow, full_bar(stage), cmask);
                        else tma_load_2d(bdst, &tmB, kb * a.k_elems, brow, full_bar(stage));
                        if (++stage == stages) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {   // ===== MMA issuer =====
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (int item = cluster_id; item < n_items; item += n_clusters) {
                const int sl = item / n_groups;
                long long r0, r1, step;
                const int ntiles = item_geom(sl, r0, r1, step);
                for (int t = 0; t < ntiles; ++t) {
                    mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + (uint32_t)acc * kGN;
                    for (int kb = 0; kb < nkb; ++kb) {
                        mbar_wait(full_bar(stage), phase);
                        tc_fence_after();
                        const uint64_t ad = make_smem_desc(smA + (uint32_t)stage * kABytes);
                        const uint64_t bd = make_smem_desc(smB + (uint32_t)stage * kBBytes);
#pragma unroll
                        for (int k4 = 0; k4 < kGKBytes / 32; ++k4)   // 32 B of K per instruction: +2 in 16-byte units
                            if (!RF_DBG(a, 2)) tc_mma<KIND>(d_tmem, ad + 2u * k4, bd + 2u * k4, a.idesc, (uint32_t)((kb | k4) != 0));
                        if (C > 1) tc_commit_mc(empty_bar(stage), cmask);
                        else tc_commit(empty_bar(stage));
                        if (++stage == stages) { stage = 0; phase ^= 1u; }
                    }
                    tc_commit(tfull_bar(acc));
                    if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
                }
            }
        }
    } else {   // ===== epilogue: thread <-> TMEM lane <-> query =====
        const int quarter = warp & 3;               // a warp may only touch TMEM lanes [32*(warp%4), +32)
        const int m = quarter * 32 + lane;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int item = cluster_id; item < n_items; item += n_clusters) {
            const int qt = (item % n_groups) * C + (int)crank, sl = item / n_groups;
            long long r0, r1, step;
            const int ntiles = item_geom(sl, r0, r1, step);
            const int q = qt * kGM + m;
            const int qc = q < a.nq ? q : a.nq - 1;
            CandState st;
            st.cnt = 0;
            st.minpos = 0;
            st.tau_key = 0;
            st.tau_s = q < a.nq ? -INFINITY : INFINITY;   // padding lanes of a partial query tile never collect
            st.gptr = (MODE == 0 && q < a.nq) ? a.gtau + q : nullptr;
            st.allow = a.allow;
            float tile_mx = -INFINITY;   // MODE 2: maximum over the block's sample tiles
            const float thr3 = (MODE == 3 && q < a.nq) ? __ldg(a.thr + qc) : INFINITY;   // padding lanes never append
            const float hi3 = (MODE == 3 && a.whi != nullptr) ? __ldg(a.whi + qc) : INFINITY;
            const float cap2 = (MODE == 2 && a.wcap != nullptr) ? __ldg(a.wcap + qc) : INFINITY;
            uint32_t* const cnt3 = MODE == 3 ? a.cnt + qc : nullptr;
            u64* const buf3 = MODE == 3 ? a.cand + (size_t)qc * a.cap : nullptr;
            uint32_t g_next = MODE != 0 ? 0u : __ldcg(a.gtau + qc);
            for (int t = 0; t < ntiles; ++t) {
                if (MODE == 0) {   // bound published by the other CTAs sweeping this query (loaded one tile ahead)
                    const uint32_t g = g_next;
                    if (g && q < a.nq) st.tau_s = fmaxf(st.tau_s, ordered_to_float(g));
                }
                mbar_wait(tfull_bar(acc), acc_phase);
                tc_fence_after();
                if (MODE == 0) g_next = __ldcg(a.gtau + qc);
                const long long trow = r0 + (long long)t * step;
                const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)acc * kGN;
                const int valid = r1 - trow < kGN ? (int)(r1 - trow) : kGN;   // rows of this tile inside the corpus
                uint32_t vb[2][32];
                if (RF_DBG(a, 1)) { tc_fence_before(); mbar_arrive(tempty_bar(acc)); if (++acc == 2) { acc = 0; acc_phase ^= 1u; } continue; }
                tmem_ld32_async(taddr, vb[0]);
#pragma unroll 2   // two chunks per iteration keep vb[c & 1] in fixed registers; a full unroll is 138 KB of code
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
                            if (c * 32 + j >= valid) v[j] = 0x7FC00000u;   // NaN: fails every >= test, ignored by fmaxf
                    }
                    if (MODE == 2 && a.allow != nullptr && c * 32 < valid) {
                        // bound pass over a masked corpus (tombstones): excluded rows must not raise a block maximum.  Tiles
                        // start at multiples of kGN, so the chunk's 32 rows are exactly one mask word.
                        const uint32_t w = __ldg(a.allow + ((trow + c * 32) >> 5));
                        if (w != 0xFFFFFFFFu) {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (!((w >> j) & 1u)) v[j] = 0x7FC00000u;
                        }
                    }
                    if (MODE == 2 && cap2 < INFINITY) {
                        // range search: a sample row that may score above range_filter must not raise a block maximum
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (__uint_as_float(v[j]) > cap2) v[j] = 0x7FC00000u;
                    }
                    // maxima of the four groups of 8 columns, then of the chunk: one compare in the common case
                    float gmx[4];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        float t = fmaxf(__uint_as_float(v[g * 8]), __uint_as_float(v[g * 8 + 1]));
#pragma unroll
                        for (int j = 2; j < 8; ++j) t = fmaxf(t, __uint_as_float(v[g * 8 + j]));
                        gmx[g] = t;
                    }
                    const float mx = fmaxf(fmaxf(gmx[0], gmx[1]), fmaxf(gmx[2], gmx[3]));
                    if (MODE == 2) { tile_mx = fmaxf(tile_mx, mx); continue; }
                    if (MODE == 3) {
                        if (mx >= thr3) {
#pragma unroll
                            for (int g = 0; g < 4; ++g) {
                                if (gmx[g] >= thr3) {
#pragma unroll
                                    for (int j = 0; j < 8; ++j) {
                                        const float sc = __uint_as_float(v[g * 8 + j]);
                                        const long long row = trow + c * 32 + g * 8 + j;
                                        // one atomic per appended row (measured: reserving slots in blocks is no faster); a
                                        // masked (tombstoned) row, or one above a range search's ceiling, never takes a slot
                                        if (sc >= thr3 && sc <= hi3 && (a.allow == nullptr || row_allowed(a.allow, row))) {
                                            const uint32_t pos = atomicAdd(cnt3, 1u);
                                            if (pos < (uint32_t)a.cap) buf3[pos] = make_key(sc + 0.0f, (uint32_t)row);
                                        }
                                    }
                                }
                            }
                        }
                        continue;
                    }
                    if (mx >= st.tau_s) {          // rare per thread; every v[j] stays in its register
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            if (gmx[g] >= st.tau_s) {
#pragma unroll
                                for (int j = 0; j < 8; ++j) {
                                    const float sc = __uint_as_float(v[g * 8 + j]);
                                    if (sc >= st.tau_s) cand_insert(st, lists, m, kp, sc, (uint32_t)(trow + c * 32 + g * 8 + j));
                                }
                            }
                        }
                    }
                }
                tc_fence_before();
                mbar_arrive(tempty_bar(acc));
                if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
            }
            if (MODE == 2 && q < a.nq) a.dump[(size_t)q * a.S + sl] = tile_mx;
            if (MODE == 0 && q < a.nq) {
                u64* out = a.cand + ((size_t)q * a.S + sl) * kp;
                for (int e = 0; e < kp; ++e) out[e] = e < st.cnt ? lists[(size_t)e * kGM + m] : 0ull;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (C > 1) cluster_sync_all();   // nobody leaves while a peer may still multicast into it or arrive on its barriers
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// ---- bound pass, second half: the rank-th largest (1-based) of the query's nb <= 1024 block maxima ---
// gtau != null (list mode): gtau[q] = that value as an ordered uint.
// thr  != null (append mode): thr[q] = value - 2 * (eps_const + eps_q[q]) - 2^-22, cnt[q] = 0.  Every row whose
//   exact score can be among the k best has an approximate score >= thr[q]:  exact_k >= approx_k - eps and
//   approx >= exact - eps, and value <= approx_k (rank = k).
__global__ void __launch_bounds__(256) bound_select_kernel(const float* __restrict__ bmax, int nb, int rank,
                                                           uint32_t* __restrict__ gtau, float* __restrict__ thr,
                                                           uint32_t* __restrict__ cnt, float eps_const,
                                                           const float* __restrict__ eps_q, const float* __restrict__ wlo) {
    __shared__ uint32_t v[1024];
    __shared__ uint32_t hist[256];
    __shared__ uint32_t s3[3];
    const int q = blockIdx.x;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) v[i] = float_to_ordered(bmax[(size_t)q * nb + i] + 0.0f);
    __syncthreads();
    const uint32_t mine = block_kth_largest([&](int i) { return v[i]; }, nb, (uint32_t)rank, hist, s3);
    if (threadIdx.x == 0) {
        if (cnt != nullptr) cnt[q] = 0u;
        if (gtau != nullptr) gtau[q] = mine;
        if (thr != nullptr) {
            const float e = eps_const + (eps_q ? eps_q[q] : 0.0f);
            const float t = __fsub_rd(__fsub_rd(ordered_to_float(mine), __fmul_ru(2.0f, e)), 2.384185791015625e-07f);
            thr[q] = wlo != nullptr ? fmaxf(t, wlo[q]) : t;   // range search: no row below the floor is worth a slot
        }
    }
}

// ---- per-query words of a range search (DESIGN.md 7c), radius < score <= range_filter.  e = eps_const + eps_q[q] + 2^-22
// bounds |approx - exact| with the fp32 rounding of the exact score to spare (directed rounding keeps every word safe):
//   lo  = radius - e        every row of the window has approx >= lo
//   hi  = range_filter + e  every row of the window has approx <= hi
//   cap = range_filter - e  a row with approx <= cap is certainly at or below range_filter
// Open bounds stay infinite.  Layout: w[0 .. nq) lo, w[nq .. 2 nq) hi, w[2 nq .. 3 nq) cap. ---------------------------------
__global__ void __launch_bounds__(128) window_words_kernel(int nq, float radius, float range_filter, float eps_const,
                                                           const float* __restrict__ eps_q, float* __restrict__ w) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const float e = __fadd_ru(__fadd_ru(eps_const, eps_q ? eps_q[q] : 0.0f), 2.384185791015625e-07f);
    w[q] = __fsub_rd(radius, e);
    w[nq + q] = __fadd_ru(range_filter, e);
    w[2 * nq + q] = __fsub_rd(range_filter, e);
}

// ---- query preparation for the tensor-core path, one launch: normalise (bit-identical to ingest_kernel<0>), zero-pad
// to whole query tiles, round to the storage type with the rounding error eps_q = |qhat - q16|_2, reset the per-batch
// flag counter and the published thresholds.  DT = storage type of the corpus (0: fp32, no 16-bit copy). ------------
template <int DT>
__global__ void __launch_bounds__(256) prep_queries_kernel(const float* __restrict__ q, int nq, int n_pad, int dim, int ld,
                                                           float* __restrict__ qhat, typename Store<DT>::T* __restrict__ q16,
                                                           float* __restrict__ eps_q, int* __restrict__ flag_count,
                                                           uint32_t* __restrict__ gtau) {
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (blockIdx.x == 0 && threadIdx.x == 0) *flag_count = 0;
    if (row >= n_pad) return;
    float* out = qhat + (size_t)row * ld;
    if (row >= nq) {   // padding row of the last query tile
        for (int i = lane; i < ld; i += kWarp) {
            out[i] = 0.0f;
            if (DT != 0) q16[(size_t)row * ld + i] = Store<DT>::from_f32(0.0f);
        }
        return;
    }
    const float* x = q + (size_t)row * dim;
    double acc = 0.0;
    for (int i = lane; i < dim; i += kWarp) {
        const double v = (double)x[i];
        acc = acc + v * v;
    }
    const double n2 = warp_butterfly_f64(acc);
    const double inv = inv_norm(n2);
    double d2 = 0.0;
    for (int i = lane; i < ld; i += kWarp) {
        const float y = i < dim ? norm_elem(x[i], inv) : 0.0f;
        out[i] = y;
        if (DT != 0) {
            const typename Store<DT>::T r = Store<DT>::from_f32(y);
            q16[(size_t)row * ld + i] = r;
            const double d = (double)y - (double)Store<DT>::to_f32(r);
            d2 += d * d;
        }
    }
    d2 = warp_butterfly_f64(d2);
    if (lane == 0) {
        eps_q[row] = DT != 0 ? (float)(sqrt(d2) * 1.0078125) + 1e-9f : 0.0f;   // * max |stored row| (<= 1 + 2^-8), rounded up
        gtau[row] = 0u;
    }
}

// ---- query conversion for the f16-kind path: q16 = RNE(qhat), eps_q = |qhat - q16|_2 ------------------
template <int DT>
__global__ void __launch_bounds__(256) qconv_kernel(const float* __restrict__ qhat, int nq, int ld,
                                                    typename Store<DT>::T* __restrict__ q16, float* __restrict__ eps_q) {
    const int lane = threadIdx.x & 31;
    const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= nq) return;
    double acc = 0.0;
    for (int i = lane; i < ld; i += kWarp) {
        const float x = qhat[(size_t)q * ld + i];
        const typename Store<DT>::T r = Store<DT>::from_f32(x);
        q16[(size_t)q * ld + i] = r;
        const double d = (double)x - (double)Store<DT>::to_f32(r);
        acc += d * d;
    }
    acc = warp_butterfly_f64(acc);
    if (lane == 0) eps_q[q] = (float)(sqrt(acc) * 1.0078125) + 1e-9f;   // * max |stored row| (<= 1 + 2^-8), rounded up
}

}  // namespace rfk
