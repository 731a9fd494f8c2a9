// K3f: the whole small-batch search in ONE kernel (<= 64 queries, k <= 128; by default <= 16 queries and queries x k <= 400,
// the measured crossover) - query preparation, tensor-core sweep with self-tightening thresholds, exact finalize and, on a
// row-sharded corpus, the cross-GPU exchange and reduce.  sm_100a only.
//
// Round 1 served these batches with seven launches (query prep, bound sweep, bound select, sweep, append finalize, two gated
// tier-2 launches): 65-90 us of latency-bound head and tail around a 0.27-2.1 ms sweep, which is what held the 8-GPU
// strong-scaling efficiency at 0.74.  Here:
//
//   prologue   every CTA prepares the queries itself: one warp per query computes 1 / |q| with the canonical fp64 reduction,
//              then all threads scale 16-byte chunks exactly as ingest does and store them straight into shared memory in the
//              tensor core's K-major SWIZZLE_128B layout, while the TMA producer already has a ring-full of corpus bytes in
//              flight.  16-bit storage: every query enters as TWO columns, hi = round(q) and lo = round(q - hi), summed in
//              the epilogue, so the query term of the error bound drops from ~1.6e-3 to an a-priori 2^-18 (SPLIT).
//   sweep      as gemm_rows.cuh: corpus rows are the MMA's M (two 128-row halves per 256-row tile), the query block its
//              N = 16 / 32 / 64, P partial accumulators per half so that no MMA waits on its predecessor.  Tiles of a slice are
//              visited in a strided permutation starting mid-slice, so a corpus sorted by similarity cannot make every row
//              beat the running bound.
//   threshold  NO bound pass.  A row is appended to its query's buffer when approx >= thr[q]; thr[q] starts at -inf and only
//              rises, always from a value that k DISTINCT rows are known to reach (a lower bound of T, the k-th best
//              approximate score), minus 2 eps: (1) the CTA's own sorted list of the k best scores it has appended; (2) the
//              best such full bound of ANY CTA, one atomicMax word per query (on a templated corpus one CTA holds the whole
//              answer); (3) G = 16 words per query, word g = max over the CTAs of group g of their ceil(k / G)-th best: the
//              MINIMUM of the G words is a bound (G different CTAs, ceil(k / G) distinct rows each) and a far tighter one for
//              large k.  Every row of the exact top-k has approx >= T - 2 eps >= thr whenever it is scored, so it is in the
//              buffer (DESIGN.md 2.4 / 2.5).  The CTA's FIRST tile is observed before anything is appended (with thr = -inf
//              148 x 256 rows per query would land on one counter): its scores go to shared memory, one warp per query finds
//              its k best, the bounds are published and, after a bounded rendezvous, the tile is appended against the best
//              bound of the grid.  Per-query bookkeeping is warp-cooperative (epilogue warp w owns queries w, w + 4, ...).
//   finalize   the last nq CTAs to bump the grid's arrival counter wait for it and finalize one query each: the buffer is
//              pre-filtered with the CTA's own final threshold and staged in shared memory (the ring is free), T by rank
//              counting or a shared-memory radix select, gather above T - 2 eps, canonical fp64 rescore (two rows in flight
//              per warp), rank sort, emit.  A buffer that overflowed (> cap rows ever within reach of the top k: massive
//              duplication) is answered by the same CTA with a canonical scan of the whole corpus - slow, exact, no launch.
//   exchange   row-sharded corpora (one process per GPU): the finalizing CTA stores its k exact hits straight into every
//              rank's gather area over NVLink (CUDA IPC mappings), publishes a per-(rank, query) flag with st.release.sys,
//              waits for the W flags of its own area, merges the W x k hits by rank counting and writes the GLOBAL top-k - a
//              sharded search is this one kernel per GPU, no collective call.
//   pipelining asynchronous entry points launch with programmatic stream serialization and the kernel releases its
//              dependents when it starts: the next search's CTAs take over SMs as this one's finish, so back-to-back
//              searches overlap one search's tail with the next one's sweep.  Consecutive searches alternate between two
//              halves of the workspace; every search leaves its control block zeroed.
#pragma once
#include "gemm_rows.cuh"

namespace rfk {

constexpr int kFMaxQ = 64;        // queries per launch
constexpr int kFThreads = 192;    // warp 0 producer, warp 1 MMA issuer, warps 2-5 epilogue; all six in prologue and finalize
constexpr int kFMaxK = 128;       // sorted per-CTA lists live in shared memory
constexpr int kFGroups = 16;      // CTA groups of the shared bound (see "threshold" above)
constexpr int kObsQ = 16;         // queries observed at a time in a CTA's first tile ...
constexpr int kObsStride = kGN + 1;   // ... [kObsQ][256 (+1: bank spread)] ordered scores in the pending area

struct FusedCtl {
    uint32_t cnt[kFMaxQ];     // rows appended per query (may exceed cap: overflow)
    uint32_t gthr[kFMaxQ][kFGroups + 1];   // published bounds per query, float_to_ordered (0 = none yet): one word per CTA group
                                           // (each CTA's ceil(k / G)-th best) and, in slot kFGroups, the best FULL bound of any CTA
                                           // (its own k-th best): on clustered data one CTA holds the whole answer
    uint32_t done;            // CTAs that have finished their sweep
    uint32_t obs_done;        // CTAs that have observed their first tile and published its bound
    uint32_t fin_done;        // finalizing CTAs that have finished
    uint32_t n_done;          // searches that have completely finished with this control block (pipelined launches, see below)
    uint32_t last_cnt[kFMaxQ];   // diagnostics of the last search: rows appended per query ...
    uint32_t last_resc[kFMaxQ];  // ... and rows rescored exactly (0xFFFFFFFF: the query took the exact scan)
    float cta_thr[160];          // diagnostics: every CTA's final threshold of query 0 ...
    uint32_t cta_app[160];       // ... and the rows it appended for query 0
    unsigned long long t[16];    // globaltimer stamps of the last search (ns): CTA 0: start, prologue done, first tile done,
                                 // sweep done; finalizer of query 0: all CTAs arrived, hits selected, rescored, emitted;
                                 // [8..]: finer stamps (setup done, norms done; count read, keys staged, T found)
};
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Queries of a small synchronous host call travel INSIDE the launch (kernel parameter space) instead of through a copy-engine
// transfer in front of the kernel: up to kFInlineFloats floats (4 queries of 768, 3 of 1024).
constexpr int kFInlineFloats = 3072;
struct alignas(16) FusedInlineQ { float v[kFInlineFloats]; };   // 16-byte aligned: the prologue reads it with 128-bit loads

struct FusedArgs {
    uint32_t idesc;             // M = 128, N = NCOL
    int num_kblocks, k_elems;   // k-blocks of 128 bytes; elements per k-block (64 for 16-bit storage, 32 for fp32)
    int dt;                     // type of `data`, the rows the exact rescore reads: 0 fp32, 1 bf16, 2 fp16
    int sdt;                    // type of the rows tmB sweeps (the 16-bit query split follows it): = dt, except 2 on an fp32
                                // collection with an fp16 copy (RAGFIN_F32_F16)
    int nq, dim, ld;
    long long n_rows;
    int S;                      // corpus slices
    long long rows_per_slice;   // multiple of kGN
    int stages;
    int k, keff;                // keff = min(k, rows a hit may come from)
    int pend;                   // pending-score slots per query and tile
    int groups, grank;          // CTA groups of the shared bound and the rank each CTA publishes: ceil(keff / groups)
    uint32_t seq_on_half;       // searches launched on this half of the double-buffered workspace before this one
    int refresh_every;          // thresholds are re-read from the grid every tile for the first 8 tiles of a slice, then every n-th
                                // tile (and whenever one of the warp's own lists changed); a stale threshold only admits more rows
    const float* q;             // [nq][dim] raw fp32 queries; null: they are in the launch's FusedInlineQ parameter
    float* qn;                  // [nq][ld] workspace: the normalised fp32 queries (written by CTA 0, read by the finalizers)
    const void* data;           // corpus [n_rows][ld]
    const uint32_t* allow;      // scalar filter bitmask or null
    u64* cand;                  // [nq][cap] append buffers
    int cap;
    FusedCtl* ctl;
    float eps_const;            // accumulation allowance (+ tf32 truncation, + the fp16 copy's rounding), see eps_approx
    long long id_base;
    long long* out_ids;         // [nq][k]
    float* out_scores;          // [nq][k]
    int* flags;                 // [nq] 1 = the query took the in-kernel exact scan
    int* flag_count;
    uint32_t* host_flag;        // synchronous host calls: device-mapped pinned word the last finalizer sets to host_seq once every
    uint32_t host_seq;          //   query's hits are in the (mapped) output buffers - the host polls it instead of waiting for the stream
    // cross-shard exchange inside the finalize (row-sharded corpora, one process per GPU; xworld <= 1: off).  Peer gather
    // areas and flags are mapped through CUDA IPC (ragfin_exchange_*); see "exchange" in the header comment.
    int xworld, xrank;
    uint32_t xstep;             // step number of this search: flag value, xstep % kXSlots selects the slot of the gather ring
    unsigned long long xrec_max;   // bytes of one rank's record in a gather area
    char* const* xpeer_area;    // [xworld] base of every rank's gather area: [kXSlots][xworld][xrec_max]
    uint32_t* const* xpeer_qflag;  // [xworld] base of every rank's per-query flags: [kXSlots][xworld][kFMaxQ]
};

// pending area: [nq][pend] appended scores per tile in steady state, [kObsQ][kObsStride] observed scores in the first tile
__host__ __device__ constexpr size_t fused_pend_words(int nq, int pend) {
    return (size_t)nq * pend > (size_t)kObsQ * kObsStride ? (size_t)nq * pend : (size_t)kObsQ * kObsStride;
}
__host__ __device__ constexpr size_t fused_state_bytes(int nq, int k, int pend) {
    return (size_t)6 * kFMaxQ * 4 + ((size_t)nq * k + fused_pend_words(nq, pend)) * 4 + 64;
}
__host__ __device__ constexpr size_t fused_smem_bytes(int num_kblocks, int ncol, int stages, int nq, int k, int pend) {
    return 1024 + (size_t)num_kblocks * ncol * kGKBytes + (size_t)stages * kBBytes + 256 + fused_state_bytes(nq, k, pend);
}

__device__ __forceinline__ void named_bar_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
// named barrier that also ORs a flag over its threads (one instruction: "did any thread of the epilogue append this tile?")
__device__ __forceinline__ bool named_bar_or(int id, int threads, bool flag) {
    uint32_t out;
    asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 q, %1, 0;\n\tbar.red.or.pred p, %2, %3, q;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(out) : "r"((uint32_t)flag), "r"(id), "r"(threads) : "memory");
    return out != 0u;
}
// tcgen05.ld without the wait: several loads in flight, then ONE tmem_ld_wait(), then tmem_ld_fence16() on every destination
// array (an empty volatile asm that names the registers in/out: no use of them can be scheduled above the wait).
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_fence16(uint32_t (&r)[16]) {
    asm volatile("" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                      "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]) :: "memory");
}
__device__ __forceinline__ uint32_t ld_acq_gpu(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// thr = value - 2 eps - 2^-22, every step rounded down (never above the real bound)
__device__ __forceinline__ float thr_below(float value, float eps) {
    return __fsub_rd(__fsub_rd(value, __fmul_ru(2.0f, eps)), 2.384185791015625e-07f);
}

// Tiles of a slice are visited in the order perm_tile(t) = (n / 2 + t * mult) % n: a stride near 0.618 n (coprime with n, so
// every tile is visited once) starting in the middle, so that the first few tiles sample the whole slice - on a corpus sorted
// by similarity a sequential sweep would see every row beat the running k-th score.
__host__ __device__ __forceinline__ int perm_tile(int t, int mult, int n) { return (int)(((long long)t * mult + n / 2) % n); }
// multiplier of the tile permutation: odd, near 0.618 n, coprime with n
__host__ __device__ __forceinline__ int perm_mult(int n) {
    if (n <= 2) return 1;
    int m = (int)(0.6180339887 * n) | 1;
    for (;; m += 2) {
        int x = m % n, y = n;
        if (x == 0) continue;
        while (x) { const int t = y % x; y = x; x = t; }
        if (y == 1) return m % n;
    }
}

// canonical_dot_row (common.cuh) for two rows at once: the same per-lane order of fp64 adds for each row (bit-identical
// results), both rows' loads issued before either chain of adds starts
template <int DT>
__device__ __forceinline__ void canonical_dot_two_rows(const void* data, uint32_t row_a, uint32_t row_b, int ld, const float* q, int lane,
                                                       double& out_a, double& out_b) {
    const typename Store<DT>::T* pa = reinterpret_cast<const typename Store<DT>::T*>(data) + (size_t)row_a * ld;
    const typename Store<DT>::T* pb = reinterpret_cast<const typename Store<DT>::T*>(data) + (size_t)row_b * ld;
    double acc_a = 0.0, acc_b = 0.0;
    int i = lane;
    for (; i + 23 * kWarp < ld; i += 24 * kWarp) {
        float xa[24], xb[24];
#pragma unroll
        for (int u = 0; u < 24; ++u) { xa[u] = Store<DT>::to_f32(pa[i + u * kWarp]); xb[u] = Store<DT>::to_f32(pb[i + u * kWarp]); }
#pragma unroll
        for (int u = 0; u < 24; ++u) {
            const double qd = (double)q[i + u * kWarp];
            acc_a = acc_a + (double)xa[u] * qd;
            acc_b = acc_b + (double)xb[u] * qd;
        }
    }
#pragma unroll 4
    for (; i < ld; i += kWarp) {
        const double qd = (double)q[i];
        acc_a = acc_a + (double)Store<DT>::to_f32(pa[i]) * qd;
        acc_b = acc_b + (double)Store<DT>::to_f32(pb[i]) * qd;
    }
    out_a = warp_butterfly_f64(acc_a);
    out_b = warp_butterfly_f64(acc_b);
}

template <int KIND, int NCOL, bool SPLIT>
__global__ void __launch_bounds__(kFThreads, 1)
sweep_fused_kernel(const __grid_constant__ CUtensorMap tmB, const FusedArgs a, const __grid_constant__ FusedInlineQ qin) {
    const float* const qsrc = a.q != nullptr ? a.q : qin.v;
    constexpr int P = NCOL <= 32 ? 4 : 2;                      // partial accumulators per half tile
    constexpr int kAcc = 2 * P * NCOL;                         // TMEM columns of one tile buffer
    constexpr int kTmemCols = 2 * kAcc <= 256 ? 256 : 512;
    constexpr int QPC = SPLIT ? 8 : 16;                        // queries per 16-column chunk
    constexpr int QTILE = NCOL * kGKBytes;                     // bytes of one k-block of the query block
    static_assert(2 * kAcc <= 512, "accumulators exceed tensor memory");
    static_assert(!(SPLIT && KIND == 1), "the hi/lo split is for 16-bit storage");

    extern __shared__ uint8_t fsm_raw[];
    const uint32_t raw = smem_u32(fsm_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* fsm = fsm_raw + (base - raw);
    const int stages = a.stages, nkb = a.num_kblocks, nq = a.nq, k = a.k;
    const uint32_t smQ = base;                                             // [nkb][NCOL x 128 B]
    const uint32_t smB = base + (uint32_t)nkb * QTILE;                     // [stages][32 KB]
    const size_t region_bytes = (size_t)nkb * QTILE + (size_t)stages * kBBytes;   // reused as scratch by the finalize
    uint64_t* bars = reinterpret_cast<uint64_t*>(fsm + region_bytes);
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (kRMaxStages + s); };
    auto tfull_bar = [&](int s) { return bar0 + 8u * (2 * kRMaxStages + s); };
    auto tempty_bar = [&](int s) { return bar0 + 8u * (2 * kRMaxStages + 2 + s); };
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kRMaxStages + 4);
    uint32_t* s_ticket = tmem_slot + 1;
    int* s_app = reinterpret_cast<int*>(tmem_slot + 2);    // diagnostics: rows this CTA appended for query 0
    // per-query threshold state
    float* thr_s = reinterpret_cast<float*>(fsm + region_bytes + 256);     // [kFMaxQ]
    float* eps_s = thr_s + kFMaxQ;                                          // [kFMaxQ]
    int* scnt = reinterpret_cast<int*>(eps_s + kFMaxQ);                     // [kFMaxQ] entries of sorted[q]
    int* pcnt = scnt + kFMaxQ;                                              // [kFMaxQ] entries appended to pend[q] this tile
    uint32_t* pub_s = reinterpret_cast<uint32_t*>(pcnt + kFMaxQ);           // [kFMaxQ] what this CTA last published for the query
    uint32_t* pubf_s = pub_s + kFMaxQ;                                      // [kFMaxQ] ... and its last published full bound
    uint32_t* sorted = pubf_s + kFMaxQ;                                     // [nq][k] descending ordered-uint scores
    uint32_t* pend = sorted + (size_t)nq * k;                               // [nq][pend]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // Pipelined launches (programmatic stream serialization, see run_fused): the NEXT search's grid may be scheduled as soon as
    // every CTA of this one has started, so its CTAs take over the SMs one by one as this search's CTAs finish their slices -
    // the prologue, the tail skew, the finalize and the exchange of one search overlap the sweep of the next, and HBM never
    // idles between back-to-back searches.  Consecutive searches alternate between two halves of the workspace and never read
    // each other's; the only shared thing is the caller's output buffer, ordered by griddepcontrol.wait before the emit.
    if (tid == 0) {
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        // the search before the previous one used this half: it must be completely done with it (it always is when the grid
        // fills the device - its last CTA has to exit before the previous search's last CTA can even start)
        while (ld_acq_gpu(&a.ctl->n_done) != a.seq_on_half) __nanosleep(200);
    }
    if (blockIdx.x == 0 && tid == 0) { a.ctl->t[0] = global_ns(); a.ctl->t[13] = 0; a.ctl->t[14] = 0; a.ctl->t[15] = 0; }
    // the prologue's first global accesses are the queries (cold): start pulling them in while barriers and tensor memory are set up
    if (a.q != nullptr)
        for (int ln = tid; ln * 32 < a.nq * a.dim; ln += kFThreads) asm volatile("prefetch.global.L1 [%0];" ::"l"(a.q + (size_t)ln * 32));
    if (tid == 0) {
        for (int s = 0; s < stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 128); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < kFMaxQ; i += kFThreads) { thr_s[i] = i < nq ? -INFINITY : INFINITY; eps_s[i] = 0.f; scnt[i] = 0; pcnt[i] = 0; pub_s[i] = 0u; pubf_s[i] = 0u; }
    if (tid == 0) *s_app = 0;
    if (blockIdx.x == 0 && tid == 0) *a.flag_count = 0;   // ordered before every finalizer's atomicAdd by the arrival counter
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (blockIdx.x == 0 && tid == 0) a.ctl->t[8] = global_ns();

    auto slice_tiles = [&](int sl, long long& r0, long long& r1) -> int {
        r0 = (long long)sl * a.rows_per_slice;
        r1 = r0 + a.rows_per_slice;
        if (r1 > a.n_rows) r1 = a.n_rows;
        return r1 > r0 ? (int)((r1 - r0 + kGN - 1) / kGN) : 0;
    };

    // ---- the producer gets the first ring-full of corpus bytes moving before anybody touches a query ----
    int pre_issued = 0;
    if (tid == 0) {
        long long r0, r1;
        const int ntiles = slice_tiles(blockIdx.x, r0, r1);
        const int mult = perm_mult(ntiles);
        for (int it = 0; it < stages && it < ntiles * nkb; ++it) {
            const int t = it / nkb, kb = it % nkb;
            const int tp = perm_tile(t, mult, ntiles);
            mbar_expect_tx(full_bar(it), kBBytes);
            tma_load_2d(smB + (uint32_t)it * kBBytes, &tmB, kb * a.k_elems, (int)(r0 + (long long)tp * kGN), full_bar(it));
            ++pre_issued;
        }
    }

    // ---- prologue: the query block, written in place in the K-major SWIZZLE_128B layout ----
    {
        uint4* qz = reinterpret_cast<uint4*>(fsm);
        for (int i = tid; i < nkb * QTILE / 16; i += kFThreads) qz[i] = make_uint4(0u, 0u, 0u, 0u);
        __syncthreads();
        const int esz = KIND == 1 ? 4 : 2;
        // pass 1, one warp per query: canonical sum of squares -> 1 / |q| (fp64), parked in the pending area
        double* inv_s = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(pend) + 7) & ~(uintptr_t)7);   // [nq]
        for (int j = warp; j < nq; j += kFThreads / 32) {
            const float* x = qsrc + (size_t)j * a.dim;
            double acc = 0.0;
            for (int i0 = lane; i0 < a.dim; i0 += 24 * kWarp) {     // 24 loads in flight (a 768-wide query: one round trip);
                float xv[24];                                       // the adds stay in increasing-i order
#pragma unroll
                for (int u = 0; u < 24; ++u) xv[u] = i0 + u * kWarp < a.dim ? x[i0 + u * kWarp] : 0.0f;
#pragma unroll
                for (int u = 0; u < 24; ++u) { const double v = (double)xv[u]; acc = acc + v * v; }   // + 0 for the tail: exact
            }
            const double n2 = warp_butterfly_f64(acc);
            if (lane == 0) inv_s[j] = inv_norm(n2);
        }
        __syncthreads();
        if (blockIdx.x == 0 && tid == 0) a.ctl->t[9] = global_ns();
        if (blockIdx.x == 0 && a.ld > a.dim)
            for (int i = tid; i < nq * (a.ld - a.dim); i += kFThreads) a.qn[(size_t)(i / (a.ld - a.dim)) * a.ld + a.dim + i % (a.ld - a.dim)] = 0.0f;
        // pass 2, all threads: y = RNE_f32(x / |q|) exactly as ingest does, hi / lo split, swizzled store
        constexpr int VE = KIND == 1 ? 4 : 8;                     // elements of one 16-byte chunk of a query row
        if (a.dim % VE == 0 && (reinterpret_cast<uintptr_t>(qsrc) & 15u) == 0) {
            // fast path: one thread per 16-byte chunk (8 bf16 / fp16 or 4 fp32 elements): 128-bit loads, one 128-bit swizzled
            // store for the hi row and one for the lo row
            constexpr int KE = KIND == 1 ? 32 : 64;
            const int cpq = a.dim / VE;                            // chunks per query
            const int total = nq * cpq;
            for (int ch0 = 0; ch0 < total; ch0 += 2 * kFThreads) {
                float xv[2][8];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int ch = ch0 + u * kFThreads + tid;
#pragma unroll
                    for (int v4 = 0; v4 < VE / 4; ++v4) {
                        const float4 f = ch < total ? reinterpret_cast<const float4*>(qsrc)[(size_t)ch * (VE / 4) + v4] : make_float4(0.f, 0.f, 0.f, 0.f);
                        xv[u][4 * v4] = f.x; xv[u][4 * v4 + 1] = f.y; xv[u][4 * v4 + 2] = f.z; xv[u][4 * v4 + 3] = f.w;
                    }
                }
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int ch = ch0 + u * kFThreads + tid;
                    const bool live = ch < total;
                    const int j = live ? ch / cpq : 0, i = (ch - j * cpq) * VE;     // query, first element of the chunk
                    if (live) {
                        const double inv = inv_s[j];
                        const int row_hi = SPLIT ? (j >> 3) * 16 + (j & 7) : j;
                        const int kb = i / KE, cc = ((i % KE) * esz) >> 4;           // k-block, 16-byte chunk inside the 128-byte row
                        uint8_t* p_hi = fsm + (size_t)kb * QTILE + (size_t)(row_hi >> 3) * 1024 + (size_t)(row_hi & 7) * 128 + ((cc ^ (row_hi & 7)) << 4);
                        float y[VE];
#pragma unroll
                        for (int e = 0; e < VE; ++e) y[e] = norm_elem(xv[u][e], inv);
                        if (blockIdx.x == 0) {
#pragma unroll
                            for (int e = 0; e < VE; e += 4) *reinterpret_cast<float4*>(a.qn + (size_t)j * a.ld + i + e) = make_float4(y[e], y[e + 1], y[e + 2], y[e + 3]);
                        }
                        if (KIND == 1) {
                            *reinterpret_cast<float4*>(p_hi) = make_float4(y[0], y[1], y[2], y[3]);
                        } else {
                            uint32_t hw[4], lw[4];
#pragma unroll
                            for (int e = 0; e < VE; e += 2) {
                                uint16_t hb[2], lb[2];
#pragma unroll
                                for (int t2 = 0; t2 < 2; ++t2) {
                                    if (a.sdt == 1) {
                                        const __nv_bfloat16 hi = __float2bfloat16_rn(y[e + t2]);
                                        const float rest = y[e + t2] - __bfloat162float(hi);             // exact
                                        const __nv_bfloat16 lo = SPLIT ? __float2bfloat16_rn(rest) : __float2bfloat16_rn(0.f);
                                        hb[t2] = __bfloat16_as_ushort(hi); lb[t2] = __bfloat16_as_ushort(lo);
                                    } else {
                                        const __half hi = __float2half_rn(y[e + t2]);
                                        const float rest = y[e + t2] - __half2float(hi);
                                        const __half lo = SPLIT ? __float2half_rn(rest) : __float2half_rn(0.f);
                                        hb[t2] = __half_as_ushort(hi); lb[t2] = __half_as_ushort(lo);
                                    }
                                }
                                hw[e >> 1] = (uint32_t)hb[0] | ((uint32_t)hb[1] << 16);
                                lw[e >> 1] = (uint32_t)lb[0] | ((uint32_t)lb[1] << 16);
                            }
                            *reinterpret_cast<uint4*>(p_hi) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
                            // the lo row is 8 MMA columns further: same position inside the next 8-row group (+1024 bytes)
                            if (SPLIT) *reinterpret_cast<uint4*>(p_hi + 1024) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
                        }
                    }
                }
            }
        } else {
            constexpr int KE = KIND == 1 ? 32 : 64;               // elements per 128-byte k-block
            constexpr int UB = 8;
            const int upq = (a.dim + kFThreads - 1) / kFThreads;  // units per query
            const int units = nq * upq;
            for (int u0 = 0; u0 < units; u0 += UB) {
                float xv[UB];
#pragma unroll
                for (int u = 0; u < UB; ++u) {
                    const int un = u0 + u, j = un / upq, i = (un - j * upq) * kFThreads + tid;
                    xv[u] = (un < units && i < a.dim) ? qsrc[(size_t)j * a.dim + i] : 0.0f;
                }
#pragma unroll
                for (int u = 0; u < UB; ++u) {
                    const int un = u0 + u;
                    if (un >= units) break;                         // block-uniform
                    const int j = un / upq, i = (un - j * upq) * kFThreads + tid;
                    if (i < a.dim) {
                        const float y = norm_elem(xv[u], inv_s[j]);
                        if (blockIdx.x == 0) a.qn[(size_t)j * a.ld + i] = y;
                        const int row_hi = SPLIT ? (j >> 3) * 16 + (j & 7) : j;
                        const int kb = i / KE, c = (i % KE) * esz;
                        uint8_t* p_hi = fsm + (size_t)kb * QTILE + (size_t)(row_hi >> 3) * 1024 + (size_t)(row_hi & 7) * 128 + ((((c >> 4) ^ (row_hi & 7)) << 4) | (c & 15));
                        if (KIND == 1) {
                            *reinterpret_cast<float*>(p_hi) = y;
                        } else {
                            // the lo row is 8 MMA columns further: same position inside the next 8-row group (+1024 bytes)
                            uint8_t* p_lo = p_hi + 1024;
                            if (a.sdt == 1) {
                                const __nv_bfloat16 hi = __float2bfloat16_rn(y);
                                const float rest = y - __bfloat162float(hi);        // exact
                                const __nv_bfloat16 lo = SPLIT ? __float2bfloat16_rn(rest) : __float2bfloat16_rn(0.f);
                                *reinterpret_cast<__nv_bfloat16*>(p_hi) = hi;
                                if (SPLIT) *reinterpret_cast<__nv_bfloat16*>(p_lo) = lo;
                            } else {
                                const __half hi = __float2half_rn(y);
                                const float rest = y - __half2float(hi);
                                const __half lo = SPLIT ? __float2half_rn(rest) : __float2half_rn(0.f);
                                *reinterpret_cast<__half*>(p_hi) = hi;
                                if (SPLIT) *reinterpret_cast<__half*>(p_lo) = lo;
                            }
                        }
                    }
                }
            }
        }
        __syncthreads();
        // |approx - exact| <= |q - hi - lo|_2 * max |stored row|_2 + the accumulation allowance.  The residual is bounded a
        // priori, element by element (round to nearest: half an ulp): bf16 keeps 8 significant bits, so |q - hi| <= 2^-9 |q|
        // and |q - hi - lo| <= 2^-18 |q|; fp16 keeps 11 (2^-12, 2^-24) but loses relative accuracy below 2^-14, where the
        // spacing is 2^-24: at most 2^-25 more per element.  |q|_2 <= 1 + 2^-22 and |row|_2 <= 1 + 2^-8: factor 1.0078125.
        {
            float eq = 0.f;
            if (KIND != 1) {
                const float rel = a.sdt == 1 ? (SPLIT ? 3.814697265625e-06f : 1.953125e-03f) : (SPLIT ? 5.9604644775390625e-08f : 2.44140625e-04f);
                const float sub = a.sdt == 1 ? 0.f : __fmul_ru(__fsqrt_ru((float)a.ld), 2.98023223876953125e-08f);
                eq = __fmul_ru(__fadd_ru(rel, sub), 1.0078125f);
            }
            for (int j = tid; j < nq; j += kFThreads) eps_s[j] = __fadd_ru(a.eps_const, eq);
        }
        __syncthreads();
        for (int i = tid; i < 2 * kFMaxQ + 2; i += kFThreads) pend[i] = 0u;   // the parking area goes back to the pending lists
        fence_proxy_async_smem();   // generic-proxy writes above -> visible to the tensor core's async-proxy reads
        __syncthreads();
        if (blockIdx.x == 0 && tid == 0) a.ctl->t[1] = global_ns();
    }

    if (warp == 0) {
        if (lane == 0) {   // ===== TMA producer =====
            int stage = 0, skip = pre_issued;
            uint32_t phase = 0;
            for (int sl = blockIdx.x; sl < a.S; sl += gridDim.x) {
                long long r0, r1;
                const int ntiles = slice_tiles(sl, r0, r1);
                const int mult = perm_mult(ntiles);
                for (int t = 0; t < ntiles; ++t) {
                    const int tp = perm_tile(t, mult, ntiles);
                    for (int kb = 0; kb < nkb; ++kb) {
                        if (skip > 0) {
                            --skip;                        // issued before the prologue (first round of the ring: slots were free)
                        } else {
                            mbar_wait(empty_bar(stage), phase ^ 1u);
                            mbar_expect_tx(full_bar(stage), kBBytes);
                            tma_load_2d(smB + (uint32_t)stage * kBBytes, &tmB, kb * a.k_elems, (int)(r0 + (long long)tp * kGN), full_bar(stage));
                        }
                        if (++stage == stages) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {   // ===== MMA issuer =====
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
                        const uint64_t qd = make_smem_desc(smQ + (uint32_t)kb * QTILE);
#pragma unroll
                        for (int k4 = 0; k4 < kGKBytes / 32; ++k4) {
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                const uint64_t cd = make_smem_desc(smB + (uint32_t)stage * kBBytes + (uint32_t)h * (kBBytes / 2));
                                const uint32_t d_tmem = tmem_base + (uint32_t)acc * kAcc + (uint32_t)h * (P * NCOL) + (uint32_t)(k4 % P) * NCOL;
                                tc_mma<KIND>(d_tmem, cd + 2u * k4, qd + 2u * k4, a.idesc, (uint32_t)(kb != 0 || k4 >= P));
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
        const int m = quarter * 32 + lane;          // row of the half tile
        const int et = tid - 64;                    // 0..127 among the epilogue threads; thread et < nq maintains query et
        const int npend = a.pend;
        int acc = 0;
        uint32_t acc_phase = 0;
        bool warm = true;                           // the CTA's first tile is observed before anything is appended
        const bool obs_holds_tile = nq <= kObsQ;    // ... and with <= kObsQ queries the observation area holds the whole tile
        // scores of the 16-column chunk c of half h of the current accumulator: QPC queries per chunk
        // the P partial accumulators of chunk c of half h: P loads in flight, no wait
        auto chunk_load = [&](int h, int c, uint32_t (&v)[P][16]) {
#pragma unroll
            for (int p = 0; p < P; ++p)
                tmem_ld16_async(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)acc * kAcc + (uint32_t)h * (P * NCOL) + (uint32_t)p * NCOL + (uint32_t)c * 16, v[p]);
        };
        auto chunk_fence = [&](uint32_t (&v)[P][16]) {
#pragma unroll
            for (int p = 0; p < P; ++p) tmem_ld_fence16(v[p]);
        };
        auto chunk_reduce = [&](const uint32_t (&v)[P][16], float (&out)[QPC]) {
            float s16[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float s = __uint_as_float(v[0][j]) + __uint_as_float(v[1][j]);
                if (P == 4) s += __uint_as_float(v[2][j]) + __uint_as_float(v[3][j]);
                s16[j] = s;
            }
#pragma unroll
            for (int j = 0; j < QPC; ++j) out[j] = SPLIT ? s16[j] + s16[j + 8] : s16[j];
        };
        auto chunk_scores = [&](int h, int c, float (&out)[QPC]) {
            uint32_t v[P][16];
            chunk_load(h, c, v);
            tmem_ld_wait();
            chunk_fence(v);
            chunk_reduce(v, out);
        };
        // ---- per-query bookkeeping, WARP-cooperative: epilogue warp ew = warp & 3 owns the queries ew, ew + 4, ew + 8, ... ----
        // (one thread walking a sorted list in shared memory is a chain of dependent ~30-cycle accesses: measured 48 us for
        // the first tile at k = 10 and 370 us at k = 100; a warp does each step in a handful of instructions.)
        const int ew = quarter;
        const int my_group = (int)(blockIdx.x % (unsigned)a.groups);
        // want-th largest (1-based) of the 256 ordered scores ob[0..256) (0 = empty): bisection on the value bits, the count of
        // values >= candidate by one warp reduction per bit.  Returns 0 when fewer than `want` entries exist.
        auto warp_kth_of_tile = [&](const uint32_t* ob, int want) -> uint32_t {
            uint32_t v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = ob[lane + 32 * i];
            uint32_t T = 0u;
#pragma unroll 1
            for (int bit = 31; bit >= 0; --bit) {
                const uint32_t cand = T | (1u << bit);
                int c = 0;
#pragma unroll
                for (int i = 0; i < 8; ++i) c += v[i] >= cand;
                if (__reduce_add_sync(kFull, c) >= want) T = cand;
            }
            return T;
        };
        // sorted[q][0..n) := the n = min(k, valid) largest of the tile's 256 scores, descending; returns n
        auto warp_seed_list = [&](int q, const uint32_t* ob) -> int {
            uint32_t* sl_ = sorted + (size_t)q * k;
            const uint32_t T = warp_kth_of_tile(ob, k);          // k-th largest, or 0: fewer than k valid scores -> take them all
            int n = 0;
            for (int pass = 0; pass < 2; ++pass) {                 // pass 0: values > T; pass 1: values == T while room remains
#pragma unroll 1
                for (int i = 0; i < 8; ++i) {
                    const uint32_t val = ob[lane + 32 * i];
                    const bool take = val != 0u && (pass == 0 ? val > T : (val == T && T != 0u));
                    const unsigned mk = __ballot_sync(kFull, take);
                    const int pos = n + __popc(mk & ((1u << lane) - 1u));
                    if (take && pos < k) sl_[pos] = val;
                    n += __popc(mk);
                }
            }
            if (n > k) n = k;
            __syncwarp();
            // rank sort in place (n <= 128: at most 4 entries per lane, held in registers across the rewrite)
            uint32_t e[4];
            int rk[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { const int jx = lane + 32 * i; e[i] = jx < n ? sl_[jx] : 0u; rk[i] = 0; }
#pragma unroll 8
            for (int mi = 0; mi < n; ++mi) {
                const uint32_t o = sl_[mi];                        // broadcast read
#pragma unroll
                for (int i = 0; i < 4; ++i) rk[i] += (o > e[i]) || (o == e[i] && mi < lane + 32 * i);
            }
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) if (lane + 32 * i < n) sl_[rk[i]] = e[i];
            __syncwarp();
            return n;
        };
        // one appended score into the query's sorted list (n entries so far; the smallest falls off a full list); returns n
        auto warp_list_add = [&](uint32_t* sl_, int n, uint32_t val) -> int {
            if (n == k && val <= sl_[k - 1]) return n;             // warp-uniform
            uint32_t e[4];
            int c = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) { const int jx = lane + 32 * i; e[i] = jx < n ? sl_[jx] : 0u; c += jx < n && e[i] > val; }
            const int pos = __reduce_add_sync(kFull, c);           // entries that stay in front of val
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) { const int jx = lane + 32 * i; if (jx >= pos && jx < n && jx + 1 < k) sl_[jx + 1] = e[i]; }
            if (lane == 0) sl_[pos] = val;
            __syncwarp();
            return n < k ? n + 1 : k;
        };
        // New thresholds for this warp's queries: own k-th best, and the minimum over the CTA groups of what each group has
        // published (read NOW, so that the next tile is filtered with the best bound the grid has found); publishes this
        // CTA's grank-th best for its group when that improved.  Two queries per step: lanes 0-15 / 16-31 read the 16 words.
        auto warp_refresh = [&]() {
            const int half = lane >> 4, gl = lane & 15;
            uint32_t gw[kFMaxQ / 8];                               // all the loads first: ONE L2 round trip per refresh
#pragma unroll
            for (int it = 0; it < kFMaxQ / 8; ++it) {
                const int q = ew + 8 * it + 4 * half;              // this half-warp's query of step `it` (may be >= nq)
                gw[it] = (q < nq && gl < a.groups) ? __ldcg(&a.ctl->gthr[q][gl]) : 0xFFFFFFFFu;
            }
            uint32_t gfull[kFMaxQ / 8];                            // the best full bound any CTA has published (lanes 0 / 16)
#pragma unroll
            for (int it = 0; it < kFMaxQ / 8; ++it) {
                const int q = ew + 8 * it + 4 * half;
                gfull[it] = (q < nq && gl == 0) ? __ldcg(&a.ctl->gthr[q][kFGroups]) : 0u;
            }
#pragma unroll
            for (int it = 0; it < kFMaxQ / 8; ++it) {
                const int q = ew + 8 * it + 4 * half;
                if (ew + 8 * it >= nq) break;                      // warp-uniform
                uint32_t g = gw[it];
#pragma unroll
                for (int off = 8; off >= 1; off >>= 1) { const uint32_t o = __shfl_xor_sync(kFull, g, off); g = o < g ? o : g; }
                if (gl == 0 && q < nq) {
                    const uint32_t* sl_ = sorted + (size_t)q * k;
                    const int n = scnt[q];
                    const float e = eps_s[q];
                    float nt = thr_s[q];
                    if (n >= a.keff && a.keff > 0) {
                        const float own = thr_below(ordered_to_float(sl_[a.keff - 1]), e);
                        nt = fmaxf(nt, own);
                        const uint32_t po = float_to_ordered(own);
                        if (po > gfull[it] && po > pubf_s[q]) { pubf_s[q] = po; atomicMax(&a.ctl->gthr[q][kFGroups], po); }
                    }
                    if (gfull[it] != 0u) nt = fmaxf(nt, ordered_to_float(gfull[it]));
                    if (n >= a.grank && a.grank > 0) {
                        const uint32_t pv = float_to_ordered(thr_below(ordered_to_float(sl_[a.grank - 1]), e));
                        if (pv > pub_s[q]) { pub_s[q] = pv; atomicMax(&a.ctl->gthr[q][my_group], pv); __threadfence(); }
                    }
                    if (g != 0u) nt = fmaxf(nt, ordered_to_float(g));   // 0: some group has not published yet
                    thr_s[q] = nt;
                }
            }
            __syncwarp();
        };
        for (int sl = blockIdx.x; sl < a.S; sl += gridDim.x) {
            long long r0, r1;
            const int ntiles = slice_tiles(sl, r0, r1);
            const int mult = perm_mult(ntiles);
            for (int t = 0; t < ntiles; ++t) {
                const int tp = perm_tile(t, mult, ntiles);
                const long long trow = r0 + (long long)tp * kGN;
                const bool stamp_tile = blockIdx.x == 0 && et == 0;
                unsigned long long ts0 = 0, ts1 = 0, ts2 = 0;
                if (stamp_tile) ts0 = global_ns();
                mbar_wait(tfull_bar(acc), acc_phase);
                tc_fence_after();
                if (stamp_tile) ts1 = global_ns();
                // rows past the slice / corpus (zero-filled by TMA) and filtered rows never qualify
                const long long row_h0 = trow + m, row_h1 = trow + 128 + m;
                const bool ok0 = row_h0 < r1 && (a.allow == nullptr || row_allowed(a.allow, row_h0));
                const bool ok1 = row_h1 < r1 && (a.allow == nullptr || row_allowed(a.allow, row_h1));
                if (warm) {
                    // ---- the CTA's first tile, pass 1 of 2: OBSERVE.  With thr = -inf every CTA would append its whole first
                    // tile (148 x 256 rows per query, all on one counter).  Instead the tile's scores go to shared memory in
                    // groups of kObsQ queries, the query's thread builds the sorted k best of the 256, and the tile is then
                    // read a second time from tensor memory (pass 2, below) against thr = kth - 2 eps.
                    for (int q0 = 0; q0 < nq; q0 += kObsQ) {
#pragma unroll 1
                        for (int h = 0; h < 2; ++h) {
#pragma unroll 1
                            for (int c = q0 / QPC; c < (q0 + kObsQ) / QPC && c < NCOL / 16; ++c) {
                                float sc[QPC];
                                chunk_scores(h, c, sc);
#pragma unroll
                                for (int j = 0; j < QPC; ++j)
                                    pend[(size_t)(c * QPC + j - q0) * kObsStride + h * 128 + m] = (h ? ok1 : ok0) ? float_to_ordered(sc[j] + 0.0f) : 0u;
                            }
                        }
                        if (obs_holds_tile) {
                            // <= kObsQ queries: the observed scores ARE the tile.  Hand the accumulator back now - the tensor core
                            // goes on with the tile after next while the bounds are agreed on - and append from shared memory below.
                            tc_fence_before();
                            mbar_arrive(tempty_bar(acc));
                        }
                        named_bar_sync(1, 128);
                        for (int q = q0 + ew; q < q0 + kObsQ && q < nq; q += 4) {
                            const int n = warp_seed_list(q, pend + (size_t)(q - q0) * kObsStride);
                            if (lane == 0) scnt[q] = n;
                        }
                        named_bar_sync(2, 128);
                    }
                    warp_refresh();
                    // Best-effort rendezvous: all CTAs observe their first tile at the same time, so a few microseconds later
                    // every bound is published and the first tile can be filtered with the best of them (on a corpus sorted
                    // by similarity - or with the coarse tf32 error bound - the LOCAL bound admits every row of the tile).
                    // The wait is bounded: a CTA that is not resident yet (another kernel on the device) only costs tightness.
                    // TMA and the tensor core keep running ahead meanwhile (second accumulator, ring).
                    named_bar_sync(1, 128);                            // every warp's bounds are published
                    if (et == 0) {
                        __threadfence();
                        atomicAdd(&a.ctl->obs_done, 1u);
                        const unsigned long long t0 = global_ns();
                        while (ld_acq_gpu(&a.ctl->obs_done) < gridDim.x && global_ns() - t0 < 4000ull) __nanosleep(100);
                    }
                    named_bar_sync(2, 128);
                    warp_refresh();
                    named_bar_sync(1, 128);
                    if (obs_holds_tile) {
                        for (int qi = 0; qi < nq; ++qi) {
                            const float th = thr_s[qi];
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                const uint32_t ov = pend[(size_t)qi * kObsStride + h * 128 + m];     // 0: row out of range / filtered
                                const float scv = ordered_to_float(ov);
                                if (ov != 0u && scv >= th) {
                                    if (qi == 0) atomicAdd(s_app, 1);
                                    const uint32_t pos = atomicAdd(a.ctl->cnt + qi, 1u);
                                    if (pos < (uint32_t)a.cap) a.cand[(size_t)qi * a.cap + pos] = make_key(scv, (uint32_t)(trow + h * 128 + m));
                                }
                            }
                        }
                    }
                }
                // ---- append pass: every row whose approximate score reaches the query's current threshold ----
                // Almost every tile has no such row: thresholds come in by vector loads, a chunk's compares fold into one mask
                // and only a non-zero mask branches (one threshold load, compare and branch per score in program order, behind
                // P serialized tensor-memory round trips per chunk, measured 3.6-6.3 us per tile at 64 columns against a tile
                // period of 7.8 us: the epilogue, not HBM, set the pace of the wide configurations).
                bool hit = false;
                if (!(warm && obs_holds_tile)) {
                    auto append_hits = [&](unsigned mask, const float (&sc)[QPC], int c, long long row) {
#pragma unroll
                        for (int j = 0; j < QPC; ++j) {
                            if (mask >> j & 1u) {
                                const int qi = c * QPC + j;
                                if (qi == 0) atomicAdd(s_app, 1);
                                const uint32_t pos = atomicAdd(a.ctl->cnt + qi, 1u);
                                if (pos < (uint32_t)a.cap) a.cand[(size_t)qi * a.cap + pos] = make_key(sc[j] + 0.0f, (uint32_t)row);
                                if (!warm) {                           // the first tile's scores are already in the sorted list
                                    const int lp = atomicAdd(pcnt + qi, 1);
                                    if (lp < npend) pend[(size_t)qi * npend + lp] = float_to_ordered(sc[j] + 0.0f);
                                }
                            }
                        }
                    };
#pragma unroll 1
                    for (int c = 0; c < NCOL / 16; ++c) {
                        float th[QPC];                                 // padding queries hold +inf
#pragma unroll
                        for (int j = 0; j < QPC; j += 4) {
                            const float4 t4 = *reinterpret_cast<const float4*>(thr_s + c * QPC + j);
                            th[j] = t4.x; th[j + 1] = t4.y; th[j + 2] = t4.z; th[j + 3] = t4.w;
                        }
                        if (P == 2) {                                  // both halves of the tile in flight: one wait per chunk
                            uint32_t v0[P][16], v1[P][16];
                            chunk_load(0, c, v0);
                            chunk_load(1, c, v1);
                            tmem_ld_wait();
                            chunk_fence(v0);
                            chunk_fence(v1);
                            float sc0[QPC], sc1[QPC];
                            chunk_reduce(v0, sc0);
                            chunk_reduce(v1, sc1);
                            unsigned m0 = 0u, m1 = 0u;
#pragma unroll
                            for (int j = 0; j < QPC; ++j) { m0 |= (unsigned)(sc0[j] >= th[j]) << j; m1 |= (unsigned)(sc1[j] >= th[j]) << j; }
                            if (!ok0) m0 = 0u;
                            if (!ok1) m1 = 0u;
                            if (m0 | m1) {
                                hit = true;
                                append_hits(m0, sc0, c, row_h0);
                                append_hits(m1, sc1, c, row_h1);
                            }
                        } else {
#pragma unroll 1
                            for (int h = 0; h < 2; ++h) {
                                float sc[QPC];
                                chunk_scores(h, c, sc);
                                unsigned mk = 0u;
#pragma unroll
                                for (int j = 0; j < QPC; ++j) mk |= (unsigned)(sc[j] >= th[j]) << j;
                                if (!(h ? ok1 : ok0)) mk = 0u;
                                if (mk) {
                                    hit = true;
                                    append_hits(mk, sc, c, h ? row_h1 : row_h0);
                                }
                            }
                        }
                    }
                    tc_fence_before();
                    mbar_arrive(tempty_bar(acc));
                }
                if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
                if (stamp_tile) ts2 = global_ns();
                // ---- threshold maintenance: the tile's appended scores enter the query's sorted list ----
                // One barrier that also tells whether ANY epilogue thread appended; a tile without appended rows that is not a
                // refresh tile ends here (nothing was written that the next tile reads).
                const bool refresh_tile = t < 8 || t % a.refresh_every == 0;
                const bool any = named_bar_or(1, 128, hit);
                if (warm) {
                    if (blockIdx.x == 0 && et == 0) a.ctl->t[2] = global_ns();
                    named_bar_sync(2, 128);
                } else if (any || refresh_tile) {
                    bool changed = false;
                    if (any) {
                        for (int q = ew; q < nq; q += 4) {
                            int pc = pcnt[q];                          // warp-uniform (shared memory, written before the barrier)
                            if (pc > 0) {
                                changed = true;
                                if (pc > npend) pc = npend;            // the surplus was dropped: only tightening information is lost
                                uint32_t* sl_ = sorted + (size_t)q * k;
                                int n = scnt[q];
                                __syncwarp();
                                for (int i = 0; i < pc; ++i) n = warp_list_add(sl_, n, pend[(size_t)q * npend + i]);
                                if (lane == 0) { scnt[q] = n; pcnt[q] = 0; }
                            }
                        }
                        __syncwarp();
                    }
                    if (changed || refresh_tile) warp_refresh();
                    named_bar_sync(2, 128);
                }
                if (stamp_tile && !warm) {   // CTA 0's epilogue, summed over its tiles: waiting for the tensor core, append pass, bookkeeping
                    a.ctl->t[13] += ts1 - ts0; a.ctl->t[14] += ts2 - ts1; a.ctl->t[15] += global_ns() - ts2;
                }
                warm = false;
            }
        }
        __threadfence();   // this thread's appended keys are visible device-wide before the CTA is counted as done
        if (blockIdx.x == 0 && et == 0) a.ctl->t[3] = global_ns();
        if (et == 0 && blockIdx.x < 160) { a.ctl->cta_thr[blockIdx.x] = thr_s[0]; a.ctl->cta_app[blockIdx.x] = (uint32_t)*s_app; }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
    }

    // ---- tail: the last n_fin CTAs to arrive finalize one query each ----
    const int n_fin = nq < (int)gridDim.x ? nq : (int)gridDim.x;
    if (tid == 0) {
        __threadfence();
        *s_ticket = atomicAdd(&a.ctl->done, 1u);
    }
    __syncthreads();
    const int ticket = (int)*s_ticket;
    const int first_fin = (int)gridDim.x - n_fin;
    if (ticket < first_fin) return;
    // scratch over the query block + ring: qv [ld] fp32 | hist [256] | s3 [3] + c2 | sel [..] u64
    fence_proxy_async_smem();   // the ring was written by TMA and read by the tensor core; from here on plain stores reuse it
    __syncthreads();
    float* qv = reinterpret_cast<float*>(fsm);
    const int ld_al = (a.ld + 3) / 4 * 4;
    uint32_t* hist = reinterpret_cast<uint32_t*>(qv + ld_al);
    uint32_t* s3 = hist + 256;
    int* s_c2 = reinterpret_cast<int*>(s3 + 3);
    u64* sel = reinterpret_cast<u64*>(fsm + (((size_t)ld_al * 4 + 256 * 4 + 16 + 15) / 16) * 16);
    const int sel_cap = (int)((region_bytes - (size_t)(reinterpret_cast<uint8_t*>(sel) - fsm)) / sizeof(u64));
    // normalised fp32 query (the rescore operand): bit-identical to what ingest would store as fp32
    // (written by CTA 0 in its prologue, before it was counted as done: visible after the acquire on the arrival counter)
    auto make_qv = [&](int qi) {
        for (int i = tid; i < a.ld; i += kFThreads) qv[i] = __ldcg(a.qn + (size_t)qi * a.ld + i);
    };
    if (tid == 0) {
        while (ld_acq_gpu(&a.ctl->done) < gridDim.x) __nanosleep(32);
        __threadfence();
    }
    __syncthreads();
    make_qv(ticket - first_fin);
    const bool stamp = ticket - first_fin == 0 && tid == 0;
    if (stamp) a.ctl->t[4] = global_ns();

    // Emit the query's hits: fin[0 .. keff) are its exact keys in order (this shard).  Single GPU: write them out.  Sharded:
    // push them to every rank, wait for every rank's, merge, write the global top-k.  Called by all threads of the CTA.
    auto emit = [&](int qi, const u64* fin, int nvalid) {
        long long* oid = a.out_ids + (size_t)qi * k;
        float* osc = a.out_scores + (size_t)qi * k;
        // the previous search on this stream (which this grid may have overtaken) has completed and its writes are visible
        // before this one touches the caller's output buffers: results land in stream order
        asm volatile("griddepcontrol.wait;" ::: "memory");
        if (a.xworld <= 1) {
            for (int i = tid; i < k; i += kFThreads) {
                const u64 key = i < nvalid ? fin[i] : 0ull;
                oid[i] = key ? a.id_base + (long long)key_row(key) : -1;
                osc[i] = key ? key_score(key) : -INFINITY;
            }
            return;
        }
        const int W = a.xworld;
        const size_t rec_q = ((size_t)k * 12 + 15) / 16 * 16;            // one query's hits inside a rank's record
        const size_t half = (size_t)(a.xstep % kXSlots) * W;             // slot of the 4-deep ring (kernels.cuh: why 4 is enough)
        for (int i = tid; i < k * W; i += kFThreads) {                    // 1. my hits -> slot `xrank` of every rank's area
            const int p = i / k, j = i % k;
            const u64 key = j < nvalid ? fin[j] : 0ull;
            char* dst = a.xpeer_area[p] + (half + a.xrank) * a.xrec_max + (size_t)qi * rec_q;
            reinterpret_cast<long long*>(dst)[j] = key ? a.id_base + (long long)key_row(key) : -1;
            reinterpret_cast<float*>(dst + (size_t)k * 8)[j] = key ? key_score(key) : -INFINITY;
        }
        __threadfence_system();
        __syncthreads();
        if (tid < W) st_release_sys(a.xpeer_qflag[tid] + (half + a.xrank) * kFMaxQ + qi, a.xstep);
        const uint32_t* myflags = a.xpeer_qflag[a.xrank] + half * kFMaxQ;
        bool arrived = true;
        if (tid < W) {                                                     // 2. every rank's hits for this query have landed
            const uint32_t* f = myflags + (size_t)tid * kFMaxQ + qi;
            unsigned long long t0 = 0, now = 0;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            while (ld_acquire_sys(f) != a.xstep) {
                __nanosleep(100);
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (now - t0 > 4000000000ull) { arrived = false; break; }  // 4 s: a peer is gone; fail the query, not the GPU
            }
        }
        const int all_in = __syncthreads_and(arrived ? 1 : 0);
        (void)ld_acquire_sys(myflags + (size_t)(tid % W) * kFMaxQ + qi);   // every thread acquires for its own loads below
        // 3. merge by rank counting: the lists are ordered and all ids are distinct
        int64_t* mids = reinterpret_cast<int64_t*>(sel);              // [W][k]   (fin is dead: it has been pushed)
        float* msc = reinterpret_cast<float*>(mids + (size_t)W * k);      // [W][k]
        const char* area = a.xpeer_area[a.xrank] + half * a.xrec_max;
        for (int i = tid; i < k * W; i += kFThreads) {
            const int p = i / k, j = i % k;
            const char* src = area + (size_t)p * a.xrec_max + (size_t)qi * rec_q;
            mids[i] = all_in ? (int64_t)__ldcg(reinterpret_cast<const long long*>(src) + j) : (int64_t)-1;
            msc[i] = all_in ? __ldcg(reinterpret_cast<const float*>(src + (size_t)k * 8) + j) : -INFINITY;
        }
        __syncthreads();
        if (tid == 0) {
            int valid = 0;
            for (int p = 0; p < W; ++p) valid += count_better<false>(mids + (size_t)p * k, msc + (size_t)p * k, k, -INFINITY, INT64_MAX);
            for (int i = valid; i < k; ++i) { oid[i] = -1; osc[i] = all_in ? -INFINITY : __int_as_float(0x7FC00000); }   // NaN: exchange timed out
        }
        for (int i = tid; i < k * W; i += kFThreads) {
            const int p = i / k, j = i % k;
            const int64_t id = mids[i];
            if (id < 0) continue;
            const float sc = msc[i];
            int rank = j;
            for (int pp = 0; pp < W && rank < k; ++pp)
                if (pp != p) rank += count_better<false>(mids + (size_t)pp * k, msc + (size_t)pp * k, k, sc, id);
            if (rank < k) { oid[rank] = id; osc[rank] = sc; }
        }
    };

    for (int qi = ticket - first_fin; qi < nq; qi += n_fin) {
        if (qi != ticket - first_fin) make_qv(qi);
        if (tid == 0) *s_c2 = 0;
        __syncthreads();
        const uint32_t m32 = __ldcg(a.ctl->cnt + qi);
        if (tid == 0) { a.ctl->last_cnt[qi] = m32; a.ctl->last_resc[qi] = 0xFFFFFFFFu; }
        if (stamp && qi == 0) a.ctl->t[10] = global_ns();
        const int keff = a.keff;
        const u64* in = a.cand + (size_t)qi * a.cap;
        bool exact_scan = m32 > (uint32_t)a.cap || (int)m32 < keff;   // block-uniform
        if (!exact_scan && keff > 0) {
            const int m = (int)m32;
            constexpr int kSmallM = 8192;
            // Pre-filter with this CTA's own final threshold thr_s[qi] (<= T - 2 eps, and by the end of the sweep - the bounds
            // are shared - very close to it): the k rows at or above T and every row within 2 eps of T pass it, most of the
            // buffer (rows appended early, under loose thresholds) does not.  What passes is staged in shared memory.
            u64* stg = sel + (sel_cap - kSmallM);
            int m1 = kSmallM + 1;
            if (sel_cap >= 2 * kSmallM) {
                const float thr_loc = thr_s[qi];
                if (tid == 0) { s3[1] = 0u; s3[0] = 0u; s3[2] = (uint32_t)keff; }
                __syncthreads();
                for (int i0 = tid; i0 < m; i0 += 4 * kFThreads) {       // four loads in flight per thread (the buffer is in L2)
                    u64 key[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) key[u] = i0 + u * kFThreads < m ? __ldcg(in + i0 + u * kFThreads) : 0ull;
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (key[u] != 0ull && key_score(key[u]) >= thr_loc) {
                            const uint32_t p_ = atomicAdd(&s3[1], 1u);
                            if (p_ < (uint32_t)kSmallM) stg[p_] = key[u];
                        }
                }
                __syncthreads();
                m1 = (int)s3[1];
            }
            if (m1 <= kSmallM && m1 >= keff) {
                // T = keff-th largest approximate score among the staged keys: rank counting for a few hundred keys, else a
                // 4-pass radix select over the ordered score bits (256-bin shared histogram)
                const int m = m1;
                if (stamp && qi == 0) a.ctl->t[11] = global_ns();
                if (m <= 2 * kFThreads) {
                    // a couple of hundred keys (k = 10): count, for one or two keys per thread, the scores above / not below
                    // it (broadcast reads); the key with #above < keff <= #not-below carries T
                    uint32_t mine[2];
                    int gt[2] = {0, 0}, ge[2] = {0, 0};
#pragma unroll
                    for (int u = 0; u < 2; ++u) mine[u] = tid + u * kFThreads < m ? (uint32_t)(stg[tid + u * kFThreads] >> 32) : 0xFFFFFFFFu;
#pragma unroll 8
                    for (int i = 0; i < m; ++i) {
                        const uint32_t o = (uint32_t)(stg[i] >> 32);
#pragma unroll
                        for (int u = 0; u < 2; ++u) { gt[u] += o > mine[u]; ge[u] += o >= mine[u]; }
                    }
#pragma unroll
                    for (int u = 0; u < 2; ++u)
                        if (tid + u * kFThreads < m && gt[u] < keff && ge[u] >= keff) s3[0] = mine[u];   // every writer holds the same value
                    __syncthreads();
                } else
#pragma unroll 1
                for (int shift = 24; shift >= 0; shift -= 8) {
                    const uint32_t prefix = s3[0], want = s3[2];
                    for (int i = tid; i < 256; i += kFThreads) hist[i] = 0u;
                    __syncthreads();
                    for (int i0 = warp * kWarp; i0 < m; i0 += kFThreads) {     // warp-uniform trip count
                        const int i = i0 + lane;
                        const uint32_t hsc = i < m ? (uint32_t)(stg[i] >> 32) : 0u;
                        const bool in = i < m && (shift == 24 || (hsc >> (shift + 8)) == (prefix >> (shift + 8)));
                        // scores of one query share their leading bytes: aggregate equal digits inside the warp, one atomic each
                        const unsigned same = __match_any_sync(kFull, in ? (int)((hsc >> shift) & 255u) : -1);
                        if (in && lane == __ffs(same) - 1) atomicAdd(&hist[(hsc >> shift) & 255u], (uint32_t)__popc(same));
                    }
                    __syncthreads();
                    if (warp == 0) {   // bin (from the top) in which the cumulative count reaches `want`; lane l owns bins 255-8l .. 248-8l
                        uint32_t c[8], sum = 0;
#pragma unroll
                        for (int b = 0; b < 8; ++b) { c[b] = hist[255 - 8 * lane - b]; sum += c[b]; }
                        uint32_t incl = sum;
#pragma unroll
                        for (int off = 1; off < 32; off <<= 1) {
                            const uint32_t o = __shfl_up_sync(kFull, incl, off);
                            if (lane >= off) incl += o;
                        }
                        const uint32_t before = incl - sum;
                        if (before < want && incl >= want) {          // exactly one lane
                            uint32_t run = before;
#pragma unroll
                            for (int b = 0; b < 8; ++b) {
                                if (run < want && run + c[b] >= want) { s3[0] = prefix | ((uint32_t)(255 - 8 * lane - b) << shift); s3[2] = want - run; }
                                run += c[b];
                            }
                        }
                    }
                    __syncthreads();
                }
                if (stamp && qi == 0) a.ctl->t[12] = global_ns();
                const float cut = thr_below(ordered_to_float(s3[0]), eps_s[qi]);
                for (int i = tid; i < m; i += kFThreads) {
                    const u64 key = stg[i];
                    if (key_score(key) >= cut) sel[atomicAdd(s_c2, 1)] = key;      // <= m <= kSmallM entries: below the staging area
                }
            } else {
                const uint32_t t_ord = block_kth_largest([&](int i) { return (uint32_t)(__ldcg(in + i) >> 32); }, m, (uint32_t)keff, hist, s3);
                const float cut = thr_below(ordered_to_float(t_ord), eps_s[qi]);
                for (int i = tid; i < m; i += kFThreads) {
                    const u64 key = __ldcg(in + i);
                    if (key_score(key) >= cut) {
                        const int pos = atomicAdd(s_c2, 1);
                        if (pos < sel_cap) sel[pos] = key;
                    }
                }
            }
            __syncthreads();
            if (stamp && qi == 0) a.ctl->t[5] = global_ns();
            const int c2 = *s_c2;
            int P2 = 32;
            while (P2 < c2) P2 <<= 1;
            if (P2 > sel_cap) exact_scan = true;   // more rows within 2 eps of the k-th score than the scratch holds: massive duplication
            else {
            // canonical rescore, one warp per row, TWO rows in flight per warp (the rows are cold in HBM: latency, not bandwidth)
            for (int c = warp; c < c2; c += 2 * (kFThreads / 32)) {
                const int c_b = c + kFThreads / 32;
                const uint32_t row_a = key_row(sel[c]), row_b = c_b < c2 ? key_row(sel[c_b]) : row_a;
                double sa, sb;
                if (a.dt == 0) canonical_dot_two_rows<0>(a.data, row_a, row_b, a.ld, qv, lane, sa, sb);
                else if (a.dt == 1) canonical_dot_two_rows<1>(a.data, row_a, row_b, a.ld, qv, lane, sa, sb);
                else canonical_dot_two_rows<2>(a.data, row_a, row_b, a.ld, qv, lane, sa, sb);
                __syncwarp();
                if (lane == 0) {
                    sel[c] = make_key((float)sa + 0.0f, row_a);
                    if (c_b < c2) sel[c_b] = make_key((float)sb + 0.0f, row_b);
                }
            }
            {
                for (int i = c2 + tid; i < P2; i += kFThreads) sel[i] = 0ull;
                __syncthreads();
                if (stamp && qi == 0) a.ctl->t[6] = global_ns();
                if (c2 <= kFThreads) {
                    // a handful of exact keys: rank by counting (keys are unique), one thread per key, two barriers
                    const u64 mine = tid < c2 ? sel[tid] : 0ull;
                    int rk = 0;
                    for (int i = 0; i < c2; ++i) rk += sel[i] > mine;
                    __syncthreads();
                    if (tid < c2) sel[rk] = mine;
                    __syncthreads();
                } else {
                    block_bitonic_sort_desc(sel, P2, tid, kFThreads);
                }
                emit(qi, sel, keff);
                if (stamp && qi == 0) a.ctl->t[7] = global_ns();
                if (tid == 0) { a.flags[qi] = 0; a.ctl->last_resc[qi] = (uint32_t)c2; }
            }
            }
        } else if (!exact_scan) {   // keff == 0: nothing to return
            emit(qi, sel, 0);
            if (tid == 0) a.flags[qi] = 0;
        }
        if (exact_scan) {
            // The buffer overflowed (more than cap rows within reach of the k-th score).  Answer exactly, here: canonical
            // score of every row, per-warp sorted lists of kpe keys, one merge.  ~0.1 s on a 15 GB corpus, no extra launch.
            __syncthreads();
            int kpe = 32;
            while (kpe < k) kpe <<= 1;
            u64* lists = sel;                                  // [6][kpe], then padded to a power of two for the sort
            const int total = (kFThreads / 32) * kpe;
            int P2 = 32;
            while (P2 < total) P2 <<= 1;
            for (int i = tid; i < P2; i += kFThreads) lists[i] = 0ull;
            __syncthreads();
            u64* mine = lists + (size_t)warp * kpe;
            for (long long r = warp; r < a.n_rows; r += kFThreads / 32) {
                if (a.allow != nullptr && !row_allowed(a.allow, r)) continue;
                double sc;
                if (a.dt == 0) sc = rescore_row<0>(a.data, r, a.ld, qv, lane);
                else if (a.dt == 1) sc = rescore_row<1>(a.data, r, a.ld, qv, lane);
                else sc = rescore_row<2>(a.data, r, a.ld, qv, lane);
                const u64 key = make_key((float)sc + 0.0f, (uint32_t)r);
                if (key > mine[kpe - 1]) warp_list_insert(mine, kpe, key, lane);
            }
            __syncthreads();
            block_bitonic_sort_desc(lists, P2, tid, kFThreads);
            emit(qi, lists, keff);
            if (tid == 0) { a.flags[qi] = 1; atomicAdd(a.flag_count, 1); }
        }
        __syncthreads();
        if (tid == 0) a.ctl->cnt[qi] = 0u;                             // leave the control block clean for the next search
        if (tid <= kFGroups) a.ctl->gthr[qi][tid] = 0u;
    }
    if (tid == 0) {
        if (a.host_flag != nullptr) __threadfence_system(); else __threadfence();   // this CTA's hits are visible (to the host) first
        if (atomicAdd(&a.ctl->fin_done, 1u) == (uint32_t)n_fin - 1u) {   // last finalizer: counters back to zero
            a.ctl->done = 0u;
            a.ctl->obs_done = 0u;
            a.ctl->fin_done = 0u;
            __threadfence();
            a.ctl->n_done = a.seq_on_half + 1u;      // this half is free for the search after the next
            if (a.host_flag != nullptr) { __threadfence_system(); *reinterpret_cast<volatile uint32_t*>(a.host_flag) = a.host_seq; }
        }
    }
}

}  // namespace rfk
