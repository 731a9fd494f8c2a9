// Large-k path (k above the fused-list limit, up to Milvus' 16384): exact from the start.
//   score_all_kernel   canonical fp64 score of every row for one query -> fp32 scores [n]
//   radix_hist_kernel  + radix_pick_kernel: 8 passes of 8 bits over the 64-bit keys
//                      (ordered(score) << 32 | ~row) find the k-th largest key exactly (keys are unique)
//   compact_kernel     keys >= threshold -> exactly k keys
//   rank_sort_kernel   rank of each key by counting (O(k^2), tiled through shared memory) -> ordered output
// Used by graph_cons.py:279-style calls (limit = 1000) on corpora of more than 256 rows.
#pragma once
#include "common.cuh"

namespace rfk {

template <int DT>
__global__ void __launch_bounds__(256) score_all_kernel(const void* __restrict__ data, int64_t n_rows, int ld,
                                                        const float* __restrict__ qhat, float* __restrict__ scores,
                                                        const uint32_t* __restrict__ allow, float radius, float range_filter) {
    const int lane = threadIdx.x & 31;
    const typename Store<DT>::T* base = reinterpret_cast<const typename Store<DT>::T*>(data);
    const int64_t stride = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n_rows; r += stride) {
        if (allow != nullptr && !row_allowed(allow, r)) {   // filtered out: below every real score
            if (lane == 0) scores[r] = -INFINITY;
            continue;
        }
        const double s = canonical_dot_row<DT>(base + (size_t)r * ld, qhat, ld, lane);
        const float s32 = (float)s + 0.0f;
        if (lane == 0) scores[r] = s32 > radius && s32 <= range_filter ? s32 : -INFINITY;   // outside a range search's window: as filtered
    }
}

struct RadixState {
    u64 prefix;        // bits of the k-th key decided so far (high to low)
    int64_t remaining; // rank still to resolve inside the current prefix
    unsigned int hist[256];
    unsigned int out_count;
};

// histogram of byte `shift/8` over the keys whose higher bytes equal the prefix
__global__ void __launch_bounds__(256) radix_hist_kernel(const float* __restrict__ scores, int64_t n, int shift,
                                                         RadixState* st) {
    __shared__ unsigned int h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const u64 prefix = st->prefix;
    const u64 himask = shift >= 56 ? 0ull : ~0ull << (shift + 8);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const u64 key = make_key(scores[i], (uint32_t)i);
        if ((key & himask) == (prefix & himask)) atomicAdd(&h[(key >> shift) & 255], 1u);
    }
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&st->hist[threadIdx.x], h[threadIdx.x]);
}

// pick the byte value that contains the wanted rank, descend
__global__ void radix_pick_kernel(int shift, RadixState* st) {
    if (threadIdx.x != 0) return;
    int64_t rem = st->remaining;
    int b = 255;
    for (; b > 0; --b) {
        const int64_t c = st->hist[b];
        if (rem <= c) break;
        rem -= c;
    }
    st->prefix |= (u64)b << shift;
    st->remaining = rem;
    for (int i = 0; i < 256; ++i) st->hist[i] = 0;
}

__global__ void __launch_bounds__(256) compact_kernel(const float* __restrict__ scores, int64_t n, RadixState* st,
                                                      u64* __restrict__ keys, int cap) {
    const u64 thr = st->prefix;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const u64 key = make_key(scores[i], (uint32_t)i);
        if (key >= thr) {
            const unsigned pos = atomicAdd(&st->out_count, 1u);
            if ((int)pos < cap) keys[pos] = key;
        }
    }
}

// out position of key i = number of keys greater than it
__global__ void __launch_bounds__(256) rank_sort_kernel(const u64* __restrict__ keys, int m, int k, int64_t id_base,
                                                        int64_t* __restrict__ out_ids, float* __restrict__ out_scores) {
    __shared__ u64 tile[1024];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const u64 mine = i < m ? keys[i] : 0ull;
    int rank = 0;
    for (int t0 = 0; t0 < m; t0 += 1024) {
        for (int j = threadIdx.x; j < 1024; j += blockDim.x) tile[j] = t0 + j < m ? keys[t0 + j] : 0ull;
        __syncthreads();
        const int lim = m - t0 < 1024 ? m - t0 : 1024;
        for (int j = 0; j < lim; ++j) rank += tile[j] > mine;
        __syncthreads();
    }
    if (i < m && rank < k) {   // a -inf key is a row outside a range search's window: padding
        const bool hit = key_score(mine) > -INFINITY;
        out_ids[rank] = hit ? id_base + (int64_t)key_row(mine) : -1;
        out_scores[rank] = hit ? key_score(mine) : -INFINITY;
    }
    if (i >= m && i < k) {   // slots past the number of rows
        out_ids[i] = -1;
        out_scores[i] = -INFINITY;
    }
}

// ---------------------------------------------------------------------------------
// Batched large-k pipeline (k > 256, up to 16384; graph_cons.py:279 asks limit = 1000): no host synchronisation per query.
//   1. the tensor-core sweep dumps approximate scores of up to 16 queries at once: approx[q][row]   (gemm.cuh MODE 1)
//   2. bk_hist_kernel x 4   radix select of T = the keff-th largest approximate score of every query (allowed rows only);
//                           pass p derives its prefix from the histogram of pass p - 1, so no pick kernels in between
//   3. bk_compact_kernel    rows with approx >= T - 2 eps  ->  candidate rows (every row of the exact top-k is among them:
//                           DESIGN.md 2.4, with the whole approximate score vector at hand instead of an append buffer)
//   4. bk_rescore_kernel    canonical fp64 score of every candidate  ->  exact keys
//   5. bk_rank_sort_kernel  the keff largest exact keys in order
// A query whose candidates exceed the buffer (thousands of rows within 2 eps of the k-th score) is flagged and answered by
// the exact one-query path above.
// ---------------------------------------------------------------------------------
struct BkState {                  // per query
    uint32_t prefix[4];           // ordered-score bits decided after pass p (high to low)
    int32_t remaining[4];         // rank still to resolve inside prefix[p]
    uint32_t hist[4][256];
    uint32_t n_cand;              // rows compacted (may exceed the buffer: overflow)
    uint32_t overflow;
    uint32_t pad[2];
};

// (prefix, remaining) after pass p from the state of pass p - 1 and hist[p]: the bin, from the top, where the cumulative count
// reaches `remaining`.  Executed by one warp; every block computes the same values.
__device__ __forceinline__ void bk_resolve(const BkState* st, int p, int want0, uint32_t* prefix_out, int* remaining_out, int lane) {
    uint32_t prefix = 0u;
    int want = want0;
    for (int pp = 0; pp <= p; ++pp) {
        if (pp < p) { prefix = st->prefix[pp]; want = st->remaining[pp]; continue; }   // stored by block 0 of the pass that computed it
        const int shift = 24 - 8 * pp;
        uint32_t c[8], sum = 0;
#pragma unroll
        for (int b = 0; b < 8; ++b) { c[b] = st->hist[pp][255 - 8 * lane - b]; sum += c[b]; }
        uint32_t incl = sum;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t o = __shfl_up_sync(kFull, incl, off);
            if (lane >= off) incl += o;
        }
        const uint32_t before = incl - sum;
        uint32_t np = 0u;
        int nw = 0;
        if ((int)before < want && (int)incl >= want) {
            uint32_t run = before;
#pragma unroll
            for (int b = 0; b < 8; ++b) {
                if ((int)run < want && (int)(run + c[b]) >= want) { np = prefix | ((uint32_t)(255 - 8 * lane - b) << shift); nw = want - (int)run; }
                run += c[b];
            }
        }
        const unsigned who = __ballot_sync(kFull, nw > 0);
        if (who) { const int src = __ffs(who) - 1; np = __shfl_sync(kFull, np, src); nw = __shfl_sync(kFull, nw, src); }
        prefix = np; want = nw;
    }
    *prefix_out = prefix;
    *remaining_out = want;
}

// pass p (0..3): histogram of byte (3 - p) of the ordered scores whose higher bytes equal the prefix decided so far.
// kGroupWords (grouping search): `approx` holds per-group ordered maxima (bk_group_max_kernel) instead of scores, n is the
// number of groups, 0 marks an empty group and is skipped; allow and wcap are unused.
template <bool kGroupWords = false>
__global__ void __launch_bounds__(256) bk_hist_kernel(const float* __restrict__ approx, int64_t n, int pass, int keff,
                                                      BkState* __restrict__ states, const uint32_t* __restrict__ allow,
                                                      const float* __restrict__ wcap) {
    __shared__ uint32_t h[256];
    __shared__ uint32_t s_prefix;
    const int q = blockIdx.y, lane = threadIdx.x & 31;
    BkState* st = states + q;
    h[threadIdx.x] = 0u;
    if (pass > 0 && threadIdx.x < 32) {
        uint32_t prefix; int rem;
        bk_resolve(st, pass - 1, keff, &prefix, &rem, lane);
        if (lane == 0) {
            s_prefix = prefix;
            if (blockIdx.x == 0) { st->prefix[pass - 1] = prefix; st->remaining[pass - 1] = rem; }
        }
    }
    __syncthreads();
    const uint32_t prefix = pass > 0 ? s_prefix : 0u;
    const int shift = 24 - 8 * pass;
    const float* sc = approx + (size_t)q * n;
    const float cap = wcap != nullptr ? wcap[q] : INFINITY;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        uint32_t o;
        if (kGroupWords) {
            o = __float_as_uint(sc[i]);
            if (o == 0u) continue;
        } else {
            if (allow != nullptr && !row_allowed(allow, i)) continue;
            if (sc[i] > cap) continue;   // range search: only rows certainly at or below range_filter count toward T
            o = float_to_ordered(sc[i] + 0.0f);
        }
        if (pass == 0 || (o >> (shift + 8)) == (prefix >> (shift + 8))) atomicAdd(&h[(o >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&st->hist[pass][threadIdx.x], h[threadIdx.x]);
}

// rows whose approximate score reaches T - 2 eps -> cand_rows[q][0 .. n_cand)
__global__ void __launch_bounds__(256) bk_compact_kernel(const float* __restrict__ approx, int64_t n, int keff, float eps_const,
                                                         const float* __restrict__ eps_q, BkState* __restrict__ states,
                                                         uint32_t* __restrict__ cand_rows, int cmax, const uint32_t* __restrict__ allow,
                                                         const float* __restrict__ wlo, const float* __restrict__ whi) {
    __shared__ float s_cut, s_hi;
    const int q = blockIdx.y, lane = threadIdx.x & 31;
    BkState* st = states + q;
    if (threadIdx.x < 32) {
        uint32_t t_ord; int rem;
        bk_resolve(st, 3, keff, &t_ord, &rem, lane);
        if (lane == 0) {
            const float e = eps_const + (eps_q ? eps_q[q] : 0.0f);
            float cut = keff > 0 ? __fsub_rd(__fsub_rd(ordered_to_float(t_ord), __fmul_ru(2.0f, e)), 2.384185791015625e-07f) : INFINITY;
            // range search: rem == 0 <=> fewer than keff rows lie certainly below the ceiling, so T is no bound and the floor
            // alone cuts; otherwise the floor may still be the tighter cut
            if (wlo != nullptr && keff > 0) cut = rem == 0 ? wlo[q] : fmaxf(cut, wlo[q]);
            s_cut = cut;
            s_hi = whi != nullptr ? whi[q] : INFINITY;
        }
    }
    __syncthreads();
    const float cut = s_cut, hi = s_hi;
    const float* sc = approx + (size_t)q * n;
    uint32_t* out = cand_rows + (size_t)q * cmax;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (allow != nullptr && !row_allowed(allow, i)) continue;
        if (sc[i] >= cut && sc[i] <= hi) {
            const uint32_t pos = atomicAdd(&st->n_cand, 1u);
            if (pos < (uint32_t)cmax) out[pos] = (uint32_t)i;
            else st->overflow = 1u;
        }
    }
}

// one warp per candidate: canonical fp64 score -> exact key (0 past the candidate count)
template <int DT>
__global__ void __launch_bounds__(256) bk_rescore_kernel(const void* __restrict__ data, int ld, const float* __restrict__ qhat,
                                                         const BkState* __restrict__ states, const uint32_t* __restrict__ cand_rows,
                                                         int cmax, u64* __restrict__ keys, float radius, float range_filter) {
    const int q = blockIdx.y, lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= cmax) return;
    const uint32_t nc = states[q].n_cand < (uint32_t)cmax ? states[q].n_cand : (uint32_t)cmax;
    u64 key = 0ull;
    if ((uint32_t)c < nc) {
        const uint32_t row = cand_rows[(size_t)q * cmax + c];
        const double s = canonical_dot_row<DT>(reinterpret_cast<const typename Store<DT>::T*>(data) + (size_t)row * ld, qhat + (size_t)q * ld, ld, lane);
        const float s32 = (float)s + 0.0f;
        key = make_key(s32 > radius && s32 <= range_filter ? s32 : -INFINITY, row);   // outside a range search's window: -inf
    }
    if (lane == 0) keys[(size_t)q * cmax + c] = key;
}

// out position of key i = number of keys greater than it (grid.y = query); flagged queries are left to the fallback
__global__ void __launch_bounds__(256) bk_rank_sort_kernel(const u64* __restrict__ keys_all, const BkState* __restrict__ states, int cmax, int k,
                                                           int keff, int64_t id_base, int64_t* __restrict__ out_ids, float* __restrict__ out_scores) {
    __shared__ u64 tile[1024];
    const int q = blockIdx.y;
    const int m = (int)(states[q].n_cand < (uint32_t)cmax ? states[q].n_cand : (uint32_t)cmax);
    const u64* keys = keys_all + (size_t)q * cmax;
    int64_t* oid = out_ids + (size_t)q * k;
    float* osc = out_scores + (size_t)q * k;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const u64 mine = i < m ? keys[i] : 0ull;
    int rank = 0;
    for (int t0 = 0; t0 < m; t0 += 1024) {
        for (int j = threadIdx.x; j < 1024; j += blockDim.x) tile[j] = t0 + j < m ? keys[t0 + j] : 0ull;
        __syncthreads();
        const int lim = m - t0 < 1024 ? m - t0 : 1024;
        for (int j = 0; j < lim; ++j) rank += tile[j] > mine;
        __syncthreads();
    }
    if (i < m && rank < keff) {   // a -inf key is a row outside a range search's window: padding
        const bool hit = key_score(mine) > -INFINITY;
        oid[rank] = hit ? id_base + (int64_t)key_row(mine) : -1;
        osc[rank] = hit ? key_score(mine) : -INFINITY;
    }
    if (i >= (m < keff ? m : keff) && i < k) {   // slots past the number of rows that exist (a window may hold fewer than keff)
        oid[i] = -1;
        osc[i] = -INFINITY;
    }
}

// ---------------------------------------------------------------------------------
// Grouping search (DESIGN.md 7d): the k best groups, one hit per group (its best row).  groups[r] is row r's code; a code
// outside [0, n_groups) never returns its row.  Every row the kernels below consider is allowed (filter and tombstones).
//
// Batched route (search_bigk_batched with a group code array), per chunk of up to 16 queries:
//   sweep (MODE 1) -> bk_group_max_kernel -> bk_hist_kernel<true> x 4 over the group maxima (T = keff-th largest non-empty
//   group maximum) -> bk_group_compact_kernel (approx >= max(T, gmax[group]) - 2 eps) -> bk_rescore_kernel ->
//   bk_group_rep_kernel (one survivor per group) -> bk_rank_sort_kernel.  Overflow: the exact path below.
// Exact path (search_grouped), one query at a time:
//   score_all_kernel -> group_best_kernel (largest exact key per group) -> radix_hist_keys_kernel + radix_pick_kernel x 8
//   over the group keys -> pad_keys_kernel + group_compact_kernel -> rank_sort_kernel.
// ---------------------------------------------------------------------------------

// gmax[q][g] = largest ordered approximate score of the allowed rows of group g (0 = none); gmax zeroed by the caller.
// One thread per row for all nb queries: the row's code and mask bit are read once.  Neighbouring rows usually share a code
// (a document's chunks are contiguous), so lanes of equal code reduce first and one of them issues the atomic, and only when
// it would raise the stored word.
__global__ void __launch_bounds__(256) bk_group_max_kernel(const float* __restrict__ approx, int64_t n, int nb,
                                                           const int32_t* __restrict__ groups, int n_groups,
                                                           const uint32_t* __restrict__ allow, uint32_t* __restrict__ gmax) {
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < n; i0 += stride) {   // warp-uniform trip count
        const int64_t i = i0 + lane;
        int g = i < n ? __ldg(groups + i) : -1;
        if ((unsigned)g >= (unsigned)n_groups || (allow != nullptr && !row_allowed(allow, i))) g = -1;
        const unsigned peers = __match_any_sync(kFull, g);
        const bool leader = g >= 0 && lane == __ffs(peers) - 1;
        for (int q = 0; q < nb; ++q) {
            const uint32_t o = g >= 0 ? float_to_ordered(approx[(size_t)q * n + i] + 0.0f) : 0u;
            const uint32_t m = __reduce_max_sync(peers, o);
            if (leader) {
                uint32_t* p = gmax + (size_t)q * n_groups + g;
                if (m > __ldcg(p)) atomicMax(p, m);
            }
        }
    }
}

// rows whose approximate score reaches max(T, gmax[q][group]) - 2 eps -> cand_rows[q][0 .. n_cand).  rem == 0 after the
// select <=> fewer than keff non-empty groups: T is no bound and the group maxima alone cut.
__global__ void __launch_bounds__(256) bk_group_compact_kernel(const float* __restrict__ approx, int64_t n, int keff, float eps_const,
                                                               const float* __restrict__ eps_q, BkState* __restrict__ states,
                                                               uint32_t* __restrict__ cand_rows, int cmax, const uint32_t* __restrict__ allow,
                                                               const int32_t* __restrict__ groups, int n_groups,
                                                               const uint32_t* __restrict__ gmax) {
    __shared__ uint32_t s_t;
    __shared__ float s_e2;
    const int q = blockIdx.y, lane = threadIdx.x & 31;
    BkState* st = states + q;
    if (threadIdx.x < 32) {
        uint32_t t_ord; int rem;
        bk_resolve(st, 3, keff, &t_ord, &rem, lane);
        if (lane == 0) {
            s_t = rem == 0 ? 0u : t_ord;
            s_e2 = __fmul_ru(2.0f, eps_const + (eps_q ? eps_q[q] : 0.0f));
        }
    }
    __syncthreads();
    const uint32_t t = s_t;
    const float e2 = s_e2;
    const float* sc = approx + (size_t)q * n;
    const uint32_t* gm = gmax + (size_t)q * n_groups;
    uint32_t* out = cand_rows + (size_t)q * cmax;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (allow != nullptr && !row_allowed(allow, i)) continue;
        const int g = __ldg(groups + i);
        if ((unsigned)g >= (unsigned)n_groups) continue;
        const uint32_t b = max(t, __ldg(gm + g));   // the row's own group is non-empty: b > 0
        const float cut = __fsub_rd(__fsub_rd(ordered_to_float(b), e2), 2.384185791015625e-07f);   // as bk_compact_kernel
        if (sc[i] >= cut) {
            const uint32_t pos = atomicAdd(&st->n_cand, 1u);
            if (pos < (uint32_t)cmax) out[pos] = (uint32_t)i;
            else st->overflow = 1u;
        }
    }
}

// Representatives: a candidate whose group holds a candidate with a larger exact key becomes make_key(-inf, row), which
// bk_rank_sort_kernel emits as padding.  Tiled O(m^2) compare (grid.y = query).  The keys are rewritten in place while other
// blocks read them: only non-maximal keys change, and a key's fate depends only on its group's maximum, which never does.
__global__ void __launch_bounds__(256) bk_group_rep_kernel(u64* __restrict__ keys_all, const BkState* __restrict__ states, int cmax,
                                                           const int32_t* __restrict__ groups) {
    __shared__ u64 tk[1024];
    __shared__ int tg[1024];
    const int q = blockIdx.y;
    const int m = (int)(states[q].n_cand < (uint32_t)cmax ? states[q].n_cand : (uint32_t)cmax);
    if (blockIdx.x * blockDim.x >= (unsigned)m) return;   // whole block past the candidates (uniform)
    u64* keys = keys_all + (size_t)q * cmax;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const u64 mine = i < m ? keys[i] : 0ull;
    const int g = i < m ? __ldg(groups + key_row(mine)) : -1;
    bool beaten = false;
    for (int t0 = 0; t0 < m; t0 += 1024) {
        for (int j = threadIdx.x; j < 1024; j += blockDim.x) {
            const u64 kj = t0 + j < m ? keys[t0 + j] : 0ull;
            tk[j] = kj;
            tg[j] = t0 + j < m ? __ldg(groups + key_row(kj)) : -2;
        }
        __syncthreads();
        const int lim = m - t0 < 1024 ? m - t0 : 1024;
        for (int j = 0; j < lim; ++j) beaten |= tg[j] == g && tk[j] > mine;
        __syncthreads();
    }
    if (i < m && beaten) keys[i] = make_key(-INFINITY, key_row(mine));
}

// gbest[g] = largest exact key (score, row) of group g over the rows score_all_kernel scored (-inf = masked); 0 = empty
__global__ void __launch_bounds__(256) group_best_kernel(const float* __restrict__ scores, int64_t n, const int32_t* __restrict__ groups,
                                                         int n_groups, u64* __restrict__ gbest) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float s = scores[i];
        const int g = __ldg(groups + i);
        if (s == -INFINITY || (unsigned)g >= (unsigned)n_groups) continue;
        const u64 key = make_key(s, (uint32_t)i);
        if (key > __ldcg(gbest + g)) atomicMax(gbest + g, key);
    }
}

// radix_hist_kernel over an array of keys (the group keys; 0 = empty group, the smallest key)
__global__ void __launch_bounds__(256) radix_hist_keys_kernel(const u64* __restrict__ keys, int64_t n, int shift, RadixState* st) {
    __shared__ unsigned int h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const u64 prefix = st->prefix;
    const u64 himask = shift >= 56 ? 0ull : ~0ull << (shift + 8);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const u64 key = keys[i];
        if ((key & himask) == (prefix & himask)) atomicAdd(&h[(key >> shift) & 255], 1u);
    }
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&st->hist[threadIdx.x], h[threadIdx.x]);
}

// keys[j] = cap - j: distinct keys below every real key, which rank_sort_kernel emits as padding.  group_compact_kernel then
// overwrites the first out_count of them, so the slots past the non-empty groups rank in order and are all written.
__global__ void __launch_bounds__(256) pad_keys_kernel(u64* __restrict__ keys, int cap) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < cap) keys[j] = (u64)(cap - j);
}

// non-empty group keys >= the selected key (0 when fewer than cap groups are non-empty: then every non-empty one)
__global__ void __launch_bounds__(256) group_compact_kernel(const u64* __restrict__ gbest, int64_t n, RadixState* st,
                                                            u64* __restrict__ keys, int cap) {
    const u64 thr = st->prefix;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const u64 key = gbest[i];
        if (key != 0ull && key >= thr) {
            const unsigned pos = atomicAdd(&st->out_count, 1u);
            if ((int)pos < cap) keys[pos] = key;
        }
    }
}

}  // namespace rfk
