// Device kernels of the exact cosine top-k path (everything except the tcgen05 GEMM).
//
//   ingest_kernel      K1  L2-normalise + cast at ingest ("chunking_storing (1).py":380-396)
//   scan_topk_kernel   K2  small-batch HBM-bound scan with fused per-warp top-K' lists
//   finalize_kernel    K4  merge of per-CTA candidates + exact fp64 rescore + certificate
//   exact_scan_kernel      tier-2: full canonical fp64 scan for queries whose certificate failed
//   merge_topk_kernel      cross-shard reduce of exact hit lists (after the NCCL all-gather)
#pragma once
#include "common.cuh"

namespace rfk {

constexpr int kScanThreads = 256;
constexpr int kScanWarps = kScanThreads / kWarp;
constexpr int kFinThreads = 1024;
constexpr int kFinWarps = kFinThreads / kWarp;

// ---------------------------------------------------------------------------------
// K1: one warp per row.  n2 = canonical fp64 sum of squares; y = RNE_store(RNE_f32(x * 1/sqrt(n2))).
// SYNTH: the source row is generated in registers from the counter hash instead of read.
// dst rows have stride ld (>= dim, multiple of 8); columns [dim, ld) are zero.
// ---------------------------------------------------------------------------------
// SYNTH with topic_rows > 0: "templated corpus" generator - row r belongs to topic r / topic_rows and is
//   centre(topic) + noise(r) * noise_scale     (noise_scale a power of two <= 1/2: the sum is exact in fp32),
// i.e. contiguous runs of topic_rows near-duplicates (cosine ~0.98 to each other at scale 1/8), inserted in topic order.
// DT = 3 (RAGFIN_F32_F16): the fp32 row exactly as DT = 0 stores it, and RNE_f16 of each stored value into dst16 - the
// same bits DT = 2 stores for the same input, since both round the same fp32 y.
template <int DT> using IngestT = typename Store<DT == 3 ? 0 : DT>::T;
template <int DT, bool SYNTH>
__global__ void __launch_bounds__(256) ingest_kernel(const float* __restrict__ src, uint64_t synth_key,
                                                     int64_t synth_row0, int dup_every, int zero_every,
                                                     int64_t n, int dim, int ld,
                                                     IngestT<DT>* __restrict__ dst,
                                                     int64_t topic_rows = 0, uint64_t topic_key = 0, float noise_scale = 0.f,
                                                     __half* __restrict__ dst16 = nullptr) {
    typedef IngestT<DT> T;
    const int lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = gw; r < n; r += nw) {
        uint64_t srow = 0;
        bool zero = false;
        const float* x = nullptr;
        if (SYNTH) {
            const uint64_t row = (uint64_t)(synth_row0 + r);
            srow = row;
            if (dup_every > 1 && row % (uint64_t)dup_every == (uint64_t)(dup_every - 1)) srow = row - 1;
            zero = zero_every > 1 && row % (uint64_t)zero_every == (uint64_t)(zero_every - 1);
        } else {
            x = src + r * (int64_t)dim;
        }
        const uint64_t topic = SYNTH && topic_rows > 0 ? srow / (uint64_t)topic_rows : 0;
        auto elem = [&](int i) -> float {
            if (SYNTH) {
                if (zero) return 0.0f;
                const float v = synth_value(synth_key, srow, dim, i);
                return topic_rows > 0 ? __fadd_rn(synth_value(topic_key, topic, dim, i), __fmul_rn(v, noise_scale)) : v;
            }
            return x[i];
        };
        double acc = 0.0;
        for (int i = lane; i < dim; i += kWarp) {
            const double v = (double)elem(i);
            acc = acc + v * v;
        }
        const double n2 = warp_butterfly_f64(acc);
        const double inv = inv_norm(n2);
        T* out = dst + r * (int64_t)ld;
        for (int i = lane * 2; i < ld; i += 2 * kWarp) {
            const float y0 = i < dim ? norm_elem(elem(i), inv) : 0.0f;
            const float y1 = i + 1 < dim ? norm_elem(elem(i + 1), inv) : 0.0f;
            if (DT == 0 || DT == 3) {
                *reinterpret_cast<float2*>(out + i) = make_float2(y0, y1);
                if (DT == 3) *reinterpret_cast<__half2*>(dst16 + r * (int64_t)ld + i) = __halves2half2(__float2half_rn(y0), __float2half_rn(y1));
            } else {
                T pr[2] = {Store<DT == 3 ? 0 : DT>::from_f32(y0), Store<DT == 3 ? 0 : DT>::from_f32(y1)};
                *reinterpret_cast<uint32_t*>(out + i) = *reinterpret_cast<uint32_t*>(pr);
            }
        }
    }
}

// ---------------------------------------------------------------------------------
// K1, vectorised (the default for host / device fp32 sources with dim % 4 == 0 and dim <= 128 * NV): one warp per row,
// the row is read ONCE with 128-bit loads (lane l, vector j holds elements [(32 j + l) * 4, +4)) and kept in registers.
// The canonical sum of squares wants lane p to add the elements i = p, p + 32, ... in increasing i (DESIGN.md 2), which
// is not the vector layout, so the warp transposes the row through its 128 NV * 16 bytes of shared memory (STS.128
// in, conflict-free LDS.32 out); every lane then scales the elements it holds in registers and stores them with one
// 64-bit (16-bit storage) or 128-bit (fp32 storage) store per vector.  Same bits as ingest_kernel.
// Algorithmic HBM bytes per row: 4 * dim read + ld * sizeof(T) written (+ ld * 2 for the fp16 copy of DT = 3).
// ---------------------------------------------------------------------------------
constexpr int kIngestThreads = 256;
constexpr int kIngestWarps = kIngestThreads / kWarp;

template <int DT, int NV>
__global__ void __launch_bounds__(kIngestThreads) ingest_vec_kernel(const float* __restrict__ src, int64_t n, int dim, int ld,
                                                                      IngestT<DT>* __restrict__ dst, __half* __restrict__ dst16 = nullptr) {
    typedef IngestT<DT> T;
    __shared__ __align__(16) float stage[kIngestWarps][NV * 128];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t gw = (int64_t)blockIdx.x * kIngestWarps + warp;
    const int64_t nw = (int64_t)gridDim.x * kIngestWarps;
    const int nvec = dim >> 2;                      // 16-byte vectors of the source row
    const int nvec_out = ld >> 2;                   // groups of 4 output elements (ld % 8 == 0)
    float* mine = stage[warp];
    for (int64_t r = gw; r < n; r += nw) {
        const float4* x = reinterpret_cast<const float4*>(src + r * (int64_t)dim);
        float4 v[NV];
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int vi = j * kWarp + lane;
            v[j] = vi < nvec ? __ldcs(x + vi) : make_float4(0.f, 0.f, 0.f, 0.f);   // streaming: read once
        }
#pragma unroll
        for (int j = 0; j < NV; ++j) *reinterpret_cast<float4*>(mine + (j * kWarp + lane) * 4) = v[j];
        __syncwarp();
        double acc = 0.0;
#pragma unroll 8
        for (int i = lane; i < dim; i += kWarp) {
            const double t = (double)mine[i];
            acc = acc + t * t;
        }
        __syncwarp();                               // the staging row is free for the next iteration
        const double n2 = warp_butterfly_f64(acc);
        const double inv = inv_norm(n2);
        T* out = dst + r * (int64_t)ld;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int vi = j * kWarp + lane;
            if (vi < nvec_out) {                    // vectors in [nvec, nvec_out) are the zero padding of the stored row
                const float y0 = norm_elem(v[j].x, inv), y1 = norm_elem(v[j].y, inv);
                const float y2 = norm_elem(v[j].z, inv), y3 = norm_elem(v[j].w, inv);
                if (DT == 0 || DT == 3) {
                    __stcs(reinterpret_cast<float4*>(out) + vi, make_float4(y0, y1, y2, y3));
                    if (DT == 3) {
                        const __half2 h01 = __halves2half2(__float2half_rn(y0), __float2half_rn(y1));
                        const __half2 h23 = __halves2half2(__float2half_rn(y2), __float2half_rn(y3));
                        __stcs(reinterpret_cast<uint2*>(dst16 + r * (int64_t)ld) + vi,
                               make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23)));
                    }
                } else {
                    typedef Store<DT == 3 ? 0 : DT> S;
                    T pr[4] = {S::from_f32(y0), S::from_f32(y1), S::from_f32(y2), S::from_f32(y3)};
                    __stcs(reinterpret_cast<uint2*>(out) + vi, *reinterpret_cast<uint2*>(pr));
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------
// fp16 copy of stored fp32 rows (ragfin_load of a RAGFIN_F32_F16 file): dst[i] = RNE_f16(src[i]), 4 elements per thread
// and step (128-bit loads, 64-bit stores) - the same bits the DT = 3 ingest stores.
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cast_f16_kernel(const float4* __restrict__ src, uint2* __restrict__ dst, int64_t n4) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 v = __ldcs(src + i);
        const __half2 h01 = __halves2half2(__float2half_rn(v.x), __float2half_rn(v.y));
        const __half2 h23 = __halves2half2(__float2half_rn(v.z), __float2half_rn(v.w));
        __stcs(dst + i, make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23)));
    }
}

// ---------------------------------------------------------------------------------
// Transposed warp reduction: every lane holds M partial sums (M a power of two <= 32);
// afterwards lane l holds the warp-wide total of value index (l >> (5 - log2 M)).
// log2(M) exchange rounds halve the live values, the remaining rounds are a plain butterfly:
// M + (5 - log2 M) - 1 shuffles instead of 5 * M.
// ---------------------------------------------------------------------------------
template <int C, int OFF>
struct TransposeReduce {
    template <int M>
    __device__ static __forceinline__ void run(float (&v)[M], int lane) {
        if (C > 1) {
            const bool upper = (lane & OFF) != 0;
#pragma unroll
            for (int i = 0; i < C / 2; ++i) {
                const float keep = upper ? v[i + C / 2] : v[i];
                const float send = upper ? v[i] : v[i + C / 2];
                v[i] = keep + __shfl_xor_sync(kFull, send, OFF);
            }
        } else {
            v[0] = v[0] + __shfl_xor_sync(kFull, v[0], OFF);
        }
        TransposeReduce<(C > 1 ? C / 2 : 1), OFF / 2>::run(v, lane);
    }
};
template <int C>
struct TransposeReduce<C, 0> {
    template <int M>
    __device__ static __forceinline__ void run(float (&)[M], int) {}
};
__host__ __device__ constexpr int ilog2(int x) { return x <= 1 ? 0 : 1 + ilog2(x / 2); }

// rows held in flight per warp iteration, by vectors per lane per row
__host__ __device__ constexpr int scan_rows(int steps) { return steps <= 1 ? 8 : steps <= 3 ? 4 : steps <= 6 ? 2 : 1; }

// ---------------------------------------------------------------------------------
// K2: small-batch scan.  Each warp streams R rows per iteration with 128-bit
// ld.global.nc loads (lane l, step j covers elements [(j*32+l)*V, +V)), holds the NQ
// normalised queries in registers as fp32, accumulates in fp32, reduces with the
// transposed butterfly and keeps a sorted top-K' key list per (warp, query) in shared
// memory behind a register threshold, so a row costs one compare in the common case.
// At the end the CTA merges its warps' lists and writes K' keys per query:
//   cand[q * cand_q_stride + blockIdx.x * kp + i],  sorted descending, 0 = empty.
// Algorithmic HBM bytes: n_rows * ld * sizeof(T) (one pass), independent of NQ.
// ---------------------------------------------------------------------------------
template <int DT, int NQ, int STEPS>
__global__ void __launch_bounds__(kScanThreads, NQ >= 4 ? 1 : 2)
scan_topk_kernel(const void* __restrict__ data, int64_t n_rows, int ld, const float* __restrict__ qhat,
                 int nq_valid, int kp, u64* __restrict__ cand, int64_t cand_q_stride,
                 const uint32_t* __restrict__ allow) {
    typedef Store<DT> S;
    constexpr int V = S::kVec;
    constexpr int R = scan_rows(STEPS);
    constexpr int M = R * NQ;
    constexpr int SH = 5 - ilog2(M);
    static_assert(M <= 32, "too many partial sums per lane");
    extern __shared__ __align__(16) u64 lists[];  // [NQ][kScanWarps][kp]

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < NQ * kScanWarps * kp; i += kScanThreads) lists[i] = 0;
    __syncthreads();

    const int nvec = ld / V;
    float qreg[NQ][STEPS * V];
#pragma unroll
    for (int q = 0; q < NQ; ++q)
#pragma unroll
        for (int j = 0; j < STEPS; ++j) {
            const int vi = j * kWarp + lane;
#pragma unroll
            for (int e = 0; e < V; ++e) qreg[q][j * V + e] = vi < nvec ? qhat[(size_t)q * ld + vi * V + e] : 0.0f;
        }

    float tau[NQ];   // padding queries (zero rows beyond nq_valid) never collect
#pragma unroll
    for (int q = 0; q < NQ; ++q) tau[q] = q < nq_valid ? -INFINITY : INFINITY;

    const char* base = reinterpret_cast<const char*>(data);
    const size_t row_bytes = (size_t)ld * sizeof(typename S::T);
    const int64_t chunks = (n_rows + R - 1) / R;
    const int64_t stride = (int64_t)gridDim.x * kScanWarps;
    for (int64_t c = (int64_t)blockIdx.x * kScanWarps + warp; c < chunks; c += stride) {
        const int64_t row0 = c * R;
        uint4 d[R][STEPS];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            int64_t rr = row0 + r;
            rr = rr < n_rows ? rr : n_rows - 1;
            const char* rp = base + (size_t)rr * row_bytes;
#pragma unroll
            for (int j = 0; j < STEPS; ++j) {
                const int vi = j * kWarp + lane;
                d[r][j] = vi < nvec ? ldg_stream(rp + (size_t)vi * 16) : make_uint4(0, 0, 0, 0);
            }
        }
        float acc[M];
#pragma unroll
        for (int i = 0; i < M; ++i) acc[i] = 0.0f;
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int j = 0; j < STEPS; ++j) {
                float f[V];
                S::unpack(d[r][j], f);
#pragma unroll
                for (int q = 0; q < NQ; ++q)
#pragma unroll
                    for (int e = 0; e < V; ++e) acc[r * NQ + q] = fmaf(f[e], qreg[q][j * V + e], acc[r * NQ + q]);
            }
        TransposeReduce<M, 16>::run(acc, lane);
        const float s = acc[0];
        const int idx = lane >> SH;
        const int myq = idx % NQ;
        float mytau = tau[0];
#pragma unroll
        for (int q = 1; q < NQ; ++q) mytau = myq == q ? tau[q] : mytau;
        const bool leader = (lane & ((1 << SH) - 1)) == 0;
        const bool hit = leader && (row0 + idx / NQ < n_rows) && (s >= mytau);
        unsigned mask = __ballot_sync(kFull, hit);
        while (mask) {
            const int l = __ffs(mask) - 1;
            mask &= mask - 1;
            const float bs = __shfl_sync(kFull, s, l) + 0.0f;
            const int bidx = l >> SH;
            const int q = bidx % NQ;
            if (allow != nullptr && !row_allowed(allow, row0 + bidx / NQ)) continue;   // scalar filter (warp-uniform)
            const u64 key = make_key(bs, (uint32_t)(row0 + bidx / NQ));
            u64* list = lists + (size_t)(q * kScanWarps + warp) * kp;
            if (key > list[kp - 1]) {
                warp_list_insert(list, kp, key, lane);
                const u64 last = list[kp - 1];
                const float nt = last ? key_score(last) : -INFINITY;
#pragma unroll
                for (int qq = 0; qq < NQ; ++qq) tau[qq] = q == qq ? nt : tau[qq];
            }
        }
    }
    __syncthreads();
#pragma unroll 1
    for (int q = 0; q < NQ; ++q) {
        u64* region = lists + (size_t)q * kScanWarps * kp;
        block_bitonic_sort_desc(region, kScanWarps * kp, threadIdx.x, kScanThreads);
        u64* out = cand + (size_t)q * cand_q_stride + (size_t)blockIdx.x * kp;
        for (int i = threadIdx.x; i < kp; i += kScanThreads) out[i] = region[i];
    }
}

// ---------------------------------------------------------------------------------
// Merge `G` descending key lists of length kp into FW per-warp lists, then one sort.
// wl: shared [kFinWarps][kp].  On return (after __syncthreads) wl[0..kp) is the top-kp.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void merge_lists(const u64* __restrict__ src, int G, int kp, u64* wl, bool sorted_lists) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int mw = 4096 / kp;                       // merging warps: their lists must fit the 4096-key buffer
    if (mw > kFinWarps) mw = kFinWarps;
    if (warp < mw) {
        u64* mine = wl + (size_t)warp * kp;
        for (int i = lane; i < kp; i += kWarp) mine[i] = 0;
        __syncwarp();
        for (int l = warp; l < G; l += mw) {
            const u64* in = src + (size_t)l * kp;
            for (int s = 0; s < kp; s += kWarp) {
                const u64 key = in[s + lane];
                const unsigned hits = __ballot_sync(kFull, key > mine[kp - 1]);
                unsigned m = hits;
                while (m) {
                    const int b = __ffs(m) - 1;
                    m &= m - 1;
                    const u64 bk = __shfl_sync(kFull, key, b);
                    if (bk > mine[kp - 1]) warp_list_insert(mine, kp, bk, lane);
                }
                if (sorted_lists && hits != kFull) break;  // sorted list: nothing further can qualify
            }
        }
    }
    __syncthreads();
    block_bitonic_sort_desc(wl, mw * kp, threadIdx.x, kFinThreads);
}

template <int DT>
__device__ __forceinline__ double rescore_row(const void* data, int64_t row, int ld, const float* q, int lane) {
    const typename Store<DT>::T* rp = reinterpret_cast<const typename Store<DT>::T*>(data) + (size_t)row * ld;
    return canonical_dot_row<DT>(rp, q, ld, lane);
}

// ---------------------------------------------------------------------------------
// K4: one CTA per query.
//  EXACT_IN = false: keys carry APPROXIMATE scores.  Select the top-kp, recompute those
//    kp dot products canonically in fp64 from the stored values, order by the exact key and
//    certify: every row outside the candidate set has approx <= tau (the kp-th approx
//    score) hence exact <= tau + eps; if exact_k > tau + eps the top-k is proven exact.
//    Otherwise flags[q] = 1 and the query goes to the exact-rescan tier.
//  EXACT_IN = true: keys already carry exact scores (tier 2); only flagged queries run.
// ---------------------------------------------------------------------------------
constexpr int kFinCap = 4096;     // survivor buffer, keys; the fallback merge uses kFinCap / kp warps
constexpr int kFinHeads = 1024;   // most candidate lists per query the head-threshold shortcut handles

// Top-kp of G candidate lists into buf[0..kp) (descending), without touching most of the input:
//  * sorted lists (scan / exact tier): the kp-th largest list HEAD is a lower bound of the kp-th
//    largest key overall (kp heads are >= it), so only each list's prefix above it can matter;
//  * unsorted lists (tensor-core path): the bound is gtau[q], the best list minimum published
//    during the sweep.
// Survivors are appended to shared memory and bitonic-sorted; if they overflow (adversarial input)
// the streaming per-warp merge below is used instead.
__device__ __forceinline__ void select_top(const u64* __restrict__ src, int G, int kp, bool sorted_lists, u64 bound,
                                           u64* buf, u64* heads, int* s_cnt, u64* s_tau) {
    const int tid = threadIdx.x;
    if (tid == 0) { *s_cnt = 0; *s_tau = bound; }
    if (sorted_lists && G >= kp && G <= kFinHeads) {
        for (int i = tid; i < G; i += kFinThreads) heads[i] = src[(size_t)i * kp];
        __syncthreads();
        for (int i = tid; i < G; i += kFinThreads) {
            const u64 my = heads[i];
            if (my == 0) continue;
            int r = 0;
            for (int j = 0; j < G; ++j) r += heads[j] > my;
            if (r == kp - 1) *s_tau = my;   // keys are unique: exactly one thread writes
        }
    }
    __syncthreads();
    const u64 tau0 = *s_tau;
    if (sorted_lists) {
        for (int l = tid; l < G; l += kFinThreads) {
            const u64* in = src + (size_t)l * kp;
            for (int e = 0; e < kp; ++e) {
                const u64 key = in[e];
                if (key == 0 || key < tau0) break;
                const int pos = atomicAdd(s_cnt, 1);
                if (pos < kFinCap) buf[pos] = key;
            }
        }
    } else {
        for (int i = tid; i < G * kp; i += kFinThreads) {
            const u64 key = src[i];
            if (key != 0 && key >= tau0) {
                const int pos = atomicAdd(s_cnt, 1);
                if (pos < kFinCap) buf[pos] = key;
            }
        }
    }
    __syncthreads();
    const int n = *s_cnt;
    if (n > kFinCap) {   // overflow: streaming merge over everything
        __syncthreads();
        merge_lists(src, G, kp, buf, sorted_lists);
        return;
    }
    int P = kp;
    while (P < n) P <<= 1;
    for (int i = n + tid; i < P; i += kFinThreads) buf[i] = 0;
    __syncthreads();
    block_bitonic_sort_desc(buf, P, tid, kFinThreads);
}

// ---------------------------------------------------------------------------------
// K4: one CTA per query.
//  EXACT_IN = false: keys carry APPROXIMATE scores.  Select the top-kp, recompute those
//    kp dot products canonically in fp64 from the stored values, order by the exact key and
//    certify: every row outside the candidate set has approx <= tau (the kp-th approx
//    score) hence exact <= tau + eps; if exact_k > tau + eps the top-k is proven exact.
//    Otherwise flags[q] = 1 and the query goes to the exact-rescan tier.
//  EXACT_IN = true: keys already carry exact scores (tier 2); only flagged queries run.
// ---------------------------------------------------------------------------------
template <bool EXACT_IN>
__global__ void __launch_bounds__(kFinThreads)
finalize_kernel(const u64* __restrict__ cand, int G, int kp, const void* __restrict__ data, int dt,
                int64_t n_rows, int scanned, int sorted_lists, const uint32_t* __restrict__ gtau, int ld,
                const float* __restrict__ qhat, float eps_const,
                const float* __restrict__ eps_q, int k, int64_t id_base, int64_t* __restrict__ out_ids,
                float* __restrict__ out_scores, int* __restrict__ flags, int* __restrict__ flag_count) {
    __shared__ __align__(16) u64 buf[kFinCap];
    __shared__ __align__(16) u64 ex[256];
    __shared__ __align__(16) u64 heads[kFinHeads];
    __shared__ int s_cnt;
    __shared__ u64 s_tau;
    const int q = blockIdx.x;
    if (EXACT_IN && flags[q] == 0) return;
    u64 bound = 0;
    if (!sorted_lists && gtau != nullptr) bound = (u64)gtau[q] << 32;   // key >= bound  <=>  score >= published bound
    select_top(cand + (size_t)q * G * kp, G, kp, sorted_lists != 0, bound, buf, heads, &s_cnt, &s_tau);
    const u64* wl = buf;

    const int keff = (int64_t)k < n_rows ? k : (int)n_rows;
    const u64* fin = wl;
    if (!EXACT_IN) {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const float* qv = qhat + (size_t)q * ld;
        for (int c = warp; c < kp; c += kFinWarps) {
            const u64 key = wl[c];
            u64 ek = 0;
            if (key) {
                const uint32_t row = key_row(key);
                double s;
                if (dt == 0) s = rescore_row<0>(data, row, ld, qv, lane);
                else if (dt == 1) s = rescore_row<1>(data, row, ld, qv, lane);
                else s = rescore_row<2>(data, row, ld, qv, lane);
                ek = make_key((float)s + 0.0f, row);
            }
            if (lane == 0) ex[c] = ek;
        }
        __syncthreads();
        block_bitonic_sort_desc(ex, kp, threadIdx.x, kFinThreads);
        if (threadIdx.x == 0) {
            bool ok = scanned && n_rows <= (int64_t)kp;
            if (!ok && scanned && keff > 0) {
                const double eps = (double)eps_const + (eps_q ? (double)eps_q[q] : 0.0);
                const double tau = (double)key_score(wl[kp - 1]);
                ok = ex[keff - 1] != 0 && (double)key_score(ex[keff - 1]) > tau + eps;
            }
            flags[q] = ok ? 0 : 1;
            if (!ok) atomicAdd(flag_count, 1);
        }
        fin = ex;
    }
    for (int i = threadIdx.x; i < k; i += kFinThreads) {
        const u64 key = i < keff ? fin[i] : 0;
        out_ids[(size_t)q * k + i] = key ? id_base + (int64_t)key_row(key) : -1;
        out_scores[(size_t)q * k + i] = key ? key_score(key) : -INFINITY;
    }
}

// ---------------------------------------------------------------------------------
// Block-wide selection of the `want`-th largest (1-based) of m 32-bit values hi_of(0..m), by histogram narrowing:
// 256 linear bins over [lo, hi], keep the bin that holds the wanted rank, repeat until the bin is one value wide
// (<= 4 passes over the data for 32-bit values).  hist: 256 words, s3: 3 words of shared memory.  Every thread
// of the block must call it (it synchronises); m >= want >= 1.
// ---------------------------------------------------------------------------------
template <typename F>
__device__ __forceinline__ uint32_t block_kth_largest(F hi_of, int m, uint32_t want0, uint32_t* hist, uint32_t* s3) {
    const int tid = threadIdx.x, nthreads = blockDim.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { s3[0] = 0xFFFFFFFFu; s3[1] = 0u; s3[2] = want0; }
    __syncthreads();
    {
        uint32_t lo = 0xFFFFFFFFu, hi = 0u;
        for (int i = tid; i < m; i += nthreads) {
            const uint32_t h = hi_of(i);
            lo = h < lo ? h : lo;
            hi = h > hi ? h : hi;
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            const uint32_t l2 = __shfl_xor_sync(kFull, lo, off), h2 = __shfl_xor_sync(kFull, hi, off);
            lo = l2 < lo ? l2 : lo;
            hi = h2 > hi ? h2 : hi;
        }
        if (lane == 0) { atomicMin(&s3[0], lo); atomicMax(&s3[1], hi); }
    }
    __syncthreads();
    for (int pass = 0; pass < 6; ++pass) {
        const uint32_t lo = s3[0], hi = s3[1], want = s3[2];
        if (lo == hi) break;                                  // block-uniform: one value left
        const uint32_t range = hi - lo;
        const int bits = 32 - __clz(range);                   // range < 2^bits
        const int sh = bits > 8 ? bits - 8 : 0;               // (range >> sh) <= 255
        for (int i = tid; i < 256; i += nthreads) hist[i] = 0;
        __syncthreads();
        for (int i = tid; i < m; i += nthreads) {
            const uint32_t h = hi_of(i);
            if (h >= lo && h <= hi) atomicAdd(&hist[(h - lo) >> sh], 1u);
        }
        __syncthreads();
        if (warp == 0) {   // bin (from the top) in which the cumulative count reaches `want`; lane l owns bins 255-8l .. 248-8l
            uint32_t c[8], sum = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { c[j] = hist[255 - 8 * lane - j]; sum += c[j]; }
            uint32_t incl = sum;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t t = __shfl_up_sync(kFull, incl, off);
                if (lane >= off) incl += t;
            }
            const uint32_t before = incl - sum;               // values in the bins above this lane's
            if (before < want && incl >= want) {              // exactly one lane
                uint32_t run = before;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (run < want && run + c[j] >= want) {
                        const uint32_t bin = (uint32_t)(255 - 8 * lane - j);
                        const uint32_t nlo = lo + (bin << sh);
                        uint32_t nhi = nlo + ((1u << sh) - 1u);
                        if (nhi > hi || nhi < nlo) nhi = hi;
                        s3[0] = nlo; s3[1] = nhi; s3[2] = want - run;
                    }
                    run += c[j];
                }
            }
        }
        __syncthreads();
    }
    return s3[0];
}

// ---------------------------------------------------------------------------------
// K4 for the append mode of the tensor-core path: one CTA of 256 threads per query, O(m) work, ~18 KB of shared
// memory (several CTAs per SM).
//   buf[q][0..m)  keys (approximate score, row) of EVERY row whose approximate score reached thr[q], any order
// With eps >= |approx - exact| for every row:  T = k-th largest approximate score (it is in the buffer, because
// thr <= T - 2 eps), and every row of the exact top-k has approx >= T - 2 eps.  So:
//   1. select T: histogram narrowing over the ordered-uint scores (256 linear bins over [lo, hi], keep the bin that
//      holds the k-th largest, repeat until the bin is one value wide: <= 4 passes over the buffer);
//   2. gather the rows with approx >= T - 2 eps (~1.6 k of them) into shared memory;
//   3. recompute those rows canonically in fp64, order by the exact key, emit k.
// Unconditionally exact - there is no certificate to fail; only an overflowing buffer (m > cap, or more than
// kAppendRescore rows above the cut: massive duplication) sends the query to tier 2.
// Range search (radius < score <= range_filter, DESIGN.md 7c; open bounds are infinite): the buffer holds the rows with
// approx in [max(thr, lo), hi] and may hold fewer than k.  T is selected among the rows CERTAINLY in the window
// (radius + e < approx <= range_filter - e); if fewer than k are, every buffer row is rescored.  The exact fp32 window is
// applied to the rescored scores before the top k are taken.
// ---------------------------------------------------------------------------------
constexpr int kAppendRescore = 2048;   // most rows one query may rescore exactly
constexpr int kFaThreads = 256;
constexpr int kFaWarps = kFaThreads / kWarp;

__global__ void __launch_bounds__(kFaThreads)
finalize_append_kernel(const u64* __restrict__ buf, const uint32_t* __restrict__ cnt, int cap,
                       const void* __restrict__ data, int dt, int64_t n_rows, int ld, const float* __restrict__ qhat,
                       float eps_const, const float* __restrict__ eps_q, int k, int64_t id_base,
                       int64_t* __restrict__ out_ids, float* __restrict__ out_scores, int* __restrict__ flags,
                       int* __restrict__ flag_count, float radius, float range_filter) {
    __shared__ __align__(16) u64 sel[kAppendRescore];
    __shared__ uint32_t hist[256];
    __shared__ uint32_t s3[3];
    __shared__ int s_c2, s_sure;
    const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool window = radius > -INFINITY || range_filter < INFINITY;
    const uint32_t m32 = cnt[q];
    const int keff = (int64_t)k < n_rows ? k : (int)n_rows;
    // fewer than k rows cannot happen with a valid bound - except in a range search, whose window may hold fewer
    const bool overflow = m32 > (uint32_t)cap || (!window && (int)m32 < keff);
    const int m = overflow ? 0 : (int)m32;
    const u64* in = buf + (size_t)q * cap;
    const float eps = eps_const + (eps_q ? eps_q[q] : 0.0f);
    if (tid == 0) { s_c2 = 0; s_sure = 0; }
    __syncthreads();
    if (window && !overflow && m > 0) {   // block-uniform
        const float ew = __fadd_ru(eps, 2.384185791015625e-07f);
        const float sure_lo = __fadd_ru(radius, ew), sure_hi = __fsub_rd(range_filter, ew);
        int c = 0;
        for (int i = tid; i < m; i += kFaThreads) { const float s = key_score(in[i]); c += s > sure_lo && s <= sure_hi; }
        c = __reduce_add_sync(kFull, c);
        if (lane == 0 && c) atomicAdd(&s_sure, c);
        __syncthreads();
        if (s_sure < keff) {   // T would not be a bound: every buffer row goes to the exact rescore
            for (int i = tid; i < m; i += kFaThreads) {
                const int pos = atomicAdd(&s_c2, 1);
                if (pos < kAppendRescore) sel[pos] = in[i];
            }
            __syncthreads();
        } else {
            const uint32_t t_ord = block_kth_largest([&](int i) {
                const float s = key_score(in[i]);
                return s > sure_lo && s <= sure_hi ? (uint32_t)(in[i] >> 32) : 0u;
            }, m, (uint32_t)keff, hist, s3);
            const float cut = __fsub_rd(__fsub_rd(ordered_to_float(t_ord), __fmul_ru(2.0f, eps)), 2.384185791015625e-07f);
            for (int i = tid; i < m; i += kFaThreads) {
                const u64 key = in[i];
                if (key_score(key) >= cut) {
                    const int pos = atomicAdd(&s_c2, 1);
                    if (pos < kAppendRescore) sel[pos] = key;
                }
            }
            __syncthreads();
        }
    }
    if (overflow || keff == 0) {   // block-uniform
        if (tid == 0) { flags[q] = overflow ? 1 : 0; if (overflow) atomicAdd(flag_count, 1); }
        if (!overflow)
            for (int i = tid; i < k; i += kFaThreads) { out_ids[(size_t)q * k + i] = -1; out_scores[(size_t)q * k + i] = -INFINITY; }
        return;
    }
    if (!window) {
        // ---- 1. T = keff-th largest approximate score, as an ordered uint ----
        const uint32_t t_ord = block_kth_largest([&](int i) { return (uint32_t)(in[i] >> 32); }, m, (uint32_t)keff, hist, s3);
        // ---- 2. gather the rows above the cut ----
        const float cut = __fsub_rd(__fsub_rd(ordered_to_float(t_ord), __fmul_ru(2.0f, eps)), 2.384185791015625e-07f);
        for (int i = tid; i < m; i += kFaThreads) {
            const u64 key = in[i];
            if (key_score(key) >= cut) {
                const int pos = atomicAdd(&s_c2, 1);
                if (pos < kAppendRescore) sel[pos] = key;
            }
        }
        __syncthreads();
    }
    const int c2 = s_c2;
    if (c2 > kAppendRescore) {   // block-uniform
        if (tid == 0) { flags[q] = 1; atomicAdd(flag_count, 1); }
        return;
    }
    // ---- 3. exact rescore, order, emit ----
    const float* qv = qhat + (size_t)q * ld;
    for (int c = warp; c < c2; c += kFaWarps) {
        const uint32_t row = key_row(sel[c]);
        double sc;
        if (dt == 0) sc = rescore_row<0>(data, row, ld, qv, lane);
        else if (dt == 1) sc = rescore_row<1>(data, row, ld, qv, lane);
        else sc = rescore_row<2>(data, row, ld, qv, lane);
        __syncwarp();
        const float s = (float)sc + 0.0f;
        if (lane == 0) sel[c] = s > radius && s <= range_filter ? make_key(s, row) : 0ull;   // the exact window
    }
    int P2 = 32;
    while (P2 < c2) P2 <<= 1;
    for (int i = c2 + tid; i < P2; i += kFaThreads) sel[i] = 0ull;
    __syncthreads();
    block_bitonic_sort_desc(sel, P2, tid, kFaThreads);
    for (int i = tid; i < k; i += kFaThreads) {
        const u64 key = i < keff ? sel[i] : 0;
        out_ids[(size_t)q * k + i] = key ? id_base + (int64_t)key_row(key) : -1;
        out_scores[(size_t)q * k + i] = key ? key_score(key) : -INFINITY;
    }
    if (tid == 0) flags[q] = 0;
}

// ---------------------------------------------------------------------------------
// Tier 2: canonical fp64 score of EVERY row for the flagged queries, exact keys, per-warp
// lists of kpe entries, CTA merge.  Exits immediately when nothing is flagged.
// cand_e[(q * gridDim.x + blockIdx.x) * kpe + i]
// ---------------------------------------------------------------------------------
template <int DT>
__global__ void __launch_bounds__(kScanThreads)
exact_scan_kernel(const void* __restrict__ data, int64_t n_rows, int ld, const float* __restrict__ qhat,
                  int nq, const int* __restrict__ flags, const int* __restrict__ flag_count, int kpe,
                  u64* __restrict__ cand_e, const uint32_t* __restrict__ allow, float radius, float range_filter) {
    if (*flag_count == 0) return;
    extern __shared__ __align__(16) u64 lists[];  // [kScanWarps][kpe]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const typename Store<DT>::T* base = reinterpret_cast<const typename Store<DT>::T*>(data);
    for (int q = 0; q < nq; ++q) {
        if (flags[q] == 0) continue;  // block-uniform
        for (int i = threadIdx.x; i < kScanWarps * kpe; i += kScanThreads) lists[i] = 0;
        __syncthreads();
        u64* mine = lists + (size_t)warp * kpe;
        const float* qv = qhat + (size_t)q * ld;
        const int64_t stride = (int64_t)gridDim.x * kScanWarps;
        for (int64_t r = (int64_t)blockIdx.x * kScanWarps + warp; r < n_rows; r += stride) {
            if (allow != nullptr && !row_allowed(allow, r)) continue;
            const double s = canonical_dot_row<DT>(base + (size_t)r * ld, qv, ld, lane);
            const float s32 = (float)s + 0.0f;
            if (!(s32 > radius && s32 <= range_filter)) continue;   // outside a range search's window (open bounds are infinite)
            const u64 key = make_key(s32, (uint32_t)r);
            if (key > mine[kpe - 1]) warp_list_insert(mine, kpe, key, lane);
        }
        __syncthreads();
        block_bitonic_sort_desc(lists, kScanWarps * kpe, threadIdx.x, kScanThreads);
        u64* out = cand_e + ((size_t)q * gridDim.x + blockIdx.x) * kpe;
        for (int i = threadIdx.x; i < kpe; i += kScanThreads) out[i] = lists[i];
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------
// Cross-shard reduce.  Each part's list is sorted by (score desc, id asc) with -1 padding at
// the end and all ids are distinct, so the global rank of an element is its own index plus,
// for every other part, the number of that part's elements that beat it (binary search).
// ---------------------------------------------------------------------------------
__device__ __forceinline__ bool hit_better(float sa, int64_t ia, float sb, int64_t ib) {
    return sa > sb || (sa == sb && ia < ib);
}
// PEER = true: the lists are written by other GPUs DURING this kernel (exchange_merge_kernel); they must be read with
// coherent loads (ld.global.cg, never the non-coherent .nc path, which PTX only allows for memory that is read-only for
// the kernel's lifetime and which the acquire on the flag does not order).
template <bool PEER> __device__ __forceinline__ int64_t ld_hit_id(const int64_t* p) { return PEER ? __ldcg(p) : *p; }
template <bool PEER> __device__ __forceinline__ float ld_hit_score(const float* p) { return PEER ? __ldcg(p) : *p; }
template <bool PEER>
__device__ __forceinline__ int count_better(const int64_t* ids, const float* sc, int k, float s, int64_t id) {
    int lo = 0, hi = k;  // first index whose element does NOT beat (s, id); padding never beats
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const int64_t im = ld_hit_id<PEER>(ids + mid);
        const bool b = im >= 0 && hit_better(ld_hit_score<PEER>(sc + mid), im, s, id);
        if (b) lo = mid + 1; else hi = mid;
    }
    return lo;
}
template <bool PEER>
__device__ __forceinline__ void merge_topk_body(const int64_t* ids, const float* scores, int nq,
                                                int parts, int k, int64_t ips, int64_t sps, int64_t query_stride,
                                                int64_t* __restrict__ out_ids, float* __restrict__ out_scores) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t per_q = (int64_t)parts * k;
    if (t >= (int64_t)nq * per_q) return;
    const int q = (int)(t / per_q);
    const int e = (int)(t % per_q);
    const int p = e / k, i = e % k;
    const int64_t* qi = ids + (size_t)q * query_stride;
    const float* qs = scores + (size_t)q * query_stride;
    if (p == 0) {  // slot i of the output: pad it if fewer than i+1 valid hits exist in total
        int valid = 0;
        for (int pp = 0; pp < parts; ++pp)
            valid += count_better<PEER>(qi + (size_t)pp * ips, qs + (size_t)pp * sps, k, -INFINITY, INT64_MAX);
        if (i >= valid) { out_ids[(size_t)q * k + i] = -1; out_scores[(size_t)q * k + i] = -INFINITY; }
    }
    const int64_t id = ld_hit_id<PEER>(qi + (size_t)p * ips + i);
    if (id < 0) return;
    const float s = ld_hit_score<PEER>(qs + (size_t)p * sps + i);
    int rank = i;
    for (int pp = 0; pp < parts && rank < k; ++pp)
        if (pp != p) rank += count_better<PEER>(qi + (size_t)pp * ips, qs + (size_t)pp * sps, k, s, id);
    if (rank < k) { out_ids[(size_t)q * k + rank] = id; out_scores[(size_t)q * k + rank] = s; }
}
__global__ void merge_topk_kernel(const int64_t* __restrict__ ids, const float* __restrict__ scores, int nq,
                                  int parts, int k, int64_t ips, int64_t sps, int64_t query_stride,
                                  int64_t* __restrict__ out_ids, float* __restrict__ out_scores) {
    merge_topk_body<false>(ids, scores, nq, parts, k, ips, sps, query_stride, out_ids, out_scores);
}

// ---------------------------------------------------------------------------------
// Cross-shard exchange over NVLink peer memory (one process per GPU, buffers opened through CUDA IPC): instead of an
// NCCL all-gather, every rank STORES its packed hit record {ids[nq*k] | scores[nq*k]} straight into slot `rank` of
// every peer's gather area and then publishes the step number in that peer's flag word (release, system scope); the
// reduce kernel spins (acquire) until all `world` flags of its own area carry the step number, then merges.
// Gather areas and flags form a ring of kXSlots = 4 slots indexed by step % 4.  With these stream-ordered kernels a rank can
// be at most one step ahead of a peer (its step t+1 reduce needs the peer's step t+1 record, sent after the peer's step t
// reduce in stream order), so two slots would do; the one-kernel search (sweep_fused.cuh) shares the ring and, when
// pipelined, keeps two searches of a rank in flight: rank A's step t+3 push can only happen after A's step t+1 search has
// completed (a search starts only when the one before its predecessor has finished with its control block), which needs
// peer B's step t+1 hits, pushed by B's step t+1 search, which could only start once B's step t-1 search - the last
// reader of slot (t+3) % 4 - had completely finished.
//   peer_area[p]  base of rank p's gather area: [kXSlots][world][record_bytes]
//   peer_flag[p]  base of rank p's flags:       [kXSlots][world] uint32
// grid = (chunks, world); blockIdx.y = destination peer.
// ---------------------------------------------------------------------------------
constexpr uint32_t kXSlots = 4;
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__global__ void __launch_bounds__(256)
exchange_push_kernel(const int64_t* __restrict__ ids, const float* __restrict__ scores, int64_t n_hits /*nq*k*/,
                     int rank, int world, size_t record_bytes, uint32_t step, char* const* __restrict__ peer_area,
                     uint32_t* const* __restrict__ peer_flag, unsigned int* __restrict__ done /*[world]*/) {
    const int p = blockIdx.y;
    char* dst = peer_area[p] + ((size_t)(step % kXSlots) * world + rank) * record_bytes;
    int64_t* dids = reinterpret_cast<int64_t*>(dst);
    float* dsc = reinterpret_cast<float*>(dst + (size_t)n_hits * 8);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_hits; i += (int64_t)gridDim.x * blockDim.x) {
        dids[i] = ids[i];
        dsc[i] = scores[i];
    }
    __threadfence_system();      // this thread's peer stores are visible system-wide before the CTA is counted
    __syncthreads();
    if (threadIdx.x == 0) {
        if (atomicAdd(&done[p], 1u) == gridDim.x - 1) {   // last CTA of this destination: publish
            done[p] = 0u;
            __threadfence_system();
            st_release_sys(peer_flag[p] + (size_t)(step % kXSlots) * world + rank, step);
        }
    }
}
__global__ void exchange_merge_kernel(const char* area, const uint32_t* flags, int nq, int world,
                                      int k, size_t record_bytes, uint32_t step, int64_t* __restrict__ out_ids,
                                      float* __restrict__ out_scores) {
    if (threadIdx.x < world) {
        const uint32_t* f = flags + (size_t)(step % kXSlots) * world + threadIdx.x;
        while (ld_acquire_sys(f) != step) __nanosleep(20);
    }
    __syncthreads();
    (void)ld_acquire_sys(flags + (size_t)(step % kXSlots) * world + threadIdx.x % world);   // every thread acquires for its own loads
    const char* base = area + (size_t)(step % kXSlots) * world * record_bytes;
    merge_topk_body<true>(reinterpret_cast<const int64_t*>(base), reinterpret_cast<const float*>(base + (size_t)nq * k * 8), nq, world, k,
                    (int64_t)(record_bytes / 8), (int64_t)(record_bytes / 4), (int64_t)k, out_ids, out_scores);
}

}  // namespace rfk
