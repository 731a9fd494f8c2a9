/*
 * C restatement of the CPU oracle (see oracle/ragfin_oracle.py for the full header).
 *
 * TEST INFRASTRUCTURE ONLY: linked/loaded by tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline leg.  The shipped library never calls into it.
 *
 * PARITY UNPINNED: the reference delegates the arithmetic to an external Milvus
 * server (pymilvus==2.3.0, reference vector_rag_mcp/requirements.txt:2); no
 * reference-owned golden vector exists for scores or rankings.  Semantics restated:
 *   Collection.search(q, "embedding", {"metric_type":"COSINE"}, k)
 *     - vector_rag_mcp/main.py:51-57, retrieve.py:28-34,
 *       "chunking_storing (1).py":411-417, graph_cons.py:275-281
 *   cosine score, descending, ties to the lower row ordinal, min(k, N) hits.
 *
 * Canonical arithmetic: 32 strided fp64 partial sums, butterfly fold 16/8/4/2/1,
 * one rounding to fp32, "+ 0.0f" to canonicalise -0.  Build WITHOUT -ffast-math.
 */
#include <float.h>
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#define LANES 32

/* ---------------- minimal pthread parallel-for (libgomp is not in this image) ---------------- */
typedef void (*range_fn)(int64_t lo, int64_t hi, void* ctx);
typedef struct { range_fn fn; int64_t lo, hi; void* ctx; } range_job;
static void* range_tramp(void* p) { range_job* j = (range_job*)p; j->fn(j->lo, j->hi, j->ctx); return 0; }
static int g_threads = 0;
void oracle_set_threads(int t) { g_threads = t; }
int oracle_get_threads(void) {
    if (g_threads > 0) return g_threads;
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n > 0 ? (int)(n > 256 ? 256 : n) : 1;
}
static void parallel_for(int64_t n, range_fn fn, void* ctx) {
    int t = oracle_get_threads();
    if (n < 4096 || t <= 1) { fn(0, n, ctx); return; }
    pthread_t th[256]; range_job jobs[256];
    int64_t per = (n + t - 1) / t; int started = 0;
    for (int i = 0; i < t; ++i) {
        int64_t lo = i * per, hi = lo + per > n ? n : lo + per;
        if (lo >= hi) break;
        jobs[i] = (range_job){fn, lo, hi, ctx};
        if (pthread_create(&th[i], 0, range_tramp, &jobs[i]) != 0) { fn(lo, hi, ctx); th[i] = 0; }
        started = i + 1;
    }
    for (int i = 0; i < started; ++i) if (th[i]) pthread_join(th[i], 0);
}

/* ---------------- synthetic generator (SURVEY.md section 8d) ---------------- */
static inline uint64_t mix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

typedef struct { uint64_t key; int64_t row0; int32_t dim, dup_every, zero_every; float* out; } synth_ctx;
static void synth_range(int64_t lo, int64_t hi, void* p) {
    synth_ctx* c = (synth_ctx*)p;
    for (int64_t r = lo; r < hi; ++r) {
        uint64_t row = (uint64_t)(c->row0 + r), src = row;
        if (c->dup_every > 1 && row % (uint64_t)c->dup_every == (uint64_t)(c->dup_every - 1)) src = row - 1;
        int zero = c->zero_every > 1 && row % (uint64_t)c->zero_every == (uint64_t)(c->zero_every - 1);
        for (int32_t j = 0; j < c->dim; ++j) {
            uint64_t h = mix64((src * (uint64_t)c->dim + (uint64_t)j) ^ c->key);
            int64_t s = (int64_t)((h & 0xFFFF) + ((h >> 16) & 0xFFFF) + ((h >> 32) & 0xFFFF) + (h >> 48));
            c->out[r * c->dim + j] = zero ? 0.0f : (float)(s - 131070) * 0x1p-16f;
        }
    }
}
void oracle_synth_rows(uint64_t seed, int64_t row0, int64_t n, int32_t dim, int32_t dup_every,
                       int32_t zero_every, float* out) {
    synth_ctx c = {mix64(seed), row0, dim, dup_every, zero_every, out};
    parallel_for(n, synth_range, &c);
}

/* ---------------- storage rounding ---------------- */
static inline float round_bf16(float x) {
    uint32_t b;
    memcpy(&b, &x, 4);
    b = (b + 0x7FFFu + ((b >> 16) & 1u)) & 0xFFFF0000u;
    memcpy(&x, &b, 4);
    return x;
}
static inline float round_f16(float x) { return (float)(_Float16)x; }
static inline float round_storage(float x, int dtype) {
    return dtype == 1 ? round_bf16(x) : dtype == 2 ? round_f16(x) : x;
}

/* ---------------- canonical reductions ---------------- */
static inline double fold32(double* v) {
    for (int off = LANES / 2; off >= 1; off >>= 1)
        for (int p = 0; p < off; ++p) v[p] = v[p] + v[p + off];
    return v[0];
}

static double canonical_dot(const float* a, const float* b, int32_t dim) {
    double v[LANES];
    for (int p = 0; p < LANES; ++p) v[p] = 0.0;
    int32_t i = 0;
    for (; i + LANES <= dim; i += LANES)
        for (int p = 0; p < LANES; ++p) v[p] = v[p] + (double)a[i + p] * (double)b[i + p];
    for (int p = 0; i + p < dim; ++p) v[p] = v[p] + (double)a[i + p] * (double)b[i + p];
    return fold32(v);
}

/* x [n, dim] fp32 -> out [n, dim] fp32 VALUES of the stored rows for `dtype`
 * (0 = f32, 1 = bf16, 2 = f16).  Ingest step implied by COSINE for
 * "chunking_storing (1).py":380-394. */
typedef struct { const float* x; int32_t dim, dtype; float* out; } norm_ctx;
static void norm_range(int64_t lo, int64_t hi, void* p) {
    norm_ctx* c = (norm_ctx*)p;
    for (int64_t r = lo; r < hi; ++r) {
        const float* xr = c->x + r * c->dim;
        double n2 = canonical_dot(xr, xr, c->dim);
        /* a zero row and a non-finite one (n2 NaN or +inf) get inv = 0; the NaN of Inf * 0 or NaN * 0 is stored as +0 */
        double inv = n2 > 0.0 && n2 <= DBL_MAX ? 1.0 / sqrt(n2) : 0.0;
        for (int32_t j = 0; j < c->dim; ++j) {
            float y = (float)((double)xr[j] * inv);
            c->out[r * c->dim + j] = round_storage(y == y ? y : 0.0f, c->dtype);
        }
    }
}
void oracle_normalize_rows(const float* x, int64_t n, int32_t dim, int32_t dtype, float* out) {
    norm_ctx c = {x, dim, dtype, out};
    parallel_for(n, norm_range, &c);
}

/* fp32 scores of one normalised query against stored rows. */
typedef struct { const float* stored; int32_t dim; const float* qhat; float* scores; } score_ctx;
static void score_range(int64_t lo, int64_t hi, void* p) {
    score_ctx* c = (score_ctx*)p;
    for (int64_t r = lo; r < hi; ++r)
        c->scores[r] = (float)canonical_dot(c->stored + r * c->dim, c->qhat, c->dim) + 0.0f;
}
void oracle_exact_scores(const float* stored, int64_t n, int32_t dim, const float* qhat, float* scores) {
    score_ctx c = {stored, dim, qhat, scores};
    parallel_for(n, score_range, &c);
}

/* better(a) over (b): higher score, then lower id */
static inline int better(float sa, int64_t ia, float sb, int64_t ib) {
    return sa > sb || (sa == sb && ia < ib);
}

/* Exact top-k of raw (un-normalised) queries over stored rows: restates
 * Collection.search(..., COSINE, k) at vector_rag_mcp/main.py:51-57.
 * ids [nq,k] (-1 padded), scores [nq,k] (-inf padded).  Returns 0, or -1 on OOM. */
int oracle_topk(const float* stored, int64_t n, int32_t dim, const float* queries, int32_t nq,
                int32_t k, int64_t id_base, int64_t* ids, float* scores) {
    float* qhat = (float*)malloc((size_t)dim * sizeof(float));
    float* s = (float*)malloc((size_t)(n > 0 ? n : 1) * sizeof(float));
    if (!qhat || !s) { free(qhat); free(s); return -1; }
    for (int32_t q = 0; q < nq; ++q) {
        oracle_normalize_rows(queries + (int64_t)q * dim, 1, dim, 0, qhat);
        oracle_exact_scores(stored, n, dim, qhat, s);
        int64_t* oi = ids + (int64_t)q * k;
        float* os = scores + (int64_t)q * k;
        int32_t m = 0;
        for (int32_t j = 0; j < k; ++j) { oi[j] = -1; os[j] = -INFINITY; }
        for (int64_t r = 0; r < n; ++r) {          /* increasing id: ties keep the earlier row */
            if (m == k && !better(s[r], r, os[k - 1], oi[k - 1] - id_base)) continue;
            int32_t pos = m < k ? m : k - 1;
            while (pos > 0 && better(s[r], r, os[pos - 1], oi[pos - 1] - id_base)) {
                os[pos] = os[pos - 1]; oi[pos] = oi[pos - 1]; --pos;
            }
            os[pos] = s[r]; oi[pos] = r + id_base;
            if (m < k) ++m;
        }
    }
    free(qhat); free(s);
    return 0;
}
