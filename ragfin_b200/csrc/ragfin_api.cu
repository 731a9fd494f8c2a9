// C ABI of the engine (include/ragfin.h): handle, workspace, kernel dispatch.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <mutex>
#include <new>
#include <utility>
#include <vector>

#include "../../include/ragfin.h"
#include "kernels.cuh"
#include "gemm.cuh"
#include "gemm_astat.cuh"
#include "gemm_rows.cuh"
#include "gemm_pair.cuh"
#include "sweep_fused.cuh"
#include "scan_tma.cuh"
#include "bigk.cuh"
#include "tombstones.cuh"

using namespace rfk;

// ------------------------------------------------------------------------------
// error plumbing: thread-local message, negative codes, no exceptions across the ABI
// ------------------------------------------------------------------------------
#define RF_LAUNCH(kern, grid, block, smem, st, ...) kern<<<grid, block, smem, st>>>(__VA_ARGS__)

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CU_TRY(expr)                                                                               \
    do {                                                                                           \
        cudaError_t e__ = (expr);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(RAGFIN_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__),     \
                        __FILE__, __LINE__);                                                       \
    } while (0)

extern "C" const char* ragfin_last_error(void) { return g_err; }
extern "C" int ragfin_abi_version(void) { return RAGFIN_ABI_VERSION; }

// ------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------
struct Buf {
    void* p = nullptr;
    size_t bytes = 0;
};

static const int kFusedMaxNq = 16, kFusedMaxNqk = 400;   // default query limits of the one-kernel search (plan_fused)

struct ragfin {
    int dim = 0, ld = 0, dtype = 0, device = 0, num_sms = 0;
    int64_t capacity = 0, count = 0, id_base = 0;
    void* data = nullptr;  // [capacity, ld] storage, row-major, L2-normalised
    // The rows the tensor-core sweeps read: {data, dtype} on dtypes 0-2; on RAGFIN_F32_F16 (dtype = RAGFIN_F32 here, so every
    // exact step keeps meaning "the fp32 rows") an fp16 copy [capacity, ld] of them, and eps_sweep bounds what reading the copy
    // instead of the rows changes in a score (see eps_sweep_const).  Only the approximate passes read these three.
    void* sweep_data = nullptr;
    int sweep_dt = 0;
    float eps_sweep = 0.f;
    bool is_view = false;  // ragfin_create_view: `data` and `sweep_data` belong to another handle (read-only here, never freed here)
    std::mutex mu;
    // workspace (grow-only)
    Buf qhat, q16, eps_q, gtau, bmax, acnt, athr, awin, allow, bk_scores, bk_state, bk_keys, bk_rows, grp, grp_codes, cand, cand_e, flags, stage_q, stage_ids, stage_scores, add_stage;
    int gemm_min_nq = 3;      // query batches of at least this many rows take the tcgen05 path (1-2: HBM-bound scan) ...
    int gemm_min_nq_large = 1;   // ... except on corpora of >= kSweepBytes, where the TMA-fed sweep wins from 1 query
    int gemm_cluster = 0;     // 0 = choose by batch size; 1, 2 or 4 = force
    bool allow_pipelined = false;          // ragfin_set_pipelined: consecutive one-kernel searches on one stream may overlap (see there)
    bool cur_pipelined = false;            // the search in flight came through an asynchronous entry point (ragfin_search)
    const uint32_t* cur_allow = nullptr;   // row mask of the search in flight (device bitmask: filter, tombstones or both), else null
    int64_t cur_allowed = 0;               // rows it allows
    bool cur_user_filter = false;          // the caller passed a filter: filtered dispatch (no bound pass, no append mode)
    bool cur_window = false;               // the search in flight is a range search (ragfin_search_range): hits must satisfy
    float cur_radius = -INFINITY, cur_range_filter = INFINITY;   //   cur_radius < score <= cur_range_filter (DESIGN.md 7c)
    const int32_t* cur_groups = nullptr;   // the search in flight is a grouping search (ragfin_search_grouped): device codes
    int32_t cur_n_groups = 0;              //   [count], one hit per code in [0, cur_n_groups) (DESIGN.md 7d)
    // Tombstones (ragfin_delete).  live_host mirrors the device mask live_dev bit for bit: ceil(capacity / 32) words in the
    // allow_bits layout, bit set = row live; rows at or past `count` are live (rows added later are).  Both stay empty until
    // the first delete, and a handle with n_dead == 0 passes a null mask to every kernel.
    std::vector<uint32_t> live_host;
    uint32_t* live_dev = nullptr;
    int64_t n_dead = 0;
    ragfin* parent = nullptr;   // a view's owner (ragfin_create_view)
    int n_views = 0;            // live views of this handle: compaction would move rows under them
    int scan_variant = 0;         // small-batch scan: 0 = automatic (= 1, measured faster), 1 = LDG kernel, 2 = TMA-fed ring
    bool use_append = true;       // tcgen05 path: append mode (threshold from the bound pass, no lists) when eligible
    bool use_bound_pass = true;   // tcgen05 path: sample pass that seeds the per-query thresholds (RAGFIN_NO_BOUND_PASS=1 disables)
    int gemm_variant = 0;     // 0 = automatic (= 3 for <= 16 queries, 4 from 129 queries), 1 = streaming (A and B through shared memory), 2 = A-stationary (A in TMEM),
                              // 3 = streaming + swapped operand roles for <= 16 queries in append mode (gemm_rows.cuh),
                              // 4 = 2-SM MMA pairs (cta_group::2) for >= 2 query tiles in append mode (gemm_pair.cuh)
    Buf fctl;                 // fused sweep: TWO control blocks (FusedCtl), zero between searches; consecutive searches alternate
    Buf fcand, fqn, fflags;   //   ... and so do their append buffers, normalised queries and overflow flags: a pipelined search
    uint32_t fused_seq = 0;   //   (ragfin_search / ragfin_search_sharded) may start while its predecessor is still finalizing
    uint32_t host_seq = 0;    // sequence number of synchronous host calls (value of the mapped completion word)
    int fused_last = 0;       // half used by the last search (diagnostics, stats)
    bool fctl_dirty = true;   // set when a launch may have left it non-zero (first use, failed call): re-zeroed before the next launch
    bool use_bigk_batched = true;   // k > 256: batched dump + select pipeline (RAGFIN_NO_BIGK_BATCHED=1: the one-query exact path)
    bool use_fused = true;    // <= 64 queries, k <= 128: the one-kernel search (sweep_fused.cuh); RAGFIN_NO_FUSED=1 disables
    int fused_min_rows = 8192;
    int fused_refresh_every = 4, fused_stage_cap = kRMaxStages;   // experiment knobs (RAGFIN_FUSED_REFRESH_EVERY / _STAGES)
    int fused_max_nq = kFusedMaxNq;     // see plan_fused; RAGFIN_FUSED_MAX_NQ overrides (<= 64)
    int fused_max_nqk = kFusedMaxNqk;   // queries x k; RAGFIN_FUSED_MAX_NQK overrides
    struct MapSlot { const void* base = nullptr; int64_t rows = 0; int ld = 0, dtype = 0, box_rows = 0; CUtensorMap map; };
    MapSlot map_cache[8];     // tensor maps are pure functions of (base, rows, ld, dtype, box): encode once
    int map_next = 0;
    Buf add_stage2[2];        // ragfin_add from host memory: two staging slices ...
    cudaStream_t copy_stream = nullptr;                       // ... filled on this stream while K1 runs on the caller's
    cudaEvent_t stage_ready[2] = {nullptr, nullptr}, stage_free[2] = {nullptr, nullptr};
    void* hstage = nullptr;   // pinned, device-mapped staging for small host calls: kernels read the queries and write the hits
                              // straight through PCIe, no copy engine launches (ragfin_search_host)
    cudaEvent_t last_done = nullptr;
    bool have_pending = false;            // pipelined searches enqueued on pending_stream since the last event record
    cudaStream_t pending_stream = nullptr;
    ragfin_search_stats stats = {0, 0, 0, 0};
    // int8 screen copy of the one-kernel search's tile filter (DESIGN.md 2.5), bf16 / fp16 collections: [i8_cap][ld8] int8 rows
    // and a {scale, residual bound} per row, rows [0, i8_rows) current.  Made at the first one-kernel search that wants it and
    // brought up to `count` by the next one after rows were added (an ordinary kernel in front of that launch); dropped by
    // compaction (rows move) and rebuilt when the capacity outgrows it.  A view shares its parent's copy when that covers it.
    int sweep_copy = RAGFIN_SWEEP_COPY_AUTO;   // ragfin_set_sweep_copy
    int8_t* i8 = nullptr;
    float2* i8side = nullptr;
    int ld8 = 0;
    int64_t i8_cap = 0, i8_rows = 0;
    bool i8_owned = false;
    // measurement hook (ragfin_profile): event pairs around the dominant kernel
    bool profiling = false;
    static const int kProfPairs = 512;
    cudaEvent_t prof_ev[2 * kProfPairs] = {};
    int prof_used = 0;
};

static void prof_begin(ragfin* h, cudaStream_t st) {
    if (h->profiling && h->prof_used < ragfin::kProfPairs) cudaEventRecord(h->prof_ev[2 * h->prof_used], st);
}
static void prof_end(ragfin* h, cudaStream_t st) {
    if (h->profiling && h->prof_used < ragfin::kProfPairs) { cudaEventRecord(h->prof_ev[2 * h->prof_used + 1], st); h->prof_used++; }
}

static size_t esize(int dtype) { return dtype == RAGFIN_F32 ? 4 : 2; }
static size_t mask_words(int64_t rows) { return (size_t)((rows + 31) / 32); }
static bool has_copy(const ragfin* h) { return h->sweep_data != h->data; }
// dtype as the caller named it (ragfin_create, the file header)
static int public_dtype(const ragfin* h) { return has_copy(h) ? RAGFIN_F32_F16 : h->dtype; }

// |q.x - q.x16| for the fp32 row x (|x|_2 <= 1 + 2^-20), its copy x16 = RNE_f16(x) and a normalised query (|q|_2 <= 1 + 2^-22):
// per element |x_i - x16_i| <= 2^-11 |x_i| (fp16 normal range, half an ulp) or <= 2^-25 (subnormal range, half the spacing
// 2^-24), so |x - x16|_2 <= 2^-11 |x|_2 + 2^-25 sqrt(ld) and |q.x - q.x16| <= |q|_2 |x - x16|_2.  Rounded up.
static float eps_sweep_const(int ld) {
    const double e = (1.0 + 2.384185791015625e-07) * (4.8828125e-04 * (1.0 + 9.5367431640625e-07) + 2.98023223876953125e-08 * sqrt((double)ld));
    return nextafterf((float)e, INFINITY);
}

static void i8_free(ragfin* h) {
    if (h->i8_owned) {
        (void)cudaDeviceSynchronize();   // no search may still be reading it
        cudaFree(h->i8);
        cudaFree(h->i8side);
    }
    h->i8 = nullptr; h->i8side = nullptr; h->i8_cap = 0; h->i8_rows = 0; h->i8_owned = false;
}

static int ensure(Buf& b, size_t bytes) {
    if (b.bytes >= bytes) return 0;
    if (b.p) {
        CU_TRY(cudaDeviceSynchronize());
        CU_TRY(cudaFree(b.p));
        b.p = nullptr;
        b.bytes = 0;
    }
    size_t want = bytes + bytes / 4;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        b.p = nullptr;
        (void)cudaGetLastError();
        return fail(RAGFIN_ENOMEM, "workspace cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    b.bytes = want;
    return 0;
}

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; (void)cudaGetLastError(); }
        ok = cudaSetDevice(dev) == cudaSuccess;
        if (!ok) (void)cudaGetLastError();
    }
    ~DeviceGuard() {
        if (prev >= 0) (void)cudaSetDevice(prev);
    }
};

// Environment knobs, read when a handle (or a view) is created.
static void read_env_knobs(ragfin* h) {
    { const char* e = getenv("RAGFIN_NO_BOUND_PASS"); if (e && atoi(e)) h->use_bound_pass = false; }
    { const char* e = getenv("RAGFIN_NO_FUSED"); if (e && atoi(e)) h->use_fused = false; }
    { const char* e = getenv("RAGFIN_NO_BIGK_BATCHED"); if (e && atoi(e)) h->use_bigk_batched = false; }
    { const char* e = getenv("RAGFIN_FUSED_MAX_NQ"); if (e && atoi(e) >= 1 && atoi(e) <= kFMaxQ) h->fused_max_nq = atoi(e); }
    { const char* e = getenv("RAGFIN_FUSED_MAX_NQK"); if (e && atoi(e) >= 1) h->fused_max_nqk = atoi(e); }
    { const char* e = getenv("RAGFIN_PIPELINED"); if (e) h->allow_pipelined = atoi(e) != 0; }
    { const char* e = getenv("RAGFIN_FUSED_REFRESH_EVERY"); if (e && atoi(e) >= 1) h->fused_refresh_every = atoi(e); }
    { const char* e = getenv("RAGFIN_FUSED_STAGES"); if (e && atoi(e) >= 2 && atoi(e) <= kRMaxStages) h->fused_stage_cap = atoi(e); }
}

extern "C" int ragfin_create(ragfin_t** out, int32_t dim, int32_t dtype, int64_t capacity_rows, int32_t device) {
    if (!out) return fail(RAGFIN_EINVAL, "out is NULL");
    *out = nullptr;
    if (dim < 1 || dim > 65536) return fail(RAGFIN_EINVAL, "dim %d out of range [1, 65536]", dim);
    if (dtype < 0 || dtype > 3) return fail(RAGFIN_EINVAL, "dtype %d is not 0 (f32), 1 (bf16), 2 (f16) or 3 (f32 + f16 copy)", dtype);
    if (capacity_rows < 1 || capacity_rows >= (int64_t)0xFFFFFFFF)
        return fail(RAGFIN_EINVAL, "capacity_rows %lld out of range [1, 2^32-1)", (long long)capacity_rows);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        (void)cudaGetLastError();
        return fail(RAGFIN_ECUDA, "no CUDA device available (%s); this engine has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= ndev) return fail(RAGFIN_EINVAL, "device %d not in [0, %d)", device, ndev);
    DeviceGuard g(device);
    if (!g.ok) return fail(RAGFIN_ECUDA, "cudaSetDevice(%d) failed", device);
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(RAGFIN_EUNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);
    ragfin* h = new (std::nothrow) ragfin();
    if (!h) return fail(RAGFIN_ENOMEM, "host allocation failed");
    h->dim = dim;
    h->ld = (dim + 7) / 8 * 8;
    h->dtype = dtype == RAGFIN_F32_F16 ? RAGFIN_F32 : dtype;
    h->device = device;
    h->num_sms = prop.multiProcessorCount;
    read_env_knobs(h);
    h->capacity = capacity_rows;
    const size_t bytes = (size_t)capacity_rows * h->ld * esize(h->dtype);
    e = cudaMalloc(&h->data, bytes);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        delete h;
        return fail(RAGFIN_ENOMEM, "cudaMalloc of %zu bytes for the corpus failed: %s", bytes, cudaGetErrorString(e));
    }
    h->sweep_data = h->data;
    h->sweep_dt = h->dtype;
    if (dtype == RAGFIN_F32_F16) {
        const size_t bytes16 = (size_t)capacity_rows * h->ld * 2;
        e = cudaMalloc(&h->sweep_data, bytes16);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            cudaFree(h->data);
            delete h;
            return fail(RAGFIN_ENOMEM, "cudaMalloc of %zu bytes for the fp16 copy failed: %s", bytes16, cudaGetErrorString(e));
        }
        h->sweep_dt = RAGFIN_F16;
        h->eps_sweep = eps_sweep_const(h->ld);
    }
    e = cudaEventCreateWithFlags(&h->last_done, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        if (has_copy(h)) cudaFree(h->sweep_data);
        cudaFree(h->data);
        delete h;
        return fail(RAGFIN_ECUDA, "cudaEventCreate failed: %s", cudaGetErrorString(e));
    }
    *out = h;
    return RAGFIN_OK;
}

// A second handle over the SAME device matrix (no copy) with its own workspace, so that searches through the two handles
// can be in flight at once on different streams (the latency-bound head and tail of one call overlap the other's sweep).
// The view sees the rows present now, is read-only (ragfin_add fails) and must be destroyed before its parent.
extern "C" int ragfin_create_view(ragfin_t* parent, ragfin_t** out) {
    if (!parent || !out) return fail(RAGFIN_EINVAL, "NULL argument");
    *out = nullptr;
    std::lock_guard<std::mutex> lk(parent->mu);
    DeviceGuard g(parent->device);
    if (!g.ok) return fail(RAGFIN_ECUDA, "cudaSetDevice(%d) failed", parent->device);
    CU_TRY(cudaDeviceSynchronize());   // every row the parent has accepted is in the matrix
    ragfin* h = new (std::nothrow) ragfin();
    if (!h) return fail(RAGFIN_ENOMEM, "host allocation failed");
    h->dim = parent->dim; h->ld = parent->ld; h->dtype = parent->dtype; h->device = parent->device; h->num_sms = parent->num_sms;
    h->capacity = parent->count > 0 ? parent->count : 1; h->count = parent->count; h->id_base = parent->id_base;
    h->data = parent->data;
    h->sweep_data = parent->sweep_data; h->sweep_dt = parent->sweep_dt; h->eps_sweep = parent->eps_sweep;
    h->is_view = true;
    h->gemm_min_nq = parent->gemm_min_nq; h->gemm_min_nq_large = parent->gemm_min_nq_large; h->gemm_cluster = parent->gemm_cluster;
    h->scan_variant = parent->scan_variant; h->use_append = parent->use_append; h->use_bound_pass = parent->use_bound_pass;
    h->gemm_variant = parent->gemm_variant;
    h->use_fused = parent->use_fused; h->use_bigk_batched = parent->use_bigk_batched; h->fused_min_rows = parent->fused_min_rows;
    h->fused_max_nq = parent->fused_max_nq; h->fused_max_nqk = parent->fused_max_nqk; h->allow_pipelined = parent->allow_pipelined;
    h->fused_refresh_every = parent->fused_refresh_every; h->fused_stage_cap = parent->fused_stage_cap;
    h->sweep_copy = parent->sweep_copy;
    if (parent->i8 && parent->i8_rows >= h->count) {   // the rows of a view never change: its parent's copy stays valid for them
        h->i8 = parent->i8; h->i8side = parent->i8side; h->ld8 = parent->ld8; h->i8_cap = parent->i8_cap; h->i8_rows = h->count;
    }
    read_env_knobs(h);
    cudaError_t e = cudaEventCreateWithFlags(&h->last_done, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        delete h;
        return fail(RAGFIN_ECUDA, "cudaEventCreate failed: %s", cudaGetErrorString(e));
    }
    if (parent->n_dead > 0) {   // the view's own copy of the tombstones: rows deleted through the parent later stay visible here
        const size_t words = mask_words(h->capacity);
        h->live_host.assign(parent->live_host.begin(), parent->live_host.begin() + words);
        e = cudaMalloc(&h->live_dev, words * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMemcpy(h->live_dev, parent->live_dev, words * sizeof(uint32_t), cudaMemcpyDeviceToDevice);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            if (h->live_dev) cudaFree(h->live_dev);
            cudaEventDestroy(h->last_done);
            delete h;
            return fail(RAGFIN_ENOMEM, "copying the tombstone mask failed: %s", cudaGetErrorString(e));
        }
        h->n_dead = parent->n_dead;
    }
    h->parent = parent;
    parent->n_views++;
    *out = h;
    return RAGFIN_OK;
}

extern "C" void ragfin_destroy(ragfin_t* h) {
    if (!h) return;
    DeviceGuard g(h->device);
    (void)cudaDeviceSynchronize();
    Buf* bufs[] = {&h->qhat, &h->q16, &h->eps_q, &h->gtau, &h->bmax, &h->acnt, &h->athr, &h->awin, &h->allow, &h->bk_scores, &h->bk_state, &h->bk_keys, &h->bk_rows, &h->grp, &h->grp_codes, &h->cand, &h->cand_e, &h->flags, &h->stage_q, &h->stage_ids, &h->stage_scores, &h->add_stage, &h->fctl, &h->fcand, &h->fqn, &h->fflags};
    for (Buf* b : bufs)
        if (b->p) cudaFree(b->p);
    i8_free(h);
    if (h->sweep_data && has_copy(h) && !h->is_view) cudaFree(h->sweep_data);
    if (h->data && !h->is_view) cudaFree(h->data);
    if (h->live_dev) cudaFree(h->live_dev);
    if (h->parent) {
        std::lock_guard<std::mutex> lk(h->parent->mu);
        h->parent->n_views--;
    }
    for (int b = 0; b < 2; ++b) {
        if (h->add_stage2[b].p) cudaFree(h->add_stage2[b].p);
        if (h->stage_ready[b]) cudaEventDestroy(h->stage_ready[b]);
        if (h->stage_free[b]) cudaEventDestroy(h->stage_free[b]);
    }
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->hstage) cudaFreeHost(h->hstage);
    if (h->last_done) cudaEventDestroy(h->last_done);
    for (cudaEvent_t e : h->prof_ev)
        if (e) cudaEventDestroy(e);
    delete h;
}

extern "C" int ragfin_count(const ragfin_t* h, int64_t* n) {
    if (!h || !n) return fail(RAGFIN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(const_cast<ragfin*>(h)->mu);   // count is written under the lock by ragfin_add
    *n = h->count;
    return RAGFIN_OK;
}

extern "C" int ragfin_live_count(const ragfin_t* h, int64_t* n) {
    if (!h || !n) return fail(RAGFIN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(const_cast<ragfin*>(h)->mu);
    *n = h->count - h->n_dead;
    return RAGFIN_OK;
}

// Tombstone rows by the ids searches return (id_base + row).  The host mirror decides what changes, so duplicates and rows
// deleted before cost nothing; only the words that changed go to the device.  The device mask is read by searches still in
// flight, so the call first waits for the handle's last operation (the completion event ragfin_add orders itself behind).
extern "C" int ragfin_delete(ragfin_t* h, const int64_t* ids_host, int64_t n, int64_t* n_deleted_out) {
    if (!h || n < 0 || (n > 0 && !ids_host)) return fail(RAGFIN_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(h->mu);
    if (h->is_view) return fail(RAGFIN_EUNSUPPORTED, "a view is read-only: delete rows through the handle that owns the matrix");
    for (int64_t i = 0; i < n; ++i)   // validate everything before anything changes
        if (ids_host[i] < h->id_base || ids_host[i] - h->id_base >= h->count)
            return fail(RAGFIN_EINVAL, "id %lld outside [%lld, %lld)", (long long)ids_host[i], (long long)h->id_base,
                        (long long)(h->id_base + h->count));
    if (n_deleted_out) *n_deleted_out = 0;
    if (n == 0) return RAGFIN_OK;
    DeviceGuard g(h->device);
    if (h->have_pending) {   // a pipelined search never chains across a delete
        CU_TRY(cudaEventRecord(h->last_done, h->pending_stream));
        h->have_pending = false;
    }
    CU_TRY(cudaEventSynchronize(h->last_done));
    const bool fresh = h->live_dev == nullptr;
    if (fresh) {   // first delete: the mask covers the capacity, every row live
        const size_t words = mask_words(h->capacity);
        cudaError_t e = cudaMalloc(&h->live_dev, words * sizeof(uint32_t));
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            h->live_dev = nullptr;
            return fail(RAGFIN_ENOMEM, "cudaMalloc of the tombstone mask failed: %s", cudaGetErrorString(e));
        }
        h->live_host.assign(words, 0xFFFFFFFFu);
    }
    int64_t del = 0;
    size_t w0 = fresh ? 0 : h->live_host.size(), w1 = fresh ? h->live_host.size() : 0;
    for (int64_t i = 0; i < n; ++i) {
        const int64_t r = ids_host[i] - h->id_base;
        const size_t w = (size_t)(r >> 5);
        const uint32_t bit = 1u << (r & 31);
        if (!(h->live_host[w] & bit)) continue;
        h->live_host[w] &= ~bit;
        ++del;
        if (w < w0) w0 = w;
        if (w + 1 > w1) w1 = w + 1;
    }
    if (w1 > w0) CU_TRY(cudaMemcpy(h->live_dev + w0, h->live_host.data() + w0, (w1 - w0) * sizeof(uint32_t), cudaMemcpyHostToDevice));
    h->n_dead += del;
    if (n_deleted_out) *n_deleted_out = del;
    return RAGFIN_OK;
}

// ceil(count / 32) words of the live mask as the kernels read it (the device copy; all ones without tombstones), bits at or
// past `count` cleared.
extern "C" int ragfin_read_live_mask(ragfin_t* h, uint32_t* out_host) {
    if (!h || !out_host) return fail(RAGFIN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(h->mu);
    const size_t words = mask_words(h->count);
    if (words == 0) return RAGFIN_OK;
    if (h->live_dev) {
        DeviceGuard g(h->device);
        CU_TRY(cudaDeviceSynchronize());
        CU_TRY(cudaMemcpy(out_host, h->live_dev, words * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    } else {
        for (size_t w = 0; w < words; ++w) out_host[w] = 0xFFFFFFFFu;
    }
    if (h->count & 31) out_host[words - 1] &= (1u << (h->count & 31)) - 1u;
    return RAGFIN_OK;
}

// Physical removal of the tombstoned rows: survivors keep their order, live row r moves to the number of live rows before
// it.  Into NEW allocations of the same capacity (the transient cost is a second copy of the matrix - of both on a
// RAGFIN_F32_F16 handle), all made before anything is freed, so a failed allocation leaves the handle as it was.
extern "C" int ragfin_compact(ragfin_t* h) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    std::lock_guard<std::mutex> lk(h->mu);
    if (h->is_view) return fail(RAGFIN_EUNSUPPORTED, "a view is read-only");
    if (h->n_views > 0) return fail(RAGFIN_EUNSUPPORTED, "%d view(s) of this collection are live: destroy them before compacting", h->n_views);
    if (h->n_dead == 0) return RAGFIN_OK;
    DeviceGuard g(h->device);
    CU_TRY(cudaDeviceSynchronize());                 // no search may still be reading the old matrix
    const size_t words = mask_words(h->count);
    std::vector<uint32_t> off(words ? words : 1);    // exclusive prefix of the per-word live counts
    uint32_t live = 0;
    for (size_t w = 0; w < words; ++w) {
        uint32_t v = h->live_host[w];
        if (w + 1 == words && (h->count & 31)) v &= (1u << (h->count & 31)) - 1u;
        off[w] = live;
        live += (uint32_t)__builtin_popcount(v);
    }
    const size_t rb = (size_t)h->ld * esize(h->dtype), rb16 = (size_t)h->ld * 2;
    void *nd = nullptr, *nd16 = nullptr, *doff = nullptr;
    cudaError_t e = cudaMalloc(&nd, (size_t)h->capacity * rb);
    if (e == cudaSuccess && has_copy(h)) e = cudaMalloc(&nd16, (size_t)h->capacity * rb16);
    if (e == cudaSuccess) e = cudaMalloc(&doff, off.size() * sizeof(uint32_t));
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        if (nd) cudaFree(nd);
        if (nd16) cudaFree(nd16);
        if (doff) cudaFree(doff);
        return fail(RAGFIN_ENOMEM, "allocation for compaction failed (it needs a second copy of the matrix): %s", cudaGetErrorString(e));
    }
    e = cudaMemcpy(doff, off.data(), off.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
    const int64_t want = (h->count + 7) / 8, cap_blocks = (int64_t)h->num_sms * 16;
    const unsigned blocks = (unsigned)(want < cap_blocks ? (want > 0 ? want : 1) : cap_blocks);
    prof_begin(h, 0);   // ragfin_profile: the gather kernels alone (the call also allocates and frees a matrix)
    if (e == cudaSuccess) {
        compact_rows_kernel<<<blocks, 256>>>((const uint4*)h->data, (uint4*)nd, (int)(rb / 16), h->count, h->live_dev, (const uint32_t*)doff);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && nd16) {
        compact_rows_kernel<<<blocks, 256>>>((const uint4*)h->sweep_data, (uint4*)nd16, (int)(rb16 / 16), h->count, h->live_dev, (const uint32_t*)doff);
        e = cudaGetLastError();
    }
    prof_end(h, 0);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    std::vector<uint32_t> ones(h->live_host.size(), 0xFFFFFFFFu);
    if (e == cudaSuccess) e = cudaMemcpy(h->live_dev, ones.data(), ones.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
    cudaFree(doff);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        cudaFree(nd);
        if (nd16) cudaFree(nd16);
        return fail(RAGFIN_ECUDA, "compaction failed: %s", cudaGetErrorString(e));
    }
    if (nd16) { CU_TRY(cudaFree(h->sweep_data)); h->sweep_data = nd16; }
    CU_TRY(cudaFree(h->data));
    h->data = nd;
    if (!nd16) h->sweep_data = nd;
    h->live_host.swap(ones);
    h->count = live;
    h->n_dead = 0;
    i8_free(h);   // rows moved: the next one-kernel search that wants the int8 copy rebuilds it
    for (ragfin::MapSlot& m : h->map_cache) m = ragfin::MapSlot();   // tensor maps of the old matrix are stale
    return RAGFIN_OK;
}

// Grow the device matrix to at least `capacity_rows` rows: new allocation + device-to-device copy of the stored rows (they
// are already normalised and rounded, so nothing is recomputed and no host copy of the embeddings is needed).
extern "C" int ragfin_reserve(ragfin_t* h, int64_t capacity_rows) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (capacity_rows < 1 || capacity_rows >= (int64_t)0xFFFFFFFF)
        return fail(RAGFIN_EINVAL, "capacity_rows %lld out of range [1, 2^32-1)", (long long)capacity_rows);
    std::lock_guard<std::mutex> lk(h->mu);
    if (h->is_view) return fail(RAGFIN_EUNSUPPORTED, "a view is read-only");
    if (capacity_rows <= h->capacity) return RAGFIN_OK;
    DeviceGuard g(h->device);
    CU_TRY(cudaDeviceSynchronize());                 // no search may still be reading the old matrix
    const size_t rb = (size_t)h->ld * esize(h->dtype);
    void* nd = nullptr;
    cudaError_t e = cudaMalloc(&nd, (size_t)capacity_rows * rb);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(RAGFIN_ENOMEM, "cudaMalloc of %zu bytes for the grown corpus failed: %s", (size_t)capacity_rows * rb, cudaGetErrorString(e));
    }
    // the fp16 copy grows with the rows; both new buffers exist before either old one is touched, so a failed allocation
    // leaves the handle as it was
    const size_t rb16 = (size_t)h->ld * 2;
    void* nd16 = nullptr;
    if (has_copy(h)) {
        e = cudaMalloc(&nd16, (size_t)capacity_rows * rb16);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            cudaFree(nd);
            return fail(RAGFIN_ENOMEM, "cudaMalloc of %zu bytes for the grown fp16 copy failed: %s", (size_t)capacity_rows * rb16, cudaGetErrorString(e));
        }
    }
    uint32_t* nm = nullptr;   // the tombstone mask grows with the rows (new rows are live)
    const size_t nwords = mask_words(capacity_rows);
    if (h->live_dev) {
        e = cudaMalloc(&nm, nwords * sizeof(uint32_t));
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            cudaFree(nd);
            if (nd16) cudaFree(nd16);
            return fail(RAGFIN_ENOMEM, "cudaMalloc of the grown tombstone mask failed: %s", cudaGetErrorString(e));
        }
    }
    if (h->count > 0) {
        e = cudaMemcpy(nd, h->data, (size_t)h->count * rb, cudaMemcpyDeviceToDevice);
        if (e == cudaSuccess && nd16) e = cudaMemcpyAsync(nd16, h->sweep_data, (size_t)h->count * rb16, cudaMemcpyDeviceToDevice, 0);
        if (e == cudaSuccess && nd16) e = cudaStreamSynchronize(0);
        if (e != cudaSuccess) {
            cudaFree(nd);
            if (nd16) cudaFree(nd16);
            if (nm) cudaFree(nm);
            (void)cudaGetLastError();
            return fail(RAGFIN_ECUDA, "device copy failed: %s", cudaGetErrorString(e));
        }
    }
    if (nm) {
        std::vector<uint32_t> grown(h->live_host);
        grown.resize(nwords, 0xFFFFFFFFu);
        e = cudaMemcpy(nm, grown.data(), nwords * sizeof(uint32_t), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            cudaFree(nd);
            if (nd16) cudaFree(nd16);
            cudaFree(nm);
            (void)cudaGetLastError();
            return fail(RAGFIN_ECUDA, "tombstone mask copy failed: %s", cudaGetErrorString(e));
        }
        CU_TRY(cudaFree(h->live_dev));
        h->live_dev = nm;
        h->live_host.swap(grown);
    }
    if (nd16) { CU_TRY(cudaFree(h->sweep_data)); h->sweep_data = nd16; }
    CU_TRY(cudaFree(h->data));
    h->data = nd;
    if (!nd16) h->sweep_data = nd;
    h->capacity = capacity_rows;
    for (ragfin::MapSlot& m : h->map_cache) m = ragfin::MapSlot();   // tensor maps of the old matrix are stale
    return RAGFIN_OK;
}

extern "C" int ragfin_set_id_base(ragfin_t* h, int64_t id_base) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (id_base < 0) return fail(RAGFIN_EINVAL, "id_base must be >= 0");
    std::lock_guard<std::mutex> lk(h->mu);
    h->id_base = id_base;
    return RAGFIN_OK;
}

// ------------------------------------------------------------------------------
// K1 launch
// ------------------------------------------------------------------------------
// dtype RAGFIN_F32_F16: fp32 rows into dst and their fp16 copy into dst16, one pass
template <bool SYNTH>
static int launch_ingest(int dtype, const float* src, uint64_t key, int64_t row0, int dup, int zero, int64_t n,
                         int dim, int ld, void* dst, int num_sms, cudaStream_t st,
                         int64_t topic_rows = 0, uint64_t topic_key = 0, float noise_scale = 0.f, void* dst16 = nullptr) {
    if (n == 0) return 0;
    const int threads = 256, wpb = threads / 32;
    int64_t blocks = (n + wpb - 1) / wpb;
    if (!SYNTH && dim % 4 == 0 && ld <= 1024 && ((uintptr_t)src & 15u) == 0) {
        // vectorised single-pass kernel (kernels.cuh ingest_vec_kernel): NV 16-byte vectors per lane cover the stored row
        const int nv = ld <= 256 ? 2 : ld <= 512 ? 4 : ld <= 768 ? 6 : 8;
        const int64_t capv = (int64_t)num_sms * 8;
        if (blocks > capv) blocks = capv;
#define RF_INGEST_VEC(DT, TT) \
        switch (nv) { \
            case 2: ingest_vec_kernel<DT, 2><<<(int)blocks, kIngestThreads, 0, st>>>(src, n, dim, ld, (TT*)dst); break; \
            case 4: ingest_vec_kernel<DT, 4><<<(int)blocks, kIngestThreads, 0, st>>>(src, n, dim, ld, (TT*)dst); break; \
            case 6: ingest_vec_kernel<DT, 6><<<(int)blocks, kIngestThreads, 0, st>>>(src, n, dim, ld, (TT*)dst); break; \
            default: ingest_vec_kernel<DT, 8><<<(int)blocks, kIngestThreads, 0, st>>>(src, n, dim, ld, (TT*)dst); break; \
        }
        if (dtype == 0) { RF_INGEST_VEC(0, float) } else if (dtype == 1) { RF_INGEST_VEC(1, __nv_bfloat16) } else if (dtype == 2) { RF_INGEST_VEC(2, __half) }
        else {
            switch (nv) {
                case 2: ingest_vec_kernel<3, 2><<<(int)blocks, kIngestThreads, 0, st>>>(src, n, dim, ld, (float*)dst, (__half*)dst16); break;
                case 4: ingest_vec_kernel<3, 4><<<(int)blocks, kIngestThreads, 0, st>>>(src, n, dim, ld, (float*)dst, (__half*)dst16); break;
                case 6: ingest_vec_kernel<3, 6><<<(int)blocks, kIngestThreads, 0, st>>>(src, n, dim, ld, (float*)dst, (__half*)dst16); break;
                default: ingest_vec_kernel<3, 8><<<(int)blocks, kIngestThreads, 0, st>>>(src, n, dim, ld, (float*)dst, (__half*)dst16); break;
            }
        }
#undef RF_INGEST_VEC
        CU_TRY(cudaGetLastError());
        return 0;
    }
    const int64_t cap = (int64_t)num_sms * 16;
    if (blocks > cap) blocks = cap;
    switch (dtype) {
        case 0: ingest_kernel<0, SYNTH><<<(int)blocks, threads, 0, st>>>(src, key, row0, dup, zero, n, dim, ld, (float*)dst, topic_rows, topic_key, noise_scale); break;
        case 1: ingest_kernel<1, SYNTH><<<(int)blocks, threads, 0, st>>>(src, key, row0, dup, zero, n, dim, ld, (__nv_bfloat16*)dst, topic_rows, topic_key, noise_scale); break;
        case 2: ingest_kernel<2, SYNTH><<<(int)blocks, threads, 0, st>>>(src, key, row0, dup, zero, n, dim, ld, (__half*)dst, topic_rows, topic_key, noise_scale); break;
        default: ingest_kernel<3, SYNTH><<<(int)blocks, threads, 0, st>>>(src, key, row0, dup, zero, n, dim, ld, (float*)dst, topic_rows, topic_key, noise_scale, (__half*)dst16); break;
    }
    CU_TRY(cudaGetLastError());
    return 0;
}

// Ordering of the handle's operations across streams: every operation waits for the previous one's completion event.  An event
// record between two kernels of one stream would also cut the programmatic dependency that lets a pipelined search start while
// its predecessor finalizes, so pipelined searches only NOTE their stream; the event is recorded later, on that stream, when an
// operation on another stream (or a non-pipelined one) needs it - a record covers everything enqueued before it.
static int wait_prev(ragfin* h, cudaStream_t st, bool pipelined = false) {
    if (h->have_pending) {
        if (pipelined && st == h->pending_stream) return 0;          // same stream: stream order is the dependency
        CU_TRY(cudaEventRecord(h->last_done, h->pending_stream));
        h->have_pending = false;
    }
    CU_TRY(cudaStreamWaitEvent(st, h->last_done, 0));
    return 0;
}
static int mark_done(ragfin* h, cudaStream_t st, bool pipelined = false) {
    if (pipelined) { h->have_pending = true; h->pending_stream = st; return 0; }
    CU_TRY(cudaEventRecord(h->last_done, st));
    return 0;
}

extern "C" int ragfin_add(ragfin_t* h, const float* rows, int64_t n, int32_t src_is_device, void* stream) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (n < 0 || (n > 0 && !rows)) return fail(RAGFIN_EINVAL, "bad rows/n");
    if (n == 0) return RAGFIN_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    if (h->is_view) return fail(RAGFIN_EUNSUPPORTED, "a view is read-only: add rows through the handle that owns the matrix");
    if (h->count + n > h->capacity)
        return fail(RAGFIN_ENOMEM, "add of %lld rows exceeds capacity (%lld of %lld used)", (long long)n,
                    (long long)h->count, (long long)h->capacity);
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if ((rc = wait_prev(h, st))) return rc;
    char* dst = (char*)h->data + (size_t)h->count * h->ld * esize(h->dtype);
    char* dst16 = has_copy(h) ? (char*)h->sweep_data + (size_t)h->count * h->ld * 2 : nullptr;
    if (src_is_device) {
        prof_begin(h, st);
        if ((rc = launch_ingest<false>(public_dtype(h), rows, 0, 0, 0, 0, n, h->dim, h->ld, dst, h->num_sms, st, 0, 0, 0.f, dst16))) return rc;
        prof_end(h, st);
    } else {
        // Staged in slices through TWO device buffers so that a huge host matrix never needs a device copy of itself and
        // the copy of slice i + 1 (on the handle's copy stream) overlaps K1 on slice i (on `st`):
        //   copy stream:  wait free[b] -> H2D into stage[b] -> record ready[b]
        //   st:           wait ready[b] -> K1 -> record free[b]
        const size_t row_b = (size_t)h->dim * 4;
        const int64_t slice = (int64_t)((64u << 20) / row_b) + 1;
        if (!h->copy_stream) {
            CU_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
            for (int b = 0; b < 2; ++b) {
                CU_TRY(cudaEventCreateWithFlags(&h->stage_ready[b], cudaEventDisableTiming));
                CU_TRY(cudaEventCreateWithFlags(&h->stage_free[b], cudaEventDisableTiming));
            }
        }
        const int64_t m_max = n < slice ? n : slice;
        for (int b = 0; b < 2; ++b)
            if ((rc = ensure(h->add_stage2[b], (size_t)m_max * row_b))) return rc;
        CU_TRY(cudaEventRecord(h->stage_free[0], st));   // both buffers are free once the work queued on st so far is done
        CU_TRY(cudaEventRecord(h->stage_free[1], st));
        int b = 0;
        for (int64_t r0 = 0; r0 < n; r0 += slice, b ^= 1) {
            const int64_t m = n - r0 < slice ? n - r0 : slice;
            CU_TRY(cudaStreamWaitEvent(h->copy_stream, h->stage_free[b], 0));
            CU_TRY(cudaMemcpyAsync(h->add_stage2[b].p, rows + (size_t)r0 * h->dim, (size_t)m * row_b, cudaMemcpyHostToDevice, h->copy_stream));
            CU_TRY(cudaEventRecord(h->stage_ready[b], h->copy_stream));
            CU_TRY(cudaStreamWaitEvent(st, h->stage_ready[b], 0));
            prof_begin(h, st);
            if ((rc = launch_ingest<false>(public_dtype(h), (const float*)h->add_stage2[b].p, 0, 0, 0, 0, m, h->dim, h->ld,
                                           dst + (size_t)r0 * h->ld * esize(h->dtype), h->num_sms, st, 0, 0, 0.f,
                                           dst16 ? dst16 + (size_t)r0 * h->ld * 2 : nullptr)))
                return rc;
            prof_end(h, st);
            CU_TRY(cudaEventRecord(h->stage_free[b], st));
        }
        CU_TRY(cudaStreamSynchronize(h->copy_stream));   // the host buffer is reusable on return
        CU_TRY(cudaStreamSynchronize(st));
    }
    h->count += n;
    return mark_done(h, st);
}

extern "C" int ragfin_add_synthetic(ragfin_t* h, uint64_t seed, int64_t row0, int64_t n, int32_t dup_every,
                                    int32_t zero_every, void* stream) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (n < 0 || row0 < 0) return fail(RAGFIN_EINVAL, "bad row0/n");
    if (n == 0) return RAGFIN_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    if (h->is_view) return fail(RAGFIN_EUNSUPPORTED, "a view is read-only: add rows through the handle that owns the matrix");
    if (h->count + n > h->capacity)
        return fail(RAGFIN_ENOMEM, "add of %lld rows exceeds capacity (%lld of %lld used)", (long long)n,
                    (long long)h->count, (long long)h->capacity);
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if ((rc = wait_prev(h, st))) return rc;
    char* dst = (char*)h->data + (size_t)h->count * h->ld * esize(h->dtype);
    char* dst16 = has_copy(h) ? (char*)h->sweep_data + (size_t)h->count * h->ld * 2 : nullptr;
    if ((rc = launch_ingest<true>(public_dtype(h), nullptr, mix64(seed), row0, dup_every, zero_every, n, h->dim, h->ld, dst,
                                  h->num_sms, st, 0, 0, 0.f, dst16)))
        return rc;
    h->count += n;
    return mark_done(h, st);
}

// "Templated corpus" generator (bench / tests): rows row0..row0+n of a matrix whose row r is
//   centre(topic = r / topic_rows) + noise(r) * 2^-noise_shift
// with centre = row `topic` of the synthetic matrix (seed + RAGFIN_TOPIC_SEED_OFFSET) and noise = row r of the synthetic
// matrix `seed`: contiguous runs of topic_rows near-duplicates in topic order (what repeated templated text looks like to
// a vector store).  Every value is exact in fp32, so the oracle rebuilds the same rows on the host.
extern "C" int ragfin_add_synthetic_topics(ragfin_t* h, uint64_t seed, int64_t row0, int64_t n, int64_t topic_rows,
                                           int32_t noise_shift, void* stream) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (n < 0 || row0 < 0 || topic_rows < 1 || noise_shift < 1 || noise_shift > 10) return fail(RAGFIN_EINVAL, "bad row0 / n / topic_rows / noise_shift");
    if (n == 0) return RAGFIN_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    if (h->is_view) return fail(RAGFIN_EUNSUPPORTED, "a view is read-only: add rows through the handle that owns the matrix");
    if (h->count + n > h->capacity)
        return fail(RAGFIN_ENOMEM, "add of %lld rows exceeds capacity (%lld of %lld used)", (long long)n,
                    (long long)h->count, (long long)h->capacity);
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if ((rc = wait_prev(h, st))) return rc;
    char* dst = (char*)h->data + (size_t)h->count * h->ld * esize(h->dtype);
    char* dst16 = has_copy(h) ? (char*)h->sweep_data + (size_t)h->count * h->ld * 2 : nullptr;
    if ((rc = launch_ingest<true>(public_dtype(h), nullptr, mix64(seed), row0, 0, 0, n, h->dim, h->ld, dst, h->num_sms, st, topic_rows,
                                  mix64(seed + RAGFIN_TOPIC_SEED_OFFSET), ldexpf(1.0f, -noise_shift), dst16)))
        return rc;
    h->count += n;
    return mark_done(h, st);
}

static int read_rows_of(ragfin* h, const void* base, int dtype, int64_t row0, int64_t n, void* out_host, int32_t* ld_out) {
    if (!h || !out_host) return fail(RAGFIN_EINVAL, "NULL argument");
    if (row0 < 0 || n < 0 || row0 + n > h->count) return fail(RAGFIN_EINVAL, "rows [%lld, %lld) outside [0, %lld)",
                                                               (long long)row0, (long long)(row0 + n), (long long)h->count);
    DeviceGuard g(h->device);
    CU_TRY(cudaDeviceSynchronize());
    const size_t rb = (size_t)h->ld * esize(dtype);
    CU_TRY(cudaMemcpy(out_host, (const char*)base + (size_t)row0 * rb, (size_t)n * rb, cudaMemcpyDeviceToHost));
    if (ld_out) *ld_out = h->ld;
    return RAGFIN_OK;
}

extern "C" int ragfin_read_rows(ragfin_t* h, int64_t row0, int64_t n, void* out_host, int32_t* ld_out) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(h->mu);
    return read_rows_of(h, h->data, h->dtype, row0, n, out_host, ld_out);
}

extern "C" int ragfin_read_sweep_rows(ragfin_t* h, int64_t row0, int64_t n, void* out_host, int32_t* ld_out) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(h->mu);
    return read_rows_of(h, h->sweep_data, h->sweep_dt, row0, n, out_host, ld_out);
}

// ------------------------------------------------------------------------------
// K2 dispatch
// ------------------------------------------------------------------------------
typedef void (*scan_fn)(const void*, int64_t, int, const float*, int, int, u64*, int64_t, const uint32_t*);
static const int kMaxScanCtasPerSm = 4;

template <int DT, int NQ>
static scan_fn pick_steps(int steps) {
    switch (steps) {
        case 1: return scan_topk_kernel<DT, NQ, 1>;
        case 2: return scan_topk_kernel<DT, NQ, 2>;
        case 3: return scan_topk_kernel<DT, NQ, 3>;
        case 4: return scan_topk_kernel<DT, NQ, 4>;
        case 6: return scan_topk_kernel<DT, NQ, 6>;
        case 8: return scan_topk_kernel<DT, NQ, 8>;
    }
    return nullptr;
}
template <int DT>
static scan_fn pick_nq(int nqt, int steps) {
    switch (nqt) {
        case 1: return pick_steps<DT, 1>(steps);
        case 2: return pick_steps<DT, 2>(steps);
        case 4: return pick_steps<DT, 4>(steps);
    }
    return nullptr;
}
static scan_fn pick_scan(int dt, int nqt, int steps) {
    switch (dt) {
        case 0: return pick_nq<0>(nqt, steps);
        case 1: return pick_nq<1>(nqt, steps);
        case 2: return pick_nq<2>(nqt, steps);
    }
    return nullptr;
}
// TMA-fed variant (scan_tma.cuh): 1 or 2 query register sets (larger batches take the tensor-core path)
template <int DT, int NQ>
static scan_fn pick_tma_steps(int steps) {
    switch (steps) {
        case 1: return scan_tma_kernel<DT, NQ, 1>;
        case 2: return scan_tma_kernel<DT, NQ, 2>;
        case 3: return scan_tma_kernel<DT, NQ, 3>;
        case 4: return scan_tma_kernel<DT, NQ, 4>;
        case 6: return scan_tma_kernel<DT, NQ, 6>;
        case 8: return scan_tma_kernel<DT, NQ, 8>;
    }
    return nullptr;
}
static scan_fn pick_scan_tma(int dt, int nqt, int steps) {
    if (nqt != 1 && nqt != 2) return nullptr;
    switch (dt) {
        case 0: return nqt == 1 ? pick_tma_steps<0, 1>(steps) : pick_tma_steps<0, 2>(steps);
        case 1: return nqt == 1 ? pick_tma_steps<1, 1>(steps) : pick_tma_steps<1, 2>(steps);
        case 2: return nqt == 1 ? pick_tma_steps<2, 1>(steps) : pick_tma_steps<2, 2>(steps);
    }
    return nullptr;
}
static int round_steps(int need) {
    static const int allowed[] = {1, 2, 3, 4, 6, 8};
    for (int s : allowed)
        if (s >= need) return s;
    return 0;
}

// candidates kept per query before the exact rescore: k plus a guard band, in lists of 32
static int cand_per_query(int k) {
    const int slack = k / 4 > 16 ? k / 4 : 16;
    const int want = k + slack;
    for (int kp = 32; kp <= 256; kp <<= 1)
        if (kp >= want) return kp;
    return 0;
}

// |fp32-accumulated dot - exact dot| for unit-norm operands (any summation order), plus the
// fp32 rounding of the exact score and one ulp so that a tie after rounding cannot hide a row.
static float eps_fp32_accumulate(int ld) { return (float)((ld + 64) * 0x1p-24 * 1.0625 + 4.76837158203125e-07); }

static const size_t kHostStageQ = 64 << 10, kHostStageOut = 64 << 10;   // mapped staging of ragfin_search_host (small requests)
static const size_t kHostStageFlag = 64;                                // ... + the completion word the one-kernel search sets

// The mapped staging of the synchronous host calls.  Its completion word starts at 0 (host_seq counts from 1): pinned memory
// freed by a destroyed handle can come back here still holding that handle's last sequence number, which would make the
// first poll succeed before the kernel has written anything.
static int alloc_hstage(ragfin* h) {
    if (cudaHostAlloc(&h->hstage, kHostStageQ + kHostStageOut + kHostStageFlag, cudaHostAllocMapped) != cudaSuccess) {
        (void)cudaGetLastError();
        h->hstage = nullptr;
        return fail(RAGFIN_ENOMEM, "pinned staging allocation failed");
    }
    memset((char*)h->hstage + kHostStageQ + kHostStageOut, 0, kHostStageFlag);
    return 0;
}
static const int kMaxQueryBatch = 4096;  // queries per pass through the pipeline (bounds the workspace)

// ------------------------------------------------------------------------------
// K3 host side: tensor maps (driver entry point, no -lcuda), slice plan, launch
// ------------------------------------------------------------------------------
typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static encode_tiled_fn get_encode_tiled() {
    static encode_tiled_fn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (encode_tiled_fn)p;
        else
            (void)cudaGetLastError();
    });
    return fn;
}

static const int kMapI8 = 4;   // make_map dtype of the int8 screen copy
// [rows, ld] row-major matrix of `dtype`; box = 128 bytes of K x box_rows rows, 128-byte swizzle, zero OOB fill
static int make_map(CUtensorMap* map, int dtype, const void* base, int64_t rows, int ld, int box_rows) {
    encode_tiled_fn enc = get_encode_tiled();
    if (!enc) return fail(RAGFIN_ECUDA, "cuTensorMapEncodeTiled is not available from the driver");
    const CUtensorMapDataType dt = dtype == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                   : dtype == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                   : dtype == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8;
    const size_t es = dtype == kMapI8 ? 1 : esize(dtype);
    const cuuint64_t dims[2] = {(cuuint64_t)ld, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * es};
    const cuuint32_t box[2] = {(cuuint32_t)(kGKBytes / es), (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(RAGFIN_ECUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return 0;
}

// make_map through the handle's cache (caller holds h->mu)
static int cached_map(ragfin* h, CUtensorMap* map, int dtype, const void* base, int64_t rows, int ld, int box_rows) {
    for (ragfin::MapSlot& m : h->map_cache)
        if (m.base == base && m.rows == rows && m.ld == ld && m.dtype == dtype && m.box_rows == box_rows) { *map = m.map; return 0; }
    int rc = make_map(map, dtype, base, rows, ld, box_rows);
    if (rc) return rc;
    ragfin::MapSlot& m = h->map_cache[h->map_next];
    h->map_next = (h->map_next + 1) % 8;
    m.base = base; m.rows = rows; m.ld = ld; m.dtype = dtype; m.box_rows = box_rows; m.map = *map;
    return 0;
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) and the occupancy query are per (device, function) facts: doing
// them once instead of on every call takes ~10 us of host time off each search (it shows in the host-path latency).
static std::mutex g_fn_mu;
static std::map<std::pair<int, const void*>, size_t> g_fn_smem;
static std::map<std::pair<std::pair<int, const void*>, size_t>, int> g_fn_occ;
static int set_dyn_smem(int device, const void* fn, size_t smem) {
    std::lock_guard<std::mutex> lk(g_fn_mu);
    auto key = std::make_pair(device, fn);
    auto it = g_fn_smem.find(key);
    if (it != g_fn_smem.end() && it->second >= smem) return 0;
    CU_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    g_fn_smem[key] = smem;
    return 0;
}
static int blocks_per_sm(int device, const void* fn, int threads, size_t smem, int* out) {
    std::lock_guard<std::mutex> lk(g_fn_mu);
    auto key = std::make_pair(std::make_pair(device, fn), smem);
    auto it = g_fn_occ.find(key);
    if (it != g_fn_occ.end()) { *out = it->second; return 0; }
    int v = 0;
    CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, fn, threads, smem));
    g_fn_occ[key] = v;
    *out = v;
    return 0;
}

struct GemmPlan {
    int QT, S, stages, grid, C;
    int64_t rows_per_slice;
};

// Items are (query tile, slice).  Pick the number of waves w (items per CTA) whose slice count S = floor(SMs*w/QT)
// leaves the fewest CTAs idle, with at least one 256-row tile per slice.
static GemmPlan plan_gemm(int nq, int64_t n, int num_sms, int kp, int C) {
    GemmPlan p;
    p.C = C;
    p.QT = (nq + kGM - 1) / kGM;
    const int groups = (p.QT + C - 1) / C;   // work items are (group of C query tiles, slice), one per cluster
    num_sms /= C;                            // = clusters that can be resident
    const int64_t n_tiles = (n + kGN - 1) / kGN;
    double best = 1e300;
    int bestS = 1;
    for (int w = 1; w <= 8; ++w) {
        int64_t S = (int64_t)num_sms * w / groups;
        if (S < 1) S = 1;
        if (S > n_tiles) S = n_tiles;
        const int64_t tps = (n_tiles + S - 1) / S;
        S = (n_tiles + tps - 1) / tps;
        const int64_t items = (int64_t)groups * S;
        // sweep length in tiles, plus a per-item charge: every extra slice of a query restarts its candidate list
        const double cost = (double)((items + num_sms - 1) / num_sms) * ((double)tps + 24.0);
        if (cost < best) { best = cost; bestS = (int)S; }
    }
    const int64_t tps = (n_tiles + bestS - 1) / bestS;
    p.S = (int)((n_tiles + tps - 1) / tps);
    p.rows_per_slice = tps * kGN;
    p.stages = kp <= 32 ? 4 : kp <= 64 ? 3 : 2;
    const int64_t items = (int64_t)groups * p.S;
    p.grid = (int)(items < num_sms ? items : num_sms) * C;
    return p;
}

// |tensor-core score - exact score| beyond the query rounding term.
// Accumulation: the products of two 16-bit (or tf32) operands are exact in fp32; what errs is their summation.  Model: every
// addend entering an accumulation step - ld products and, per 16-element MMA step, the running sum, i.e. ld * 17 / 16 addends -
// is aligned to the largest exponent of the step and TRUNCATED there, losing less than one fp32 ulp of a magnitude that never
// exceeds sum |x_i q_i| <= |x|_2 |q|_2 <= 1.0078 (stored rows: <= 1 + 2^-8; queries: <= 1 + 2^-22): less than 2^-23 * 1.0078
// each, so |error| < 1.0625 * ld * 2^-23 * 1.0078 (9.8e-5 at ld = 768) for ANY summation order and grouping.  The allowance
// below is twice that model (2^-22 per element, + 64 elements, + one ulp so that rounding the exact score cannot create a
// tie); tests/test_parity_gpu.py::test_tensor_core_error_stays_inside_the_allowance measures the real error on adversarial
// (all-positive, maximal partial sums) and random operands through the raw-score hook and requires it to stay below a
// quarter of the allowance.  Round 1 used 2^-21 per element.
// fp32 storage (kind::tf32): both operands are truncated to 10 explicit mantissa bits, 2^-10 relative each.
static float eps_gemm_const(int dtype, int ld) {
    double e = (ld + 64) * 2.384185791015625e-07 * 1.0625 + 4.76837158203125e-07;   // (ld + 64) * 2^-22 * 17/16 + 2^-21
    if (dtype == 0) e += 2.0 * 9.765625e-04 * 1.0625;                               // 2 * 2^-10
    return (float)e;
}
// |approximate score - exact score| beyond the query rounding term, for the rows the sweeps read: + eps_sweep when they are
// the fp16 copy of fp32 rows (the exact score is the fp32 row's)
static float eps_approx(int sweep_dt, int ld, float eps_sweep) {
    const float e = eps_gemm_const(sweep_dt, ld);
    if (eps_sweep == 0.f) return e;
    return nextafterf((float)((double)e + (double)eps_sweep), INFINITY);
}
static float eps_approx(const ragfin* h) { return eps_approx(h->sweep_dt, h->ld, h->eps_sweep); }

// TMA coordinates are signed 32-bit: shards of 2^31 rows or more stay on the scan path (int64 row arithmetic)
static bool gemm_rows_ok(const ragfin* h) { return h->count > 0 && h->count < ((int64_t)1 << 31) - kGN; }
static bool gemm_supported(const ragfin* h, int kp) { return kp <= 128 && gemm_rows_ok(h); }

// Scores the nb normalised queries in h->qhat against the corpus on the tensor cores.  Fills
// h->cand as [nb][S][kp] (unsorted lists) and h->eps_q; returns S through *G.  dump != null: write raw scores instead.
// Corpus size from which even 1-2 queries take the tensor-core sweep: its TMA ring streams at 7.3 TB/s against the
// LDG scan's 6.9, but it carries ~35 us more fixed cost per call (bound pass, append finalize).  Measured (bf16,
// 768-d, batch 1, whole call): 10M rows 2.16 vs 2.31 ms; 2.5M rows 0.606 vs 0.632 ms; 1.25M rows (1.9 GB, the shard
// of the 8-GPU split) 0.340 vs 0.355 ms, batch 2: 0.339 vs 0.389 ms.
static const size_t kSweepBytes = (size_t)1 << 30;

static const int kAppendCap = 16384;   // append mode: keys one query may collect before it overflows to tier 2
static const int kAppendMaxK = 256;    // largest k the append mode serves (tier 2, its overflow path, keeps 256 keys)

// Append mode needs the bound pass (no scalar filter) and at least 4 k corpus tiles to draw 2 k sample blocks from.
// Tombstones alone keep it: the bound pass and the append epilogues honour the mask (DESIGN.md, "Deleted rows").
static bool append_eligible(const ragfin* h, int k) {
    const int64_t n_tiles = (h->count + kGN - 1) / kGN;
    return h->use_bound_pass && h->use_append && !h->cur_user_filter && k <= kAppendMaxK && n_tiles >= 4 * (int64_t)k &&
           h->count < ((int64_t)1 << 31) - kGN;
}

// Cluster size of the single-CTA-MMA kernel by the number of query tiles.  Measured interleaved on 10M x 768 bf16
// (profiles/r02/policy_sweep.log): pairs beat quads at every batch (512: 6.71 vs 7.67 ms, 768: 9.5 vs 14.5, 4096: 47.9 vs 55.0;
// round 1's table, measured in separate runs, had quads ahead at 3-7 tiles) and the 2-SM MMA kernel (gemm_pair.cuh) beats both
// (see run_gemm), so this policy only serves what the pair kernel does not: list mode (filters, small corpora) and fp32 dumps.
static int auto_cluster(int QT0) { return QT0 >= 2 ? 2 : 1; }

// Sample ("bound") pass geometry: nblk blocks of g sample tiles each; sample tile j is corpus tile j * bstride, so the
// tiles are distinct and the last (possibly partial) tile is never sampled.  Callers guarantee n_tiles >= 4 * rank.
static void bound_geometry(int64_t n_tiles, int rank, bool append, int QT0, int k, int* nblk_out, int* g_out, int64_t* bstride_out) {
    // blocks: 16 x rank keeps the rank best sample rows in distinct blocks (expected collisions rank / 32)
    int64_t want_blk = 16 * (int64_t)rank;
    if (want_blk < 256) want_blk = 256;
    if (want_blk > 1024) want_blk = 1024;
    int nblk = (int)(n_tiles / 2 < want_blk ? n_tiles / 2 : want_blk);
    // Sample fraction f.  A query collects ~1.6 * k / f rows; the bound pass costs f of a sweep.  HBM-bound
    // batches (one query tile) have epilogue slack, so f only has to keep the buffer well under kAppendCap;
    // tensor-bound batches pay ~2.6e-3 ms per unit of k / f in the epilogue's slow path (measured: 13 ms at
    // k = 100, f = 2 %), which puts the optimum near 0.8 % * sqrt(k) (2.5 % for k = 10, 8 % for k = 100).
    double frac = append ? (double)k / 5000.0 : 0.0;
    const double frac_min = (append && QT0 == 1) ? 1.0 / 256.0 : 1.0 / 96.0;   // one query tile: the pass is pure latency
    if (frac < frac_min) frac = frac_min;
    if (append && QT0 >= 2) {
        const double opt = 0.008 * sqrt((double)k);
        if (opt > frac) frac = opt;
    }
    int64_t sample = (int64_t)(frac * (double)n_tiles);
    if (sample < nblk) sample = nblk;
    if (sample > n_tiles / 2) sample = n_tiles / 2;
    int g = (int)((sample + nblk / 2) / nblk);
    if (g < 1) g = 1;
    while (g > 1 && (int64_t)nblk * g > n_tiles / 2) --g;
    int64_t bstride = (n_tiles - 1) / ((int64_t)nblk * g);   // the last (possibly partial) tile is never sampled
    if (bstride < 1) bstride = 1;
    *nblk_out = nblk; *g_out = g; *bstride_out = bstride;
}

// Scores the nb normalised queries in h->qhat against the corpus on the tensor cores and leaves per-query candidates
// for the finalize step: list mode fills h->cand as [nb][S][kp] (unsorted lists, S returned through *G); append
// mode (*appended = true) fills h->cand as [nb][kAppendCap] with h->acnt[q] keys each.  dump != null: raw scores.
static int run_gemm(ragfin* h, int nb, int k, int kp, int* G, bool* appended, float* dump, cudaStream_t st, bool prepped = false) {
    int rc;
    const int64_t n = h->count;
    *appended = false;
    // cluster size along the query-tile axis: multicast pays once several query tiles share a slice
    const int QT0 = (nb + kGM - 1) / kGM;
    int C = h->gemm_cluster ? h->gemm_cluster : auto_cluster(QT0);
    // 2-SM MMA sweep (gemm_pair.cuh, tcgen05 cta_group::2) for >= 2 query tiles: the default since the interleaved sweep of
    // profiles/r02/policy_sweep.log - faster than the best single-CTA configuration at every batch from 129 to 4096 queries
    // (256: 3.07 vs 3.49 ms, 1024: 11.97 vs 14.00, 2048: 21.8 vs 25.4, 4096: 45.3 vs 47.9 = 1 390 TFLOP/s); variant 1 forces
    // the single-CTA kernel
    // the single-CTA kernel, and so does a forced cluster size other than 2
    const bool want_pair = (h->gemm_variant == 4 || ((h->gemm_variant == 0 || h->gemm_variant == 3) && (h->gemm_cluster == 0 || h->gemm_cluster == 2))) && QT0 >= 2;
    if (want_pair) C = 2;
    typedef void (*gemm_fn)(const CUtensorMap, const CUtensorMap, const GemmArgs);
#define RF_PICK_MODE(KIND, CC) (mode == 0 ? gemm_topk_kernel<KIND, 0, CC> : mode == 1 ? gemm_topk_kernel<KIND, 1, CC> : mode == 2 ? gemm_topk_kernel<KIND, 2, CC> : gemm_topk_kernel<KIND, 3, CC>)
    auto pick = [&](int c, int mode) -> gemm_fn {
        if (h->sweep_dt == 0) return c == 4 ? RF_PICK_MODE(1, 4) : c == 2 ? RF_PICK_MODE(1, 2) : RF_PICK_MODE(1, 1);
        return c == 4 ? RF_PICK_MODE(0, 4) : c == 2 ? RF_PICK_MODE(0, 2) : RF_PICK_MODE(0, 1);
    };
#undef RF_PICK_MODE
    // Sample ("bound") pass geometry.  nblk blocks of g sample tiles each, evenly strided over the corpus; the
    // rank-th largest block maximum bounds the rank-th best score from below.  Needs at least twice as many blocks
    // as the rank and samples at most half of the corpus; skipped under a scalar filter and for the dump hook.  Under
    // tombstones alone it runs with the mask: excluded sample rows never raise a block maximum.
    const int64_t n_tiles = (n + kGN - 1) / kGN;
    const bool can_bound = !dump && h->use_bound_pass && !h->cur_user_filter;
    const bool append = !dump && append_eligible(h, k);
    const bool bound = append || (can_bound && n_tiles >= 4 * (int64_t)kp);
    const int rank = append ? k : kp;
    int nblk = 0, g = 1;
    int64_t bstride = 1;
    if (bound) bound_geometry(n_tiles, rank, append, QT0, k, &nblk, &g, &bstride);
    int stages0 = append ? 4 : kp <= 32 ? 4 : kp <= 64 ? 3 : 2;
#ifdef RAGFIN_TIMING_EXPERIMENTS
    { const char* e = getenv("RAGFIN_GEMM_STAGES"); if (e && atoi(e) >= 2 && atoi(e) <= stages0) stages0 = atoi(e); }
#endif
    const int kp_smem = append ? 0 : kp;      // append mode keeps no lists in shared memory
    const size_t smem = gemm_smem_bytes(stages0, kp_smem);
    const int mode = dump ? 1 : append ? 3 : 0;
    gemm_fn fn = pick(C, mode);
    if ((rc = set_dyn_smem(h->device, (const void*)fn, smem))) return rc;
    int resident_clusters = h->num_sms;
    if (C > 1) {   // how many clusters of C CTAs the device can hold at once (GPC packing may strand SMs)
        cudaLaunchConfig_t qc = {};
        qc.gridDim = dim3(h->num_sms / C * C);
        qc.blockDim = dim3(kGemmThreads);
        qc.dynamicSmemBytes = smem;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        qc.attrs = at; qc.numAttrs = 1;
        int nc = 0;
        CU_TRY(cudaOccupancyMaxActiveClusters(&nc, (const void*)fn, &qc));
        if (nc < 1) { C = 1; fn = pick(1, mode); if ((rc = set_dyn_smem(h->device, (const void*)fn, smem))) return rc; }
        else resident_clusters = nc;
    }
    GemmPlan p = plan_gemm(nb, n, C > 1 ? resident_clusters * C : h->num_sms, kp, C);
    p.stages = stages0;
    // A operand: the query tiles, padded with zero rows to whole tiles (search_locked zeroes qhat's padding; the
    // 16-bit copy is zeroed here) so that no TMA box of the A operand is partly out of bounds
    const int nb_pad = p.QT * kGM;
    const float* qhat = (const float*)h->qhat.p;
    const void* a_base = qhat;
    if (prepped) {   // prep_queries_kernel already produced qhat, q16, eps_q and cleared gtau
        if (h->sweep_dt != 0) a_base = h->q16.p;
    } else if ((rc = ensure(h->eps_q, (size_t)nb * sizeof(float)))) {
        return rc;
    } else if (h->sweep_dt != 0) {
        if ((rc = ensure(h->q16, (size_t)nb_pad * h->ld * 2))) return rc;
        if (nb_pad > nb) CU_TRY(cudaMemsetAsync((char*)h->q16.p + (size_t)nb * h->ld * 2, 0, (size_t)(nb_pad - nb) * h->ld * 2, st));
        const int wpb = 8;
        if (h->sweep_dt == 1)
            qconv_kernel<1><<<(nb + wpb - 1) / wpb, wpb * 32, 0, st>>>(qhat, nb, h->ld, (__nv_bfloat16*)h->q16.p, (float*)h->eps_q.p);
        else
            qconv_kernel<2><<<(nb + wpb - 1) / wpb, wpb * 32, 0, st>>>(qhat, nb, h->ld, (__half*)h->q16.p, (float*)h->eps_q.p);
        CU_TRY(cudaGetLastError());
        h->stats.launches++;
        a_base = h->q16.p;
    } else {
        CU_TRY(cudaMemsetAsync(h->eps_q.p, 0, (size_t)nb * sizeof(float), st));
    }
    CUtensorMap tmA, tmB;
    if ((rc = cached_map(h, &tmA, h->sweep_dt, a_base, nb_pad, h->ld, kGM))) return rc;
    if ((rc = cached_map(h, &tmB, h->sweep_dt, h->sweep_data, n, h->ld, kGN / C))) return rc;   // each CTA fetches 1/C of a tile
    if (append) {
        if ((rc = ensure(h->cand, (size_t)nb * kAppendCap * sizeof(u64)))) return rc;
        if ((rc = ensure(h->acnt, (size_t)nb * sizeof(uint32_t)))) return rc;
        if ((rc = ensure(h->athr, (size_t)nb * sizeof(float)))) return rc;
    } else if (!dump) {
        if ((rc = ensure(h->cand, (size_t)nb * p.S * kp * sizeof(u64)))) return rc;
    }
    GemmArgs a;
    a.idesc = make_idesc(h->sweep_dt == 0 ? 2 : h->sweep_dt == 1 ? 1 : 0);
    a.k_elems = kGKBytes / (int)esize(h->sweep_dt);
    a.num_kblocks = (h->ld + a.k_elems - 1) / a.k_elems;
    a.nq = nb;
    a.n_rows = n;
    a.QT = p.QT;
    a.S = p.S;
    a.rows_per_slice = p.rows_per_slice;
    a.stages = p.stages;
    a.kp = kp_smem;
    if ((rc = ensure(h->gtau, (size_t)nb * sizeof(uint32_t)))) return rc;
    if (!append && !prepped) CU_TRY(cudaMemsetAsync(h->gtau.p, 0, (size_t)nb * sizeof(uint32_t), st));
    a.cand = (u64*)h->cand.p;
    a.gtau = (uint32_t*)h->gtau.p;
    a.allow = h->cur_allow;
    a.dump = dump;
    a.bound_tps = 0; a.bound_tiles = 0; a.bound_stride = 0;
    a.thr = (const float*)h->athr.p; a.cnt = (uint32_t*)h->acnt.p; a.cap = kAppendCap;
    a.wcap = nullptr; a.whi = nullptr;
    a.dbg = 0;
#ifdef RAGFIN_TIMING_EXPERIMENTS   // scripts/gemm_dbg_sweep.py: switch pipeline stages off (INVALID results, timing only)
    { const char* e = getenv("RAGFIN_GEMM_DEBUG"); a.dbg = e ? atoi(e) : 0; }
#endif
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;

    const float* wlo = nullptr;
    if (append && h->cur_window) {   // range search: per-query window words (window_words_kernel) for the three passes below
        if ((rc = ensure(h->awin, (size_t)3 * nb * sizeof(float)))) return rc;
        float* w = (float*)h->awin.p;
        RF_LAUNCH(window_words_kernel, (nb + 127) / 128, 128, 0, st, nb, h->cur_radius, h->cur_range_filter, eps_approx(h),
                                                                   (const float*)h->eps_q.p, w);
        CU_TRY(cudaGetLastError());
        h->stats.launches++;
        wlo = w; a.whi = w + nb; a.wcap = w + 2 * nb;
    }
    if (bound) {
        const int groups = (p.QT + C - 1) / C;
        const int clusters = C > 1 ? resident_clusters : h->num_sms;
        GemmArgs b = a;
        b.S = nblk;                 // one item per (group of query tiles, block)
        b.bound_tps = g;
        b.bound_tiles = nblk * g;
        b.bound_stride = bstride;
        if ((rc = ensure(h->bmax, (size_t)nb * nblk * sizeof(float)))) return rc;
        b.dump = (float*)h->bmax.p;
        gemm_fn bfn = pick(C, 2);
        if ((rc = set_dyn_smem(h->device, (const void*)bfn, smem))) return rc;
        const int64_t items = (int64_t)groups * nblk;
        cfg.gridDim = dim3((unsigned)(items < clusters ? items : clusters) * C);
        CU_TRY(cudaLaunchKernelEx(&cfg, bfn, tmA, tmB, b));
        RF_LAUNCH(bound_select_kernel, nb, 256, 0, st, (const float*)h->bmax.p, nblk, rank, append ? nullptr : (uint32_t*)h->gtau.p,
                                                 append ? (float*)h->athr.p : nullptr, append ? (uint32_t*)h->acnt.p : nullptr,
                                                 eps_approx(h), (const float*)h->eps_q.p, wlo);
        CU_TRY(cudaGetLastError());
        h->stats.launches += 2;
    }
    if (append && (h->gemm_variant == 3 || h->gemm_variant == 0) && nb <= kRN && C == 1 && rows_stages(a.num_kblocks) >= 3) {
        // <= 16 queries, operand roles swapped (gemm_rows.cuh): corpus rows are the MMA's M, the queries its N = 16
        RowsArgs r;
        r.idesc = make_idesc_n(h->sweep_dt == 0 ? 2 : h->sweep_dt == 1 ? 1 : 0, kRN);
        r.num_kblocks = a.num_kblocks; r.k_elems = a.k_elems; r.nq = nb; r.n_rows = n;
        r.S = p.S; r.rows_per_slice = p.rows_per_slice; r.stages = rows_stages(a.num_kblocks);
        r.cand = a.cand; r.thr = a.thr; r.cnt = a.cnt; r.cap = a.cap; r.allow = a.allow; r.whi = a.whi;
        CUtensorMap tmQ;
        if ((rc = cached_map(h, &tmQ, h->sweep_dt, a_base, nb_pad, h->ld, kRN))) return rc;
        typedef void (*rows_fn)(const CUtensorMap, const CUtensorMap, const RowsArgs);
        rows_fn rfn = h->sweep_dt == 0 ? gemm_rows_kernel<1> : gemm_rows_kernel<0>;
        const size_t rsmem = rows_smem_bytes(r.num_kblocks, r.stages);
        if ((rc = set_dyn_smem(h->device, (const void*)rfn, rsmem))) return rc;
        prof_begin(h, st);
        RF_LAUNCH(rfn, p.grid, kGemmThreads, rsmem, st, tmQ, tmB, r);
        prof_end(h, st);
    } else if (want_pair && C == 2 && (append || dump)) {
        // gemm variant 4 (gemm_pair.cuh): one M = 256 MMA per cluster, each CTA holds half of the corpus tile
        GemmArgs pa = a;
        pa.idesc = make_idesc_pair(h->sweep_dt == 0 ? 2 : h->sweep_dt == 1 ? 1 : 0);
        pa.stages = kPMaxStages;
        gemm_fn pfn = h->sweep_dt == 0 ? (dump ? gemm_pair_kernel<1, 1> : gemm_pair_kernel<1, 3>)
                                    : (dump ? gemm_pair_kernel<0, 1> : gemm_pair_kernel<0, 3>);
        const size_t psmem = pair_smem_bytes(pa.stages);
        if ((rc = set_dyn_smem(h->device, (const void*)pfn, psmem))) return rc;
        cfg.dynamicSmemBytes = psmem;
        cfg.gridDim = dim3(p.grid);
        prof_begin(h, st);
        CU_TRY(cudaLaunchKernelEx(&cfg, pfn, tmA, tmB, pa));
        prof_end(h, st);
    } else {
        cfg.gridDim = dim3(p.grid);
        prof_begin(h, st);
        CU_TRY(cudaLaunchKernelEx(&cfg, fn, tmA, tmB, a));
        prof_end(h, st);
    }
    CU_TRY(cudaGetLastError());
    h->stats.launches++;
    *G = p.S;
    *appended = append;
    return 0;
}

static bool astat_supported(const ragfin* h, int kp) {
    return h->dtype != 0 && h->ld <= 2 * kAColsMax && (kp == 32 || kp == 64 || kp == 128) && h->count > 0;
}

// A-stationary tcgen05 path (gemm_astat.cuh): same contract as run_gemm.
static int run_gemm_astat(ragfin* h, int nb, int kp, int* G, float* dump, cudaStream_t st) {
    int rc;
    const int64_t n = h->count;
    const int QT0 = (nb + kGM - 1) / kGM;
    int C = h->gemm_cluster ? h->gemm_cluster : (QT0 >= 8 ? 4 : QT0 >= 2 ? 2 : 1);
    typedef void (*astat_fn)(const CUtensorMap, const AstatArgs);
    auto pick = [&](int c) -> astat_fn {
        if (dump) return gemm_astat_kernel<true, 1>;
        return c == 4 ? gemm_astat_kernel<false, 4> : c == 2 ? gemm_astat_kernel<false, 2> : gemm_astat_kernel<false, 1>;
    };
    if (dump) C = 1;
    const size_t smem = astat_smem_bytes(kp);
    astat_fn fn = pick(C);
    if ((rc = set_dyn_smem(h->device, (const void*)fn, smem))) return rc;
    int resident_clusters = h->num_sms;
    if (C > 1) {
        cudaLaunchConfig_t qc = {};
        qc.gridDim = dim3(h->num_sms / C * C);
        qc.blockDim = dim3(kGemmThreads);
        qc.dynamicSmemBytes = smem;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        qc.attrs = at; qc.numAttrs = 1;
        int nc = 0;
        CU_TRY(cudaOccupancyMaxActiveClusters(&nc, (const void*)fn, &qc));
        if (nc < 1) { C = 1; fn = pick(1); if ((rc = set_dyn_smem(h->device, (const void*)fn, smem))) return rc; }
        else resident_clusters = nc;
    }
    const GemmPlan p = plan_gemm(nb, n, C > 1 ? resident_clusters * C : h->num_sms, kp, C);
    const float* qhat = (const float*)h->qhat.p;
    if ((rc = ensure(h->eps_q, (size_t)nb * sizeof(float)))) return rc;
    if ((rc = ensure(h->q16, (size_t)nb * h->ld * 2))) return rc;
    const int wpb = 8;
    if (h->dtype == 1)
        qconv_kernel<1><<<(nb + wpb - 1) / wpb, wpb * 32, 0, st>>>(qhat, nb, h->ld, (__nv_bfloat16*)h->q16.p, (float*)h->eps_q.p);
    else
        qconv_kernel<2><<<(nb + wpb - 1) / wpb, wpb * 32, 0, st>>>(qhat, nb, h->ld, (__half*)h->q16.p, (float*)h->eps_q.p);
    CU_TRY(cudaGetLastError());
    h->stats.launches++;
    CUtensorMap tmB;
    if ((rc = cached_map(h, &tmB, h->dtype, h->data, n, h->ld, kSN / C))) return rc;
    if (!dump) {
        if ((rc = ensure(h->cand, (size_t)nb * p.S * kp * sizeof(u64)))) return rc;
    }
    if ((rc = ensure(h->gtau, (size_t)nb * sizeof(uint32_t)))) return rc;
    CU_TRY(cudaMemsetAsync(h->gtau.p, 0, (size_t)nb * sizeof(uint32_t), st));
    AstatArgs a;
    a.idesc = make_idesc_n(h->dtype == 1 ? 1 : 0, kSN);
    a.num_kblocks = (h->ld + 63) / 64;
    a.ld = h->ld;
    a.nq = nb;
    a.n_rows = n;
    a.QT = p.QT;
    a.S = p.S;
    a.rows_per_slice = p.rows_per_slice;
    a.slots = astat_slots(kp);
    a.kp = kp;
    a.q16 = (const uint16_t*)h->q16.p;
    a.cand = (u64*)h->cand.p;
    a.gtau = (uint32_t*)h->gtau.p;
    a.allow = h->cur_allow;
    a.dump = dump;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(p.grid);
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    prof_begin(h, st);
    CU_TRY(cudaLaunchKernelEx(&cfg, fn, tmB, a));
    prof_end(h, st);
    CU_TRY(cudaGetLastError());
    h->stats.launches++;
    *G = p.S;
    return 0;
}

static bool use_astat(const ragfin* h, int kp) {
    if (h->gemm_variant != 2) return false;   // measured slower: only when asked for
    return astat_supported(h, kp);
}

// ------------------------------------------------------------------------------
// Cross-shard exchange state (CUDA IPC gather areas over NVLink peer memory), used by the one-kernel search's finalize
// and by the stand-alone exchange kernels further down
// ------------------------------------------------------------------------------
struct ragfin_exchange {
    int rank = 0, world = 0, device = 0;
    size_t record_max = 0, bytes = 0;
    char* local = nullptr;               // [2][world][record_max] gather area | [2][world] u32 flags | [2][world][kFMaxQ] u32 per-query flags
    char* peer_base[64] = {};            // base of every rank's block in this process's address space
    bool opened[64] = {};
    char** d_peer_area = nullptr;
    uint32_t** d_peer_flag = nullptr;
    uint32_t** d_peer_qflag = nullptr;
    unsigned int* d_done = nullptr;
    uint32_t step = 0;
    bool connected = false;
    const void* owner = nullptr;         // the collection whose one-kernel searches use this exchange (first one to do so)
    bool have_stream = false;            // the slot-ring argument (kernels.cuh: how far a rank can run ahead of a peer) holds only
    cudaStream_t stream = nullptr;       // if every step of this rank is issued on ONE stream: recorded at step 1, checked after
    std::mutex mu;
};

// ------------------------------------------------------------------------------
// K3f: the one-kernel search for <= 64 queries and k <= 128 (sweep_fused.cuh)
// ------------------------------------------------------------------------------
struct FusedPlan {
    int ncol = 0, stages = 0, pend = 0, cap = 0;
    bool split = false;
    size_t smem = 0;
};

// Column count / split / ring depth for nb queries, or ncol = 0 when the shape does not fit one CTA's shared memory.
// Measured (profiles/r02, 1.25M- and 10M-row corpora): the one-kernel search wins up to 16 queries at k = 10 (0.306 vs 0.343 ms
// at 1 query, 0.330 vs 0.343 at 16 on the 1.25M-row shard) and up to ~4 queries at k = 100 (0.347 vs 0.413 ms at 1 query); beyond
// that its per-query bookkeeping in the first tile and the finalize outweigh the launches it saves (32 queries: 0.383 vs 0.343;
// 16 queries at k = 100: 0.504 vs 0.416).  Default limits: <= 16 queries and queries x k <= 400; RAGFIN_FUSED_MAX_NQ /
// RAGFIN_FUSED_MAX_NQK override them (the wider configurations stay compiled in and tested).
// i8: the plan of the int8 tile filter (split only; its query block and state take shared memory too).
static FusedPlan plan_fused(int sweep_dt, int ld, int max_nq, int max_nqk, int stage_cap, int nb, int k, bool i8 = false) {
    FusedPlan best;
    const int nkb8 = ((ld + 15) / 16 * 16 + kGKBytes - 1) / kGKBytes;
    if (nb < 1 || nb > (max_nq < kFMaxQ ? max_nq : kFMaxQ) || k > kFMaxK || (int64_t)nb * k > max_nqk) return best;
    const int es = (int)esize(sweep_dt);
    const int k_elems = kGKBytes / es;
    const int nkb = (ld + k_elems - 1) / k_elems;
    const int pend = nb <= 16 ? 64 : 32;
    const bool can_split = sweep_dt != 0;
    // candidates in order of preference: split (tight error bound) first, then plain
    const int cols_split[3] = {16, 32, 64}, cols_plain[3] = {16, 32, 64};
    for (int pass = 0; pass < 2; ++pass) {
        const bool split = pass == 0;
        if (split && !can_split) continue;
        if (i8 && !split) continue;
        for (int ci = 0; ci < 3; ++ci) {
            const int ncol = split ? cols_split[ci] : cols_plain[ci];
            if ((split ? ncol / 2 : ncol) < nb) continue;
            for (int stages = stage_cap; stages >= 2; --stages) {
                const size_t smem = fused_smem_bytes(nkb, ncol, stages, nb, k, pend) +
                                    (i8 ? (size_t)nkb8 * ncol * kGKBytes + sizeof(FusedI8State) + 16 : 0);
                if (smem > (size_t)227 * 1024) continue;
                const size_t region = (size_t)nkb * ncol * kGKBytes + (size_t)stages * kBBytes;
                const size_t hdr = (((size_t)((ld + 3) / 4 * 4) * 4 + 256 * 4 + 16 + 15) / 16) * 16;
                if (region < hdr + 4096 * sizeof(u64)) continue;      // the finalize's scratch (rows within 2 eps of the k-th score)
                // every CTA appends ~k rows of its first tile, so the buffer scales with k (148 CTAs x 128 = 19 k rows)
                const int cap = k <= 16 ? kAppendCap : 4 * kAppendCap;
                if ((size_t)nb * cap > (size_t)kFMaxQ * kAppendCap) continue;   // one half of the double-buffered append workspace
                FusedPlan f;
                f.ncol = ncol; f.split = split; f.stages = stages; f.pend = pend; f.cap = cap; f.smem = smem;
                return f;
            }
        }
    }
    return best;
}
static FusedPlan plan_fused(const ragfin* h, int nb, int k) {
    return plan_fused(h->sweep_dt, h->ld, h->fused_max_nq, h->fused_max_nqk, h->fused_stage_cap, nb, k);
}

// Query term of the one-kernel search's eps: |approx - exact| <= |q - hi - lo|_2 * max |stored row|_2 + the accumulation
// allowance, where the query enters the MMA as hi = RNE(q) (plain) or hi + lo with lo = RNE(q - hi) (split; q - hi is exact
// in fp32).  Round to nearest with p significant bits is off by at most half an ulp, 2^-p |y| (bf16 p = 8, fp16 p = 11).
// Split: with 2^e <= |y|, |q - hi| <= 2^(e-p); either it equals 2^(e-p) (then lo = q - hi exactly) or it lies at least one
// binade lower, where lo is off by at most 2^(e-2p-1) <= 2^-(2p+1) |y|.  Subnormal results lose relative accuracy: at most
// half the subnormal spacing more per element, absolute (fp16 2^-25, bf16 2^-134).
// Per element |q_i - hi_i (- lo_i)| <= rel |q_i| + sub, so |q - hi (- lo)|_2 <= rel |q|_2 + sub sqrt(ld); |q|_2 <= 1 + 2^-22
// and |row|_2 <= 1 + 2^-8: factor 1.0078125.  fp32 sweeps (kind::tf32) have no query term here: eps_gemm_const charges the
// operand truncation.  tests/test_query_rounding_cpu.py checks rel and sub on every fp32 value of the binades that matter.
static void fused_query_rounding(int sweep_dt, bool split, double* rel, double* sub) {
    *rel = sweep_dt == 0 ? 0.0 : sweep_dt == 1 ? (split ? 0x1p-17 : 0x1p-8) : (split ? 0x1p-23 : 0x1p-11);
    *sub = sweep_dt == 0 ? 0.0 : sweep_dt == 1 ? 0x1p-134 : 0x1p-25;
}
static float eps_fused_query(int sweep_dt, bool split, int ld) {
    double rel, sub;
    fused_query_rounding(sweep_dt, split, &rel, &sub);
    if (rel == 0.0) return 0.f;
    return nextafterf((float)((rel + sub * sqrt((double)ld)) * 1.0078125), INFINITY);
}

// fp32 evaluation of the int8 score w = (s sq) (H + L / 256) in the kernel: five roundings (two int -> float conversions,
// the add, two products) of 2^-24 each on terms bounded by (sq |hi|_2 + sq |lo|_2 / 256) (s |x8|_2), where s |x8|_2 <=
// |x|_2 + e <= 1.0078125 (1 + sqrt(ld) / 254) and sq |hi|_2 + sq |lo|_2 / 256 <= 1 + 2^-20 + sqrt(ld) / 127.  Rounded up.
static float eps_i8_conv(int ld) {
    const double r = sqrt((double)ld);
    const double e = 5.01 * 0x1p-24 * 1.0078125 * (1.0 + r / 250.0) * (1.00001 + r / 125.0);
    return nextafterf((float)e, INFINITY);
}

// Rows from which a collection's one-kernel search screens tiles with the int8 copy (RAGFIN_SWEEP_COPY_AUTO)
static const int64_t kI8MinRows = (int64_t)1 << 20;
static bool i8_wanted(const ragfin* h) {
    if (h->sweep_copy == 0 || has_copy(h) || (h->dtype != RAGFIN_BF16 && h->dtype != RAGFIN_F16)) return false;
    return h->sweep_copy == 1 || h->count >= kI8MinRows;
}
// Bring the int8 copy up to `count` rows (kernel on st).  Returns false when it cannot be allocated: the search then sweeps
// the 16-bit rows.  *built: a kernel was enqueued in front of the search.
static bool i8_prepare(ragfin* h, cudaStream_t st, bool* built) {
    *built = false;
    if (h->i8 && h->i8_owned && h->i8_cap < h->capacity) i8_free(h);   // ragfin_reserve grew the collection
    if (!h->i8) {
        const int64_t cap = h->capacity;
        h->ld8 = (h->ld + 15) / 16 * 16;
        cudaError_t e = cudaMalloc(&h->i8, (size_t)cap * h->ld8);
        if (e == cudaSuccess) e = cudaMalloc(&h->i8side, (size_t)cap * sizeof(float2));
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            if (h->i8) cudaFree(h->i8);
            h->i8 = nullptr; h->i8side = nullptr;
            return false;
        }
        h->i8_cap = cap; h->i8_rows = 0; h->i8_owned = true;
    }
    if (h->i8_rows < h->count) {
        const int64_t n = h->count - h->i8_rows, wpb = 8;
        const int64_t want = (n + wpb - 1) / wpb, cap_blocks = (int64_t)h->num_sms * 16;
        const int blocks = (int)(want < cap_blocks ? want : cap_blocks);
        if (h->dtype == RAGFIN_BF16)
            quantize_i8_kernel<1><<<blocks, wpb * 32, 0, st>>>((const __nv_bfloat16*)h->data, h->ld, h->i8_rows, n, h->i8, h->ld8, h->i8side);
        else
            quantize_i8_kernel<2><<<blocks, wpb * 32, 0, st>>>((const __half*)h->data, h->ld, h->i8_rows, n, h->i8, h->ld8, h->i8side);
        if (cudaGetLastError() != cudaSuccess) return false;
        h->i8_rows = h->count;
        *built = true;
    }
    return true;
}

static bool fused_eligible(const ragfin* h, int nb, int k) {
    return h->use_fused && h->count >= h->fused_min_rows && gemm_rows_ok(h) && plan_fused(h, nb, k).ncol != 0;
}

typedef void (*fused_fn)(const CUtensorMap, const FusedArgs, const FusedInlineQ, const CUtensorMap);
static fused_fn pick_fused(int dtype, int ncol, bool split, bool i8) {
    if (dtype == 0) return ncol == 16 ? sweep_fused_kernel<1, 16, false, false> : ncol == 32 ? sweep_fused_kernel<1, 32, false, false> : sweep_fused_kernel<1, 64, false, false>;
    if (i8) return ncol == 16 ? sweep_fused_kernel<0, 16, true, true> : ncol == 32 ? sweep_fused_kernel<0, 32, true, true> : sweep_fused_kernel<0, 64, true, true>;
    if (split) return ncol == 16 ? sweep_fused_kernel<0, 16, true, false> : ncol == 32 ? sweep_fused_kernel<0, 32, true, false> : sweep_fused_kernel<0, 64, true, false>;
    return ncol == 16 ? sweep_fused_kernel<0, 16, false, false> : ncol == 32 ? sweep_fused_kernel<0, 32, false, false> : sweep_fused_kernel<0, 64, false, false>;
}

// pipelined: the asynchronous entry points.  The launch carries programmatic stream serialization and the kernel releases its
// dependents when it starts, so the CTAs of the next search on the stream take over the SMs one by one as this search's CTAs
// finish: one search's prologue, tail skew, finalize and exchange overlap the next one's sweep.  Synchronous host calls (one
// search, then a stream synchronisation) use a plain launch.
// q_inline_host != null: the queries are host memory and travel in the launch's parameter space (no copy in front of the kernel);
// host_flag_dev != null: the last finalizer sets that device-mapped word to host_seq (synchronous host calls poll it).
static int run_fused(ragfin* h, const float* q_dev, int nb, int k, int64_t n_eff, int64_t* out_ids, float* out_scores,
                     cudaStream_t st, bool pipelined, ragfin_exchange* x = nullptr, uint32_t xstep = 0,
                     const float* q_inline_host = nullptr, uint32_t* host_flag_dev = nullptr, uint32_t host_seq = 0) {
    int rc;
    FusedPlan f = plan_fused(h, nb, k);
    if (f.ncol == 0) return fail(RAGFIN_EUNSUPPORTED, "no fused sweep for %d queries, k = %d", nb, k);
    const int64_t n = h->count;
    // int8 tile filter: same eps, same answers, the 16-bit rows read only for tiles within reach of a threshold
    bool use8 = false;
    if (i8_wanted(h)) {
        const FusedPlan f8 = plan_fused(h->sweep_dt, h->ld, h->fused_max_nq, h->fused_max_nqk, h->fused_stage_cap, nb, k, true);
        bool built = false;
        if (f8.ncol == f.ncol && f8.split && i8_prepare(h, st, &built)) {
            f = f8;
            use8 = true;
            if (built) pipelined = false;   // the copy's kernel ran in front of this launch: an ordinary launch
        }
    }
    const size_t cand_half = (size_t)kFMaxQ * 4 * kAppendCap * sizeof(u64) / 4;   // per half: up to 16 queries x 65 536 keys (= 64 x 16 384)
    const size_t qn_half = (size_t)kFMaxQ * h->ld * sizeof(float);
    if ((size_t)nb * f.cap * sizeof(u64) > cand_half) return fail(RAGFIN_EUNSUPPORTED, "append buffers of %d queries x %d keys exceed the workspace half", nb, f.cap);
    if ((rc = ensure(h->fcand, 2 * cand_half)) || (rc = ensure(h->fqn, 2 * qn_half)) || (rc = ensure(h->fflags, 2 * (kFMaxQ + 1) * sizeof(int)))) return rc;
    if (!h->fctl.p) { if ((rc = ensure(h->fctl, 2 * sizeof(FusedCtl)))) return rc; h->fctl_dirty = true; }
    if (h->fctl_dirty) {
        CU_TRY(cudaMemsetAsync(h->fctl.p, 0, 2 * sizeof(FusedCtl), st));
        h->fctl_dirty = false; h->fused_seq = 0;
        pipelined = false;     // the kernel reads the control block from its first instruction: full dependency on the memset
    }
    const uint32_t seq = h->fused_seq++;
    const int half = (int)(seq & 1u);
    h->fused_last = half;
    const GemmPlan p = plan_gemm(nb, n, h->num_sms, 32, 1);
    CUtensorMap tmB, tmB8;
    if ((rc = cached_map(h, &tmB, h->sweep_dt, h->sweep_data, n, h->ld, kGN))) return rc;
    tmB8 = tmB;
    if (use8 && (rc = cached_map(h, &tmB8, kMapI8, h->i8, n, h->ld8, kGN))) return rc;
    FusedArgs a;
    a.idesc = make_idesc_n(h->sweep_dt == 0 ? 2 : h->sweep_dt == 1 ? 1 : 0, f.ncol);
    a.k_elems = kGKBytes / (int)esize(h->sweep_dt);
    a.num_kblocks = (h->ld + a.k_elems - 1) / a.k_elems;
    a.dt = h->dtype;
    a.sdt = h->sweep_dt;
    a.nq = nb; a.dim = h->dim; a.ld = h->ld;
    a.n_rows = n;
    a.S = p.S; a.rows_per_slice = p.rows_per_slice;
    a.stages = f.stages;
    a.k = k; a.keff = (int)((int64_t)k < n_eff ? k : n_eff);
    a.pend = f.pend;
    a.groups = p.grid < kFGroups ? p.grid : kFGroups;
    if (a.keff > 0 && a.groups > a.keff) a.groups = a.keff;
    if (a.groups < 1) a.groups = 1;
    a.grank = a.keff > 0 ? (a.keff + a.groups - 1) / a.groups : 0;
    a.seq_on_half = seq >> 1;
    a.refresh_every = h->fused_refresh_every;
    a.q = q_inline_host ? nullptr : q_dev;
    a.host_flag = host_flag_dev; a.host_seq = host_seq;
    a.qn = (float*)((char*)h->fqn.p + half * qn_half);
    a.data = h->data;
    a.allow = h->cur_allow;
    a.cand = (u64*)((char*)h->fcand.p + half * cand_half); a.cap = f.cap;
    a.ctl = (FusedCtl*)h->fctl.p + half;
    a.eps_const = eps_approx(h);
    a.eps_query = eps_fused_query(h->sweep_dt, f.split, h->ld);
    a.id_base = h->id_base;
    a.out_ids = (long long*)out_ids; a.out_scores = out_scores;
    a.flags = (int*)h->fflags.p + half * (kFMaxQ + 1); a.flag_count = a.flags + kFMaxQ;
    a.xworld = 0; a.xrank = 0; a.xstep = 0; a.xrec_max = 0; a.xpeer_area = nullptr; a.xpeer_qflag = nullptr;
    if (x != nullptr && x->world > 1) {
        a.xworld = x->world; a.xrank = x->rank; a.xstep = xstep; a.xrec_max = x->record_max;
        a.xpeer_area = x->d_peer_area; a.xpeer_qflag = x->d_peer_qflag;
    }
    a.idesc8 = make_idesc_i8(f.ncol);
    a.num_kblocks8 = use8 ? (h->ld8 + kGKBytes - 1) / kGKBytes : 0;
    a.side8 = use8 ? h->i8side : nullptr;
    a.i8_conv = eps_i8_conv(h->ld);
    fused_fn fn = pick_fused(h->sweep_dt, f.ncol, f.split, use8);
    if ((rc = set_dyn_smem(h->device, (const void*)fn, f.smem))) return rc;
    h->fctl_dirty = true;          // until the launch is known to have been accepted
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(p.grid); cfg.blockDim = dim3(kFThreads); cfg.dynamicSmemBytes = f.smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pipelined ? 1 : 0;
    static thread_local FusedInlineQ qin;          // 12 KB: copied into the launch only up to what the queries occupy matters
    if (q_inline_host) memcpy(qin.v, q_inline_host, (size_t)nb * h->dim * sizeof(float));
    prof_begin(h, st);
    CU_TRY(cudaLaunchKernelEx(&cfg, fn, tmB, a, qin, tmB8));
    prof_end(h, st);
    CU_TRY(cudaGetLastError());
    h->fctl_dirty = false;
    h->stats.launches++;
    h->stats.path = 3;
    h->stats.cand_per_query = f.cap;
    return 0;
}

// ------------------------------------------------------------------------------
// Large-k path: exact scores of every row, radix select of the k-th key, rank sort.  One query at a time.
// ------------------------------------------------------------------------------
static int search_bigk(ragfin* h, const float* q_dev, int nq, int k, int64_t* out_ids, float* out_scores, cudaStream_t st) {
    int rc;
    const int64_t n = h->count;
    const int64_t n_eff = h->cur_allow ? h->cur_allowed : n;
    const int m = (int64_t)k < n_eff ? k : (int)n_eff;   // hits that exist
    h->stats.path = 2;
    h->stats.cand_per_query = m;
    h->stats.queries_rescanned = 0;
    if ((rc = ensure(h->qhat, (size_t)h->ld * sizeof(float)))) return rc;
    if ((rc = ensure(h->bk_scores, (size_t)n * sizeof(float)))) return rc;
    if ((rc = ensure(h->bk_state, sizeof(RadixState)))) return rc;
    if ((rc = ensure(h->bk_keys, (size_t)m * sizeof(u64)))) return rc;
    float* qhat = (float*)h->qhat.p;
    float* scores = (float*)h->bk_scores.p;
    RadixState* state = (RadixState*)h->bk_state.p;
    u64* keys = (u64*)h->bk_keys.p;
    const int blocks = h->num_sms * 8;
    for (int q = 0; q < nq; ++q) {
        if ((rc = launch_ingest<false>(0, q_dev + (size_t)q * h->dim, 0, 0, 0, 0, 1, h->dim, h->ld, qhat, h->num_sms, st))) return rc;
        switch (h->dtype) {
            case 0: score_all_kernel<0><<<blocks, 256, 0, st>>>(h->data, n, h->ld, qhat, scores, h->cur_allow, h->cur_radius, h->cur_range_filter); break;
            case 1: score_all_kernel<1><<<blocks, 256, 0, st>>>(h->data, n, h->ld, qhat, scores, h->cur_allow, h->cur_radius, h->cur_range_filter); break;
            default: score_all_kernel<2><<<blocks, 256, 0, st>>>(h->data, n, h->ld, qhat, scores, h->cur_allow, h->cur_radius, h->cur_range_filter); break;
        }
        CU_TRY(cudaGetLastError());
        RadixState init;
        memset(&init, 0, sizeof(init));
        init.remaining = m;
        CU_TRY(cudaMemcpyAsync(state, &init, sizeof(init), cudaMemcpyHostToDevice, st));
        CU_TRY(cudaStreamSynchronize(st));   // `init` lives on this stack frame
        for (int shift = 56; shift >= 0; shift -= 8) {
            radix_hist_kernel<<<blocks, 256, 0, st>>>(scores, n, shift, state);
            radix_pick_kernel<<<1, 32, 0, st>>>(shift, state);
        }
        if (m > 0) compact_kernel<<<blocks, 256, 0, st>>>(scores, n, state, keys, m);
        const int span = m > k ? m : k;
        rank_sort_kernel<<<(span + 255) / 256, 256, 0, st>>>(keys, m, k, h->id_base, out_ids + (size_t)q * k, out_scores + (size_t)q * k);
        CU_TRY(cudaGetLastError());
        h->stats.launches += 20;
    }
    return 0;
}

// Grouping search, exact path (DESIGN.md 7d): exact scores of every row, the best key of every group, radix select of the
// m-th largest group key, rank sort.  One query at a time; serves small corpora, RAGFIN_NO_BIGK_BATCHED=1 and the batched
// route's overflow.
static int search_grouped(ragfin* h, const float* q_dev, int nq, int k, int64_t* out_ids, float* out_scores, cudaStream_t st) {
    int rc;
    const int64_t n = h->count, ng = h->cur_n_groups;
    const int m = (int64_t)k < ng ? k : (int)ng;   // hits that may exist
    h->stats.path = 2;
    h->stats.cand_per_query = m;
    h->stats.queries_rescanned = 0;
    if ((rc = ensure(h->qhat, (size_t)h->ld * sizeof(float)))) return rc;
    if ((rc = ensure(h->bk_scores, (size_t)n * sizeof(float)))) return rc;
    if ((rc = ensure(h->bk_state, sizeof(RadixState)))) return rc;
    if ((rc = ensure(h->bk_keys, (size_t)m * sizeof(u64)))) return rc;
    if ((rc = ensure(h->grp, (size_t)ng * sizeof(u64)))) return rc;
    float* qhat = (float*)h->qhat.p;
    float* scores = (float*)h->bk_scores.p;
    RadixState* state = (RadixState*)h->bk_state.p;
    u64* keys = (u64*)h->bk_keys.p;
    u64* gbest = (u64*)h->grp.p;
    const int blocks = h->num_sms * 8;
    for (int q = 0; q < nq; ++q) {
        if ((rc = launch_ingest<false>(0, q_dev + (size_t)q * h->dim, 0, 0, 0, 0, 1, h->dim, h->ld, qhat, h->num_sms, st))) return rc;
        switch (h->dtype) {
            case 0: score_all_kernel<0><<<blocks, 256, 0, st>>>(h->data, n, h->ld, qhat, scores, h->cur_allow, -INFINITY, INFINITY); break;
            case 1: score_all_kernel<1><<<blocks, 256, 0, st>>>(h->data, n, h->ld, qhat, scores, h->cur_allow, -INFINITY, INFINITY); break;
            default: score_all_kernel<2><<<blocks, 256, 0, st>>>(h->data, n, h->ld, qhat, scores, h->cur_allow, -INFINITY, INFINITY); break;
        }
        CU_TRY(cudaMemsetAsync(gbest, 0, (size_t)ng * sizeof(u64), st));
        group_best_kernel<<<blocks, 256, 0, st>>>(scores, n, h->cur_groups, (int)ng, gbest);
        CU_TRY(cudaGetLastError());
        RadixState init;
        memset(&init, 0, sizeof(init));
        init.remaining = m;
        CU_TRY(cudaMemcpyAsync(state, &init, sizeof(init), cudaMemcpyHostToDevice, st));
        CU_TRY(cudaStreamSynchronize(st));   // `init` lives on this stack frame
        for (int shift = 56; shift >= 0; shift -= 8) {
            radix_hist_keys_kernel<<<blocks, 256, 0, st>>>(gbest, ng, shift, state);
            radix_pick_kernel<<<1, 32, 0, st>>>(shift, state);
        }
        pad_keys_kernel<<<(m + 255) / 256, 256, 0, st>>>(keys, m);
        group_compact_kernel<<<blocks, 256, 0, st>>>(gbest, ng, state, keys, m);
        const int span = m > k ? m : k;
        rank_sort_kernel<<<(span + 255) / 256, 256, 0, st>>>(keys, m, k, h->id_base, out_ids + (size_t)q * k, out_scores + (size_t)q * k);
        CU_TRY(cudaGetLastError());
        h->stats.launches += 23;
    }
    return 0;
}

// Batched large-k path (bigk.cuh, second half): up to 16 queries per tensor-core sweep, approximate scores dumped, radix
// select + compaction + exact rescore + rank sort per query with grid.y = query; ONE stream synchronisation at the end to
// read the overflow flags (flagged queries - thousands of rows within 2 eps of the k-th score - take the exact one-query path).
// A grouping search (h->cur_groups, DESIGN.md 7d) adds the group maxima, selects T among them, cuts each row at its group's
// maximum too, keeps one candidate per group, and sends flagged queries to search_grouped.
static const int kBigChunk = 16;
static int search_bigk_batched(ragfin* h, const float* q_dev, int nq, int k, int64_t* out_ids, float* out_scores, cudaStream_t st) {
    int rc;
    const int64_t n = h->count;
    const int64_t n_eff = h->cur_allow ? h->cur_allowed : n;
    const int keff = (int)((int64_t)k < n_eff ? k : n_eff);
    // rows within 2 eps below the k-th score: the score density grows with k (~ +40 % of k at k = 16384 on 10M random rows
    // with the unsplit 16-bit query's eps)
    const int slack = keff > 4096 ? keff : 4096;
    const int cmax = keff + slack;
    h->stats.path = 2;
    h->stats.cand_per_query = cmax;
    h->stats.queries_rescanned = 0;
    const int nbq = kGM;                                   // the sweep pads the query tile to 128 rows
    if ((rc = ensure(h->qhat, (size_t)nbq * h->ld * sizeof(float)))) return rc;
    if ((rc = ensure(h->eps_q, (size_t)nbq * sizeof(float))) || (rc = ensure(h->gtau, (size_t)nbq * sizeof(uint32_t)))) return rc;
    if (h->sweep_dt != 0 && (rc = ensure(h->q16, (size_t)nbq * h->ld * 2))) return rc;
    if ((rc = ensure(h->flags, (size_t)(kMaxQueryBatch + 1) * sizeof(int)))) return rc;
    if ((rc = ensure(h->bk_scores, (size_t)kBigChunk * n * sizeof(float)))) return rc;
    if ((rc = ensure(h->bk_state, (size_t)nq * sizeof(BkState)))) return rc;
    if ((rc = ensure(h->bk_rows, (size_t)kBigChunk * cmax * sizeof(uint32_t)))) return rc;
    if ((rc = ensure(h->bk_keys, (size_t)kBigChunk * cmax * sizeof(u64)))) return rc;
    if (h->cur_window && (rc = ensure(h->awin, (size_t)3 * kBigChunk * sizeof(float)))) return rc;
    const int ng = h->cur_n_groups;
    if (h->cur_groups && (rc = ensure(h->grp, (size_t)kBigChunk * ng * sizeof(uint32_t)))) return rc;
    uint32_t* gmax = (uint32_t*)h->grp.p;
    float* qhat = (float*)h->qhat.p;
    float* scores = (float*)h->bk_scores.p;
    BkState* states = (BkState*)h->bk_state.p;
    int* flag_count = (int*)h->flags.p + kMaxQueryBatch;
    CU_TRY(cudaMemsetAsync(states, 0, (size_t)nq * sizeof(BkState), st));
    const int blocks = h->num_sms * 8;
    const float eps = eps_approx(h);
    for (int q0 = 0; q0 < nq; q0 += kBigChunk) {
        const int nb = nq - q0 < kBigChunk ? nq - q0 : kBigChunk;
        const int wpb = 8, pblocks = (nbq + wpb - 1) / wpb;
        const float* qsrc = q_dev + (size_t)q0 * h->dim;
        switch (h->sweep_dt) {
            case 0: prep_queries_kernel<0><<<pblocks, wpb * 32, 0, st>>>(qsrc, nb, nbq, h->dim, h->ld, qhat, nullptr, (float*)h->eps_q.p, flag_count, (uint32_t*)h->gtau.p); break;
            case 1: prep_queries_kernel<1><<<pblocks, wpb * 32, 0, st>>>(qsrc, nb, nbq, h->dim, h->ld, qhat, (__nv_bfloat16*)h->q16.p, (float*)h->eps_q.p, flag_count, (uint32_t*)h->gtau.p); break;
            default: prep_queries_kernel<2><<<pblocks, wpb * 32, 0, st>>>(qsrc, nb, nbq, h->dim, h->ld, qhat, (__half*)h->q16.p, (float*)h->eps_q.p, flag_count, (uint32_t*)h->gtau.p); break;
        }
        CU_TRY(cudaGetLastError());
        int G = 0;
        bool ap = false;
        if ((rc = run_gemm(h, nb, 10, 32, &G, &ap, scores, st, true))) return rc;        // MODE 1: approx[q][row]
        const float* w = nullptr;   // range search: per-query window words {lo, hi, cap}
        if (h->cur_window) {
            w = (const float*)h->awin.p;
            RF_LAUNCH(window_words_kernel, (nb + 127) / 128, 128, 0, st, nb, h->cur_radius, h->cur_range_filter, eps,
                                                                       (const float*)h->eps_q.p, (float*)h->awin.p);
            CU_TRY(cudaGetLastError());
            h->stats.launches++;
        }
        BkState* stq = states + q0;
        if (h->cur_groups) {
            CU_TRY(cudaMemsetAsync(gmax, 0, (size_t)nb * ng * sizeof(uint32_t), st));
            bk_group_max_kernel<<<blocks, 256, 0, st>>>(scores, n, nb, h->cur_groups, ng, h->cur_allow, gmax);
            for (int pass = 0; pass < 4; ++pass)
                bk_hist_kernel<true><<<dim3(blocks, nb), 256, 0, st>>>((const float*)gmax, ng, pass, keff, stq, nullptr, nullptr);
            bk_group_compact_kernel<<<dim3(blocks, nb), 256, 0, st>>>(scores, n, keff, eps, (const float*)h->eps_q.p, stq, (uint32_t*)h->bk_rows.p,
                                                                      cmax, h->cur_allow, h->cur_groups, ng, gmax);
            h->stats.launches += 2;
        } else {
            for (int pass = 0; pass < 4; ++pass)
                bk_hist_kernel<<<dim3(blocks, nb), 256, 0, st>>>(scores, n, pass, keff, stq, h->cur_allow, w ? w + 2 * nb : nullptr);
            bk_compact_kernel<<<dim3(blocks, nb), 256, 0, st>>>(scores, n, keff, eps, (const float*)h->eps_q.p, stq, (uint32_t*)h->bk_rows.p, cmax, h->cur_allow,
                                                                w, w ? w + nb : nullptr);
        }
        const dim3 rg((cmax + 7) / 8, nb);
        switch (h->dtype) {
            case 0: bk_rescore_kernel<0><<<rg, 256, 0, st>>>(h->data, h->ld, qhat, stq, (const uint32_t*)h->bk_rows.p, cmax, (u64*)h->bk_keys.p, h->cur_radius, h->cur_range_filter); break;
            case 1: bk_rescore_kernel<1><<<rg, 256, 0, st>>>(h->data, h->ld, qhat, stq, (const uint32_t*)h->bk_rows.p, cmax, (u64*)h->bk_keys.p, h->cur_radius, h->cur_range_filter); break;
            default: bk_rescore_kernel<2><<<rg, 256, 0, st>>>(h->data, h->ld, qhat, stq, (const uint32_t*)h->bk_rows.p, cmax, (u64*)h->bk_keys.p, h->cur_radius, h->cur_range_filter); break;
        }
        if (h->cur_groups) {
            bk_group_rep_kernel<<<dim3((cmax + 255) / 256, nb), 256, 0, st>>>((u64*)h->bk_keys.p, stq, cmax, h->cur_groups);
            h->stats.launches++;
        }
        const int span = cmax > k ? cmax : k;
        bk_rank_sort_kernel<<<dim3((span + 255) / 256, nb), 256, 0, st>>>((const u64*)h->bk_keys.p, stq, cmax, k, keff, h->id_base,
                                                                          out_ids + (size_t)q0 * k, out_scores + (size_t)q0 * k);
        CU_TRY(cudaGetLastError());
        h->stats.launches += 9;
    }
    // overflow flags: the one host round trip of this path
    std::vector<BkState> host(nq);
    CU_TRY(cudaMemcpyAsync(host.data(), states, (size_t)nq * sizeof(BkState), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    int redone = 0;
    const int launches = h->stats.launches;
    for (int q = 0; q < nq; ++q) {
        if (!host[q].overflow) continue;
        ++redone;
        if ((rc = (h->cur_groups ? search_grouped : search_bigk)(h, q_dev + (size_t)q * h->dim, 1, k, out_ids + (size_t)q * k,
                                                                 out_scores + (size_t)q * k, st))) return rc;
    }
    h->stats.path = 2;
    h->stats.cand_per_query = cmax;
    h->stats.queries_rescanned = redone;
    h->stats.launches = launches + 20 * redone;
    return 0;
}

static int search_locked(ragfin* h, const float* q_dev, int nq, int k, int64_t* out_ids, float* out_scores,
                         cudaStream_t st) {
    int rc;
    const int64_t n = h->count;
    h->stats.launches = 0;
    h->stats.path = 0;
    h->stats.queries_rescanned = -1;
    const int V = h->dtype == 0 ? 4 : 8;
    const int nvec = h->ld / V;
    const int steps = round_steps((nvec + 31) / 32);
    const int64_t n_eff = h->cur_allow ? h->cur_allowed : n;   // rows a hit may come from
    if ((rc = ensure(h->flags, (size_t)(kMaxQueryBatch + 1) * sizeof(int)))) return rc;
    if (h->cur_groups) {   // grouping search (DESIGN.md 7d): the large-k route on corpora worth a sweep, else the exact path
        if (h->use_bigk_batched && n >= 4096 && gemm_rows_ok(h)) return search_bigk_batched(h, q_dev, nq, k, out_ids, out_scores, st);
        return search_grouped(h, q_dev, nq, k, out_ids, out_scores, st);
    }
    const int min_nq_all = (size_t)n * h->ld * esize(h->dtype) >= kSweepBytes ? h->gemm_min_nq_large : h->gemm_min_nq;
    const bool ap = append_eligible(h, k) && nq >= min_nq_all;   // tensor-core append mode: no K' lists needed
    if (h->cur_window && !ap) {
        // Range search (DESIGN.md 7c): the append path when the batch would take it, else the large-k pipeline with the
        // window, which serves every k, filter and corpus size.  Never the one-kernel search.
        if (h->use_bigk_batched && n >= 4096 && gemm_rows_ok(h)) return search_bigk_batched(h, q_dev, nq, k, out_ids, out_scores, st);
        return search_bigk(h, q_dev, nq, k, out_ids, out_scores, st);
    }
    if (!h->cur_window && nq <= h->fused_max_nq && fused_eligible(h, nq, k)) {   // the one-kernel search (sweep_fused.cuh): prep, sweep, finalize, exact fallback
        return run_fused(h, q_dev, nq, k, n_eff, out_ids, out_scores, st, h->cur_pipelined);
    }
    int kp = cand_per_query(k);
    if (kp == 0 && n <= 256) kp = 256;   // every row is a candidate: any k (graph_cons.py:279 asks limit=1000 of 16 rows)
    if (kp == 0 && !ap) {
        // k beyond the list / append modes: batched dump + select on corpora worth a tensor-core sweep, else one query at a time
        if (h->use_bigk_batched && n >= 4096 && gemm_rows_ok(h)) return search_bigk_batched(h, q_dev, nq, k, out_ids, out_scores, st);
        return search_bigk(h, q_dev, nq, k, out_ids, out_scores, st);
    }
    if (kp == 0) kp = 256;
    h->stats.cand_per_query = kp;
    int kpe = 32;                                          // tier-2 list length: a power of two (bitonic merges)
    while (kpe < k && kpe < 256) kpe <<= 1;                // k > 256 only occurs with n <= 256
    if ((rc = ensure(h->flags, (size_t)(kMaxQueryBatch + 1) * sizeof(int)))) return rc;
    int* flags = (int*)h->flags.p;
    int* flag_count = flags + kMaxQueryBatch;

    for (int q0 = 0; q0 < nq; q0 += kMaxQueryBatch) {
        const int nb = nq - q0 < kMaxQueryBatch ? nq - q0 : kMaxQueryBatch;
        const int nb4 = (nb + 3) / 4 * 4;
        const size_t corpus_bytes = (size_t)h->count * h->ld * esize(h->dtype);
        const int min_nq = corpus_bytes >= kSweepBytes ? h->gemm_min_nq_large : h->gemm_min_nq;
        // a range search's last chunk takes the append path whatever its size (its window is not applied elsewhere)
        const bool via_gemm = (h->cur_window || nb >= min_nq) && (gemm_supported(h, kp) || (ap && h->count > 0));
        const int nbq = via_gemm ? (nb + kGM - 1) / kGM * kGM : nb4;   // tensor-core path: whole 128-query tiles
        // 1. normalise the queries (same kernel as ingest, fp32 out, stride ld); pad with zero rows
        if ((rc = ensure(h->qhat, (size_t)nbq * h->ld * sizeof(float)))) return rc;
        float* qhat = (float*)h->qhat.p;
        const bool prepped = via_gemm && !(!ap && use_astat(h, kp));   // the 16-bit query copy is made here too
        {   // one launch: normalise + pad + [16-bit copy + eps_q] + counters (flags[q] itself is written by finalize for every q)
            if ((rc = ensure(h->eps_q, (size_t)nbq * sizeof(float))) || (rc = ensure(h->gtau, (size_t)nbq * sizeof(uint32_t)))) return rc;
            if (prepped && h->sweep_dt != 0 && (rc = ensure(h->q16, (size_t)nbq * h->ld * 2))) return rc;
            const int wpb = 8, blocks = (nbq + wpb - 1) / wpb;
            const float* qsrc = q_dev + (size_t)q0 * h->dim;
            switch (prepped ? h->sweep_dt : 0) {
                case 0: RF_LAUNCH(prep_queries_kernel<0>, blocks, wpb * 32, 0, st, qsrc, nb, nbq, h->dim, h->ld, qhat, nullptr, (float*)h->eps_q.p, flag_count, (uint32_t*)h->gtau.p); break;
                case 1: RF_LAUNCH(prep_queries_kernel<1>, blocks, wpb * 32, 0, st, qsrc, nb, nbq, h->dim, h->ld, qhat, (__nv_bfloat16*)h->q16.p, (float*)h->eps_q.p, flag_count, (uint32_t*)h->gtau.p); break;
                default: RF_LAUNCH(prep_queries_kernel<2>, blocks, wpb * 32, 0, st, qsrc, nb, nbq, h->dim, h->ld, qhat, (__half*)h->q16.p, (float*)h->eps_q.p, flag_count, (uint32_t*)h->gtau.p); break;
            }
            CU_TRY(cudaGetLastError());
            h->stats.launches++;
        }

        int G = 0, sorted_lists = 1;
        bool scanned = false, appended = false;
        float eps = 0.f;
        const float* eps_q = nullptr;
        if (via_gemm) {
            // 2a. tensor-core path
            if (!ap && use_astat(h, kp)) { if ((rc = run_gemm_astat(h, nb, kp, &G, nullptr, st))) return rc; }
            else if ((rc = run_gemm(h, nb, k, kp, &G, &appended, nullptr, st, prepped))) return rc;
            h->stats.path = 1;
            sorted_lists = 0;
            scanned = true;
            eps = eps_approx(h);
            eps_q = (const float*)h->eps_q.p;
        } else {
            // 2b. scan in groups of <= 4 queries.  Candidate layout [nb4][G][kp]; a group whose kernel
            //     variant fits fewer CTAs than G leaves the surplus lists empty (zeroed here).
            //     Every group of a batch uses the same grid (the smallest occupancy among the variants used), so
            //     the candidate buffer is exactly [nb4][G][kp] and every list is written by its CTA.
            scanned = n > 0 && steps > 0;
            eps = eps_fp32_accumulate(h->ld);
            G = 1;
            // TMA-fed scan: whole batch of 1 or 2 queries, ring of 4 stages must fit in shared memory
            const size_t row_bytes = (size_t)h->ld * esize(h->dtype);
            const size_t tsm = scanned ? ts_smem_bytes(steps, row_bytes, nb, kp) : 0;
            scan_fn tfn = (scanned && h->scan_variant == 2 && nb <= 2 && tsm <= (size_t)227 * 1024) ? pick_scan_tma(h->dtype, nb, steps) : nullptr;
            if (tfn) {
                G = h->num_sms;
                if ((rc = ensure(h->cand, (size_t)nb4 * G * kp * sizeof(u64)))) return rc;
                if ((rc = set_dyn_smem(h->device, (const void*)tfn, tsm))) return rc;
                prof_begin(h, st);
                tfn<<<G, kTsThreads, tsm, st>>>(h->data, n, h->ld, qhat, nb, kp, (u64*)h->cand.p, (int64_t)G * kp, h->cur_allow);
                prof_end(h, st);
                CU_TRY(cudaGetLastError());
                h->stats.launches++;
            } else {
            if (scanned) {
                int per_sm_min = kMaxScanCtasPerSm;
                const int last = nb - (nb - 1) / 4 * 4;                      // queries in the last group: 1..4
                const int variants[2] = {nb > 4 ? 4 : 0, last >= 3 ? 4 : last};  // every group but the last uses 4
                for (int nqt : variants) {
                    if (nqt == 0) continue;
                    scan_fn fn = pick_scan(h->dtype, nqt, steps);
                    if (!fn) return fail(RAGFIN_EUNSUPPORTED, "no scan kernel for dtype %d nq %d steps %d", h->dtype, nqt, steps);
                    const size_t smem = (size_t)nqt * kScanWarps * kp * sizeof(u64);
                    if ((rc = set_dyn_smem(h->device, (const void*)fn, smem))) return rc;
                    int per_sm = 0;
                    if ((rc = blocks_per_sm(h->device, (const void*)fn, kScanThreads, smem, &per_sm))) return rc;
                    if (per_sm < 1) return fail(RAGFIN_ECUDA, "scan kernel does not fit on an SM (smem %zu)", smem);
                    if (per_sm < per_sm_min) per_sm_min = per_sm;
                }
                G = h->num_sms * per_sm_min;
            }
            if ((rc = ensure(h->cand, (size_t)nb4 * G * kp * sizeof(u64)))) return rc;
            if (!scanned) CU_TRY(cudaMemsetAsync(h->cand.p, 0, (size_t)nb4 * G * kp * sizeof(u64), st));
            if (scanned) {
                for (int g0 = 0; g0 < nb; g0 += 4) {
                    const int left = nb - g0;
                    const int nqt = left >= 3 ? 4 : left;  // 1, 2 or 4 query register sets (3 pads to 4)
                    scan_fn fn = pick_scan(h->dtype, nqt, steps);
                    const size_t smem = (size_t)nqt * kScanWarps * kp * sizeof(u64);
                    prof_begin(h, st);
                    RF_LAUNCH(fn, G, kScanThreads, smem, st, h->data, n, h->ld, qhat + (size_t)g0 * h->ld, left < nqt ? left : nqt, kp,
                                                       (u64*)h->cand.p + (size_t)g0 * G * kp,
                                                       (int64_t)G * kp, h->cur_allow);
                    prof_end(h, st);
                    CU_TRY(cudaGetLastError());
                    h->stats.launches++;
                }
            }
            }
        }
        // 3. merge + exact rescore + certificate (an unscanned, non-empty corpus flags every query)
        if (appended) {
            RF_LAUNCH(finalize_append_kernel, nb, kFaThreads, 0, st,
                (const u64*)h->cand.p, (const uint32_t*)h->acnt.p, kAppendCap, h->data, h->dtype, n_eff, h->ld, qhat, eps, eps_q, k,
                h->id_base, out_ids + (size_t)q0 * k, out_scores + (size_t)q0 * k, flags, flag_count, h->cur_radius, h->cur_range_filter);
            CU_TRY(cudaGetLastError());
            h->stats.launches++;
        } else {
            RF_LAUNCH(finalize_kernel<false>, nb, kFinThreads, 0, st,
                (const u64*)h->cand.p, G, kp, h->data, h->dtype, n_eff, (scanned || n == 0) ? 1 : 0, sorted_lists,
                sorted_lists ? nullptr : (const uint32_t*)h->gtau.p, h->ld, qhat, eps, eps_q, k, h->id_base, out_ids + (size_t)q0 * k, out_scores + (size_t)q0 * k, flags, flag_count);
            CU_TRY(cudaGetLastError());
            h->stats.launches++;
        }
        // 4. tier 2 (device-side gated: both kernels exit at once when no query is flagged)
        if (n > 0) {
            const int Ge = h->num_sms * 2;
            if ((rc = ensure(h->cand_e, (size_t)nb * Ge * kpe * sizeof(u64)))) return rc;
            const size_t smem = (size_t)kScanWarps * kpe * sizeof(u64);
            switch (h->dtype) {
                case 0: RF_LAUNCH(exact_scan_kernel<0>, Ge, kScanThreads, smem, st, h->data, n, h->ld, qhat, nb, flags, flag_count, kpe, (u64*)h->cand_e.p, h->cur_allow,
                                          h->cur_radius, h->cur_range_filter); break;
                case 1: RF_LAUNCH(exact_scan_kernel<1>, Ge, kScanThreads, smem, st, h->data, n, h->ld, qhat, nb, flags, flag_count, kpe, (u64*)h->cand_e.p, h->cur_allow,
                                          h->cur_radius, h->cur_range_filter); break;
                default: RF_LAUNCH(exact_scan_kernel<2>, Ge, kScanThreads, smem, st, h->data, n, h->ld, qhat, nb, flags, flag_count, kpe, (u64*)h->cand_e.p, h->cur_allow,
                                          h->cur_radius, h->cur_range_filter); break;
            }
            CU_TRY(cudaGetLastError());
            RF_LAUNCH(finalize_kernel<true>, nb, kFinThreads, 0, st, (const u64*)h->cand_e.p, Ge, kpe, h->data, h->dtype, n_eff, 1, 1, nullptr,
                                                              h->ld, qhat, 0.0f, nullptr, k, h->id_base,
                                                                out_ids + (size_t)q0 * k, out_scores + (size_t)q0 * k,
                                                                flags, flag_count);
            CU_TRY(cudaGetLastError());
            h->stats.launches += 2;
        }
    }
    return 0;
}

// ------------------------------------------------------------------------------
// persistence
// ------------------------------------------------------------------------------
struct FileHeader {
    char magic[8];
    uint32_t version, dim, ld, dtype;
    int64_t count, id_base;
    uint8_t pad[24];
};
static_assert(sizeof(FileHeader) == 64, "header is 64 bytes");

extern "C" int ragfin_save(ragfin_t* h, const char* path) {
    if (!h || !path) return fail(RAGFIN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    CU_TRY(cudaDeviceSynchronize());
    FILE* f = fopen(path, "wb");
    if (!f) return fail(RAGFIN_EINVAL, "cannot open %s for writing", path);
    FileHeader hd;
    memset(&hd, 0, sizeof(hd));
    memcpy(hd.magic, "RAGFINB2", 8);
    hd.version = h->n_dead > 0 ? 2 : 1; hd.dim = (uint32_t)h->dim; hd.ld = (uint32_t)h->ld; hd.dtype = (uint32_t)public_dtype(h);   // rows: the fp32 ones
    hd.count = h->count; hd.id_base = h->id_base;
    if (h->n_dead > 0) memcpy(hd.pad, &h->n_dead, sizeof(h->n_dead));   // version 2: tombstone count, then the live mask after the rows
    int rc = 0;
    if (fwrite(&hd, sizeof(hd), 1, f) != 1) rc = fail(RAGFIN_EINVAL, "write to %s failed", path);
    const size_t rb = (size_t)h->ld * esize(h->dtype);
    const int64_t slice = (int64_t)((64u << 20) / rb) + 1;
    void* host = nullptr;
    if (!rc && cudaMallocHost(&host, (size_t)slice * rb) != cudaSuccess) { (void)cudaGetLastError(); rc = fail(RAGFIN_ENOMEM, "pinned staging allocation failed"); }
    for (int64_t r0 = 0; !rc && r0 < h->count; r0 += slice) {
        const int64_t m = h->count - r0 < slice ? h->count - r0 : slice;
        if (cudaMemcpy(host, (char*)h->data + (size_t)r0 * rb, (size_t)m * rb, cudaMemcpyDeviceToHost) != cudaSuccess) { (void)cudaGetLastError(); rc = fail(RAGFIN_ECUDA, "device read failed"); break; }
        if (fwrite(host, rb, (size_t)m, f) != (size_t)m) rc = fail(RAGFIN_EINVAL, "write to %s failed", path);
    }
    if (host) cudaFreeHost(host);
    if (!rc && h->n_dead > 0) {
        std::vector<uint32_t> m(h->live_host.begin(), h->live_host.begin() + mask_words(h->count));
        if (h->count & 31) m.back() &= (1u << (h->count & 31)) - 1u;
        if (fwrite(m.data(), sizeof(uint32_t), m.size(), f) != m.size()) rc = fail(RAGFIN_EINVAL, "write to %s failed", path);
    }
    if (fclose(f) != 0 && !rc) rc = fail(RAGFIN_EINVAL, "close of %s failed", path);
    return rc;
}

extern "C" int ragfin_load(ragfin_t** out, const char* path, int64_t capacity_rows, int32_t device) {
    if (!out || !path) return fail(RAGFIN_EINVAL, "NULL argument");
    *out = nullptr;
    FILE* f = fopen(path, "rb");
    if (!f) return fail(RAGFIN_EINVAL, "cannot open %s", path);
    FileHeader hd;
    if (fread(&hd, sizeof(hd), 1, f) != 1 || memcmp(hd.magic, "RAGFINB2", 8) != 0 || (hd.version != 1 && hd.version != 2) || hd.dtype > 3 ||
        hd.ld != (hd.dim + 7) / 8 * 8 || hd.count < 0) {
        fclose(f);
        return fail(RAGFIN_EINVAL, "%s is not a ragfin matrix file", path);
    }
    ragfin* h = nullptr;
    const int64_t cap = capacity_rows > hd.count ? capacity_rows : (hd.count > 0 ? hd.count : 1);
    int rc = ragfin_create(&h, (int32_t)hd.dim, (int32_t)hd.dtype, cap, device);
    if (rc) { fclose(f); return rc; }
    DeviceGuard g(device);
    const size_t rb = (size_t)h->ld * esize(h->dtype);
    const int64_t slice = (int64_t)((64u << 20) / rb) + 1;
    void* host = nullptr;
    if (cudaMallocHost(&host, (size_t)slice * rb) != cudaSuccess) { (void)cudaGetLastError(); rc = fail(RAGFIN_ENOMEM, "pinned staging allocation failed"); }
    for (int64_t r0 = 0; !rc && r0 < hd.count; r0 += slice) {
        const int64_t m = hd.count - r0 < slice ? hd.count - r0 : slice;
        if (fread(host, rb, (size_t)m, f) != (size_t)m) { rc = fail(RAGFIN_EINVAL, "%s is truncated", path); break; }
        if (cudaMemcpy((char*)h->data + (size_t)r0 * rb, host, (size_t)m * rb, cudaMemcpyHostToDevice) != cudaSuccess) { (void)cudaGetLastError(); rc = fail(RAGFIN_ECUDA, "device write failed"); }
    }
    if (host) cudaFreeHost(host);
    int64_t n_dead = 0;
    if (!rc && hd.version == 2) {   // tombstones: the live mask follows the rows
        memcpy(&n_dead, hd.pad, sizeof(n_dead));
        const size_t words = mask_words(hd.count), cap_words = mask_words(h->capacity);
        std::vector<uint32_t> m(cap_words, 0xFFFFFFFFu);
        int64_t live = 0;
        if (fread(m.data(), sizeof(uint32_t), words, f) != words) rc = fail(RAGFIN_EINVAL, "%s is truncated", path);
        for (size_t w = 0; !rc && w < words; ++w) {
            if (w + 1 == words && (hd.count & 31)) m[w] |= ~((1u << (hd.count & 31)) - 1u);   // rows past count are live
            live += __builtin_popcount(w + 1 == words && (hd.count & 31) ? m[w] & ((1u << (hd.count & 31)) - 1u) : m[w]);
        }
        if (!rc && (n_dead < 1 || live != hd.count - n_dead)) rc = fail(RAGFIN_EINVAL, "%s: the live mask does not match the tombstone count", path);
        if (!rc) {
            cudaError_t e = cudaMalloc(&h->live_dev, cap_words * sizeof(uint32_t));
            if (e == cudaSuccess) e = cudaMemcpy(h->live_dev, m.data(), cap_words * sizeof(uint32_t), cudaMemcpyHostToDevice);
            if (e != cudaSuccess) { (void)cudaGetLastError(); rc = fail(RAGFIN_ECUDA, "tombstone mask upload failed: %s", cudaGetErrorString(e)); }
            h->live_host.swap(m);
        }
    }
    fclose(f);
    if (!rc && has_copy(h) && hd.count > 0) {   // the fp16 copy is not in the file: rebuilt from the fp32 rows (ld % 8 == 0)
        const int64_t n4 = hd.count * h->ld / 4;
        const int64_t cap_blocks = (int64_t)h->num_sms * 8, want = (n4 + 255) / 256;
        cast_f16_kernel<<<(unsigned)(want < cap_blocks ? want : cap_blocks), 256>>>((const float4*)h->data, (uint2*)h->sweep_data, n4);
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { (void)cudaGetLastError(); rc = fail(RAGFIN_ECUDA, "rebuilding the fp16 copy failed: %s", cudaGetErrorString(e)); }
    }
    if (rc) { ragfin_destroy(h); return rc; }
    h->count = hd.count;
    h->id_base = hd.id_base;
    h->n_dead = n_dead;
    *out = h;
    return RAGFIN_OK;
}

// Test hook: raw tensor-core scores [nq, count] of the queries against every row (device memory out).
extern "C" int ragfin_debug_gemm_scores(ragfin_t* h, const float* q_dev, int32_t nq, float* out_scores_dev, void* stream) {
    if (!h || !q_dev || !out_scores_dev || nq < 1) return fail(RAGFIN_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (h->count == 0) return fail(RAGFIN_EINVAL, "empty collection");
    if ((rc = wait_prev(h, st))) return rc;
    const int nqp = (nq + kGM - 1) / kGM * kGM;
    if ((rc = ensure(h->qhat, (size_t)nqp * h->ld * sizeof(float)))) return rc;
    if (nqp > nq) CU_TRY(cudaMemsetAsync((float*)h->qhat.p + (size_t)nq * h->ld, 0, (size_t)(nqp - nq) * h->ld * sizeof(float), st));
    if ((rc = launch_ingest<false>(0, q_dev, 0, 0, 0, 0, nq, h->dim, h->ld, (float*)h->qhat.p, h->num_sms, st))) return rc;
    int G = 0;
    if (use_astat(h, 32)) { if ((rc = run_gemm_astat(h, nq, 32, &G, out_scores_dev, st))) return rc; }
    else { bool ap = false; if ((rc = run_gemm(h, nq, 10, 32, &G, &ap, out_scores_dev, st))) return rc; }
    return mark_done(h, st);
}

// Test hook, pure host arithmetic (no device needed): the tcgen05 path's work plan and bound-pass geometry for a shape
// on a device of `num_sms` SMs.  out[10] = {C, QT, S, rows_per_slice, grid, append (by size), bound, nblk, g, bstride}.
extern "C" int ragfin_debug_plan(int32_t nq, int64_t n_rows, int32_t num_sms, int32_t k, int32_t cluster, int64_t* out) {
    if (!out || nq < 1 || n_rows < 1 || num_sms < 4 || k < 1 || k > 16384 || !(cluster == 0 || cluster == 1 || cluster == 2 || cluster == 4))
        return fail(RAGFIN_EINVAL, "bad argument");
    int kp = cand_per_query(k);
    if (kp == 0) kp = 256;
    const int QT0 = (nq + kGM - 1) / kGM;
    const int C = cluster ? cluster : auto_cluster(QT0);
    const int64_t n_tiles = (n_rows + kGN - 1) / kGN;
    const bool append = k <= kAppendMaxK && n_tiles >= 4 * (int64_t)k && n_rows < ((int64_t)1 << 31) - kGN;   // append_eligible, size part
    const bool bound = append || n_tiles >= 4 * (int64_t)kp;
    const GemmPlan p = plan_gemm(nq, n_rows, num_sms / C * C, kp, C);
    int nblk = 0, g = 1;
    int64_t bstride = 1;
    if (bound) bound_geometry(n_tiles, append ? k : kp, append, QT0, k, &nblk, &g, &bstride);
    const int64_t v[10] = {C, p.QT, p.S, p.rows_per_slice, p.grid, append, bound, nblk, g, bstride};
    for (int i = 0; i < 10; ++i) out[i] = v[i];
    return RAGFIN_OK;
}

// Test hook, pure host arithmetic (no device needed): what the one-kernel search does for nq queries, top-k, on a collection
// of `dtype` (public code) and `dim`, with the query limits max_nq / max_nqk (0: the defaults, 16 and 400) and the default
// ring depth.  out[5] = {ncol (0: the shape does not take it), split, stages, pend, cap}; out_eps[4] = {rel, sub (the
// per-element query-rounding bound rel |y| + sub), query term, eps_approx} for the variant planned (the plain one if none is).
extern "C" int ragfin_debug_fused_plan(int32_t dtype, int32_t dim, int32_t nq, int32_t k, int32_t max_nq, int32_t max_nqk,
                                       int64_t* out, double* out_eps) {
    if (!out || !out_eps || dtype < 0 || dtype > 3 || dim < 1 || dim > 65536 || nq < 1 || k < 1 || max_nq < 0 || max_nq > kFMaxQ || max_nqk < 0)
        return fail(RAGFIN_EINVAL, "bad argument");
    const int ld = (dim + 7) / 8 * 8;
    const int sweep_dt = dtype == RAGFIN_F32_F16 ? RAGFIN_F16 : dtype;
    const FusedPlan f = plan_fused(sweep_dt, ld, max_nq ? max_nq : kFusedMaxNq, max_nqk ? max_nqk : kFusedMaxNqk, kRMaxStages, nq, k);
    const int64_t v[5] = {f.ncol, f.split, f.stages, f.pend, f.cap};
    for (int i = 0; i < 5; ++i) out[i] = v[i];
    fused_query_rounding(sweep_dt, f.split, &out_eps[0], &out_eps[1]);
    out_eps[2] = eps_fused_query(sweep_dt, f.split, ld);
    out_eps[3] = eps_approx(sweep_dt, ld, dtype == RAGFIN_F32_F16 ? eps_sweep_const(ld) : 0.f);
    return RAGFIN_OK;
}

// Dispatch knob: query batches of at least `min_nq` rows use the tcgen05 path (default 3, and 1 on corpora of >= 1 GiB; INT32_MAX = never).
extern "C" int ragfin_set_gemm_min_batch(ragfin_t* h, int32_t min_nq) {
    if (!h || min_nq < 0) return fail(RAGFIN_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(h->mu);
    h->gemm_min_nq = min_nq ? min_nq : 3;          // 0 restores the defaults
    h->gemm_min_nq_large = min_nq ? min_nq : 1;
    return RAGFIN_OK;
}

// Tuning knob: the tcgen05 path's threshold-seeding sample pass (default on; results are identical either way).
extern "C" int ragfin_set_bound_pass(ragfin_t* h, int32_t enable) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    std::lock_guard<std::mutex> lk(h->mu);
    h->use_bound_pass = enable != 0;
    return RAGFIN_OK;
}

// Tuning knob: append mode of the tcgen05 path (default on; needs the bound pass; results are identical).
extern "C" int ragfin_set_append_mode(ragfin_t* h, int32_t enable) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    std::lock_guard<std::mutex> lk(h->mu);
    h->use_append = enable != 0;
    return RAGFIN_OK;
}

// Diagnostics of the last one-kernel search: rows appended per query (out_appended[nq]) and rows rescored exactly
// (out_rescored[nq]; -1 = the query took the in-kernel exact scan).  Synchronises the device.
// Test hook, pure host arithmetic (no device needed): the order in which the one-kernel search visits the n tiles of a slice
// (out[n]).  Exactness rests on it being a permutation - every tile scored exactly once.
extern "C" int ragfin_debug_fused_tile_order(int32_t n_tiles, int32_t* out) {
    if (!out || n_tiles < 1) return fail(RAGFIN_EINVAL, "bad argument");
    const int mult = perm_mult(n_tiles);
    for (int t = 0; t < n_tiles; ++t) out[t] = perm_tile(t, mult, n_tiles);
    return RAGFIN_OK;
}

// Phase stamps of the last one-kernel search, ns relative to the kernel's start (out[16], see FusedCtl::t).
extern "C" int ragfin_debug_fused_times(ragfin_t* h, int64_t* out) {
    if (!h || !out) return fail(RAGFIN_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    if (!h->fctl.p) return fail(RAGFIN_EINVAL, "no one-kernel search has run on this handle");
    CU_TRY(cudaDeviceSynchronize());
    FusedCtl c;
    CU_TRY(cudaMemcpy(&c, (FusedCtl*)h->fctl.p + h->fused_last, sizeof(c), cudaMemcpyDeviceToHost));
    for (int i = 0; i < 13; ++i) out[i] = (int64_t)(c.t[i] - c.t[0]);
    for (int i = 13; i < 16; ++i) out[i] = (int64_t)c.t[i];   // sums over CTA 0's tiles, not stamps
    return RAGFIN_OK;
}

// Per-CTA diagnostics of the last one-kernel search: final threshold of query 0 and rows appended for it (out arrays of 160).
extern "C" int ragfin_debug_fused_ctas(ragfin_t* h, float* out_thr, int32_t* out_app) {
    if (!h || !out_thr || !out_app) return fail(RAGFIN_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    if (!h->fctl.p) return fail(RAGFIN_EINVAL, "no one-kernel search has run on this handle");
    CU_TRY(cudaDeviceSynchronize());
    FusedCtl* c = new FusedCtl;
    cudaError_t e = cudaMemcpy(c, (FusedCtl*)h->fctl.p + h->fused_last, sizeof(*c), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) for (int i = 0; i < 160; ++i) { out_thr[i] = c->cta_thr[i]; out_app[i] = (int32_t)c->cta_app[i]; }
    delete c;
    CU_TRY(e);
    return RAGFIN_OK;
}

extern "C" int ragfin_debug_fused_counts(ragfin_t* h, int32_t nq, int64_t* out_appended, int64_t* out_rescored) {
    if (!h || !out_appended || !out_rescored || nq < 1 || nq > kFMaxQ) return fail(RAGFIN_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    if (!h->fctl.p) return fail(RAGFIN_EINVAL, "no one-kernel search has run on this handle");
    CU_TRY(cudaDeviceSynchronize());
    FusedCtl c;
    CU_TRY(cudaMemcpy(&c, (FusedCtl*)h->fctl.p + h->fused_last, sizeof(c), cudaMemcpyDeviceToHost));
    for (int i = 0; i < nq; ++i) {
        out_appended[i] = c.last_cnt[i];
        out_rescored[i] = c.last_resc[i] == 0xFFFFFFFFu ? -1 : (int64_t)c.last_resc[i];
    }
    return RAGFIN_OK;
}

// Tuning knob: the one-kernel search for <= 64 queries and k <= 128 (sweep_fused.cuh; default on; results are identical).
// min_rows: corpora below this many rows keep the multi-kernel paths (0 = leave unchanged).
extern "C" int ragfin_set_fused(ragfin_t* h, int32_t enable, int64_t min_rows) {
    if (!h || min_rows < 0) return fail(RAGFIN_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(h->mu);
    h->use_fused = enable != 0;
    if (min_rows > 0) h->fused_min_rows = (int)(min_rows > 0x7FFFFFFF ? 0x7FFFFFFF : min_rows);
    return RAGFIN_OK;
}

// Opt-in: consecutive one-kernel searches issued through the asynchronous entry points (ragfin_search, ragfin_search_sharded)
// on ONE stream are launched with programmatic stream serialization - search n + 1 starts sweeping while search n finalizes
// (and, sharded, exchanges hits), so HBM never idles between them; results still land in stream order.  The price is a
// contract: such a search may begin BEFORE the operation enqueued just ahead of it on the stream has completed, so its query
// buffer must already hold the queries when the PREVIOUS search on this handle was enqueued (written by a copy or kernel
// ordered before that search, or by the host) - a kernel that produces the queries between two searches needs pipelining off
// (the default), or its own stream synchronisation.  The corpus, filters and workspaces are the library's own business: a
// search that follows anything but this handle's previous one-kernel search on the same stream is launched normally.
extern "C" int ragfin_set_sweep_copy(ragfin_t* h, int32_t mode) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (mode != 0 && mode != 1 && mode != RAGFIN_SWEEP_COPY_AUTO)
        return fail(RAGFIN_EINVAL, "mode %d is not 0 (off), 1 (on) or RAGFIN_SWEEP_COPY_AUTO (%d)", mode, RAGFIN_SWEEP_COPY_AUTO);
    std::lock_guard<std::mutex> lk(h->mu);
    h->sweep_copy = mode;
    return RAGFIN_OK;
}

extern "C" int ragfin_debug_sweep_copy(ragfin_t* h, int64_t row0, int64_t n, int8_t* out_rows_host, float* out_side_host, int32_t* ld8_out) {
    if (!h || !ld8_out || row0 < 0 || n < 0 || (n > 0 && (!out_rows_host || !out_side_host))) return fail(RAGFIN_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->i8) return fail(RAGFIN_EUNSUPPORTED, "this collection has no int8 copy (it is made by the first one-kernel search that uses it)");
    if (row0 + n > h->i8_rows) return fail(RAGFIN_EINVAL, "rows [%lld, %lld) outside the %lld rows of the int8 copy", (long long)row0, (long long)(row0 + n), (long long)h->i8_rows);
    *ld8_out = h->ld8;
    if (n == 0) return RAGFIN_OK;
    DeviceGuard g(h->device);
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpy(out_rows_host, h->i8 + (size_t)row0 * h->ld8, (size_t)n * h->ld8, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(out_side_host, h->i8side + row0, (size_t)n * sizeof(float2), cudaMemcpyDeviceToHost));
    return RAGFIN_OK;
}

extern "C" int ragfin_debug_fused_tiles(ragfin_t* h, int64_t* out) {
    if (!h || !out) return fail(RAGFIN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(h->mu);
    out[0] = out[1] = 0;
    if (!h->fctl.p) return RAGFIN_OK;
    DeviceGuard g(h->device);
    CU_TRY(cudaDeviceSynchronize());
    FusedCtl c;
    CU_TRY(cudaMemcpy(&c, (FusedCtl*)h->fctl.p + h->fused_last, sizeof(FusedCtl), cudaMemcpyDeviceToHost));
    out[0] = c.last_refined;
    out[1] = c.last_screened;
    return RAGFIN_OK;
}

extern "C" int ragfin_set_pipelined(ragfin_t* h, int32_t enable) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    std::lock_guard<std::mutex> lk(h->mu);
    h->allow_pipelined = enable != 0;
    return RAGFIN_OK;
}

// Tuning knob: small-batch scan kernel.  0 = automatic, 1 = register-path loads (scan_topk_kernel), 2 = TMA-fed ring
// (scan_tma_kernel; 1-2 queries).  Results are identical.
extern "C" int ragfin_set_scan_variant(ragfin_t* h, int32_t variant) {
    if (!h || variant < 0 || variant > 2) return fail(RAGFIN_EINVAL, "variant must be 0, 1 or 2");
    std::lock_guard<std::mutex> lk(h->mu);
    h->scan_variant = variant;
    return RAGFIN_OK;
}

// Tuning knob: which tcgen05 kernel serves large batches (0 automatic, 1 streaming, 2 A-stationary when eligible,
// 3 swapped roles for <= 16 queries, 4 2-SM MMA pairs for >= 2 query tiles in append mode).
extern "C" int ragfin_set_gemm_variant(ragfin_t* h, int32_t variant) {
    if (!h || variant < 0 || variant > 4) return fail(RAGFIN_EINVAL, "variant must be 0 ... 4");
    std::lock_guard<std::mutex> lk(h->mu);
    h->gemm_variant = variant;
    return RAGFIN_OK;
}

// Tuning knob: thread-block cluster size of the tcgen05 path (0 = automatic, else 1, 2 or 4).
extern "C" int ragfin_set_gemm_cluster(ragfin_t* h, int32_t cluster) {
    if (!h || !(cluster == 0 || cluster == 1 || cluster == 2 || cluster == 4)) return fail(RAGFIN_EINVAL, "cluster must be 0, 1, 2 or 4");
    std::lock_guard<std::mutex> lk(h->mu);
    h->gemm_cluster = cluster;
    return RAGFIN_OK;
}

static int set_filter(ragfin* h, const uint32_t* allow_bits, int64_t n_allowed, int bits_on_device, cudaStream_t st);
static void clear_filter(ragfin* h);

extern "C" int ragfin_search(ragfin_t* h, const float* q, int32_t nq, int32_t k, int64_t* out_ids, float* out_scores,
                             void* stream) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (nq < 0 || (nq > 0 && (!q || !out_ids || !out_scores))) return fail(RAGFIN_EINVAL, "NULL buffer");
    if (k < 1 || k > 16384) return fail(RAGFIN_EINVAL, "k = %d outside [1, 16384]", k);
    if (nq == 0) return RAGFIN_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    // Pipelined launch of the one-kernel search (opt-in, ragfin_set_pipelined): only behind this handle's own previous
    // one-kernel search on the same stream - after an add, a filter, another path or another stream the launch is an ordinary
    // one (a programmatic launch does not wait for its predecessor's memory flush, and this kernel reads its inputs at once).
    const bool pipe = h->allow_pipelined && nq <= h->fused_max_nq && fused_eligible(h, nq, k);
    const bool chained = pipe && h->have_pending && st == h->pending_stream;
    if ((rc = wait_prev(h, st, pipe))) return rc;
    if ((rc = set_filter(h, nullptr, 0, 1, st))) return rc;   // tombstones, if any
    h->cur_pipelined = chained;
    rc = search_locked(h, q, nq, k, out_ids, out_scores, st);
    h->cur_pipelined = false;
    clear_filter(h);
    if (rc) return rc;
    return mark_done(h, st, pipe);
}

// Synchronous host calls of the one-kernel search: wait for the completion word the last finalizing CTA writes into
// device-mapped pinned memory (a posted PCIe write, ~1 us after the hits) instead of for the stream (kernel teardown + driver
// wake-up).  The stream is queried now and then so that a failed launch cannot spin forever.
static int poll_host_flag(const volatile uint32_t* flag, uint32_t seq, cudaStream_t st) {
    for (unsigned spins = 1;; ++spins) {
        if (*flag == seq) { __atomic_thread_fence(__ATOMIC_ACQUIRE); return 0; }
        __builtin_ia32_pause();
        if ((spins & 0x3FFFu) == 0) {
            const cudaError_t e = cudaStreamQuery(st);
            if (e == cudaSuccess) return *flag == seq ? 0 : fail(RAGFIN_ECUDA, "the search kernel finished without publishing its results");
            if (e != cudaErrorNotReady) { (void)cudaGetLastError(); return fail(RAGFIN_ECUDA, "search kernel failed: %s", cudaGetErrorString(e)); }
        }
    }
}

// The fused-path body of the two synchronous host entry points (hstage = mapped staging: [queries | hits | flag]).
static int fused_host_call(ragfin* h, ragfin_exchange* x, const float* q_host, int nq, int k, int64_t* out_ids_host, float* out_scores_host,
                           cudaStream_t st) {
    int rc;
    const size_t qb = (size_t)nq * h->dim * sizeof(float), ib = (size_t)nq * k * sizeof(int64_t), sb = (size_t)nq * k * sizeof(float);
    void* dptr = nullptr;
    CU_TRY(cudaHostGetDevicePointer(&dptr, h->hstage, 0));
    char* hq = (char*)h->hstage;
    char* ho = hq + kHostStageQ;
    volatile uint32_t* hflag = (volatile uint32_t*)(ho + kHostStageOut);
    char* dout = (char*)dptr + kHostStageQ;
    uint32_t* dflag = (uint32_t*)(dout + kHostStageOut);
    const float* q_dev = nullptr;
    const float* q_inline = nullptr;
    if ((size_t)nq * h->dim <= (size_t)kFInlineFloats) {
        q_inline = q_host;                                   // the queries ride in the launch: no transfer in front of the kernel
    } else {
        // every CTA reads the queries: one small copy-engine transfer into HBM instead of ~150 reads of the same bytes over PCIe
        memcpy(hq, q_host, qb);
        if ((rc = ensure(h->stage_q, qb))) return rc;
        CU_TRY(cudaMemcpyAsync(h->stage_q.p, hq, qb, cudaMemcpyHostToDevice, st));
        q_dev = (const float*)h->stage_q.p;
    }
    const uint32_t seq = ++h->host_seq;
    h->stats.launches = 0;
    h->stats.queries_rescanned = -1;
    if (x != nullptr) {
        if (!x->connected) return fail(RAGFIN_EINVAL, "exchange is not connected");
        if (x->have_stream && x->stream != st)
            return fail(RAGFIN_EINVAL, "every step of an exchange must be issued on the same CUDA stream (its slot ring relies on stream order)");
        if (x->owner != nullptr && x->owner != h)
            return fail(RAGFIN_EINVAL, "an exchange serves the one-kernel searches of ONE collection (its gather ring counts on a handle's limit of two searches in flight)");
        x->owner = h;
        x->have_stream = true; x->stream = st;
        const uint32_t step = ++x->step;
        rc = run_fused(h, q_dev, nq, k, h->count, (int64_t*)dout, (float*)(dout + ib), st, false, x, step, q_inline, dflag, seq);
    } else {
        const int64_t n_eff = h->cur_allow ? h->cur_allowed : h->count;
        rc = run_fused(h, q_dev, nq, k, n_eff, (int64_t*)dout, (float*)(dout + ib), st, false, nullptr, 0, q_inline, dflag, seq);
    }
    if (rc) return rc;
    if ((rc = poll_host_flag(hflag, seq, st))) return rc;
    memcpy(out_ids_host, ho, ib);
    memcpy(out_scores_host, ho + ib, sb);
    return 0;
}

static int search_host_locked(ragfin* h, const float* q_host, int nq, int k, int64_t* out_ids_host, float* out_scores_host,
                              cudaStream_t st);
extern "C" int ragfin_search_host(ragfin_t* h, const float* q_host, int32_t nq, int32_t k, int64_t* out_ids_host,
                                  float* out_scores_host) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (nq < 0 || (nq > 0 && (!q_host || !out_ids_host || !out_scores_host))) return fail(RAGFIN_EINVAL, "NULL buffer");
    if (k < 1 || k > 16384) return fail(RAGFIN_EINVAL, "k = %d outside [1, 16384]", k);
    if (nq == 0) return RAGFIN_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    cudaStream_t st = 0;
    int rc;
    if ((rc = wait_prev(h, st))) return rc;
    if ((rc = set_filter(h, nullptr, 0, 1, st))) return rc;   // tombstones, if any
    rc = search_host_locked(h, q_host, nq, k, out_ids_host, out_scores_host, st);
    clear_filter(h);
    return rc;
}

static int search_host_locked(ragfin* h, const float* q_host, int nq, int k, int64_t* out_ids_host, float* out_scores_host,
                              cudaStream_t st) {
    int rc;
    const size_t qb = (size_t)nq * h->dim * sizeof(float), ib = (size_t)nq * k * sizeof(int64_t), sb = (size_t)nq * k * sizeof(float);
    if (qb <= kHostStageQ && ib + sb <= kHostStageOut) {
        // small request: three copy-engine launches (~20 us) would cost more than the bytes; the kernels read the queries
        // from, and write the hits to, device-mapped pinned memory
        if (!h->hstage) {
            (void)alloc_hstage(h);
        }
        void* dptr = nullptr;
        if (h->hstage && cudaHostGetDevicePointer(&dptr, h->hstage, 0) == cudaSuccess) {
            if (!h->cur_window && !h->cur_groups && nq <= h->fused_max_nq && fused_eligible(h, nq, k)) {
                if ((rc = fused_host_call(h, nullptr, q_host, nq, k, out_ids_host, out_scores_host, st))) return rc;
                return mark_done(h, st);
            }
            char* hq = (char*)h->hstage;
            char* ho = hq + kHostStageQ;
            memcpy(hq, q_host, qb);
            char* dq = (char*)dptr;
            char* dout = dq + kHostStageQ;
            const float* qsrc = (const float*)dq;
            if ((rc = search_locked(h, qsrc, nq, k, (int64_t*)dout, (float*)(dout + ib), st))) return rc;
            CU_TRY(cudaStreamSynchronize(st));
            memcpy(out_ids_host, ho, ib);
            memcpy(out_scores_host, ho + ib, sb);
            return mark_done(h, st);
        }
        (void)cudaGetLastError();
    }
    if ((rc = ensure(h->stage_q, qb)) || (rc = ensure(h->stage_ids, ib)) || (rc = ensure(h->stage_scores, sb))) return rc;
    CU_TRY(cudaMemcpyAsync(h->stage_q.p, q_host, qb, cudaMemcpyHostToDevice, st));
    if ((rc = search_locked(h, (const float*)h->stage_q.p, nq, k, (int64_t*)h->stage_ids.p, (float*)h->stage_scores.p, st))) return rc;
    CU_TRY(cudaMemcpyAsync(out_ids_host, h->stage_ids.p, ib, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(out_scores_host, h->stage_scores.p, sb, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return mark_done(h, st);
}

// The row mask of one search, installed before dispatch and cleared after it by every search entry point.
//  - no filter, no tombstones: null (every row);
//  - tombstones only: the live mask, with the UNFILTERED dispatch (bound pass and append mode honour the mask);
//  - a filter (bit r of allow_bits, ceil(count / 32) 32-bit words, set <=> row r may be returned): the filtered dispatch,
//    with the mask allow AND live when the handle has tombstones.  n_allowed counts the caller's bits; the rows left after
//    the AND are counted here: on the host for a host mask, by mask_and_popc_kernel for a device mask (one stream
//    synchronisation, only on handles with tombstones).
static int set_filter(ragfin* h, const uint32_t* allow_bits, int64_t n_allowed, int bits_on_device, cudaStream_t st) {
    h->cur_user_filter = allow_bits != nullptr;
    if (!allow_bits) {
        h->cur_allow = h->n_dead > 0 ? h->live_dev : nullptr;
        h->cur_allowed = h->n_dead > 0 ? h->count - h->n_dead : 0;
        return 0;
    }
    if (n_allowed < 0 || n_allowed > h->count) return fail(RAGFIN_EINVAL, "n_allowed %lld outside [0, %lld]", (long long)n_allowed, (long long)h->count);
    const size_t words = mask_words(h->count);
    int rc;
    if (h->n_dead > 0 && bits_on_device) {
        const size_t cnt_off = (words + 1) / 2 * 2 * sizeof(uint32_t);   // the 8-byte count after the words
        if ((rc = ensure(h->allow, cnt_off + sizeof(unsigned long long)))) return rc;
        unsigned long long* dcnt = (unsigned long long*)((char*)h->allow.p + cnt_off);
        CU_TRY(cudaMemsetAsync(dcnt, 0, sizeof(*dcnt), st));
        if (words > 0) {
            const int64_t want = ((int64_t)words + 255) / 256, cap_blocks = (int64_t)h->num_sms * 4;
            mask_and_popc_kernel<<<(unsigned)(want < cap_blocks ? want : cap_blocks), 256, 0, st>>>(allow_bits, h->live_dev, (uint32_t*)h->allow.p,
                                                                                                 (int64_t)words, h->count, dcnt);
            CU_TRY(cudaGetLastError());
        }
        unsigned long long live_allowed = 0;
        CU_TRY(cudaMemcpyAsync(&live_allowed, dcnt, sizeof(live_allowed), cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        h->cur_allow = (const uint32_t*)h->allow.p;
        h->cur_allowed = (int64_t)live_allowed;
        return 0;
    }
    if (bits_on_device) { h->cur_allow = allow_bits; h->cur_allowed = n_allowed; return 0; }
    if ((rc = ensure(h->allow, (words ? words : 1) * sizeof(uint32_t)))) return rc;
    if (h->n_dead > 0) {
        std::vector<uint32_t> m(words);
        int64_t live_allowed = 0;
        for (size_t w = 0; w < words; ++w) {
            uint32_t v = allow_bits[w] & h->live_host[w];
            if (w + 1 == words && (h->count & 31)) v &= (1u << (h->count & 31)) - 1u;
            m[w] = v;
            live_allowed += __builtin_popcount(v);
        }
        CU_TRY(cudaMemcpyAsync(h->allow.p, m.data(), words * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        CU_TRY(cudaStreamSynchronize(st));   // `m` is pageable and local
        h->cur_allowed = live_allowed;
    } else {
        CU_TRY(cudaMemcpyAsync(h->allow.p, allow_bits, words * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        h->cur_allowed = n_allowed;
    }
    h->cur_allow = (const uint32_t*)h->allow.p;
    return 0;
}
static void clear_filter(ragfin* h) {
    h->cur_allow = nullptr;
    h->cur_allowed = 0;
    h->cur_user_filter = false;
}

extern "C" int ragfin_search_filtered(ragfin_t* h, const float* q, int32_t nq, int32_t k, const uint32_t* allow_bits_dev,
                                      int64_t n_allowed, int64_t* out_ids, float* out_scores, void* stream) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (nq < 0 || (nq > 0 && (!q || !out_ids || !out_scores))) return fail(RAGFIN_EINVAL, "NULL buffer");
    if (k < 1 || k > 16384) return fail(RAGFIN_EINVAL, "k = %d outside [1, 16384]", k);
    if (nq == 0) return RAGFIN_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if ((rc = wait_prev(h, st))) return rc;
    if ((rc = set_filter(h, allow_bits_dev, n_allowed, 1, st))) return rc;
    rc = search_locked(h, q, nq, k, out_ids, out_scores, st);
    clear_filter(h);
    if (rc) return rc;
    return mark_done(h, st);
}

extern "C" int ragfin_search_filtered_host(ragfin_t* h, const float* q_host, int32_t nq, int32_t k,
                                           const uint32_t* allow_bits_host, int64_t n_allowed, int64_t* out_ids_host,
                                           float* out_scores_host) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (nq < 0 || (nq > 0 && (!q_host || !out_ids_host || !out_scores_host))) return fail(RAGFIN_EINVAL, "NULL buffer");
    if (k < 1 || k > 16384) return fail(RAGFIN_EINVAL, "k = %d outside [1, 16384]", k);
    if (nq == 0) return RAGFIN_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    cudaStream_t st = 0;
    int rc;
    if ((rc = wait_prev(h, st))) return rc;
    const size_t qb = (size_t)nq * h->dim * sizeof(float), ib = (size_t)nq * k * sizeof(int64_t), sb = (size_t)nq * k * sizeof(float);
    if ((rc = ensure(h->stage_q, qb)) || (rc = ensure(h->stage_ids, ib)) || (rc = ensure(h->stage_scores, sb))) return rc;
    if ((rc = set_filter(h, allow_bits_host, n_allowed, 0, st))) return rc;
    CU_TRY(cudaMemcpyAsync(h->stage_q.p, q_host, qb, cudaMemcpyHostToDevice, st));
    rc = search_locked(h, (const float*)h->stage_q.p, nq, k, (int64_t*)h->stage_ids.p, (float*)h->stage_scores.p, st);
    clear_filter(h);
    if (rc) return rc;
    CU_TRY(cudaMemcpyAsync(out_ids_host, h->stage_ids.p, ib, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(out_scores_host, h->stage_scores.p, sb, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return mark_done(h, st);
}

// Range search (DESIGN.md 7c): the k best rows with radius < score <= range_filter.  Both bounds open: the plain entry
// points themselves.  Otherwise the window is installed next to the row mask for the one dispatch (search_locked).
// The window is checked first: it needs neither a handle nor a device.
static int check_range_args(const ragfin* h, const float* q, int nq, int k, const ragfin_range* range,
                            const void* out_ids, const void* out_scores) {
    if (!range) return fail(RAGFIN_EINVAL, "NULL range");
    const float radius = range->radius, range_filter = range->range_filter;
    if (radius != radius || range_filter != range_filter) return fail(RAGFIN_EINVAL, "radius and range_filter must not be NaN");
    if (!(range_filter > radius)) return fail(RAGFIN_EINVAL, "range_filter (%g) must be greater than radius (%g)", (double)range_filter, (double)radius);
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (nq < 0 || (nq > 0 && (!q || !out_ids || !out_scores))) return fail(RAGFIN_EINVAL, "NULL buffer");
    if (k < 1 || k > 16384) return fail(RAGFIN_EINVAL, "k = %d outside [1, 16384]", k);
    return 0;
}
static bool range_open(float radius, float range_filter) { return radius == -INFINITY && range_filter == INFINITY; }
static void set_window(ragfin* h, float radius, float range_filter) {
    h->cur_window = true; h->cur_radius = radius; h->cur_range_filter = range_filter;
}
static void clear_window(ragfin* h) {
    h->cur_window = false; h->cur_radius = -INFINITY; h->cur_range_filter = INFINITY;
}

extern "C" int ragfin_search_range(ragfin_t* h, const float* q, int32_t nq, int32_t k, const ragfin_range* range,
                                   const uint32_t* allow_bits_dev, int64_t n_allowed, int64_t* out_ids, float* out_scores,
                                   void* stream) {
    int rc;
    if ((rc = check_range_args(h, q, nq, k, range, out_ids, out_scores))) return rc;
    const float radius = range->radius, range_filter = range->range_filter;
    if (range_open(radius, range_filter))
        return allow_bits_dev ? ragfin_search_filtered(h, q, nq, k, allow_bits_dev, n_allowed, out_ids, out_scores, stream)
                              : ragfin_search(h, q, nq, k, out_ids, out_scores, stream);
    if (nq == 0) return RAGFIN_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = wait_prev(h, st))) return rc;
    if ((rc = set_filter(h, allow_bits_dev, n_allowed, 1, st))) return rc;
    set_window(h, radius, range_filter);
    rc = search_locked(h, q, nq, k, out_ids, out_scores, st);
    clear_window(h);
    clear_filter(h);
    if (rc) return rc;
    return mark_done(h, st);
}

extern "C" int ragfin_search_range_host(ragfin_t* h, const float* q_host, int32_t nq, int32_t k, const ragfin_range* range,
                                        const uint32_t* allow_bits_host, int64_t n_allowed, int64_t* out_ids_host,
                                        float* out_scores_host) {
    int rc;
    if ((rc = check_range_args(h, q_host, nq, k, range, out_ids_host, out_scores_host))) return rc;
    const float radius = range->radius, range_filter = range->range_filter;
    if (range_open(radius, range_filter))
        return allow_bits_host ? ragfin_search_filtered_host(h, q_host, nq, k, allow_bits_host, n_allowed, out_ids_host, out_scores_host)
                               : ragfin_search_host(h, q_host, nq, k, out_ids_host, out_scores_host);
    if (nq == 0) return RAGFIN_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    cudaStream_t st = 0;
    if ((rc = wait_prev(h, st))) return rc;
    if ((rc = set_filter(h, allow_bits_host, n_allowed, 0, st))) return rc;
    set_window(h, radius, range_filter);
    rc = search_host_locked(h, q_host, nq, k, out_ids_host, out_scores_host, st);
    clear_window(h);
    clear_filter(h);
    return rc;
}

// Grouping search (DESIGN.md 7d): the k best groups, each represented by its best row.  The codes are installed next to the
// row mask for the one dispatch (search_locked).  The codes are checked first: that needs neither a handle nor a device.
static int check_group_args(const ragfin* h, const float* q, int nq, int k, const int32_t* groups, int n_groups,
                            const void* out_ids, const void* out_scores) {
    if (!groups) return fail(RAGFIN_EINVAL, "NULL group codes");
    if (n_groups < 1) return fail(RAGFIN_EINVAL, "n_groups = %d must be at least 1", n_groups);
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    if (nq < 0 || (nq > 0 && (!q || !out_ids || !out_scores))) return fail(RAGFIN_EINVAL, "NULL buffer");
    if (k < 1 || k > 16384) return fail(RAGFIN_EINVAL, "k = %d outside [1, 16384]", k);
    return 0;
}
static void set_groups(ragfin* h, const int32_t* groups_dev, int n_groups) { h->cur_groups = groups_dev; h->cur_n_groups = n_groups; }
static void clear_groups(ragfin* h) { h->cur_groups = nullptr; h->cur_n_groups = 0; }

extern "C" int ragfin_search_grouped(ragfin_t* h, const float* q, int32_t nq, int32_t k, const int32_t* group_of_row_dev,
                                     int32_t n_groups, const uint32_t* allow_bits_dev, int64_t n_allowed, int64_t* out_ids,
                                     float* out_scores, void* stream) {
    int rc;
    if ((rc = check_group_args(h, q, nq, k, group_of_row_dev, n_groups, out_ids, out_scores))) return rc;
    if (nq == 0) return RAGFIN_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = wait_prev(h, st))) return rc;
    if ((rc = set_filter(h, allow_bits_dev, n_allowed, 1, st))) return rc;
    set_groups(h, group_of_row_dev, n_groups);
    rc = search_locked(h, q, nq, k, out_ids, out_scores, st);
    clear_groups(h);
    clear_filter(h);
    if (rc) return rc;
    return mark_done(h, st);
}

extern "C" int ragfin_search_grouped_host(ragfin_t* h, const float* q_host, int32_t nq, int32_t k, const int32_t* group_of_row,
                                          int32_t groups_on_device, int32_t n_groups, const uint32_t* allow_bits_host,
                                          int64_t n_allowed, int64_t* out_ids_host, float* out_scores_host) {
    int rc;
    if ((rc = check_group_args(h, q_host, nq, k, group_of_row, n_groups, out_ids_host, out_scores_host))) return rc;
    if (nq == 0) return RAGFIN_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    cudaStream_t st = 0;
    if ((rc = wait_prev(h, st))) return rc;
    const int32_t* codes = group_of_row;
    if (!groups_on_device && h->count > 0) {
        if ((rc = ensure(h->grp_codes, (size_t)h->count * sizeof(int32_t)))) return rc;
        CU_TRY(cudaMemcpyAsync(h->grp_codes.p, group_of_row, (size_t)h->count * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        codes = (const int32_t*)h->grp_codes.p;
    }
    if ((rc = set_filter(h, allow_bits_host, n_allowed, 0, st))) return rc;
    set_groups(h, codes, n_groups);
    rc = search_host_locked(h, q_host, nq, k, out_ids_host, out_scores_host, st);
    clear_groups(h);
    clear_filter(h);
    return rc;
}

extern "C" int ragfin_last_search_stats(ragfin_t* h, ragfin_search_stats* out) {
    if (!h || !out) return fail(RAGFIN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    if (h->stats.path == 3 && h->fflags.p) {
        CU_TRY(cudaDeviceSynchronize());
        int fc = 0;
        CU_TRY(cudaMemcpy(&fc, (int*)h->fflags.p + h->fused_last * (kFMaxQ + 1) + kFMaxQ, sizeof(int), cudaMemcpyDeviceToHost));
        h->stats.queries_rescanned = fc;
    } else if (h->flags.p && h->stats.path != 2) {
        CU_TRY(cudaDeviceSynchronize());
        int fc = 0;
        CU_TRY(cudaMemcpy(&fc, (int*)h->flags.p + kMaxQueryBatch, sizeof(int), cudaMemcpyDeviceToHost));
        h->stats.queries_rescanned = fc;  // of the last query batch (<= 256 queries)
    }
    *out = h->stats;
    return RAGFIN_OK;
}

extern "C" int ragfin_profile(ragfin_t* h, int32_t enable) {
    if (!h) return fail(RAGFIN_EINVAL, "NULL handle");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    if (enable && !h->prof_ev[0])
        for (cudaEvent_t& e : h->prof_ev) CU_TRY(cudaEventCreate(&e));
    h->profiling = enable != 0;
    h->prof_used = 0;
    return RAGFIN_OK;
}

extern "C" int ragfin_profile_read(ragfin_t* h, double* total_ms, int32_t* launches) {
    if (!h || !total_ms || !launches) return fail(RAGFIN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceGuard g(h->device);
    CU_TRY(cudaDeviceSynchronize());
    double sum = 0.0;
    for (int i = 0; i < h->prof_used; ++i) {
        float ms = 0.f;
        CU_TRY(cudaEventElapsedTime(&ms, h->prof_ev[2 * i], h->prof_ev[2 * i + 1]));
        sum += ms;
    }
    *total_ms = sum;
    *launches = h->prof_used;
    h->prof_used = 0;
    return RAGFIN_OK;
}

extern "C" int ragfin_merge_topk(const int64_t* ids, const float* scores, int32_t nq, int32_t parts, int32_t k,
                                 int64_t ids_part_stride, int64_t scores_part_stride, int64_t query_stride,
                                 int64_t* out_ids, float* out_scores, int32_t device, void* stream) {
    if (nq < 0 || parts < 1 || k < 1) return fail(RAGFIN_EINVAL, "bad nq/parts/k");
    if (ids_part_stride < k || scores_part_stride < k || query_stride < k) return fail(RAGFIN_EINVAL, "strides must be >= k");
    if (nq == 0) return RAGFIN_OK;
    if (!ids || !scores || !out_ids || !out_scores) return fail(RAGFIN_EINVAL, "NULL buffer");
    DeviceGuard g(device);
    if (!g.ok) return fail(RAGFIN_ECUDA, "cudaSetDevice(%d) failed", device);
    const int64_t total = (int64_t)nq * parts * k;
    const int threads = 256;
    merge_topk_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
        ids, scores, nq, parts, k, ids_part_stride, scores_part_stride, query_stride, out_ids, out_scores);
    CU_TRY(cudaGetLastError());
    return RAGFIN_OK;
}

// ------------------------------------------------------------------------------
// Cross-shard exchange over peer memory (CUDA IPC + NVLink P2P stores), see exchange_push_kernel
// ------------------------------------------------------------------------------
extern "C" int ragfin_exchange_create(ragfin_exchange_t** out, int32_t rank, int32_t world, int64_t record_bytes_max, int32_t device) {
    if (!out) return fail(RAGFIN_EINVAL, "out is NULL");
    *out = nullptr;
    if (world < 1 || world > 64 || rank < 0 || rank >= world) return fail(RAGFIN_EINVAL, "rank %d / world %d out of range (world <= 64)", rank, world);
    if (record_bytes_max < 16) return fail(RAGFIN_EINVAL, "record_bytes_max must be >= 16");
    DeviceGuard g(device);
    if (!g.ok) return fail(RAGFIN_ECUDA, "cudaSetDevice(%d) failed", device);
    ragfin_exchange* x = new (std::nothrow) ragfin_exchange();
    if (!x) return fail(RAGFIN_ENOMEM, "host allocation failed");
    x->rank = rank; x->world = world; x->device = device;
    x->record_max = ((size_t)record_bytes_max + 15) / 16 * 16;
    const size_t area = kXSlots * (size_t)world * x->record_max;
    x->bytes = area + kXSlots * (size_t)world * sizeof(uint32_t) + kXSlots * (size_t)world * kFMaxQ * sizeof(uint32_t);
    cudaError_t e = cudaMalloc((void**)&x->local, x->bytes);
    if (e == cudaSuccess) e = cudaMemset(x->local, 0, x->bytes);
    if (e == cudaSuccess) e = cudaMalloc((void**)&x->d_peer_area, world * sizeof(char*));
    if (e == cudaSuccess) e = cudaMalloc((void**)&x->d_peer_flag, world * sizeof(uint32_t*));
    if (e == cudaSuccess) e = cudaMalloc((void**)&x->d_peer_qflag, world * sizeof(uint32_t*));
    if (e == cudaSuccess) e = cudaMalloc((void**)&x->d_done, world * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMemset(x->d_done, 0, world * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        if (x->local) cudaFree(x->local);
        if (x->d_peer_area) cudaFree(x->d_peer_area);
        if (x->d_peer_flag) cudaFree(x->d_peer_flag);
        if (x->d_peer_qflag) cudaFree(x->d_peer_qflag);
        if (x->d_done) cudaFree(x->d_done);
        delete x;
        return fail(RAGFIN_ENOMEM, "exchange allocation failed: %s", cudaGetErrorString(e));
    }
    *out = x;
    return RAGFIN_OK;
}

extern "C" int ragfin_exchange_handle(ragfin_exchange_t* x, void* handle_out) {
    if (!x || !handle_out) return fail(RAGFIN_EINVAL, "NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == RAGFIN_IPC_HANDLE_BYTES, "IPC handle size");
    DeviceGuard g(x->device);
    cudaIpcMemHandle_t hd;
    CU_TRY(cudaIpcGetMemHandle(&hd, x->local));
    memcpy(handle_out, &hd, sizeof(hd));
    return RAGFIN_OK;
}

extern "C" int ragfin_exchange_connect(ragfin_exchange_t* x, const void* handles) {
    if (!x || !handles) return fail(RAGFIN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(x->mu);
    if (x->connected) return fail(RAGFIN_EINVAL, "exchange is already connected");
    DeviceGuard g(x->device);
    const size_t area = kXSlots * (size_t)x->world * x->record_max;
    char* areas[64];
    uint32_t* flags[64];
    uint32_t* qflags[64];
    for (int p = 0; p < x->world; ++p) {
        if (p == x->rank) {
            x->peer_base[p] = x->local;
        } else {
            cudaIpcMemHandle_t hd;
            memcpy(&hd, (const char*)handles + (size_t)p * sizeof(hd), sizeof(hd));
            void* ptr = nullptr;
            cudaError_t e = cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) {
                (void)cudaGetLastError();
                return fail(RAGFIN_ECUDA, "cudaIpcOpenMemHandle for rank %d failed: %s (no peer access between the GPUs?)", p, cudaGetErrorString(e));
            }
            x->peer_base[p] = (char*)ptr;
            x->opened[p] = true;
        }
        areas[p] = x->peer_base[p];
        flags[p] = reinterpret_cast<uint32_t*>(x->peer_base[p] + area);
        qflags[p] = flags[p] + kXSlots * (size_t)x->world;
    }
    CU_TRY(cudaMemcpy(x->d_peer_area, areas, x->world * sizeof(char*), cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(x->d_peer_flag, flags, x->world * sizeof(uint32_t*), cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(x->d_peer_qflag, qflags, x->world * sizeof(uint32_t*), cudaMemcpyHostToDevice));
    x->connected = true;
    return RAGFIN_OK;
}

extern "C" int ragfin_exchange_allgather_merge(ragfin_exchange_t* x, const int64_t* ids_dev, const float* scores_dev, int32_t nq,
                                               int32_t k, int64_t* out_ids, float* out_scores, void* stream) {
    if (!x || !ids_dev || !scores_dev || !out_ids || !out_scores) return fail(RAGFIN_EINVAL, "NULL argument");
    if (nq < 1 || k < 1) return fail(RAGFIN_EINVAL, "bad nq/k");
    std::lock_guard<std::mutex> lk(x->mu);
    if (!x->connected) return fail(RAGFIN_EINVAL, "exchange is not connected");
    const int64_t n_hits = (int64_t)nq * k;
    const size_t record = ((size_t)n_hits * 12 + 15) / 16 * 16;
    if (record > x->record_max) return fail(RAGFIN_EINVAL, "record of %zu bytes exceeds the exchange's %zu", record, x->record_max);
    DeviceGuard g(x->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (x->have_stream && x->stream != st)
        return fail(RAGFIN_EINVAL, "every step of an exchange must be issued on the same CUDA stream (its slot ring relies on stream order)");
    x->have_stream = true; x->stream = st;
    const uint32_t step = ++x->step;
    int chunks = (int)((n_hits + 255) / 256);
    if (chunks > 64) chunks = 64;
    exchange_push_kernel<<<dim3(chunks, x->world), 256, 0, st>>>(ids_dev, scores_dev, n_hits, x->rank, x->world, x->record_max, step,
                                                                 x->d_peer_area, x->d_peer_flag, x->d_done);
    CU_TRY(cudaGetLastError());
    const int64_t total = n_hits * x->world;
    const uint32_t* flags = reinterpret_cast<const uint32_t*>(x->local + kXSlots * (size_t)x->world * x->record_max);
    exchange_merge_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(x->local, flags, nq, x->world, k, x->record_max, step,
                                                                           out_ids, out_scores);
    CU_TRY(cudaGetLastError());
    return RAGFIN_OK;
}

// Whether (nq, k) on this handle would take the one-kernel search.  Ranks of a sharded search must agree before they use
// ragfin_search_sharded (shard sizes differ by a row): the host layer reduces this over the ranks once per shape.
extern "C" int ragfin_fused_eligible(ragfin_t* h, int32_t nq, int32_t k, int32_t* out) {
    if (!h || !out || nq < 1 || k < 1) return fail(RAGFIN_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(h->mu);
    *out = (nq <= kFMaxQ && fused_eligible(h, nq, k)) ? 1 : 0;
    return RAGFIN_OK;
}

static int sharded_locked(ragfin* h, ragfin_exchange* x, const float* q_dev, int nq, int k, int64_t* out_ids, float* out_scores,
                          cudaStream_t st, bool pipelined) {
    if (!x->connected) return fail(RAGFIN_EINVAL, "exchange is not connected");
    if (x->device != h->device) return fail(RAGFIN_EINVAL, "exchange and collection live on different devices");
    if (h->n_dead > 0) return fail(RAGFIN_EUNSUPPORTED, "sharded search over a shard with deleted rows: compact first");
    if (nq > kFMaxQ || !fused_eligible(h, nq, k))
        return fail(RAGFIN_EUNSUPPORTED, "shape (nq = %d, k = %d) does not take the one-kernel search on this shard", nq, k);
    const size_t record = (size_t)nq * (((size_t)k * 12 + 15) / 16 * 16);
    if (record > x->record_max) return fail(RAGFIN_EINVAL, "record of %zu bytes exceeds the exchange's %zu", record, x->record_max);
    if (x->have_stream && x->stream != st)
        return fail(RAGFIN_EINVAL, "every step of an exchange must be issued on the same CUDA stream (its slot ring relies on stream order)");
    if (x->owner != nullptr && x->owner != h)
        return fail(RAGFIN_EINVAL, "an exchange serves the one-kernel searches of ONE collection (its gather ring counts on a handle's limit of two searches in flight)");
    x->owner = h;
    x->have_stream = true; x->stream = st;
    int rc;
    if ((rc = ensure(h->flags, (size_t)(kMaxQueryBatch + 1) * sizeof(int)))) return rc;
    h->stats.launches = 0;
    const int64_t n_eff = h->count;
    const uint32_t step = ++x->step;
    return run_fused(h, q_dev, nq, k, n_eff, out_ids, out_scores, st, pipelined, x, step);
}

// Row-sharded search in ONE kernel per GPU (sweep_fused.cuh): this rank's shard is swept, the finalizing CTAs push the
// shard's exact hits into every rank's gather area over NVLink, wait for the other ranks' and write the GLOBAL top-k.
// Collective: every rank of the exchange must call it with the same (nq, k) and queries, once per step, on one stream.
extern "C" int ragfin_search_sharded(ragfin_t* h, ragfin_exchange_t* x, const float* q, int32_t nq, int32_t k, int64_t* out_ids,
                                     float* out_scores, void* stream) {
    if (!h || !x) return fail(RAGFIN_EINVAL, "NULL handle");
    if (nq < 1 || !q || !out_ids || !out_scores) return fail(RAGFIN_EINVAL, "NULL buffer");
    if (k < 1 || k > 16384) return fail(RAGFIN_EINVAL, "k = %d outside [1, 16384]", k);
    std::lock_guard<std::mutex> lk(h->mu);
    std::lock_guard<std::mutex> lx(x->mu);
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    const bool pipe = h->allow_pipelined;
    const bool chained = pipe && h->have_pending && st == h->pending_stream;   // as in ragfin_search
    if ((rc = wait_prev(h, st, pipe))) return rc;
    if ((rc = sharded_locked(h, x, q, nq, k, out_ids, out_scores, st, chained))) return rc;
    return mark_done(h, st, pipe);
}

// Same with HOST buffers (what a serving process calls): queries staged through pinned memory, the global hits written by
// the kernel straight into device-mapped pinned memory, one stream synchronisation.
extern "C" int ragfin_search_sharded_host(ragfin_t* h, ragfin_exchange_t* x, const float* q_host, int32_t nq, int32_t k,
                                          int64_t* out_ids_host, float* out_scores_host) {
    if (!h || !x) return fail(RAGFIN_EINVAL, "NULL handle");
    if (nq < 1 || !q_host || !out_ids_host || !out_scores_host) return fail(RAGFIN_EINVAL, "NULL buffer");
    if (k < 1 || k > 16384) return fail(RAGFIN_EINVAL, "k = %d outside [1, 16384]", k);
    std::lock_guard<std::mutex> lk(h->mu);
    std::lock_guard<std::mutex> lx(x->mu);
    DeviceGuard g(h->device);
    cudaStream_t st = 0;
    int rc;
    if ((rc = wait_prev(h, st))) return rc;
    const size_t qb = (size_t)nq * h->dim * sizeof(float), ib = (size_t)nq * k * sizeof(int64_t), sb = (size_t)nq * k * sizeof(float);
    if (qb > kHostStageQ || ib + sb > kHostStageOut) return fail(RAGFIN_EUNSUPPORTED, "request too large for the mapped staging");
    if (x->device != h->device) return fail(RAGFIN_EINVAL, "exchange and collection live on different devices");
    if (h->n_dead > 0) return fail(RAGFIN_EUNSUPPORTED, "sharded search over a shard with deleted rows: compact first");
    if (nq > h->fused_max_nq || !fused_eligible(h, nq, k))
        return fail(RAGFIN_EUNSUPPORTED, "shape (nq = %d, k = %d) does not take the one-kernel search on this shard", nq, k);
    if ((size_t)nq * (((size_t)k * 12 + 15) / 16 * 16) > x->record_max) return fail(RAGFIN_EINVAL, "record exceeds the exchange's %zu bytes", x->record_max);
    if (!h->hstage && (rc = alloc_hstage(h))) return rc;
    if ((rc = fused_host_call(h, x, q_host, nq, k, out_ids_host, out_scores_host, st))) return rc;
    // a finalizing CTA that waited 4 s for a peer's hits gives up and marks the query's empty slots with NaN scores
    for (size_t i = 0; i < (size_t)nq * k; ++i)
        if (out_scores_host[i] != out_scores_host[i]) {
            (void)mark_done(h, st);
            return fail(RAGFIN_ECUDA, "sharded search: the exchange timed out waiting for a peer rank's hits (query %zu); is every rank calling with the same shape?", i / k);
        }
    return mark_done(h, st);
}

extern "C" void ragfin_exchange_destroy(ragfin_exchange_t* x) {
    if (!x) return;
    DeviceGuard g(x->device);
    (void)cudaDeviceSynchronize();
    for (int p = 0; p < x->world; ++p)
        if (x->opened[p]) (void)cudaIpcCloseMemHandle(x->peer_base[p]);
    if (x->local) cudaFree(x->local);
    if (x->d_peer_area) cudaFree(x->d_peer_area);
    if (x->d_peer_flag) cudaFree(x->d_peer_flag);
    if (x->d_peer_qflag) cudaFree(x->d_peer_qflag);
    if (x->d_done) cudaFree(x->d_done);
    (void)cudaGetLastError();
    delete x;
}
