/*
 * ragfin.h - C ABI of the B200-native exact cosine top-k engine.
 *
 * This is the drop-in boundary for rag-fin's vector-RAG hot path.  The reference has no
 * FFI layer of its own: its operator API for this path is the pymilvus 2.3.0 call
 *
 *     Collection.search(data, "embedding", {"metric_type": "COSINE"}, limit, output_fields=...)
 *
 * made at   retrieve.py:28-34,  vector_rag_mcp/main.py:51-57,
 *           "chunking_storing (1).py":411-417,  graph_cons.py:275-281
 * plus the ingest calls  Collection.insert / flush / load  ("chunking_storing (1).py":383-396)
 * and  Collection.num_entities  (vector_rag_mcp/main.py:113,120,164).
 * The Python shim `ragfin_b200.milvus_compat.Collection` reproduces that surface and binds
 * exactly the entry points below through ctypes (see INTEGRATION.md).
 *
 * Conventions: every function returns 0 on success and a negative RAGFIN_E* code on
 * failure; the message is available from ragfin_last_error() (thread local).  No C++
 * exception crosses the boundary.  Plain pointers and sizes only.  The engine owns the
 * device-resident corpus matrix behind the opaque handle; the caller owns every buffer it
 * passes in.  `stream` is a cudaStream_t cast to void* (NULL = legacy default stream).
 * A handle may be used from several host threads: searches are serialised against each
 * other and against add (FastMCP runs tools on a worker pool, vector_rag_mcp/main.py:134).
 *
 * There is NO CPU fallback: without a CUDA device every call that touches data fails
 * with RAGFIN_ECUDA.
 */
#ifndef RAGFIN_H
#define RAGFIN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ragfin ragfin_t;

/* RAGFIN_F32_F16: fp32 rows plus an fp16 copy of them (see ragfin_create). */
enum { RAGFIN_F32 = 0, RAGFIN_BF16 = 1, RAGFIN_F16 = 2, RAGFIN_F32_F16 = 3 };

enum {
    RAGFIN_OK = 0,
    RAGFIN_EINVAL = -1,   /* bad argument                                   */
    RAGFIN_ECUDA = -2,    /* CUDA runtime / driver error, or no device      */
    RAGFIN_ENOMEM = -3,   /* capacity_rows exceeded or device allocation failed */
    RAGFIN_EUNSUPPORTED = -4
};

/* ABI version of this header; bumped on any signature change.  Version 4 also carries the row-deletion entry points
 * (ragfin_delete, ragfin_live_count, ragfin_read_live_mask, ragfin_compact) and the range-search entry points
 * (ragfin_search_range, ragfin_search_range_host): they were added without changing any existing signature, so the version
 * stays 4. */
#define RAGFIN_ABI_VERSION 4
int ragfin_abi_version(void);

/* Create an empty collection of `dim`-wide embeddings stored as `dtype` on CUDA device
 * `device`, with room for `capacity_rows` rows (HBM is reserved up front: one contiguous
 * row-major [capacity, ld] matrix, ld = dim rounded up to 8).
 * dtype RAGFIN_F32_F16 holds two matrices: the fp32 rows exactly as RAGFIN_F32 stores them, and an fp16 copy
 * [capacity, ld] (each element RNE-rounded from the stored fp32 value: bit for bit what RAGFIN_F16 stores for the same
 * input).  The tensor-core sweeps stream the copy (16-bit bytes, kind::f16); every exact step - rescore, exact tiers,
 * small-batch scan - reads the fp32 rows, so results are bit-identical to a RAGFIN_F32 collection.  Cost: 6 bytes per
 * element (46.1 GB at 10M x 768, against 30.7 GB for fp32), which is why it is opt-in.
 * Replaces: Collection(name, CollectionSchema([... FieldSchema("embedding", FLOAT_VECTOR,
 * dim=384) ...])) + create_index(COSINE)  - "chunking_storing (1).py":14-29. */
int ragfin_create(ragfin_t** out, int32_t dim, int32_t dtype, int64_t capacity_rows, int32_t device);

/* Append n fp32 rows ([n, dim] row-major; host memory, or device memory when
 * src_is_device != 0).  Each row is L2-normalised (fp64 canonical sum, see DESIGN.md) and
 * rounded once to the storage type by the ingest kernel.  Row ids are insertion ordinals.
 * A row with any NaN or +-Inf component is stored as the zero row (every element 0: it scores exactly 0 against every query);
 * nothing is validated or reported, so a device source stays asynchronous.
 * Replaces: collection.insert([... embeddings ...]); flush(); load()
 * - "chunking_storing (1).py":383-396. */
int ragfin_add(ragfin_t* h, const float* rows, int64_t n, int32_t src_is_device, void* stream);

/* Append rows row0..row0+n of the deterministic synthetic matrix `seed` (SURVEY.md 8d),
 * generated on the device and passed through the same ingest kernel.  dup_every /
 * zero_every (0 = off) plant duplicate and all-zero rows.  Bench/test data only. */
int ragfin_add_synthetic(ragfin_t* h, uint64_t seed, int64_t row0, int64_t n, int32_t dup_every,
                         int32_t zero_every, void* stream);

/* Bench / test data with the structure of a templated text corpus (the reference's chunks are the same templates filled
 * with each quarter's figures: FinRag_knowledge_graph/chunks.json): row r = centre(r / topic_rows) + noise(r) * 2^-noise_shift,
 * centre = row `topic` of the synthetic matrix (seed + RAGFIN_TOPIC_SEED_OFFSET), noise = row r of the synthetic matrix
 * `seed`; contiguous runs of topic_rows near-duplicates inserted in topic order.  Exact in fp32 (1 <= noise_shift <= 10). */
#define RAGFIN_TOPIC_SEED_OFFSET 0x7091C5ull
int ragfin_add_synthetic_topics(ragfin_t* h, uint64_t seed, int64_t row0, int64_t n, int64_t topic_rows, int32_t noise_shift,
                                void* stream);

/* Number of rows held.  Replaces: Collection.num_entities - vector_rag_mcp/main.py:164. */
int ragfin_count(const ragfin_t* h, int64_t* n);

/* Row deletion.  ragfin_delete tombstones rows by the ids searches return (id_base + row): from then on no search entry point
 * returns them, and searches keep the unfiltered kernel dispatch (the bound pass and the append-mode epilogues read the
 * tombstone mask).  Duplicate ids and ids deleted before are allowed; *n_deleted_out (may be NULL) counts the rows this call
 * deleted.  An id outside [id_base, id_base + count) fails the whole call with RAGFIN_EINVAL and changes nothing; a view
 * returns RAGFIN_EUNSUPPORTED.  The call waits for the handle's searches in flight (the mask they read changes), under the
 * same lock as ragfin_add.  Rows added later are live.  The handle keeps a host mirror of the mask; the device mask
 * (capacity / 8 bytes) is allocated on the first delete, and a handle that never deletes allocates nothing for it.
 * ragfin_count keeps counting the rows stored; ragfin_live_count returns stored minus tombstoned.
 * ragfin_read_live_mask copies ceil(count / 32) words in the allow_bits layout (bit set = row live) - test hook.
 * A filtered search on a handle with tombstones searches allow AND live; n_allowed still counts the caller's bits (the library
 * counts what survives the AND itself: on the host for _filtered_host, with one extra stream synchronisation for the device
 * mask of _filtered).  ragfin_search_sharded[_host] on a handle with tombstones returns RAGFIN_EUNSUPPORTED: compact first.
 * ragfin_compact removes the tombstoned rows physically: survivors keep their order, new row r is the r-th live row (ids
 * become id_base + new ordinal), the capacity is unchanged and the tombstones are cleared.  It builds the compacted matrix in a
 * second allocation, so it needs a second copy of the matrix transiently (of both matrices on RAGFIN_F32_F16: 92 GB at
 * 10M x 768), and synchronises the device.  RAGFIN_EUNSUPPORTED on a view or while views of the handle are live.
 * Replaces: Collection.delete(expr) / upsert(data) / compact() of pymilvus 2.3. */
int ragfin_delete(ragfin_t* h, const int64_t* ids_host, int64_t n, int64_t* n_deleted_out);
int ragfin_live_count(const ragfin_t* h, int64_t* n);
int ragfin_read_live_mask(ragfin_t* h, uint32_t* out_host);
int ragfin_compact(ragfin_t* h);

/* Grow the matrix to at least capacity_rows rows: a new device allocation and a device-to-device copy of the stored rows
 * (bits unchanged, nothing re-normalised, no host copy of the embeddings).  No-op when the capacity is already there.
 * Replaces: Milvus growing a collection's segments under repeated insert() - "chunking_storing (1).py":383-396. */
int ragfin_reserve(ragfin_t* h, int64_t capacity_rows);

/* Global id of local row 0 (row-sharded corpora: shard r sets its base). Default 0. */
int ragfin_set_id_base(ragfin_t* h, int64_t id_base);

/* Exact cosine top-k.  q: [nq, dim] fp32 row-major DEVICE memory (raw, un-normalised
 * queries).  out_ids [nq, k] int64 and out_scores [nq, k] fp32 are DEVICE memory; hits are
 * in descending score, ties broken by lower id; slots beyond min(k, N) hold id -1 and
 * score -inf.  Asynchronous on `stream` for k <= 224; larger k (up to 16384, the Milvus limit) takes
 * an exact radix-select path that synchronises the stream once per query.
 * A query with any NaN or +-Inf component is searched as the zero query: every row scores exactly 0 (this holds for every
 * search entry point).
 * Replaces: Collection.search(q, "embedding", {"metric_type":"COSINE"}, k)
 * - vector_rag_mcp/main.py:51-57 (and the three other call sites listed above). */
int ragfin_search(ragfin_t* h, const float* q, int32_t nq, int32_t k, int64_t* out_ids,
                  float* out_scores, void* stream);

/* Same, with HOST buffers: copies the queries in, searches, copies the hits out and
 * synchronises.  This is the call the Python shim makes for numpy / list input. */
int ragfin_search_host(ragfin_t* h, const float* q_host, int32_t nq, int32_t k, int64_t* out_ids_host,
                       float* out_scores_host);

/* Scalar-filtered search (Milvus `search(..., expr=...)`; "next" row N1 of the scope table): only rows
 * whose bit is set in `allow_bits` (ceil(count / 32) little-endian 32-bit words, bit r of word r/32 = row r)
 * may be returned; n_allowed = number of set bits.  The bitmask is consumed inside the top-k epilogues, the
 * corpus is still read once.  Results equal the unfiltered search restricted to the allowed rows.
 * _filtered: device bitmask, asynchronous; _filtered_host: host buffers, synchronous. */
int ragfin_search_filtered(ragfin_t* h, const float* q, int32_t nq, int32_t k, const uint32_t* allow_bits_dev,
                           int64_t n_allowed, int64_t* out_ids, float* out_scores, void* stream);
int ragfin_search_filtered_host(ragfin_t* h, const float* q_host, int32_t nq, int32_t k,
                                const uint32_t* allow_bits_host, int64_t n_allowed, int64_t* out_ids_host,
                                float* out_scores_host);

/* Range search (pymilvus `search(..., {"metric_type": "COSINE", "params": {"radius": r, "range_filter": f}}, limit=k)`):
 * the k best rows whose score s satisfies  radius < s <= range_filter,  ordered by (score desc, id asc); slots past the
 * number of rows in the window hold id -1 and score -inf.  s is the exact fp32 score every search returns and the compares
 * are fp32 compares on it: a row scoring exactly `radius` is excluded, one scoring exactly `range_filter` is included.
 * radius = -INFINITY is no floor, range_filter = +INFINITY no ceiling; with both open the call IS ragfin_search[_host]
 * (or _filtered[_host] when allow_bits is given), bit for bit.  allow_bits (may be NULL) and n_allowed mean what they mean for
 * ragfin_search_filtered[_host]; tombstoned rows are never returned.  RAGFIN_EINVAL for a NULL range, a NaN bound or
 * range_filter <= radius.
 * Dispatch (DESIGN.md 7c): the tensor-core append path with the window applied in its bound pass and epilogues when the
 * batch would take it (k <= 256, no filter, a corpus of >= 4 k tiles), else the large-k pipeline with the window; never the
 * one-kernel search.  ragfin_last_search_stats reports path 1 (append) or 2 (large-k) and queries_rescanned.  Works on views;
 * the sharded entry points have no range form.
 * The window travels by pointer to a ragfin_range in host memory, read before the call returns: every parameter of this
 * ABI is a pointer or a 32- / 64-bit integer, the rule tests/test_abi_cpu.py checks every ctypes binding against.  FFI
 * callers pass the address of two consecutive fp32 values {radius, range_filter} (ctypes: (c_float * 2)(r, f)).  A NULL
 * range is RAGFIN_EINVAL.  The window is validated before the handle, so a bad window fails the same way with any handle.
 * _range: device buffers and bitmask, asynchronous on `stream` (the large-k route synchronises it); _range_host: host
 * buffers and bitmask, synchronous. */
typedef struct {
    float radius;         /* exclusive floor; -INFINITY = none */
    float range_filter;   /* inclusive ceiling; +INFINITY = none */
} ragfin_range;
int ragfin_search_range(ragfin_t* h, const float* q, int32_t nq, int32_t k, const ragfin_range* range,
                        const uint32_t* allow_bits_dev, int64_t n_allowed, int64_t* out_ids, float* out_scores, void* stream);
int ragfin_search_range_host(ragfin_t* h, const float* q_host, int32_t nq, int32_t k, const ragfin_range* range,
                             const uint32_t* allow_bits_host, int64_t n_allowed, int64_t* out_ids_host, float* out_scores_host);

/* Cross-shard reduce: merge `parts` exact hit lists per query (device memory; -1 ids are
 * padding) into the global top-k, ordered by (score desc, id asc).  Hit j of part p for query q
 * is at element  q * query_stride + p * ids_part_stride + j  of `ids` and
 * q * query_stride + p * scores_part_stride + j  of `scores`: an all-gather buffer
 * [parts][nq][k] has both part strides nq*k and query_stride k; a concatenation [nq][parts*k] has
 * part strides k and query_stride parts*k; a packed per-rank record {ids[nq*k] | scores[nq*k]} of
 * B bytes (one all-gather) has ids_part_stride B/8 and scores_part_stride B/4.  Used after the NCCL all-gather of per-rank hits
 * (Milvus proxy reduce in the reference deployment, SURVEY.md 2a). */
int ragfin_merge_topk(const int64_t* ids, const float* scores, int32_t nq, int32_t parts, int32_t k,
                      int64_t ids_part_stride, int64_t scores_part_stride, int64_t query_stride,
                      int64_t* out_ids, float* out_scores, int32_t device, void* stream);

/* Cross-shard exchange over NVLink peer memory, one process per GPU on one box - the fused alternative to
 * "NCCL all-gather + ragfin_merge_topk" (like it, it stands in for the querynode -> proxy top-k reduce of a sharded
 * Milvus deployment of the reference; that reduce is not in the reference repository, SURVEY.md 2a / 8e).  Every rank allocates a gather area, publishes its CUDA IPC handle, and
 * opens its peers' (ragfin_exchange_connect takes the `world` handles, RAGFIN_IPC_HANDLE_BYTES each, in rank order;
 * the caller moves them between processes, e.g. torch.distributed.all_gather_object, and runs a barrier after
 * connect and before destroy).  ragfin_exchange_allgather_merge then STORES this rank's exact hits {ids [nq,k] |
 * scores [nq,k]} into every peer's area, publishes a per-step flag (release, system scope) and reduces the `world`
 * records that arrived in its own area as soon as their flags are up (acquire) - two small kernels, no collective
 * library call.  All ranks must call it in the same order with the same (nq, k); nq*k*12 <= record_bytes_max. */
typedef struct ragfin_exchange ragfin_exchange_t;
#define RAGFIN_IPC_HANDLE_BYTES 64
int ragfin_exchange_create(ragfin_exchange_t** out, int32_t rank, int32_t world, int64_t record_bytes_max, int32_t device);
int ragfin_exchange_handle(ragfin_exchange_t* x, void* handle_out /* RAGFIN_IPC_HANDLE_BYTES */);
int ragfin_exchange_connect(ragfin_exchange_t* x, const void* handles /* world * RAGFIN_IPC_HANDLE_BYTES */);
int ragfin_exchange_allgather_merge(ragfin_exchange_t* x, const int64_t* ids_dev, const float* scores_dev, int32_t nq,
                                    int32_t k, int64_t* out_ids_dev, float* out_scores_dev, void* stream);
/* Whether a search of nq queries with limit k on this handle takes the one-kernel search (csrc/sweep_fused.cuh).  The
 * ranks of a sharded search must agree before they call ragfin_search_sharded (shard sizes differ by a row), so the host
 * layer reduces *out over the ranks once per (nq, k). */
int ragfin_fused_eligible(ragfin_t* h, int32_t nq, int32_t k, int32_t* out);

/* Row-sharded search in ONE kernel per GPU: this rank's shard is swept by the one-kernel search, whose finalizing CTAs store
 * the shard's exact hits into every rank's gather area over NVLink (the exchange's CUDA IPC mappings), wait for the other
 * ranks' hits and write the GLOBAL top-k into out_ids / out_scores on every rank - no collective call, no separate reduce
 * kernel.  Collective: every rank calls it once per step with the same (nq <= 64, k <= 128) and the same queries, always
 * on the same stream and with the same handle (one exchange serves one collection: its four-slot gather ring is safe because
 * a handle never has more than two searches in flight); fails with RAGFIN_EUNSUPPORTED when the shape does not take the
 * one-kernel search on this shard.
 * _host: host buffers, queries staged through pinned memory, hits written by the kernel into device-mapped pinned memory,
 * one stream synchronisation.
 * Replaces: the querynode -> proxy reduce behind Collection.search on a sharded Milvus deployment
 * (vector_rag_mcp/main.py:51-57; SURVEY.md 8e), i.e. local search + NCCL all-gather + ragfin_merge_topk. */
int ragfin_search_sharded(ragfin_t* h, ragfin_exchange_t* x, const float* q, int32_t nq, int32_t k, int64_t* out_ids,
                          float* out_scores, void* stream);
int ragfin_search_sharded_host(ragfin_t* h, ragfin_exchange_t* x, const float* q_host, int32_t nq, int32_t k,
                               int64_t* out_ids_host, float* out_scores_host);

void ragfin_exchange_destroy(ragfin_exchange_t* x);

/* Copy rows row0..row0+n of the STORED matrix, raw storage bytes [n, ld], to host memory
 * (test hook for ingest parity).  *ld_out receives the row stride in elements.  RAGFIN_F32_F16: the fp32 rows. */
int ragfin_read_rows(ragfin_t* h, int64_t row0, int64_t n, void* out_host, int32_t* ld_out);
/* Same for the rows the tensor-core sweeps read: the fp16 copy on a RAGFIN_F32_F16 handle ([n, ld] fp16), the stored
 * rows otherwise (test hook). */
int ragfin_read_sweep_rows(ragfin_t* h, int64_t row0, int64_t n, void* out_host, int32_t* ld_out);

/* Grouping search (Milvus' group_by_field, DESIGN.md 7d): the k best GROUPS, one hit per group.  Row r belongs to the
 * group group_of_row[r]: `count` int32 codes, one per stored row, passed per search like allow_bits (the handle keeps no
 * codes; ragfin_add, ragfin_compact and the file format are unchanged).
 *  - A group's score is the exact fp32 score of its best row: the largest (score desc, row asc) among its allowed, live
 *    rows.  The hit of a group is that row; hits are ordered (score desc, id asc) and slots past the number of non-empty
 *    groups hold (-1, -inf).
 *  - A row whose code lies outside [0, n_groups) is never returned (as if filtered out): codes need no validation pass.
 *  - allow_bits (NULL = every row) and tombstones compose as with ragfin_search_filtered.
 *  - codes[r] = r with n_groups = count is the plain search, bit for bit; a single group is the plain top-1.
 * Codes: ragfin_search_grouped takes device memory; ragfin_search_grouped_host takes host memory (copied in) or, with
 * groups_on_device = 1, device memory, so that a caller keeping the codes resident uploads nothing per search.  A NULL code
 * pointer or n_groups < 1 gives RAGFIN_EINVAL, checked before the handle.  ragfin_last_search_stats reports path 2, and
 * queries_rescanned counts queries that overflowed the batched route into the exact path.  No sharded form; grouping is
 * not combined with a range window.  Workspace: 16 * n_groups * 4 bytes next to the large-k route's score dump. */
int ragfin_search_grouped(ragfin_t* h, const float* q, int32_t nq, int32_t k, const int32_t* group_of_row_dev, int32_t n_groups,
                          const uint32_t* allow_bits_dev, int64_t n_allowed, int64_t* out_ids, float* out_scores, void* stream);
int ragfin_search_grouped_host(ragfin_t* h, const float* q_host, int32_t nq, int32_t k, const int32_t* group_of_row,
                               int32_t groups_on_device, int32_t n_groups, const uint32_t* allow_bits_host, int64_t n_allowed,
                               int64_t* out_ids_host, float* out_scores_host);

/* Counters of the most recent search on this handle: kernel launches issued, queries that
 * took the exact-rescan tier (certificate failed), which scoring path ran
 * (0 = small-batch scan, 1 = tcgen05 GEMM, 2 = large-k radix select).  Reading queries_rescanned synchronises. */
typedef struct {
    int32_t launches;
    int32_t path;
    int32_t queries_rescanned;
    int32_t cand_per_query;   /* K' : candidates kept per query before the exact rescore */
} ragfin_search_stats;
int ragfin_last_search_stats(ragfin_t* h, ragfin_search_stats* out);

/* Measurement hook: when enabled, every search records a CUDA event pair around its dominant
 * scoring kernel (the scan or the GEMM) on the launching stream.  ragfin_profile_read
 * synchronises, returns the summed kernel time and the number of timed launches since the last
 * read, and resets both.  Used by bench.py for the roofline figure; off by default. */
int ragfin_profile(ragfin_t* h, int32_t enable);
int ragfin_profile_read(ragfin_t* h, double* total_ms, int32_t* launches);

/* Persistence of the device-resident matrix (stands in for Milvus' flush()/load() durability,
 * "chunking_storing (1).py":395-396, retrieve.py:18-19).  File = 64-byte header {magic "RAGFINB2", version,
 * dim, ld, dtype, count, id_base} + the stored rows [count, ld] exactly as they sit in HBM.  A handle without tombstones
 * writes version 1; with tombstones, version 2: the tombstone count (int64) in the header's first spare bytes (offset 40)
 * and ceil(count / 32) live-mask words after the rows.  ragfin_load reads both versions.  So a
 * reloaded collection returns bit-identical results without re-normalising.  A RAGFIN_F32_F16 file has header dtype 3 and
 * holds the fp32 rows only; ragfin_load rebuilds the fp16 copy from them on the device (same bits as at ingest).
 * ragfin_load creates a new handle on `device` with room for max(capacity_rows, count) rows. */
int ragfin_save(ragfin_t* h, const char* path);
int ragfin_load(ragfin_t** out, const char* path, int64_t capacity_rows, int32_t device);

/* Dispatch knob: query batches of at least `min_nq` rows take the tcgen05 tensor-core path, smaller
 * ones the HBM-bound scan.  Default: 3, and 1 on corpora of >= 1 GiB (there the TMA-fed sweep is faster even for
 * one query: 2.16 vs 2.31 ms on 10M x 768 bf16, 0.340 vs 0.355 ms on 1.25M rows).  Setting it overrides both; 0 restores the defaults.  Both paths return identical results. */
int ragfin_set_gemm_min_batch(ragfin_t* h, int32_t min_nq);

/* Tuning knob: thread-block cluster size of the tcgen05 path along the query-tile axis (corpus tiles
 * are TMA-multicast across the cluster).  0 = automatic (default), else 1, 2 or 4. */
int ragfin_set_gemm_cluster(ragfin_t* h, int32_t cluster);

/* Tuning knob: tcgen05 kernel variant. 1 = streaming (query and corpus tiles through shared memory, any
 * dtype / width); 2 = A-stationary (query tile resident in tensor memory; 16-bit storage, dim <= 768; measured
 * slower); 3 = streaming, and batches of <= 16 queries in append mode run with the operand roles swapped (corpus
 * rows are the MMA's M dimension, the queries its N = 16: a sixteenth of the tensor work per byte, full SM clock);
 * 4 = batches of >= 2 query tiles in append mode sweep with a 2-SM MMA (tcgen05 cta_group::2, M = 256: each CTA of a
 * pair holds its own query tile and half of the corpus tile; csrc/gemm_pair.cuh).
 * 0 = automatic (default): 3 for <= 16 queries, 4 from 129 queries - measured interleaved on 10M x 768 bf16
 * (profiles/r02/policy_sweep.log) the 2-SM kernel beats the best single-CTA configuration at every batch from 129 to 4096
 * queries (4096: 45.3 vs 47.9 ms = 1 390 TFLOP/s).  Results are identical. */
int ragfin_set_gemm_variant(ragfin_t* h, int32_t variant);

/* Tuning knob: small-batch (1-2 query) scan kernel.  0 = automatic (default; currently 1), 1 = 128-bit register-path
 * loads (scan_topk_kernel), 2 = shared-memory ring filled by cp.async.bulk (scan_tma_kernel; measured no faster).
 * Results are identical. */
int ragfin_set_scan_variant(ragfin_t* h, int32_t variant);

/* Tuning knob: the tensor-core path first scores an evenly strided ~1 % sample of corpus tiles and seeds every
 * query's candidate threshold with the K'-th largest per-tile maximum (a valid lower bound of the global K'-th
 * score).  1 = on (default), 0 = off.  Results are identical; only the epilogue's bookkeeping cost changes. */
int ragfin_set_bound_pass(ragfin_t* h, int32_t enable);

/* Tuning knob: with the bound pass on, unfiltered searches over corpora of at least 1024 * k rows run the
 * tensor-core sweep in "append" mode: every row whose approximate score reaches (k-th largest sample maximum -
 * 2 * error bound) is appended to a per-query buffer, and the finalize step sorts, cuts at (k-th approximate score -
 * 2 * error bound) and rescans those rows exactly - exact by construction, no certificate.  1 = on (default),
 * 0 = per-query K' lists in shared memory + certificate.  Results are identical. */
int ragfin_set_append_mode(ragfin_t* h, int32_t enable);

/* Tuning knob: batches of <= 64 queries with k <= 128 over corpora of >= min_rows rows (default 8192) are answered by ONE
 * kernel (csrc/sweep_fused.cuh): query preparation, tensor-core sweep with self-tightening thresholds, exact finalize and
 * the exact fallback all inside it - no bound pass, no separate finalize, no gated launches.  1 = on (default), 0 = the
 * multi-kernel paths.  min_rows = 0 leaves the row limit unchanged.  Results are identical.
 * Replaces: the same Collection.search call sites; this is the batch-1 path of vector_rag_mcp/main.py:51-57. */
int ragfin_set_fused(ragfin_t* h, int32_t enable, int64_t min_rows);

/* Opt-in pipelining of consecutive one-kernel searches issued through ragfin_search / ragfin_search_sharded on ONE stream
 * (default off; RAGFIN_PIPELINED=1 turns it on for new handles): search n + 1 is launched with programmatic stream
 * serialization and starts sweeping while search n finalizes and exchanges hits; results land in stream order.  Contract: a
 * pipelined search may begin before the operation enqueued just ahead of it on the stream has completed, so its query buffer
 * must already hold the queries when the PREVIOUS search on this handle was enqueued (written by work ordered before that
 * search, or by the host).  Queries produced by a kernel enqueued between two searches need pipelining off.  Only a search
 * that directly follows this handle's own one-kernel search on the same stream is launched this way; after an add, a delete, a filter,
 * another path or another stream the launch is an ordinary one.  Results are identical either way.
 * Replaces: nothing in the reference (its searches are sequential gRPC calls - vector_rag_mcp/main.py:51-57). */
int ragfin_set_pipelined(ragfin_t* h, int32_t enable);

/* The one-kernel search's int8 tile filter on bf16 / fp16 collections (csrc/sweep_fused.cuh, DESIGN.md 2.5): tiles are first
 * swept from an int8 copy of the rows (half the bytes) with a rigorous bound on each row's 16-bit score, and read in 16 bits
 * only where some row can reach a query's threshold.  The copy ([capacity] x ceil16(dim) int8 + 8 bytes per row) is made
 * by the first one-kernel search that uses it and kept current by the searches after ragfin_add / ragfin_reserve /
 * ragfin_compact; files do not change.  mode 1 = on, 0 = off, RAGFIN_SWEEP_COPY_AUTO (default) = on from 2^20 rows.
 * Results are identical either way; a copy that cannot be allocated leaves the search on the 16-bit rows. */
#define RAGFIN_SWEEP_COPY_AUTO (-1)
int ragfin_set_sweep_copy(ragfin_t* h, int32_t mode);
/* Test hook: rows [row0, row0 + n) of the int8 copy, out_rows_host [n][*ld8_out] int8, and their {scale, residual bound},
 * out_side_host [n][2] float.  RAGFIN_EUNSUPPORTED when the collection has no copy.  Synchronises. */
int ragfin_debug_sweep_copy(ragfin_t* h, int64_t row0, int64_t n, int8_t* out_rows_host, float* out_side_host, int32_t* ld8_out);
/* Diagnostics of the last one-kernel search, out[2]: 256-row tiles read in 16 bits (every CTA's first tile and the refined
 * ones; without the int8 filter, all) and tiles screened from the int8 copy.  Synchronises. */
int ragfin_debug_fused_tiles(ragfin_t* h, int64_t* out);

/* Test / bench hook: per-query diagnostics of the last one-kernel search on this handle - rows appended to the query's
 * buffer during the sweep and rows rescored exactly by the finalize (-1: the buffer overflowed and the query was answered
 * by the in-kernel exact scan).  Synchronises. */
int ragfin_debug_fused_counts(ragfin_t* h, int32_t nq, int64_t* out_appended, int64_t* out_rescored);
/* Phase stamps of the last one-kernel search in ns since the kernel's start, out[16]: CTA 0 {start, prologue done, first tile
 * done, sweep done}, finalizer of query 0 {all CTAs arrived, hits selected, rescored, emitted}, then finer stamps {setup done,
 * norms done, count read, keys staged, T found} (csrc/sweep_fused.cuh FusedCtl::t).  Synchronises. */
int ragfin_debug_fused_times(ragfin_t* h, int64_t* out);
/* Test hook, no device needed: the order in which the one-kernel search visits the n_tiles tiles of a slice (out[n_tiles]); the
 * CPU suite checks that it is a permutation for every slice length (every tile scored exactly once) and starts mid-slice. */
int ragfin_debug_fused_tile_order(int32_t n_tiles, int32_t* out);
/* Per-CTA diagnostics of the last one-kernel search (arrays of 160): final threshold of query 0, rows appended for it. */
int ragfin_debug_fused_ctas(ragfin_t* h, float* out_thr, int32_t* out_app);

/* Test hook: raw (approximate, fp32-accumulated) tensor-core scores of nq queries against every
 * stored row, out_scores_dev [nq, count] device memory.  Validates the TMA / tcgen05 plumbing. */
int ragfin_debug_gemm_scores(ragfin_t* h, const float* q_dev, int32_t nq, float* out_scores_dev, void* stream);

/* Test hook, pure host arithmetic (needs no device): how the tcgen05 path would split a search of nq queries over
 * n_rows rows on a device with num_sms SMs - cluster size, query tiles, corpus slices, grid - and the geometry of its
 * sample ("bound") pass.  out[10] = {C, QT, S, rows_per_slice, grid, append_by_size, bound, nblk, g, bstride}.
 * The CPU suite checks the invariants exactness rests on: slices cover every row once, sample tiles are distinct and
 * never the last (partial) tile, at least 2 x rank sample blocks. */
int ragfin_debug_plan(int32_t nq, int64_t n_rows, int32_t num_sms, int32_t k, int32_t cluster, int64_t* out);
/* Test hook, pure host arithmetic (needs no device): the one-kernel search's plan for nq queries and top-k on a collection of
 * `dtype` (RAGFIN_F32 .. RAGFIN_F32_F16) and `dim`, under the query limits max_nq and max_nqk (0: the defaults, 16 queries and
 * queries x k <= 400; RAGFIN_FUSED_MAX_NQ / _NQK set them per handle) and the default ring depth.
 * out[5] = {ncol (0: the search takes another path), split (1: the query enters as hi + lo), stages, pend, cap};
 * out_eps[4] = {rel, sub, query term, eps_approx}: the per-element query-rounding bound |y - hi (- lo)| <= rel |y| + sub of the
 * planned variant (plain when none), the query term of eps it gives, and the rest of eps (accumulation allowance, tf32
 * truncation, fp16-copy rounding).  The kernel's eps is their sum, rounded up. */
int ragfin_debug_fused_plan(int32_t dtype, int32_t dim, int32_t nq, int32_t k, int32_t max_nq, int32_t max_nqk, int64_t* out,
                            double* out_eps);

/* A second handle over the SAME device matrix (no copy) with its own workspace: searches through the parent and the
 * view (or two views) may be in flight at once on different streams, so the latency-bound head and tail of one call
 * (query preparation, bound pass, finalize, exchange) overlap the neighbour's sweep.  Replaces nothing in the reference
 * (a Milvus querynode serves concurrent searches from one loaded segment the same way).  The view sees the rows present
 * when it is made (and the tombstones present then: it keeps its own copy of the mask), inherits the parent's tuning knobs,
 * is read-only (ragfin_add, ragfin_delete and ragfin_compact return RAGFIN_EUNSUPPORTED), blocks ragfin_compact on its parent
 * while it lives (ragfin_reserve of a parent with live views remains the caller's hazard) and must
 * be destroyed before its parent.  Measured (scripts/pipeline_check.py, profiles/r02): 1.25M-row shard, batch 1, three
 * handles on three streams: 0.284 ms per query against 0.327 ms on one handle. */
int ragfin_create_view(ragfin_t* parent, ragfin_t** out);

void ragfin_destroy(ragfin_t* h);

const char* ragfin_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* RAGFIN_H */
