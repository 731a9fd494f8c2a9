"""CPU oracle for rag-fin's vector-RAG hot path: exact cosine top-k.

TEST INFRASTRUCTURE ONLY.  Nothing in the shipped package (``ragfin_b200/``) may
import this module; only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` do, and only as the
checker or the timed CPU baseline.

PARITY UNPINNED.  The reference never computes a similarity itself: every call
site hands the query embedding to an external Milvus server through
``pymilvus==2.3.0`` (reference ``vector_rag_mcp/requirements.txt:2``), whose code
is not under /root/reference and is not installed in this image.  The call sites
this module restates are

  * ``retrieve.py:26-47``            SimpleRAG.search_and_answer (search + hit unpack)
  * ``vector_rag_mcp/main.py:48-70`` VectorRAG.search
  * ``chunking_storing (1).py:399-424`` search_financial_query; schema ``:14-22``,
    index ``IVF_FLAT / COSINE / nlist=128`` ``:29``, column-major insert ``:383-396``
  * ``graph_cons.py:272-293``        hybrid_query_simple (limit=1000)

and the reference holds no test, golden vector or fixture that pins a score or
a ranking at that boundary (``test_vector.py`` only prints).  The published
algorithm restated here is Milvus/knowhere brute-force COSINE (what the
reference gets on its 16-row collection, below the IVF build threshold):

  score(q, x) = <q, x> / (|q| |x|);  larger is better;  return min(k, N) hits in
  descending score; equal scores resolve to the smaller primary key, which for
  insertion-ordered keys is the lower row ordinal.

Canonical arithmetic (shared bit-for-bit by this file, ``ragfin_oracle.c`` and
the CUDA rescore kernel) so that "bit-exact" is a property and not luck:

  * LANES = 32 partial sums; partial p accumulates, in increasing i, the terms
    with i % 32 == p, in IEEE fp64.  Every term is a product of two values that
    are exactly representable in fp32 (24-bit significands), so the product is
    exact in fp64 and an fma equals multiply-then-add.
  * The 32 partials are folded by a butterfly: 16, 8, 4, 2, 1
    (v[p] = v[p] + v[p ^ off]); fp64 addition is commutative, so every lane
    holds the same value.
  * Row normalisation: n2 = canonical sum of squares; stored = RNE_storage(
    RNE_fp32(double(x) * (1 / sqrt(n2)))); a zero row stays zero (score 0).
    A row with any NaN or +-Inf component (n2 NaN or +inf) is stored as a zero
    row: inv = 0, and the NaN of Inf * 0 or NaN * 0 becomes +0.
    bf16 / fp16 storage rounds the fp32 value once more (RNE).
  * Query normalisation: same, to fp32.
  * score = RNE_fp32(canonical_dot(stored_row, q_hat)) + 0.0f   (kills -0).
  * order: (-score_fp32, +row_id).
"""
from __future__ import annotations

import numpy as np

LANES = 32
DTYPES = ("f32", "bf16", "f16")
DTYPE_CODE = {"f32": 0, "bf16": 1, "f16": 2}
ITEMSIZE = {"f32": 4, "bf16": 2, "f16": 2}

# ----------------------------------------------------------------------------
# deterministic synthetic data (SURVEY.md §8d): counter-based hash -> sum of four
# 16-bit uniforms, centred, scaled by 2^-16.  Every value is an 18-bit integer
# times 2^-16, hence exact in fp32 (and identical on CPU and GPU).
# ----------------------------------------------------------------------------
_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _mix64(z: np.ndarray) -> np.ndarray:
    """splitmix64 output function (Steele, Lea, Flood 2014) on uint64 arrays."""
    with np.errstate(over="ignore"):
        z = (z + np.uint64(0x9E3779B97F4A7C15)) & _M64
        z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M64
        z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M64
        return z ^ (z >> np.uint64(31))


def synth_source_row(rows: np.ndarray, dup_every: int) -> np.ndarray:
    """Adversarial duplicates: row r with r % dup_every == dup_every-1 repeats row r-1."""
    rows = np.asarray(rows, dtype=np.uint64)
    if dup_every and dup_every > 1:
        is_dup = (rows % np.uint64(dup_every)) == np.uint64(dup_every - 1)
        rows = np.where(is_dup, rows - np.uint64(1), rows)
    return rows


def synth_rows(seed: int, row0: int, n: int, dim: int, dup_every: int = 0,
               zero_every: int = 0) -> np.ndarray:
    """fp32 [n, dim] block of the synthetic matrix with the given seed, rows row0..row0+n."""
    rows = np.arange(row0, row0 + n, dtype=np.uint64)
    src = synth_source_row(rows, dup_every)
    cols = np.arange(dim, dtype=np.uint64)
    with np.errstate(over="ignore"):
        ctr = src[:, None] * np.uint64(dim) + cols[None, :]
        key = _mix64(np.asarray([seed], dtype=np.uint64))[0]
        h = _mix64(ctr ^ key)
    s = ((h & np.uint64(0xFFFF)) + ((h >> np.uint64(16)) & np.uint64(0xFFFF))
         + ((h >> np.uint64(32)) & np.uint64(0xFFFF)) + (h >> np.uint64(48)))
    out = (s.astype(np.int64) - 131070).astype(np.float32) * np.float32(2.0 ** -16)
    if zero_every and zero_every > 1:
        z = (rows % np.uint64(zero_every)) == np.uint64(zero_every - 1)
        out[z] = 0.0
    return out


# ----------------------------------------------------------------------------
# storage rounding
# ----------------------------------------------------------------------------
def f32_to_bf16_bits(x: np.ndarray) -> np.ndarray:
    """RNE fp32 -> bf16, returned as uint16 bit patterns (no NaN handling needed)."""
    b = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    r = (b + np.uint32(0x7FFF) + ((b >> np.uint32(16)) & np.uint32(1))) >> np.uint32(16)
    return r.astype(np.uint16)


def bf16_bits_to_f32(b: np.ndarray) -> np.ndarray:
    return (np.ascontiguousarray(b, dtype=np.uint16).astype(np.uint32) << np.uint32(16)).view(np.float32)


def round_to_storage(x32: np.ndarray, dtype: str) -> np.ndarray:
    """fp32 -> the fp32 value of what the given storage type holds (RNE)."""
    x32 = np.ascontiguousarray(x32, dtype=np.float32)
    if dtype == "f32":
        return x32
    if dtype == "bf16":
        return bf16_bits_to_f32(f32_to_bf16_bits(x32))
    if dtype == "f16":
        return x32.astype(np.float16).astype(np.float32)
    raise ValueError(f"unknown storage dtype {dtype!r}")


def storage_bits(x32: np.ndarray, dtype: str) -> np.ndarray:
    """fp32 (already storage-exact) -> raw storage array as the device holds it."""
    if dtype == "f32":
        return np.ascontiguousarray(x32, dtype=np.float32)
    if dtype == "bf16":
        return f32_to_bf16_bits(x32)
    if dtype == "f16":
        return np.ascontiguousarray(x32, dtype=np.float32).astype(np.float16)
    raise ValueError(dtype)


# ----------------------------------------------------------------------------
# canonical fp64 reductions
# ----------------------------------------------------------------------------
def _canonical_fold(prod64: np.ndarray) -> np.ndarray:
    """prod64: [..., D] fp64 exact products -> [...] canonical sum."""
    d = prod64.shape[-1]
    pad = (-d) % LANES
    if pad:
        prod64 = np.concatenate(
            [prod64, np.zeros(prod64.shape[:-1] + (pad,), dtype=np.float64)], axis=-1)
    steps = prod64.shape[-1] // LANES
    p = prod64.reshape(prod64.shape[:-1] + (steps, LANES))
    acc = np.zeros(prod64.shape[:-1] + (LANES,), dtype=np.float64)
    for j in range(steps):                      # sequential, increasing i
        acc = acc + p[..., j, :]
    off = LANES // 2
    while off >= 1:                             # butterfly 16, 8, 4, 2, 1
        acc = acc[..., :off] + acc[..., off:2 * off]
        off //= 2
    return acc[..., 0]


def canonical_sumsq(x32: np.ndarray) -> np.ndarray:
    x = np.asarray(x32, dtype=np.float32).astype(np.float64)
    return _canonical_fold(x * x)


def canonical_dot(rows32: np.ndarray, q32: np.ndarray) -> np.ndarray:
    """rows32 [n, D] fp32-exact stored values, q32 [D] fp32 -> fp64 [n]."""
    r = np.asarray(rows32, dtype=np.float32).astype(np.float64)
    q = np.asarray(q32, dtype=np.float32).astype(np.float64)
    return _canonical_fold(r * q[None, :])


def normalize_rows(x32: np.ndarray, dtype: str = "f32") -> np.ndarray:
    """Ingest normalisation; returns the fp32 VALUES of the stored rows.

    Restates the unit-norm step that COSINE implies for
    ``chunking_storing (1).py:380-394`` (encode -> insert).
    """
    x32 = np.ascontiguousarray(x32, dtype=np.float32)
    if x32.ndim == 1:
        x32 = x32[None, :]
    n2 = canonical_sumsq(x32)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        inv = np.where((n2 > 0.0) & np.isfinite(n2), 1.0 / np.sqrt(n2), 0.0)
        y = (x32.astype(np.float64) * inv[:, None]).astype(np.float32)
    y[np.isnan(y)] = 0.0                     # Inf * 0 and NaN * 0 in a non-finite row: stored as +0
    return round_to_storage(y, dtype)


def exact_scores(stored32: np.ndarray, qhat32: np.ndarray) -> np.ndarray:
    """fp32 scores of one normalised query against stored rows (canonical)."""
    s = canonical_dot(stored32, qhat32).astype(np.float32)
    return s + np.float32(0.0)


def cosine_topk(queries32: np.ndarray, stored32: np.ndarray, k: int, block: int = 8192,
                id_base: int = 0):
    """Exact top-k of every query over the stored (already normalised) rows.

    Restates ``Collection.search(data, "embedding", {"metric_type": "COSINE"}, k)``
    as used at ``vector_rag_mcp/main.py:51-57``.  Returns ids int64 [nq, k] and
    scores fp32 [nq, k], padded with id=-1 / score=-inf when k > N.
    """
    q = np.ascontiguousarray(queries32, dtype=np.float32)
    if q.ndim == 1:
        q = q[None, :]
    qhat = normalize_rows(q, "f32")
    n = stored32.shape[0]
    nq = q.shape[0]
    ids = np.full((nq, k), -1, dtype=np.int64)
    scores = np.full((nq, k), -np.inf, dtype=np.float32)
    for qi in range(nq):
        s = np.empty(n, dtype=np.float32)
        for b0 in range(0, n, block):
            s[b0:b0 + block] = exact_scores(stored32[b0:b0 + block], qhat[qi])
        order = np.lexsort((np.arange(n), -s.astype(np.float64)))[:k]
        m = order.shape[0]
        ids[qi, :m] = order + id_base
        scores[qi, :m] = s[order]
    return ids, scores


def merge_topk(ids_list, scores_list, k: int):
    """Merge per-shard (ids, scores) lists: the cross-segment reduce (SURVEY §2a)."""
    ids = np.concatenate(ids_list, axis=1)
    sc = np.concatenate(scores_list, axis=1)
    nq = ids.shape[0]
    out_i = np.full((nq, k), -1, dtype=np.int64)
    out_s = np.full((nq, k), -np.inf, dtype=np.float32)
    for qi in range(nq):
        valid = ids[qi] >= 0
        vi, vs = ids[qi][valid], sc[qi][valid]
        order = np.lexsort((vi, -vs.astype(np.float64)))[:k]
        out_i[qi, :order.shape[0]] = vi[order]
        out_s[qi, :order.shape[0]] = vs[order]
    return out_i, out_s
