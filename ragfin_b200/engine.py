"""Device-resident exact cosine top-k index: the Python face of the C ABI.

`Index` owns one handle (one GPU, one row shard).  Arrays go in and out as numpy (host) or
torch CUDA tensors (device); torch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import numpy as np

from . import _lib

# "f32+f16": fp32 rows (every exact step, so results equal "f32") plus an fp16 copy the tensor-core sweeps stream;
# 6 bytes per element (include/ragfin.h, RAGFIN_F32_F16)
DTYPE_CODE = {"f32": 0, "fp32": 0, "float32": 0, "bf16": 1, "bfloat16": 1, "f16": 2, "fp16": 2, "float16": 2, "f32+f16": 3}
_DTYPE_NAME = ("f32", "bf16", "f16", "f32+f16")   # by header code
MAX_TOPK = 16384  # Milvus' own limit on `limit`


def _stream_ptr(stream) -> int:
    if stream is None:
        import torch
        return int(torch.cuda.current_stream().cuda_stream)
    return int(getattr(stream, "cuda_stream", stream))


def _host_queries(queries, dim: int):
    """Host queries -> (object keeping the memory alive, address, nq).  numpy / lists go through numpy; a torch CPU tensor
    (e.g. pinned) is taken as it is when it is already fp32 and contiguous - `data_ptr()` costs a tenth of numpy's
    `.ctypes.data`, which matters once a whole 8-GPU search is 0.3 ms."""
    if hasattr(queries, "data_ptr"):
        import torch
        q = queries if queries.dim() != 1 else queries[None, :]
        if q.is_cuda or q.dtype != torch.float32 or not q.is_contiguous():
            q = q.detach().to("cpu", torch.float32).contiguous()
        if q.dim() != 2 or q.shape[1] != dim:
            raise ValueError(f"queries must be [nq, {dim}], got {tuple(q.shape)}")
        return q, q.data_ptr(), q.shape[0]
    q = np.ascontiguousarray(queries, dtype=np.float32)
    if q.ndim == 1:
        q = q[None, :]
    if q.ndim != 2 or q.shape[1] != dim:
        raise ValueError(f"queries must be [nq, {dim}], got {q.shape}")
    return q, q.ctypes.data, q.shape[0]


def _window(radius, range_filter):
    """Range-search bounds as the C ABI takes them (a ragfin_range): fp32 (round to nearest even), None = open (-inf / +inf).
    The library rejects a NaN bound and range_filter <= radius."""
    lo = -np.inf if radius is None else float(np.float32(radius))
    hi = np.inf if range_filter is None else float(np.float32(range_filter))
    return (ctypes.c_float * 2)(lo, hi)


def _host_out(out, nq: int, k: int, np_dtype, what: str):
    """Caller-owned result buffer (numpy array or torch CPU tensor, C-contiguous [nq, k]) or a fresh numpy one -> (obj, address)."""
    if out is None:
        out = np.empty((nq, k), dtype=np_dtype)
        return out, out.ctypes.data
    if hasattr(out, "data_ptr"):
        import torch
        want = torch.int64 if np_dtype is np.int64 else torch.float32
        if out.is_cuda or out.dtype != want or tuple(out.shape) != (nq, k) or not out.is_contiguous():
            raise ValueError(f"{what} must be a C-contiguous host {np.dtype(np_dtype).name} buffer of shape [nq, k]")
        return out, out.data_ptr()
    if out.shape != (nq, k) or out.dtype != np_dtype or not out.flags.c_contiguous:
        raise ValueError(f"{what} must be a C-contiguous host {np.dtype(np_dtype).name} buffer of shape [nq, k]")
    return out, out.ctypes.data


class Index:
    """Exact cosine top-k over a device-resident, L2-normalised embedding matrix.

    Mirrors what the reference gets from a loaded Milvus collection with a COSINE index
    (reference "chunking_storing (1).py":14-29, retrieve.py:17-19)."""

    def __init__(self, dim: int, dtype: str = "f32", capacity: int = 1 << 20, device: int = 0):
        if dtype not in DTYPE_CODE:
            raise ValueError(f"dtype must be one of {sorted(DTYPE_CODE)}, got {dtype!r}")
        self._L = _lib.load()
        self.dim, self.dtype, self.capacity, self.device = int(dim), dtype, int(capacity), int(device)
        h = ctypes.c_void_p()
        _lib.check(self._L.ragfin_create(ctypes.byref(h), self.dim, DTYPE_CODE[dtype], self.capacity, self.device))
        self._h = h

    # -- persistence -----------------------------------------------------------------
    def save(self, path: str) -> None:
        """Write the stored (normalised, rounded) matrix to `path`; `Index.load` restores it bit for bit."""
        _lib.check(self._L.ragfin_save(self._h, str(path).encode()))

    @classmethod
    def load(cls, path: str, capacity: int = 0, device: int = 0) -> "Index":
        L = _lib.load()
        h = ctypes.c_void_p()
        _lib.check(L.ragfin_load(ctypes.byref(h), str(path).encode(), int(capacity), int(device)))
        self = cls.__new__(cls)
        self._L, self._h, self.device = L, h, int(device)
        with open(path, "rb") as f:
            hd = f.read(64)
        self.dim = int.from_bytes(hd[12:16], "little")
        self.dtype = _DTYPE_NAME[int.from_bytes(hd[20:24], "little")]
        self.capacity = max(int(capacity), int.from_bytes(hd[24:32], "little", signed=True), 1)
        self._id_base = int.from_bytes(hd[32:40], "little", signed=True)
        return self

    def view(self) -> "Index":
        """A second handle over the same device matrix (no copy) with its own workspace: searches through `self` and the
        view may be in flight at once on different CUDA streams.  Read-only; sees the rows present now; keeps `self` alive."""
        h = ctypes.c_void_p()
        _lib.check(self._L.ragfin_create_view(self._h, ctypes.byref(h)))
        v = Index.__new__(Index)
        v._L, v._h, v._parent = self._L, h, self
        v.dim, v.dtype, v.device, v.capacity = self.dim, self.dtype, self.device, max(len(self), 1)
        v._id_base = getattr(self, "_id_base", 0)
        return v

    # -- lifecycle -------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None):
            self._L.ragfin_destroy(self._h)
            self._h = None
            self._parent = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self) -> int:
        n = ctypes.c_int64()
        _lib.check(self._L.ragfin_count(self._h, ctypes.byref(n)))
        return int(n.value)

    num_entities = property(__len__)

    # -- deletion --------------------------------------------------------------------
    def delete(self, ids) -> int:
        """Tombstone rows by the ids searches return; no search returns them afterwards.  Duplicates and rows deleted before
        are allowed; returns the number of rows this call deleted.  An out-of-range id raises and deletes nothing."""
        a = np.ascontiguousarray(np.asarray(ids, dtype=np.int64).reshape(-1))
        n = ctypes.c_int64()
        _lib.check(self._L.ragfin_delete(self._h, a.ctypes.data, a.size, ctypes.byref(n)))
        return int(n.value)

    @property
    def live_count(self) -> int:
        """Rows stored minus rows deleted (`len(self)` keeps counting the rows stored until `compact`)."""
        n = ctypes.c_int64()
        _lib.check(self._L.ragfin_live_count(self._h, ctypes.byref(n)))
        return int(n.value)

    def live_mask(self) -> np.ndarray:
        """bool [len(self)]: True where the row is live (read from the device mask the kernels use)."""
        n = len(self)
        words = np.zeros(max((n + 31) // 32, 1), np.uint32)
        _lib.check(self._L.ragfin_read_live_mask(self._h, words.ctypes.data))
        return np.unpackbits(words.view(np.uint8), bitorder="little")[:n].astype(bool)

    def compact(self) -> np.ndarray:
        """Remove the deleted rows from the device matrix; survivors keep their order and row r becomes the r-th survivor.
        Returns the surviving OLD ids in ascending order (new id i was old id out[i])."""
        survivors = np.flatnonzero(self.live_mask()).astype(np.int64) + getattr(self, "_id_base", 0)
        _lib.check(self._L.ragfin_compact(self._h))
        return survivors

    def reserve(self, capacity: int) -> None:
        """Grow the device matrix to at least `capacity` rows (device-to-device copy of the stored rows, bits unchanged)."""
        _lib.check(self._L.ragfin_reserve(self._h, int(capacity)))
        self.capacity = max(self.capacity, int(capacity))

    def set_id_base(self, base: int) -> None:
        _lib.check(self._L.ragfin_set_id_base(self._h, int(base)))
        self._id_base = int(base)

    # -- ingest (K1) -----------------------------------------------------------------
    def add(self, rows, stream=None) -> None:
        """Append fp32 rows [n, dim]: numpy / nested lists (host) or a torch CUDA tensor."""
        if hasattr(rows, "is_cuda"):
            import torch
            if not rows.is_cuda:
                rows = rows.numpy()
            else:
                if rows.dim() != 2 or rows.shape[1] != self.dim:
                    raise ValueError(f"rows must be [n, {self.dim}], got {tuple(rows.shape)}")
                if rows.device.index != self.device:
                    raise ValueError(f"rows live on cuda:{rows.device.index}, index on cuda:{self.device}")
                rows = rows.to(torch.float32).contiguous()
                with torch.cuda.device(self.device):
                    if stream is None:
                        stream = torch.cuda.current_stream()
                    elif not hasattr(stream, "synchronize"):      # a raw cudaStream_t
                        stream = torch.cuda.ExternalStream(int(stream))
                    _lib.check(self._L.ragfin_add(self._h, rows.data_ptr(), rows.shape[0], 1, _stream_ptr(stream)))
                    stream.synchronize()  # `rows` may be freed by the caller
                return
        a = np.ascontiguousarray(rows, dtype=np.float32)
        if a.ndim == 1:
            a = a[None, :]
        if a.ndim != 2 or a.shape[1] != self.dim:
            raise ValueError(f"rows must be [n, {self.dim}], got {a.shape}")
        _lib.check(self._L.ragfin_add(self._h, a.ctypes.data, a.shape[0], 0, None))

    def add_synthetic(self, seed: int, row0: int, n: int, dup_every: int = 0, zero_every: int = 0) -> None:
        _lib.check(self._L.ragfin_add_synthetic(self._h, seed, row0, n, dup_every, zero_every, None))

    def add_synthetic_topics(self, seed: int, row0: int, n: int, topic_rows: int, noise_shift: int = 3) -> None:
        """Templated-corpus generator (bench / tests): row r = centre(r // topic_rows) + noise(r) * 2**-noise_shift, see
        include/ragfin.h; `ragfin_b200.synthetic.synth_topic_rows` builds the same rows on the host."""
        _lib.check(self._L.ragfin_add_synthetic_topics(self._h, seed, row0, n, topic_rows, noise_shift, None))

    def read_rows(self, row0: int, n: int) -> np.ndarray:
        """Stored rows as fp32 values [n, dim] (test hook for ingest parity); the fp32 rows of an "f32+f16" index."""
        code = DTYPE_CODE[self.dtype]
        return self._read(self._L.ragfin_read_rows, 0 if code == 3 else code, row0, n)

    def read_sweep_rows(self, row0: int, n: int) -> np.ndarray:
        """The rows the tensor-core sweeps read, as fp32 values [n, dim] (test hook): the fp16 copy of an "f32+f16" index,
        the stored rows otherwise."""
        code = DTYPE_CODE[self.dtype]
        return self._read(self._L.ragfin_read_sweep_rows, 2 if code == 3 else code, row0, n)

    def _read(self, fn, code: int, row0: int, n: int) -> np.ndarray:
        ld = (self.dim + 7) // 8 * 8
        raw = np.empty((n, ld), dtype=np.float32 if code == 0 else np.uint16)
        ldo = ctypes.c_int32()
        _lib.check(fn(self._h, row0, n, raw.ctypes.data, ctypes.byref(ldo)))
        assert ldo.value == ld
        if code == 0:
            out = raw
        elif code == 1:
            out = (raw.astype(np.uint32) << np.uint32(16)).view(np.float32)
        else:
            out = raw.view(np.float16).astype(np.float32)
        assert not out[:, self.dim:].any(), "padding columns must be zero"
        return np.ascontiguousarray(out[:, :self.dim])

    # -- search ----------------------------------------------------------------------
    def _check_k(self, k: int) -> int:
        k = int(k)
        if not 1 <= k <= MAX_TOPK:
            raise ValueError(f"top_k must be in [1, {MAX_TOPK}], got {k}")
        return k

    def search(self, queries, k: int, out_ids: Optional[np.ndarray] = None,
               out_scores: Optional[np.ndarray] = None, allow: Optional[np.ndarray] = None,
               radius: Optional[float] = None, range_filter: Optional[float] = None,
               group_by=None, n_groups: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray]:
        """Host path: queries numpy / list / torch CPU tensor [nq, dim] -> (ids int64 [nq, k], scores fp32 [nq, k]).
        Hits are in descending score, ties to the lower id; slots past min(k, N) hold (-1, -inf).
        `out_ids` / `out_scores` may be caller-owned (e.g. pinned) C-contiguous numpy arrays or torch CPU tensors; they are
        returned as passed, fresh numpy arrays otherwise.
        `allow`: optional bool array [N]; only rows with allow[r] may be returned (scalar-filtered search).
        `radius` / `range_filter`: range search, only rows with radius < score <= range_filter (both rounded to fp32 with
        np.float32; None = open) may be returned, and slots past the rows in the window hold (-1, -inf).
        `group_by` / `n_groups`: grouping search, the k best groups with one hit each (the group's best row); `group_by` is
        row r's group code, int32 [N] as a numpy array (copied in) or a CUDA tensor (read in place).  Rows whose code lies
        outside [0, n_groups) are never returned; slots past the non-empty groups hold (-1, -inf).  Composes with `allow`,
        not with a range window."""
        k = self._check_k(k)
        grouped = self._check_groups(group_by, n_groups, radius, range_filter)
        q, qp, nq = _host_queries(queries, self.dim)
        ids, ip = _host_out(out_ids, nq, k, np.int64, "out_ids")
        scores, sp = _host_out(out_scores, nq, k, np.float32, "out_scores")
        if grouped is not None:
            codes, cp, on_device = grouped
            packed, n_allowed = self._pack_allow(allow) if allow is not None else (None, 0)
            _lib.check(self._L.ragfin_search_grouped_host(self._h, qp, nq, k, cp, on_device, int(n_groups),
                                                          packed.ctypes.data if packed is not None else None, n_allowed, ip, sp))
            return ids, scores
        if radius is not None or range_filter is not None:
            window = _window(radius, range_filter)
            packed, n_allowed = self._pack_allow(allow) if allow is not None else (None, 0)
            _lib.check(self._L.ragfin_search_range_host(self._h, qp, nq, k, window,
                                                        packed.ctypes.data if packed is not None else None, n_allowed, ip, sp))
            return ids, scores
        if allow is not None:
            packed, n_allowed = self._pack_allow(allow)
            _lib.check(self._L.ragfin_search_filtered_host(self._h, qp, nq, k, packed.ctypes.data, n_allowed, ip, sp))
            return ids, scores
        _lib.check(self._L.ragfin_search_host(self._h, qp, nq, k, ip, sp))
        return ids, scores

    def _check_groups(self, group_by, n_groups, radius, range_filter):
        """Grouping arguments -> None (plain search) or (object keeping the codes alive, address, on_device)."""
        if group_by is None:
            if n_groups is not None:
                raise ValueError("n_groups needs group_by")
            return None
        if radius is not None or range_filter is not None:
            raise ValueError("group_by cannot be combined with radius / range_filter")
        if n_groups is None or not 1 <= int(n_groups) <= np.iinfo(np.int32).max:
            raise ValueError(f"n_groups must be in [1, 2^31 - 1], got {n_groups!r}")
        n = len(self)
        if hasattr(group_by, "is_cuda") and group_by.is_cuda:
            import torch
            if group_by.dtype != torch.int32 or tuple(group_by.shape) != (n,):
                raise ValueError(f"group_by must be an int32 tensor of shape [{n}], got {group_by.dtype} {tuple(group_by.shape)}")
            if group_by.device.index != self.device:
                raise ValueError(f"group_by lives on cuda:{group_by.device.index}, index on cuda:{self.device}")
            g = group_by.contiguous()
            return g, g.data_ptr(), 1
        g = np.asarray(group_by.numpy() if hasattr(group_by, "numpy") else group_by)
        if g.dtype != np.int32 or g.shape != (n,):
            raise ValueError(f"group_by must be an int32 array of shape [{n}], got {g.dtype} {g.shape}")
        g = np.ascontiguousarray(g)
        if n == 0:
            g = np.zeros(1, np.int32)   # the library wants a non-NULL pointer; nothing is read
        return g, g.ctypes.data, 0

    def _pack_allow(self, allow):
        """bool [N] -> (ceil(N / 32) little-endian uint32 words, number of set bits), the allow_bits layout."""
        mask = np.ascontiguousarray(allow, dtype=bool)
        if mask.shape != (len(self),):
            raise ValueError(f"allow must be a bool array of shape [{len(self)}], got {mask.shape}")
        packed = np.packbits(mask, bitorder="little")
        packed = np.concatenate([packed, np.zeros((-len(packed)) % 4, np.uint8)]).view(np.uint32)
        if packed.size == 0:
            packed = np.zeros(1, np.uint32)
        return packed, int(mask.sum())

    def search_device(self, queries, k: int, out_ids=None, out_scores=None, stream=None,
                      radius: Optional[float] = None, range_filter: Optional[float] = None,
                      group_by=None, n_groups: Optional[int] = None):
        """Device path: `queries` is a torch CUDA fp32 tensor [nq, dim]; returns torch CUDA tensors.
        Asynchronous on the given (default: current) stream.  `radius` / `range_filter`: range search, as in search().
        `group_by` (CUDA int32 tensor [N]) / `n_groups`: grouping search, as in search()."""
        import torch
        k = self._check_k(k)
        if group_by is not None and not (hasattr(group_by, "is_cuda") and group_by.is_cuda):
            raise ValueError("search_device takes group_by as a CUDA int32 tensor")
        grouped = self._check_groups(group_by, n_groups, radius, range_filter)
        if not queries.is_cuda or queries.dtype != torch.float32 or queries.dim() != 2 or queries.shape[1] != self.dim:
            raise ValueError(f"queries must be a CUDA fp32 tensor [nq, {self.dim}]")
        queries = queries.contiguous()
        nq = queries.shape[0]
        if out_ids is None:
            out_ids = torch.empty((nq, k), dtype=torch.int64, device=queries.device)
        if out_scores is None:
            out_scores = torch.empty((nq, k), dtype=torch.float32, device=queries.device)
        with torch.cuda.device(self.device):
            if grouped is not None:
                _lib.check(self._L.ragfin_search_grouped(self._h, queries.data_ptr(), nq, k, grouped[1], int(n_groups), None, 0,
                                                         out_ids.data_ptr(), out_scores.data_ptr(), _stream_ptr(stream)))
                return out_ids, out_scores
            if radius is not None or range_filter is not None:
                _lib.check(self._L.ragfin_search_range(self._h, queries.data_ptr(), nq, k, _window(radius, range_filter), None, 0,
                                                       out_ids.data_ptr(), out_scores.data_ptr(), _stream_ptr(stream)))
                return out_ids, out_scores
            _lib.check(self._L.ragfin_search(self._h, queries.data_ptr(), nq, k, out_ids.data_ptr(),
                                             out_scores.data_ptr(), _stream_ptr(stream)))
        return out_ids, out_scores

    def set_gemm_min_batch(self, min_nq: int) -> None:
        """Query batches of at least `min_nq` rows use the tcgen05 path (0 restores the defaults: 3, and 1 on
        corpora of >= 1 GiB)."""
        _lib.check(self._L.ragfin_set_gemm_min_batch(self._h, int(min_nq)))

    def set_gemm_cluster(self, cluster: int) -> None:
        """Thread-block cluster size of the tcgen05 path (0 = automatic, else 1, 2 or 4)."""
        _lib.check(self._L.ragfin_set_gemm_cluster(self._h, int(cluster)))

    def set_gemm_variant(self, variant: int) -> None:
        """tcgen05 kernel variant: 0 automatic, 1 streaming, 2 A-stationary (query tile in tensor memory),
        3 streaming with swapped operand roles for batches of <= 16 queries, 4 2-SM MMA pairs (csrc/gemm_pair.cuh,
        tcgen05 cta_group::2; never chosen automatically)."""
        _lib.check(self._L.ragfin_set_gemm_variant(self._h, int(variant)))

    def set_bound_pass(self, enable: bool) -> None:
        """tcgen05 path: threshold-seeding sample pass on/off (default on; results identical)."""
        _lib.check(self._L.ragfin_set_bound_pass(self._h, 1 if enable else 0))

    def set_scan_variant(self, variant: int) -> None:
        """Small-batch scan kernel: 0 automatic, 1 register-path loads, 2 TMA-fed shared-memory ring."""
        _lib.check(self._L.ragfin_set_scan_variant(self._h, int(variant)))

    def set_fused(self, enable: bool, min_rows: int = 0) -> None:
        """One-kernel search for <= 64 queries, k <= 128 (csrc/sweep_fused.cuh) on/off (default on; results identical);
        min_rows > 0 also sets the smallest corpus it serves."""
        _lib.check(self._L.ragfin_set_fused(self._h, 1 if enable else 0, int(min_rows)))

    def set_pipelined(self, enable: bool) -> None:
        """Opt-in: consecutive one-kernel searches issued through `search_device` (or the sharded device call) on one stream
        overlap - the next one sweeps while this one finalizes; results land in stream order.  Contract (include/ragfin.h,
        ragfin_set_pipelined): the query tensor must already hold its values when the PREVIOUS search on this index was
        issued - do not enable it when a kernel enqueued between two searches produces the queries.  Default off."""
        _lib.check(self._L.ragfin_set_pipelined(self._h, 1 if enable else 0))

    def set_sweep_copy(self, mode) -> None:
        """The one-kernel search's int8 tile filter (bf16 / fp16): True = on, False = off, "auto" (default) = on from 2^20
        rows.  Results are identical; the int8 copy of the rows is made by the first search that uses it."""
        m = -1 if mode == "auto" else (1 if mode else 0)
        _lib.check(self._L.ragfin_set_sweep_copy(self._h, m))

    def sweep_copy_rows(self, row0: int, n: int):
        """Rows [row0, row0 + n) of the int8 copy: (int8 [n, ld8], float32 [n, 2] = per-row scale and residual bound)."""
        ld8 = ctypes.c_int32(0)
        _lib.check(self._L.ragfin_debug_sweep_copy(self._h, int(row0), 0, None, None, ctypes.byref(ld8)))
        rows = np.zeros((n, ld8.value), np.int8)
        side = np.zeros((n, 2), np.float32)
        _lib.check(self._L.ragfin_debug_sweep_copy(self._h, int(row0), int(n), rows.ctypes.data, side.ctypes.data, ctypes.byref(ld8)))
        return rows, side

    def fused_tiles(self):
        """Tiles of the last one-kernel search: (read in 16 bits, screened from the int8 copy)."""
        out = np.zeros(2, np.int64)
        _lib.check(self._L.ragfin_debug_fused_tiles(self._h, out.ctypes.data))
        return int(out[0]), int(out[1])

    def fused_eligible(self, nq: int, k: int) -> bool:
        """Whether (nq, k) takes the one-kernel search on this handle (csrc/sweep_fused.cuh)."""
        out = ctypes.c_int32()
        _lib.check(self._L.ragfin_fused_eligible(self._h, int(nq), int(k), ctypes.byref(out)))
        return bool(out.value)

    def fused_counts(self, nq: int):
        """Diagnostics of the last one-kernel search: (rows appended per query, rows rescored per query; -1 = exact scan)."""
        a, r = np.zeros(nq, np.int64), np.zeros(nq, np.int64)
        _lib.check(self._L.ragfin_debug_fused_counts(self._h, int(nq), a.ctypes.data, r.ctypes.data))
        return a, r

    def fused_ctas(self):
        """Per-CTA diagnostics of the last one-kernel search: (final threshold of query 0, rows appended for it), 160 slots."""
        t, c = np.zeros(160, np.float32), np.zeros(160, np.int32)
        _lib.check(self._L.ragfin_debug_fused_ctas(self._h, t.ctypes.data, c.ctypes.data))
        return t, c

    def fused_times(self):
        """Phase stamps of the last one-kernel search (us since kernel start): start, prologue, first tile, sweep end (CTA 0);
        all arrived, selected, rescored, emitted (finalizer of query 0); entries 13-15: CTA 0's epilogue summed over its tiles -
        waiting for the tensor core, append pass, bookkeeping."""
        t = np.zeros(16, np.int64)
        _lib.check(self._L.ragfin_debug_fused_times(self._h, t.ctypes.data))
        return (t / 1e3).round(1).tolist()

    def set_append_mode(self, enable: bool) -> None:
        """tcgen05 path: append mode (no lists, threshold from the bound pass) on/off (default on; results identical)."""
        _lib.check(self._L.ragfin_set_append_mode(self._h, 1 if enable else 0))

    def debug_gemm_scores(self, queries):
        """Test hook: raw tensor-core scores [nq, N] (torch CUDA fp32) of CUDA fp32 queries [nq, dim]."""
        import torch
        queries = queries.contiguous()
        out = torch.empty((queries.shape[0], len(self)), dtype=torch.float32, device=queries.device)
        with torch.cuda.device(self.device):
            _lib.check(self._L.ragfin_debug_gemm_scores(self._h, queries.data_ptr(), queries.shape[0], out.data_ptr(),
                                                        _stream_ptr(None)))
        return out

    def profile(self, enable: bool = True) -> None:
        """Record CUDA events around the dominant scoring kernel of every search (bench.py)."""
        _lib.check(self._L.ragfin_profile(self._h, 1 if enable else 0))

    def profile_read(self):
        """(summed kernel ms, timed launches) since the last read; synchronises."""
        ms, n = ctypes.c_double(), ctypes.c_int32()
        _lib.check(self._L.ragfin_profile_read(self._h, ctypes.byref(ms), ctypes.byref(n)))
        return float(ms.value), int(n.value)

    def stats(self) -> dict:
        s = _lib.SearchStats()
        _lib.check(self._L.ragfin_last_search_stats(self._h, ctypes.byref(s)))
        return {"launches": s.launches, "path": s.path, "queries_rescanned": s.queries_rescanned,
                "cand_per_query": s.cand_per_query}


def fused_plan(dtype: str, dim: int, nq: int, k: int, max_nq: int = 0, max_nqk: int = 0) -> dict:
    """What the one-kernel search does for nq queries and top-k on a `dtype` collection of `dim` (no device needed; include/
    ragfin.h, ragfin_debug_fused_plan): ncol (0: another path serves the shape), split (the query enters as hi + lo), stages,
    pend, cap, and its eps split into the per-element query-rounding bound rel |y| + sub, the query term and eps_approx.
    max_nq / max_nqk: the handle's query limits (0: the defaults)."""
    L = _lib.load()
    out, eps = (ctypes.c_int64 * 5)(), (ctypes.c_double * 4)()
    _lib.check(L.ragfin_debug_fused_plan(DTYPE_CODE[dtype], int(dim), int(nq), int(k), int(max_nq), int(max_nqk), out, eps))
    plan = dict(zip(("ncol", "split", "stages", "pend", "cap"), (int(v) for v in out)))
    plan.update(zip(("rel", "sub", "eps_query", "eps_approx"), (float(v) for v in eps)))
    return plan


def merge_topk(ids, scores, parts: int, k: int, stream=None, out_ids=None, out_scores=None):
    """Cross-shard reduce of exact hit lists (torch CUDA tensors, ids int64 / scores fp32).

    Accepts either the all-gather layout [parts, nq, k] or a concatenation [nq, parts*k]."""
    import torch
    ids, scores = ids.contiguous(), scores.contiguous()
    if ids.dim() == 3:
        assert ids.shape[0] == parts and ids.shape[2] == k and scores.shape == ids.shape
        nq, part_stride, query_stride = ids.shape[1], ids.shape[1] * k, k
    else:
        nq = ids.shape[0]
        assert ids.shape == (nq, parts * k) and scores.shape == ids.shape
        part_stride, query_stride = k, parts * k
    return _merge_raw(ids.data_ptr(), scores.data_ptr(), nq, parts, k, part_stride, part_stride, query_stride,
                      ids.device, stream, out_ids, out_scores)


def _merge_raw(ids_ptr, scores_ptr, nq, parts, k, ids_ps, scores_ps, qs, device, stream=None, out_ids=None, out_scores=None):
    import torch
    L = _lib.load()
    if out_ids is None:
        out_ids = torch.empty((nq, k), dtype=torch.int64, device=device)
    if out_scores is None:
        out_scores = torch.empty((nq, k), dtype=torch.float32, device=device)
    _lib.check(L.ragfin_merge_topk(ids_ptr, scores_ptr, nq, parts, k, ids_ps, scores_ps, qs,
                                   out_ids.data_ptr(), out_scores.data_ptr(), device.index, _stream_ptr(stream)))
    return out_ids, out_scores


class PackedHits:
    """One byte buffer per rank holding {ids int64 [nq, k] | scores fp32 [nq, k]} (padded to 16 B) so that the
    cross-shard exchange is a single all-gather; `gathered` is the [world, record] receive buffer."""

    def __init__(self, nq: int, k: int, world: int, device):
        import torch
        self.nq, self.k, self.world = nq, k, world
        self.record = (nq * k * 12 + 15) // 16 * 16
        self.local = torch.empty(self.record, dtype=torch.uint8, device=device)
        self.gathered = torch.empty(world * self.record, dtype=torch.uint8, device=device)
        self.ids = self.local[: nq * k * 8].view(torch.int64).view(nq, k)
        self.scores = self.local[nq * k * 8: nq * k * 12].view(torch.float32).view(nq, k)

    def merge(self, stream=None):
        base = self.gathered.data_ptr()
        return _merge_raw(base, base + self.nq * self.k * 8, self.nq, self.world, self.k, self.record // 8,
                          self.record // 4, self.k, self.gathered.device, stream)


class PeerExchange:
    """Cross-shard exchange over NVLink peer memory (include/ragfin.h, ragfin_exchange_*): each rank stores its hit record
    into every peer's gather area through CUDA IPC mappings and reduces what arrived in its own - two small kernels
    instead of an NCCL all-gather + reduce.  One process per GPU of ONE box; construction is collective over `group`
    (handles travel through torch.distributed) and raises on every rank if any rank cannot map its peers."""

    def __init__(self, device: int, max_record_bytes: int = 8 << 20, group=None):
        import torch
        import torch.distributed as dist
        self._L = _lib.load()
        self.device = int(device)
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.max_record_bytes = int(max_record_bytes)
        self._x = ctypes.c_void_p()
        ok, err = 1, ""
        try:
            _lib.check(self._L.ragfin_exchange_create(ctypes.byref(self._x), self.rank, self.world, self.max_record_bytes, self.device))
            mine = ctypes.create_string_buffer(64)
            _lib.check(self._L.ragfin_exchange_handle(self._x, mine))
            payload = bytes(mine.raw)
        except Exception as e:   # noqa: BLE001 - reported collectively below
            ok, err, payload = 0, str(e), b""
        handles = [None] * self.world
        dist.all_gather_object(handles, payload, group=group)
        if ok and all(len(h) == 64 for h in handles):
            try:
                _lib.check(self._L.ragfin_exchange_connect(self._x, b"".join(handles)))
            except Exception as e:   # noqa: BLE001
                ok, err = 0, str(e)
        else:
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device=torch.device("cuda", self.device))
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)   # also the barrier after connect
        if int(flag.item()) != 1:
            self.close()
            raise RuntimeError(f"peer-memory exchange unavailable on at least one rank ({err or 'a peer failed'})")

    def allgather_merge(self, ids, scores, stream=None):
        """ids int64 [nq, k], scores fp32 [nq, k] (this rank's exact hits, CUDA) -> global (ids, scores) [nq, k]."""
        import torch
        nq, k = ids.shape
        out_ids = torch.empty((nq, k), dtype=torch.int64, device=ids.device)
        out_scores = torch.empty((nq, k), dtype=torch.float32, device=ids.device)
        _lib.check(self._L.ragfin_exchange_allgather_merge(self._x, ids.data_ptr(), scores.data_ptr(), nq, k,
                                                           out_ids.data_ptr(), out_scores.data_ptr(), _stream_ptr(stream)))
        return out_ids, out_scores

    def search_sharded(self, index, queries, k: int, out_ids=None, out_scores=None, stream=None):
        """Row-sharded search in one kernel per GPU (ragfin_search_sharded): `queries` CUDA fp32 [nq, dim], the same on
        every rank; returns the GLOBAL (ids, scores) [nq, k] on every rank.  Collective over the exchange's ranks."""
        import torch
        if not queries.is_cuda or queries.dtype != torch.float32 or queries.dim() != 2 or queries.shape[1] != index.dim:
            raise ValueError(f"queries must be a CUDA fp32 tensor [nq, {index.dim}]")
        nq = queries.shape[0]
        if out_ids is None:
            out_ids = torch.empty((nq, k), dtype=torch.int64, device=queries.device)
        if out_scores is None:
            out_scores = torch.empty((nq, k), dtype=torch.float32, device=queries.device)
        queries = queries.contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self._L.ragfin_search_sharded(index._h, self._x, queries.data_ptr(), nq, int(k), out_ids.data_ptr(),
                                                     out_scores.data_ptr(), _stream_ptr(stream)))
        return out_ids, out_scores

    def search_sharded_host(self, index, queries, k: int, out_ids=None, out_scores=None):
        """Same through host buffers (numpy in, numpy out, synchronous): ragfin_search_sharded_host."""
        k = int(k)
        q, qp, nq = _host_queries(queries, index.dim)
        ids, ip = _host_out(out_ids, nq, k, np.int64, "out_ids")
        scores, sp = _host_out(out_scores, nq, k, np.float32, "out_scores")
        _lib.check(self._L.ragfin_search_sharded_host(index._h, self._x, qp, nq, k, ip, sp))
        return ids, scores

    def close(self):
        if getattr(self, "_x", None) is not None and self._x:
            self._L.ragfin_exchange_destroy(self._x)
            self._x = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:   # noqa: BLE001
            pass
