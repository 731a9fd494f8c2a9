"""pymilvus-shaped front end over the B200 engine: the reference's operator API for the hot path.

The reference reaches its vector store only through this subset of pymilvus 2.3.0
(reference vector_rag_mcp/requirements.txt:2); each name below behaves like the pymilvus
object the reference uses, so a maintainer switches with

    from ragfin_b200.milvus_compat import connections, Collection, CollectionSchema, FieldSchema, DataType, utility

  connections.connect                      retrieve.py:17, vector_rag_mcp/main.py:43, "chunking_storing (1).py":11
  FieldSchema / CollectionSchema / DataType  "chunking_storing (1).py":14-28
  utility.has_collection / drop_collection  "chunking_storing (1).py":25-26
  Collection(name[, schema])               retrieve.py:18, "chunking_storing (1).py":28
  .create_index(field, params)             "chunking_storing (1).py":29      (metric must be COSINE)
  .insert(column-major data)               "chunking_storing (1).py":383-394
  .flush() / .load()                       "chunking_storing (1).py":395-396, retrieve.py:19
  .num_entities                            vector_rag_mcp/main.py:113,120,164, test_vector.py:29
  .search(data, anns_field, param, limit, output_fields=)   retrieve.py:28-34, vector_rag_mcp/main.py:51-57,
                                           "chunking_storing (1).py":411-417, graph_cons.py:275-281
  .search(..., {"metric_type": "COSINE", "params": {"radius": r, "range_filter": f}}, limit)   range search: at most
                                           `limit` hits with r < score <= f, best first (pymilvus 2.3; both bounds are
                                           rounded to fp32 and compared with the fp32 scores; range_filter needs radius)
  .query(expr, output_fields=, limit=)     test_vector.py:35-39, graph_cons.py:308-311
  .delete(expr) / .upsert(data) / .compact()   keeping a corpus current: restated filings, re-cut chunks, withdrawn
                                           documents (pymilvus 2.3 names; not called by the reference itself)

Hits expose .id, .distance, .score, .entity.<field> and .entity.get(field) exactly as the
call sites read them (retrieve.py:39-43, graph_cons.py:287-292).  Scalar columns live on the
host; only the embedding column goes to the GPU.  Row id = insertion ordinal; equal scores
resolve to the earlier-inserted row (SURVEY.md 8c).  delete() tombstones rows (the engine's search never returns them);
num_entities keeps counting them, as Milvus does, until compact() removes them and renumbers the survivors.

The engine is exact: index_type / nlist / nprobe (and the other keys of a search's "params" but radius and range_filter)
are accepted and ignored.
"""
from __future__ import annotations

import re
import threading
from enum import IntEnum
from typing import Any, Callable, Dict, List, Optional, Sequence

import numpy as np

MAX_LIMIT = 16384  # Milvus' cap on `limit`


class MilvusException(Exception):
    """Mirror of pymilvus.exceptions.MilvusException (code, message)."""

    def __init__(self, code: int = 1, message: str = ""):
        super().__init__(f"<MilvusException: (code={code}, message={message})>")
        self.code, self.message = code, message


class SchemaNotReadyException(MilvusException):
    pass


class ParamError(MilvusException):
    pass


def _refuse_non_finite(vectors: np.ndarray, what: str) -> None:
    """Milvus refuses float vectors holding NaN or +-Inf.  The engine would treat such a vector as the zero vector
    (include/ragfin.h), a silent answer for what is almost always a broken embedding, so the shim refuses host data.
    CUDA tensors are not checked: that would cost a pass and a synchronisation, and the engine's rule holds for them."""
    bad = ~np.isfinite(vectors)
    if bad.any():
        row = int(np.argwhere(bad)[0][0])
        raise MilvusException(message=f"{what}: vector {row} holds NaN or Inf; float vectors must be finite")


class DataType(IntEnum):
    NONE = 0
    BOOL = 1
    INT8 = 2
    INT16 = 3
    INT32 = 4
    INT64 = 5
    FLOAT = 10
    DOUBLE = 11
    STRING = 20
    VARCHAR = 21
    JSON = 23
    BINARY_VECTOR = 100
    FLOAT_VECTOR = 101


class FieldSchema:
    def __init__(self, name: str, dtype: DataType, description: str = "", **kwargs):
        self.name, self.dtype, self.description = name, DataType(dtype), description
        self.is_primary = bool(kwargs.get("is_primary", False))
        self.auto_id = bool(kwargs.get("auto_id", False))
        self.max_length = kwargs.get("max_length")
        self.dim = kwargs.get("dim")
        self.params = {k: v for k, v in kwargs.items() if k in ("max_length", "dim")}
        if self.dtype == DataType.FLOAT_VECTOR and (not isinstance(self.dim, int) or self.dim < 1):
            raise ParamError(message=f"FLOAT_VECTOR field {name!r} needs dim >= 1")

    def __repr__(self):
        return f"FieldSchema({self.name!r}, {self.dtype.name}, {self.params})"


class CollectionSchema:
    def __init__(self, fields: Sequence[FieldSchema], description: str = "", **kwargs):
        self.fields, self.description = list(fields), description
        names = [f.name for f in self.fields]
        if len(set(names)) != len(names):
            raise ParamError(message="duplicate field names")
        prim = [f for f in self.fields if f.is_primary]
        if len(prim) != 1:
            raise SchemaNotReadyException(message="exactly one primary field is required")
        vec = [f for f in self.fields if f.dtype == DataType.FLOAT_VECTOR]
        if len(vec) != 1:
            raise SchemaNotReadyException(message="exactly one FLOAT_VECTOR field is supported")
        self.primary_field, self.vector_field = prim[0], vec[0]


class _Connections:
    """connections.connect("default", host=..., port=...): there is no server; the alias records
    which CUDA device collections are created on (kwarg `device`, default 0)."""

    def __init__(self):
        self._alias: Dict[str, dict] = {}

    def connect(self, alias: str = "default", **kwargs):
        self._alias[alias] = dict(kwargs)

    def disconnect(self, alias: str = "default"):
        self._alias.pop(alias, None)

    def has_connection(self, alias: str = "default") -> bool:
        return alias in self._alias

    def device(self, alias: str = "default") -> int:
        return int(self._alias.get(alias, {}).get("device", 0))


connections = _Connections()

_REGISTRY: Dict[str, "_Store"] = {}
_REG_LOCK = threading.Lock()

# engine defaults for collections created through the shim (override per collection with kwargs)
DEFAULTS = {"storage_dtype": "f32", "initial_capacity": 4096}


def _default_index_factory(dim: int, dtype: str, capacity: int, device: int):
    from .engine import Index
    return Index(dim, dtype, capacity=capacity, device=device)


class _Store:
    """State of one named collection (what the Milvus server would hold)."""

    def __init__(self, name, schema, storage_dtype, capacity, device, index_factory):
        self.name, self.schema = name, schema
        self.storage_dtype, self.capacity, self.device = storage_dtype, capacity, device
        self.index_factory = index_factory
        self.columns: Dict[str, list] = {f.name: [] for f in schema.fields if f.dtype != DataType.FLOAT_VECTOR}
        self.pending: list = []               # embedding blocks inserted but not yet flushed: numpy fp32 or CUDA tensors
        self.n_inserted = 0
        self.index = None
        self.metric: Optional[str] = None
        self.pk_to_row: Dict[Any, int] = {}      # live rows only: a deleted row's key may be inserted again
        self.dead: set = set()                    # tombstoned rows (mirrors the engine's live mask) until compact()
        # value -> ascending rows, per scalar field, built on the first filter over that field and kept current by
        # insert(): a filtered search costs the matching rows, not a pass over every row of the column
        self.scalar_index: Dict[str, Dict[Any, List[int]]] = {}
        self.lock = threading.RLock()

    def rows_with(self, field: str, wanted, n: int) -> List[int]:
        """Rows (ascending) among the first n whose `field` equals one of `wanted`."""
        with self.lock:
            inv = self.scalar_index.get(field)
            if inv is None:
                inv = {}
                for r, v in enumerate(self.columns[field]):
                    inv.setdefault(v, []).append(r)
                self.scalar_index[field] = inv
            lists = []
            for w in dict.fromkeys(wanted):                          # a literal listed twice selects its rows once
                try:
                    rows = inv.get(w)
                except TypeError:                                    # unhashable literal: matches nothing
                    rows = None
                if rows:
                    lists.append(rows)
            if not lists:
                return []
            out = lists[0] if len(lists) == 1 else sorted(r for rows in lists for r in rows)
            if out and out[-1] >= n:
                import bisect
                out = out[:bisect.bisect_left(out, n)]
            return list(out)

    def flush(self):
        """Upload the pending blocks through K1.  The collection keeps NO host copy of the embeddings: when the rows
        outgrow the device matrix it is grown on the device (`Index.reserve`: new allocation + device-to-device copy of
        the stored, already normalised rows), so nothing is re-normalised and host memory stays flat."""
        with self.lock:
            if not self.pending:
                return
            need = self.n_inserted
            if self.index is None:
                while self.capacity < need:
                    self.capacity *= 2
                self.index = self.index_factory(self.schema.vector_field.dim, self.storage_dtype, self.capacity, self.device)
            elif need > self.capacity:
                while self.capacity < need:
                    self.capacity *= 2
                self.index.reserve(self.capacity)
            for b in self.pending:
                self.index.add(b)
            self.pending = []


def save_collection(name: str, directory: str) -> None:
    """Durability stand-in for a Milvus flush: `<dir>/<name>.ragfin` (device matrix) + `<dir>/<name>.columns.json`."""
    import json, os
    st = _REGISTRY[name]
    with st.lock:
        st.flush()
        os.makedirs(directory, exist_ok=True)
        if st.index is not None:
            st.index.save(os.path.join(directory, name + ".ragfin"))   # with deletions: a version-2 file carrying the live mask
        fields = [{"name": f.name, "dtype": int(f.dtype), "is_primary": f.is_primary, "params": f.params} for f in st.schema.fields]
        with open(os.path.join(directory, name + ".columns.json"), "w") as f:
            json.dump({"fields": fields, "description": st.schema.description, "columns": st.columns,
                       "n": st.n_inserted, "storage_dtype": st.storage_dtype, "metric": st.metric,
                       "deleted": sorted(st.dead)}, f)


def load_collection(name: str, directory: str, device: int = 0, using: str = "default", index_loader=None) -> "Collection":
    """Re-open a saved collection without re-embedding or re-normalising (results are bit-identical).  Deleted rows stay
    deleted: the matrix file's live mask is checked against the rows recorded in columns.json.  `index_loader(path, capacity,
    device)` replaces `Index.load` (tests)."""
    import json, os
    if index_loader is None:
        from .engine import Index
        index_loader = lambda path, capacity, device: Index.load(path, capacity=capacity, device=device)   # noqa: E731
    with open(os.path.join(directory, name + ".columns.json")) as f:
        meta = json.load(f)
    fields = [FieldSchema(x["name"], DataType(x["dtype"]), is_primary=x["is_primary"], **x["params"]) for x in meta["fields"]]
    utility.drop_collection(name)
    col = Collection(name, CollectionSchema(fields, meta["description"]), using=using, storage_dtype=meta["storage_dtype"], device=device)
    st = col._st
    st.columns = meta["columns"]
    st.scalar_index = {}
    st.n_inserted = int(meta["n"])
    st.metric = meta["metric"]
    st.dead = set(int(r) for r in meta.get("deleted", []))
    pk = st.schema.primary_field.name
    st.pk_to_row = {v: i for i, v in enumerate(st.columns[pk]) if i not in st.dead}
    mpath = os.path.join(directory, name + ".ragfin")
    if st.n_inserted and os.path.exists(mpath):
        st.index = index_loader(mpath, max(st.capacity, st.n_inserted), device)
        st.capacity = st.index.capacity
        dead_in_file = set(np.flatnonzero(~np.asarray(st.index.live_mask(), dtype=bool)).tolist())
        if dead_in_file != st.dead:
            raise MilvusException(message=f"{mpath}: its deleted rows ({len(dead_in_file)}) disagree with {name}.columns.json ({len(st.dead)})")
    return col


class _Utility:
    def has_collection(self, name: str, using: str = "default") -> bool:
        return name in _REGISTRY

    def drop_collection(self, name: str, using: str = "default") -> None:
        with _REG_LOCK:
            st = _REGISTRY.pop(name, None)
        if st is not None and st.index is not None:
            st.index.close()

    def list_collections(self, using: str = "default") -> List[str]:
        return sorted(_REGISTRY)


utility = _Utility()


class Entity:
    """hit.entity: attribute access (retrieve.py:40-42) and .get() (graph_cons.py:288-291).

    A view of one row of the collection's scalar columns restricted to the requested output fields: values are looked up
    when they are read (rows are append-only, so a row's values never change), which keeps a `limit=1000` result
    (graph_cons.py:275-281) from costing a dict of every field of every hit before the caller has looked at one."""
    __slots__ = ("_cols", "_row", "_names")

    def __init__(self, fields, row: Optional[int] = None, names=None):
        if row is None:                                   # Entity({"field": value, ...}): a detached record
            self._cols, self._row, self._names = {k: (v,) for k, v in fields.items()}, 0, tuple(fields)
        else:                                             # Entity(columns, row, names): row `row` of the collection
            self._cols, self._row, self._names = fields, row, names

    @property
    def fields(self) -> Dict[str, Any]:
        return {f: self._cols[f][self._row] for f in self._names}

    def __getattr__(self, name):
        if name.startswith("_"):                          # an unset slot (copy / pickle protocols probing): not a field
            raise AttributeError(name)
        if name in self._names:
            return self._cols[name][self._row]
        raise MilvusException(message=f"Field {name} is not in return entity")

    def get(self, name, default=None):
        return self._cols[name][self._row] if name in self._names else default

    def to_dict(self):
        return self.fields

    def __repr__(self):
        return f"Entity({self.fields!r})"


class Hit:
    __slots__ = ("id", "distance", "entity")

    def __init__(self, pk, distance: float, entity: Entity):
        self.id, self.distance, self.entity = pk, distance, entity

    @property
    def score(self) -> float:
        return self.distance

    def to_dict(self):
        return {"id": self.id, "distance": self.distance, "entity": self.entity.to_dict()}

    def __repr__(self):
        return f"id: {self.id}, distance: {self.distance}, entity: {self.entity.to_dict()}"


class Hits(list):
    @property
    def ids(self):
        return [h.id for h in self]

    @property
    def distances(self):
        return [h.distance for h in self]


class SearchResult(list):
    """results[0] is the Hits of the first query (retrieve.py:38)."""


class MutationResult:
    def __init__(self, primary_keys, insert_count: Optional[int] = None, delete_count: int = 0, upsert_count: int = 0):
        self.primary_keys = list(primary_keys)
        self.insert_count = len(self.primary_keys) if insert_count is None else insert_count
        self.delete_count = delete_count
        self.upsert_count = upsert_count


class CompactionState:
    """What get_compaction_state() reports: compaction here is synchronous, so it has always completed."""

    def __init__(self, completed: int):
        self.state = "Completed"
        self.executing_plan_no, self.timeout_plan_no, self.completed_plan_no = 0, 0, completed

    def __repr__(self):
        return f"CompactionState(state={self.state}, completed_plan_no={self.completed_plan_no})"


_STR = r"\"[^\"]*\"|'[^']*'"
_NUM = r"[-+]?(?:\d+\.?\d*(?:[eE][-+]?\d+)?|\.\d+(?:[eE][-+]?\d+)?)"
_LIT = rf"(?:{_STR}|{_NUM})"
_EXPR_IN = re.compile(rf"^\s*(\w+)\s+in\s+\[\s*((?:{_LIT}\s*(?:,\s*{_LIT}\s*)*)?)\]\s*$", re.S)
_EXPR_EQ = re.compile(rf"^\s*(\w+)\s*==\s*({_LIT})\s*$", re.S)
_LIT_RE = re.compile(_LIT, re.S)


def _parse_literal(tok: str):
    tok = tok.strip()
    if len(tok) >= 2 and tok[0] == tok[-1] and tok[0] in "\"'":
        return tok[1:-1]
    try:
        return int(tok)
    except ValueError:
        try:
            return float(tok)
        except ValueError:
            raise MilvusException(message=f"cannot parse expression: invalid literal {tok!r}") from None


def _range_window(params: dict) -> Dict[str, float]:
    """radius / range_filter of a search's "params" as Index.search keywords ({} for a plain search).  Both must be real
    numbers (bool is refused), neither NaN, and range_filter > radius after rounding to fp32, the precision the engine
    compares in; a radius of +inf or a range_filter of -inf after that rounding leaves no score to return and is refused;
    range_filter without radius is refused rather than dropped, as Milvus would."""
    if not isinstance(params, dict):
        raise MilvusException(message=f"search params must be a dict, got {type(params).__name__}")
    if "radius" not in params:
        if "range_filter" in params:
            raise MilvusException(message="range_filter needs radius: a range search is radius < score <= range_filter")
        return {}
    out = {}
    for key in ("radius", "range_filter"):
        if key not in params:
            continue
        v = params[key]
        if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, float, np.integer, np.floating)):
            raise MilvusException(message=f"{key} must be a number, got {v!r}")
        with np.errstate(over="ignore"):      # a finite value beyond the fp32 range rounds to +-inf, checked below
            v32 = np.float32(v)
        if np.isnan(v32):
            raise MilvusException(message=f"{key} must not be NaN")
        out[key] = float(v32)
    if out["radius"] == np.inf:
        raise MilvusException(message=f"radius must be below +inf in fp32, got {params['radius']!r}: no score exceeds it")
    if out.get("range_filter", 0.0) == -np.inf:
        raise MilvusException(message=f"range_filter must be above -inf in fp32, got {params['range_filter']!r}")
    if "range_filter" in out and not out["range_filter"] > out["radius"]:
        raise MilvusException(message=f"range_filter must be greater than radius for COSINE: radius {params['radius']!r}, "
                                      f"range_filter {params['range_filter']!r}")
    return out


class Collection:
    def __init__(self, name: str, schema: Optional[CollectionSchema] = None, using: str = "default", **kwargs):
        self.name, self._using = name, using
        with _REG_LOCK:
            st = _REGISTRY.get(name)
            if st is None:
                if schema is None:
                    raise SchemaNotReadyException(
                        message=f"Collection '{name}' not exist, or you can pass in schema to create one.")
                st = _Store(name, schema,
                            kwargs.get("storage_dtype", DEFAULTS["storage_dtype"]),
                            int(kwargs.get("initial_capacity", DEFAULTS["initial_capacity"])),
                            int(kwargs.get("device", connections.device(using))),
                            kwargs.get("index_factory", _default_index_factory))
                _REGISTRY[name] = st
        self._st = st

    # -- schema / index ---------------------------------------------------------------
    @property
    def schema(self) -> CollectionSchema:
        return self._st.schema

    @property
    def description(self) -> str:
        return self._st.schema.description

    def create_index(self, field_name: str, index_params: Optional[dict] = None, **kwargs):
        if field_name != self._st.schema.vector_field.name:
            raise MilvusException(message=f"cannot create index on non-vector field {field_name!r}")
        metric = str((index_params or {}).get("metric_type", "COSINE")).upper()
        if metric != "COSINE":
            raise MilvusException(message=f"metric_type {metric} is not supported: this engine serves COSINE only")
        self._st.metric = metric      # index_type / nlist are irrelevant: the search is exact

    def has_index(self, **kwargs) -> bool:
        return self._st.metric is not None

    # -- ingest -----------------------------------------------------------------------
    def insert(self, data, partition_name=None, timeout=None, **kwargs) -> MutationResult:
        st = self._st
        emb, pks, cols, n = self._parse(data)
        with st.lock:
            # ---- validate every column before anything is touched: a Milvus insert is all-or-nothing
            staged = self._validate(pks, cols)
            for pk in pks:
                if pk in st.pk_to_row:
                    raise MilvusException(message=f"duplicate primary key {pk!r}")
            self._commit(staged, pks, emb, n)
        return MutationResult(pks)

    def upsert(self, data, partition_name=None, timeout=None, **kwargs) -> MutationResult:
        """Insert rows, replacing the live rows whose primary keys they carry: those rows are deleted (tombstoned) and the
        new ones appended.  Validated in full first; all-or-nothing like insert()."""
        st = self._st
        emb, pks, cols, n = self._parse(data)
        with st.lock:
            staged = self._validate(pks, cols)
            st.flush()                                    # the rows being replaced are on the device
            old = sorted(st.pk_to_row[pk] for pk in pks if pk in st.pk_to_row)
            if old:
                st.index.delete(old)
                st.dead.update(old)
            self._commit(staged, pks, emb, n)
        return MutationResult(pks, delete_count=len(old), upsert_count=n)

    def delete(self, expr: str, partition_name=None, timeout=None, **kwargs) -> MutationResult:
        """Delete the live rows matching `expr` (`pk in [...]` or `field == literal`): no search or query returns them from
        now on.  num_entities keeps counting them until compact()."""
        st = self._st
        if not isinstance(expr, str) or not expr.strip():
            raise MilvusException(message="delete needs an expression")
        with st.lock:
            st.flush()
            rows = sorted(set(self._rows_matching(expr.strip(), st.n_inserted)) - st.dead)   # a key listed twice: once
            if rows:
                st.index.delete(rows)
                st.dead.update(rows)
            pk_col = st.columns[st.schema.primary_field.name]
            pks = [pk_col[r] for r in rows]
            for pk in pks:
                st.pk_to_row.pop(pk, None)
        return MutationResult(pks, insert_count=0, delete_count=len(rows))

    def compact(self, timeout=None, **kwargs) -> None:
        """Remove deleted rows for good: the engine compacts its matrix (survivors keep their order), the scalar columns,
        primary-key map and scalar filter index follow with the same old-to-new row map.  Synchronous."""
        st = self._st
        with st.lock:
            st.flush()
            st.compactions = getattr(st, "compactions", 0) + 1
            if not st.dead:
                return
            survivors = [int(r) for r in st.index.compact()]
            if len(survivors) != st.n_inserted - len(st.dead):
                raise MilvusException(message=f"compaction kept {len(survivors)} rows, expected {st.n_inserted - len(st.dead)}")
            new_of = {r: i for i, r in enumerate(survivors)}
            st.columns = {name: [c[r] for r in survivors] for name, c in st.columns.items()}   # earlier hits keep the old lists
            st.scalar_index = {f: {v: [new_of[r] for r in rows if r in new_of] for v, rows in inv.items()}
                               for f, inv in st.scalar_index.items()}
            for inv in st.scalar_index.values():
                for v in [v for v, rows in inv.items() if not rows]:
                    del inv[v]
            st.pk_to_row = {v: i for i, v in enumerate(st.columns[st.schema.primary_field.name])}
            st.n_inserted = len(survivors)
            st.dead = set()

    def get_compaction_state(self, timeout=None, **kwargs) -> CompactionState:
        return CompactionState(getattr(self._st, "compactions", 0))

    def wait_for_compaction_completed(self, timeout=None, **kwargs) -> CompactionState:
        return self.get_compaction_state()

    def _parse(self, data):
        """Rows of an insert / upsert -> (embeddings, primary keys, columns in schema order, n); shapes checked."""
        st = self._st
        fields = st.schema.fields
        if isinstance(data, dict):
            data = [data]
        if len(data) > 0 and isinstance(data[0], dict):          # row-major list of dicts
            cols = [[row[f.name] for row in data] for f in fields]
        else:                                                     # column-major, schema field order
            cols = list(data)
        if len(cols) != len(fields):
            raise ParamError(message=f"expected {len(fields)} columns ({[f.name for f in fields]}), got {len(cols)}")
        n = len(cols[0])
        if any(len(c) != n for c in cols):
            raise ParamError(message="all columns must have the same number of rows")
        vi = fields.index(st.schema.vector_field)
        dim = st.schema.vector_field.dim
        emb = cols[vi]
        if hasattr(emb, "is_cuda") and emb.is_cuda:
            # embeddings produced on the GPU (a torch encoder) stay there: K1 reads them through ragfin_add(src_is_device=1)
            import torch
            if emb.dim() != 2 or tuple(emb.shape) != (n, dim):
                raise ParamError(message=f"embedding column must be [{n}, {dim}], got {tuple(emb.shape)}")
            emb = emb.detach().to(torch.float32).contiguous().clone()      # the caller may reuse its buffer after insert()
        else:
            if hasattr(emb, "detach"):
                emb = emb.detach().numpy()
            emb = np.array(emb, dtype=np.float32, order="C")               # a private copy: pending until flush()
            if n and (emb.ndim != 2 or emb.shape != (n, dim)):
                raise ParamError(message=f"embedding column must be [{n}, {dim}], got {emb.shape}")
            _refuse_non_finite(emb, "insert")
        pks = list(cols[fields.index(st.schema.primary_field)])
        return emb, pks, cols, n

    def _validate(self, pks, cols) -> dict:
        """Checks that need no collection state beyond the schema; returns the scalar columns to append."""
        st = self._st
        if len(set(pks)) != len(pks):
            raise MilvusException(message="duplicate primary keys inside one insert")
        staged = {}
        for f, c in zip(st.schema.fields, cols):
            if f.dtype == DataType.FLOAT_VECTOR:
                continue
            c = list(c)
            if f.dtype == DataType.VARCHAR and f.max_length:
                for v in c:
                    if len(str(v)) > f.max_length:
                        raise MilvusException(message=f"length of varchar field {f.name} exceeds max length {f.max_length}")
            staged[f.name] = c
        return staged

    def _commit(self, staged: dict, pks, emb, n: int) -> None:
        st = self._st
        for name, c in staged.items():
            st.columns[name].extend(c)
            inv = st.scalar_index.get(name)
            if inv is not None:
                for j, v in enumerate(c):
                    inv.setdefault(v, []).append(st.n_inserted + j)
        for j, pk in enumerate(pks):
            st.pk_to_row[pk] = st.n_inserted + j
        if n:
            st.pending.append(emb)
        st.n_inserted += n

    def flush(self, timeout=None, **kwargs):
        self._st.flush()

    def load(self, partition_names=None, replica_number=1, timeout=None, **kwargs):
        self._st.flush()

    def release(self, timeout=None, **kwargs):
        pass

    def drop(self, timeout=None, **kwargs):
        utility.drop_collection(self.name)

    @property
    def num_entities(self) -> int:
        st = self._st
        with st.lock:                                         # a flush on another thread swaps `pending` under the same lock
            return st.n_inserted - sum(len(b) for b in st.pending)

    @property
    def is_empty(self) -> bool:
        return self.num_entities == 0

    # -- hot path ---------------------------------------------------------------------
    def search(self, data, anns_field: str, param: dict, limit: int, expr: Optional[str] = None,
               partition_names=None, output_fields: Optional[List[str]] = None, timeout=None,
               round_decimal: int = -1, **kwargs) -> SearchResult:
        st = self._st
        if anns_field != st.schema.vector_field.name:
            raise MilvusException(message=f"failed to get field schema by name: fieldName({anns_field}) not found")
        metric = str((param or {}).get("metric_type", st.metric or "COSINE")).upper()
        if metric != "COSINE":
            raise MilvusException(message=f"metric type not match: expected=COSINE, actual={metric}")
        if not isinstance(limit, (int, np.integer)) or not 1 <= int(limit) <= MAX_LIMIT:
            raise MilvusException(message=f"`limit` value {limit} is illegal: topk [1, {MAX_LIMIT}]")
        out_fields = list(output_fields or [])
        for f in out_fields:
            if f not in st.columns:
                raise MilvusException(message=f"field {f} not exist")
        window = _range_window((param or {}).get("params") or {})
        q = np.ascontiguousarray(data, dtype=np.float32)
        if q.ndim == 1:
            q = q[None, :]
        if q.ndim != 2 or q.shape[1] != st.schema.vector_field.dim:
            raise MilvusException(message=f"vector dimension mismatch: expected {st.schema.vector_field.dim}, got {q.shape}")
        _refuse_non_finite(q, "search")
        with st.lock:
            st.flush()
            res = SearchResult()
            if st.index is None or st.n_inserted == 0:
                for _ in range(q.shape[0]):
                    res.append(Hits())
                return res
            # deleted rows: the engine holds their tombstones and never returns them, filtered or not
            if expr and expr.strip():     # scalar filter -> row bitmask consumed inside the top-k epilogues
                allow = np.zeros(st.n_inserted, dtype=bool)
                allow[self._rows_matching(expr.strip(), st.n_inserted)] = True
                ids, scores = st.index.search(q, int(limit), allow=allow, **window)
            else:
                ids, scores = st.index.search(q, int(limit), **window)
            pk_col = st.columns[st.schema.primary_field.name]
            cols, names = st.columns, tuple(out_fields)
            for qi in range(q.shape[0]):
                rows_q, sc_q = ids[qi].tolist(), scores[qi].tolist()      # Python ints / floats (fp32 scores widened exactly)
                if rows_q and rows_q[-1] < 0:                            # padded: fewer than `limit` rows (allowed, in the window)
                    rows_q = rows_q[:next(i for i, r in enumerate(rows_q) if r < 0)]
                if round_decimal >= 0:
                    sc_q = [round(s_, round_decimal) for s_ in sc_q]
                res.append(Hits([Hit(pk_col[row], sc, Entity(cols, row, names)) for row, sc in zip(rows_q, sc_q)]))
            return res

    def _rows_matching(self, expr: str, n: int) -> List[int]:
        """Rows (ascending) among the first n that satisfy `field in [...]` or `field == literal`."""
        st = self._st
        pk_name = st.schema.primary_field.name
        # The two forms the reference uses (graph_cons.py:306-311 `id in [...]`, plus `field == literal`), matched in FULL:
        # anything else - and / or / not, comparisons, unquoted strings, trailing text - is rejected instead of being
        # swallowed into a literal (which would silently select no rows).
        m_in, m_eq = _EXPR_IN.match(expr), _EXPR_EQ.match(expr)
        if m_in:
            field = m_in.group(1)
            wanted = [_parse_literal(t) for t in _LIT_RE.findall(m_in.group(2))]
        elif m_eq:
            field, wanted = m_eq.group(1), [_parse_literal(m_eq.group(2))]
        else:
            raise MilvusException(message=f"cannot parse expression: {expr} (supported: `field in [literals]`, `field == literal`)")
        if field not in st.columns:
            raise MilvusException(message=f"field {field} not exist")
        if field == pk_name:
            return sorted(r for r in (st.pk_to_row.get(w) for w in wanted) if r is not None and r < n)
        return st.rows_with(field, wanted, n)

    # -- scalar lookups (host side; "next" row N1) --------------------------------------
    def query(self, expr: str = "", output_fields: Optional[List[str]] = None, partition_names=None,
              timeout=None, limit: Optional[int] = None, offset: int = 0, **kwargs) -> List[dict]:
        st = self._st
        pk_name = st.schema.primary_field.name
        out_fields = list(output_fields or [])
        if pk_name not in out_fields:
            out_fields = [pk_name] + out_fields
        for f in out_fields:
            if f not in st.columns:
                raise MilvusException(message=f"field {f} not exist")
        with st.lock:
            n = self.num_entities
            expr = (expr or "").strip()
            if expr == "":
                if limit is None:
                    raise MilvusException(message="empty expression should be used with limit")
                rows = list(range(n))
            else:
                rows = self._rows_matching(expr, n)
            if st.dead:
                rows = [r for r in rows if r not in st.dead]
            rows = rows[offset:]
            if limit is not None:
                rows = rows[:int(limit)]
            return [{f: st.columns[f][r] for f in out_fields} for r in rows]
