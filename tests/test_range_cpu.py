"""CPU suite for range search (radius < score <= range_filter) in the pymilvus-shaped shim: parameter validation, fp32
rounding of the bounds, composition with expr and with deletions.  The engine is replaced by an oracle-backed stand-in that
accepts radius / range_filter, so the shim's handling of `params` is what is under test; tests/test_range_gpu.py checks the
engine itself.  Also: argument checks of the two new C entry points through the real library (no device needed)."""
import ctypes
import math
import os

import numpy as np
import pytest

from oracle import ragfin_oracle as O
from ragfin_b200 import milvus_compat as mc

DIM = 64


def range_topk(q, stored, k, radius=-np.inf, range_filter=np.inf, allow=None):
    """Oracle: the k best rows with radius < s <= range_filter (fp32 compares on the exact fp32 score), by (score desc,
    id asc), padded with (-1, -inf).  Built on exact_scores over every row."""
    q = np.atleast_2d(np.asarray(q, np.float32))
    qhat = O.normalize_rows(q, "f32")
    lo, hi = np.float32(radius), np.float32(range_filter)
    ids = np.full((len(q), k), -1, np.int64)
    sc = np.full((len(q), k), -np.inf, np.float32)
    for i in range(len(q)):
        s = O.exact_scores(stored, qhat[i])
        ok = (s > lo) & (s <= hi)
        if allow is not None:
            ok &= allow
        rows = np.flatnonzero(ok)
        order = rows[np.lexsort((rows, -s[rows].astype(np.float64)))][:k]
        ids[i, :len(order)] = order
        sc[i, :len(order)] = s[order]
    return ids, sc


class RangeIndex:
    """The `Index` surface the shim uses, with deletion and range search."""

    def __init__(self, dim, dtype, capacity, device):
        self.dim, self.dtype, self.capacity = dim, dtype, capacity
        self.rows = np.zeros((0, dim), np.float32)
        self.live = np.zeros(0, bool)
        self.calls = []

    def add(self, rows):
        rows = np.asarray(rows, np.float32)
        self.rows = np.concatenate([self.rows, O.normalize_rows(rows, self.dtype)])
        self.live = np.concatenate([self.live, np.ones(len(rows), bool)])

    def reserve(self, capacity):
        self.capacity = max(self.capacity, capacity)

    def __len__(self):
        return len(self.rows)

    @property
    def live_count(self):
        return int(self.live.sum())

    def delete(self, ids):
        ids = np.unique(np.asarray(ids, np.int64).reshape(-1))
        n = int(self.live[ids].sum())
        self.live[ids] = False
        return n

    def live_mask(self):
        return self.live.copy()

    def search(self, q, k, allow=None, **window):
        self.calls.append(window)
        for v in window.values():   # the shim hands the engine fp32 values
            assert isinstance(v, float) and float(np.float32(v)) == v
        mask = self.live if allow is None else (np.asarray(allow, bool) & self.live)
        return range_topk(q, self.rows, k, window.get("radius", -np.inf), window.get("range_filter", np.inf), mask)

    def close(self):
        pass


def fields():
    F, D = mc.FieldSchema, mc.DataType
    return [F("id", D.VARCHAR, max_length=32, is_primary=True), F("embedding", D.FLOAT_VECTOR, dim=DIM),
            F("period", D.VARCHAR, max_length=20)]


def make(name="rng", n=60, seed=5):
    if mc.utility.has_collection(name):
        mc.utility.drop_collection(name)
    col = mc.Collection(name, mc.CollectionSchema(fields(), "range"), index_factory=RangeIndex, initial_capacity=16)
    col.create_index("embedding", {"metric_type": "COSINE"})
    emb = O.synth_rows(seed, 0, n, DIM)
    col.insert([[f"c{i}" for i in range(n)], emb, [f"Q{i % 4 + 1}" for i in range(n)]])
    col.flush()
    return col, emb


def scores_of(col, emb, q):
    return O.exact_scores(O.normalize_rows(emb, "f32"), O.normalize_rows(q, "f32")[0])


def search(col, q, params, limit=10, **kw):
    return col.search(q, "embedding", {"metric_type": "COSINE", "params": params}, limit=limit, **kw)


def test_range_oracle_matches_brute_force():
    rng = np.random.default_rng(0)
    stored = O.normalize_rows(O.synth_rows(1, 0, 300, DIM, dup_every=7), "f32")
    q = O.synth_rows(2, 0, 3, DIM)
    qhat = O.normalize_rows(q, "f32")
    for radius, rf in ((-np.inf, np.inf), (0.0, 0.2), (-0.1, np.inf), (-np.inf, 0.05), (0.3, 0.31)):
        allow = rng.random(300) < 0.7
        ids, sc = range_topk(q, stored, 20, radius, rf, allow)
        for i in range(3):
            s = [float(np.dot(stored[r].astype(np.float64), qhat[i].astype(np.float64))) for r in range(300)]
            s32 = O.exact_scores(stored, qhat[i])
            assert max(abs(a - b) for a, b in zip(s, s32)) < 1e-6
            want = sorted((r for r in range(300) if allow[r] and radius < s32[r] <= rf), key=lambda r: (-s32[r], r))[:20]
            assert ids[i, :len(want)].tolist() == want and (ids[i, len(want):] == -1).all()
            assert (sc[i, len(want):] == -np.inf).all()
    ids, sc = range_topk(q, stored, 5)
    want_ids, want_sc = O.cosine_topk(q, stored, 5)
    assert np.array_equal(ids, want_ids) and np.array_equal(sc.view(np.uint32), want_sc.view(np.uint32))


@pytest.mark.parametrize("params, what", [
    ({"range_filter": 0.9}, "needs radius"),
    ({"radius": 0.5, "range_filter": 0.5}, "greater than radius"),
    ({"radius": 0.5, "range_filter": 0.4}, "greater than radius"),
    ({"radius": float("nan")}, "NaN"),
    ({"radius": 0.1, "range_filter": float("nan")}, "NaN"),
    ({"radius": "0.5"}, "number"),
    ({"radius": None}, "number"),
    ({"radius": True}, "number"),
    ({"radius": 0.1, "range_filter": False}, "number"),
    # distinct Python floats that round to the same fp32 value: an empty window in the engine's precision
    ({"radius": 0.8, "range_filter": 0.8 + 1e-12}, "greater than radius"),
    # bounds that leave nothing to return once rounded to fp32
    ({"radius": float("inf")}, "radius must be below"),
    ({"radius": 1e39}, "radius must be below"),
    ({"radius": -2.0, "range_filter": float("-inf")}, "range_filter must be above"),
    ({"radius": -1e40, "range_filter": -1e39}, "range_filter must be above"),
])
def test_bad_params_raise(params, what):
    col, _ = make()
    with pytest.raises(mc.MilvusException, match=what):
        search(col, O.synth_rows(9, 0, 1, DIM), params)


def test_params_without_radius_is_a_plain_search():
    col, emb = make()
    q = O.synth_rows(9, 0, 2, DIM)
    plain = col.search(q, "embedding", {"metric_type": "COSINE"}, limit=10)
    got = search(col, q, {"nprobe": 16, "ef": 64})
    assert [h.ids for h in got] == [h.ids for h in plain]
    assert [h.distances for h in got] == [h.distances for h in plain]
    assert col._st.index.calls[-1] == {} and col._st.index.calls[-2] == {}


def test_window_selects_rows_strictly_above_radius_and_up_to_range_filter():
    col, emb = make()
    q = O.synth_rows(9, 0, 1, DIM)
    s = scores_of(col, emb, q)
    order = np.lexsort((np.arange(len(s)), -s.astype(np.float64)))
    radius, rf = float(s[order[12]]), float(s[order[3]])     # excludes rank 12 (the radius), includes rank 3 (the ceiling)
    got = search(col, q, {"radius": radius, "range_filter": rf}, limit=20)[0]
    assert got.ids == [f"c{r}" for r in order[3:12]]
    assert got.distances == [float(s[r]) for r in order[3:12]]
    got = search(col, q, {"radius": radius}, limit=5)[0]       # a floor alone
    assert got.ids == [f"c{r}" for r in order[:5]]
    got = search(col, q, {"radius": -1.5, "range_filter": -1.0}, limit=5)[0]   # an empty window
    assert got.ids == []


def test_python_float_bounds_compare_as_fp32():
    col, emb = make()
    q = O.synth_rows(9, 0, 1, DIM)
    s = scores_of(col, emb, q)
    top = np.float32(s.max())
    r64 = float(top) - 1e-12                                   # below the score as a double, equal to it in fp32
    assert np.float32(r64) == top and r64 < float(top)
    got = search(col, q, {"radius": r64}, limit=5)[0]
    assert float(top) not in got.distances                      # radius == score in fp32: excluded
    assert col._st.index.calls[-1] == {"radius": float(top)}
    got = search(col, q, {"radius": -1.0, "range_filter": r64}, limit=1)[0]
    assert got.distances == [float(top)]                         # range_filter == score in fp32: included
    r = search(col, q, {"radius": 0.8, "range_filter": 0.9})
    assert col._st.index.calls[-1] == {"radius": float(np.float32(0.8)), "range_filter": float(np.float32(0.9))}
    assert all(np.float32(0.8) < np.float32(d) <= np.float32(0.9) for d in r[0].distances)


def test_window_with_expr_deletes_and_round_decimal():
    col, emb = make()
    q = O.synth_rows(9, 0, 2, DIM)
    col.delete('id in ["c0", "c1", "c2", "c3", "c4", "c5", "c6", "c7"]')
    stored = O.normalize_rows(emb, "f32")
    allow = np.array([i % 4 in (0, 1) and i >= 8 for i in range(len(emb))])
    got = search(col, q, {"radius": -0.05, "range_filter": 0.1}, limit=7, expr='period in ["Q1", "Q2"]')
    ids, sc = range_topk(q, stored, 7, np.float32(-0.05), np.float32(0.1), allow)
    for h, i, s in zip(got, ids, sc):
        assert h.ids == [f"c{r}" for r in i if r >= 0]
        assert h.distances == [float(x) for x in s[i >= 0]]
    got = search(col, q, {"radius": -0.05, "range_filter": 0.1}, limit=7, expr='period in ["Q1", "Q2"]', round_decimal=3)
    for h, s, i in zip(got, sc, ids):
        assert h.distances == [round(float(x), 3) for x in s[i >= 0]]
    got = search(col, q, {"radius": -0.05}, limit=100)             # deleted rows never come back
    live = np.arange(len(emb)) >= 8
    ids, _ = range_topk(q, stored, 100, np.float32(-0.05), np.inf, live)
    assert [h.ids for h in got] == [[f"c{r}" for r in i if r >= 0] for i in ids]


def test_library_validates_the_window_without_a_device():
    """The window is checked before the handle: a NULL range, a NaN bound and range_filter <= radius each fail with EINVAL
    and their own message; a valid window then reaches the handle check."""
    from ragfin_b200 import _lib
    if not os.path.exists(_lib.SO_PATH):
        pytest.skip("library not built")
    L = _lib.load()
    q = (ctypes.c_float * DIM)()
    ids = (ctypes.c_int64 * 4)()
    sc = (ctypes.c_float * 4)()
    cases = [(None, "NULL range"), ((math.nan, 0.5), "NaN"), ((0.1, math.nan), "NaN"), ((0.5, 0.5), "greater than radius"),
             ((0.5, 0.4), "greater than radius"), ((math.inf, math.inf), "greater than radius"), ((0.1, 0.5), "NULL handle"),
             ((-math.inf, math.inf), "NULL handle")]
    for window, msg in cases:
        w = None if window is None else (ctypes.c_float * 2)(*window)
        assert L.ragfin_search_range(None, q, 1, 4, w, None, 0, ids, sc, None) == _lib.EINVAL
        assert msg in L.ragfin_last_error().decode(), (window, L.ragfin_last_error())
        assert L.ragfin_search_range_host(None, q, 1, 4, w, None, 0, ids, sc) == _lib.EINVAL
        assert msg in L.ragfin_last_error().decode(), (window, L.ragfin_last_error())
