"""CPU suite for grouping search: the reference answer (tests/_grouping.py grouped_topk) against a brute-force loop, the
identities that pin its semantics, the shim's group_by_field (validation and composition with expr, deletes,
round_decimal and output_fields) through an oracle-backed stand-in index, and the library's argument checks of the two
new entry points (no device needed). tests/test_grouped_gpu.py checks the engine itself."""
import ctypes
import os

import numpy as np
import pytest

from _grouping import grouped_topk
from oracle import ragfin_oracle as O
from ragfin_b200 import milvus_compat as mc

DIM = 64


def brute(S, codes, n_groups, k, allow=None):
    """Grouping search by definition: each group's best (score desc, row asc) row, groups ordered the same way."""
    out = []
    for s in np.atleast_2d(S):
        best = {}
        for r in range(len(s)):
            g = int(codes[r])
            if not 0 <= g < n_groups or (allow is not None and not allow[r]):
                continue
            if g not in best or (s[r], -r) > (s[best[g]], -best[g]):
                best[g] = r
        rows = sorted(best.values(), key=lambda r: (-float(s[r]), r))[:k]
        out.append(rows + [-1] * (k - len(rows)))
    return np.array(out, np.int64)


def test_grouped_topk_matches_brute_force_with_ties():
    rng = np.random.default_rng(0)
    for trial in range(30):
        n = int(rng.integers(1, 200))
        ng = int(rng.integers(1, 40))
        S = rng.integers(-4, 5, (3, n)).astype(np.float32) / np.float32(8)   # coarse scores: ties inside and across groups
        codes = rng.integers(-3, ng + 3, n).astype(np.int32)                 # some codes out of range
        allow = rng.random(n) < 0.8 if trial % 2 else None
        k = int(rng.integers(1, 50))
        ids, sc = grouped_topk(S, codes, ng, k, allow=allow)
        want = brute(S, codes, ng, k, allow)
        assert np.array_equal(ids, want), (trial, ids, want)
        for i in range(3):
            hit = ids[i] >= 0
            assert np.array_equal(sc[i][hit], S[i][ids[i][hit]]) and (sc[i][~hit] == -np.inf).all()


def test_identities():
    stored = O.normalize_rows(O.synth_rows(1, 0, 500, DIM, dup_every=7), "f32")
    q = O.synth_rows(2, 0, 3, DIM)
    qhat = O.normalize_rows(q, "f32")
    S = np.stack([O.exact_scores(stored, v) for v in qhat])
    for k in (1, 10, 600):
        ids, sc = grouped_topk(S, np.arange(500, dtype=np.int32), 500, k)
        wi, ws = O.cosine_topk(q, stored, k)
        assert np.array_equal(ids, wi) and np.array_equal(sc.view(np.uint32), ws.view(np.uint32))
    ids, sc = grouped_topk(S, np.zeros(500, np.int32), 1, 5)
    wi, ws = O.cosine_topk(q, stored, 1)
    assert np.array_equal(ids[:, :1], wi) and (ids[:, 1:] == -1).all() and (sc[:, 1:] == -np.inf).all()


class GroupIndex:
    """The `Index` surface the shim uses, with deletion, filters and grouping, answered by the oracle."""

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

    def delete(self, ids):
        ids = np.unique(np.asarray(ids, np.int64).reshape(-1))
        n = int(self.live[ids].sum())
        self.live[ids] = False
        return n

    def live_mask(self):
        return self.live.copy()

    def compact(self):
        keep = np.flatnonzero(self.live)
        self.rows, self.live = self.rows[keep], self.live[keep]
        return keep

    def search(self, q, k, allow=None, group_by=None, n_groups=None, **window):
        self.calls.append(dict(window, grouped=group_by is not None))
        assert not window or group_by is None
        mask = self.live if allow is None else (np.asarray(allow, bool) & self.live)
        qhat = O.normalize_rows(np.atleast_2d(q), "f32")
        S = np.stack([O.exact_scores(self.rows, v) for v in qhat])
        if group_by is None:
            return grouped_topk(S, np.arange(len(self.rows)), len(self.rows), k, allow=mask)
        codes = np.asarray(group_by.cpu()).astype(np.int32)
        assert codes.shape == (len(self.rows),)
        return grouped_topk(S, codes, n_groups, k, allow=mask)

    def close(self):
        pass


def fields():
    F, D = mc.FieldSchema, mc.DataType
    return [F("id", D.VARCHAR, max_length=32, is_primary=True), F("embedding", D.FLOAT_VECTOR, dim=DIM),
            F("period", D.VARCHAR, max_length=20), F("doc", D.INT64), F("weight", D.FLOAT), F("meta", D.JSON)]


def make(name="grp", n=60, seed=5):
    if mc.utility.has_collection(name):
        mc.utility.drop_collection(name)
    col = mc.Collection(name, mc.CollectionSchema(fields(), "grouped"), index_factory=GroupIndex, initial_capacity=16)
    col.create_index("embedding", {"metric_type": "COSINE"})
    emb = O.synth_rows(seed, 0, n, DIM, dup_every=9)
    col.insert([[f"c{i}" for i in range(n)], emb, [f"Q{i % 4 + 1}" for i in range(n)], [i // 6 for i in range(n)],
                [0.5] * n, [{}] * n])
    col.flush()
    return col, emb


def want_groups(emb, q, values, k, allow=None):
    """(rows, scores) of the oracle grouping over a list of field values (codes in first-seen order)."""
    first = {}
    codes = np.array([first.setdefault(v, len(first)) for v in values], np.int32)
    S = O.exact_scores(O.normalize_rows(emb, "f32"), O.normalize_rows(q, "f32")[0])
    ids, sc = grouped_topk(S, codes, len(first), k, allow=allow)
    keep = ids[0] >= 0
    return ids[0][keep].tolist(), sc[0][keep].tolist()


def search(col, q, limit=10, **kw):
    return col.search(q, "embedding", {"metric_type": "COSINE"}, limit=limit, **kw)


def test_group_by_field_one_hit_per_group():
    col, emb = make()
    q = O.synth_rows(9, 0, 1, DIM)
    n = len(emb)
    for field, values in (("period", [f"Q{i % 4 + 1}" for i in range(n)]), ("doc", [i // 6 for i in range(n)])):
        rows, sc = want_groups(emb, q, values, 10)
        got = search(col, q, group_by_field=field, output_fields=[field])[0]
        assert got.ids == [f"c{r}" for r in rows] and got.distances == sc
        assert [h.entity.get(field) for h in got] == [values[r] for r in rows]
        assert len(set(values[r] for r in rows)) == len(rows)
    assert col._st.index.calls[-1]["grouped"]
    plain = search(col, q, unknown_keyword=1)[0]                   # other keywords are still ignored
    assert not col._st.index.calls[-1]["grouped"] and len(plain) == 10


def test_group_by_composes_with_expr_deletes_round_decimal_and_inserts():
    col, emb = make()
    q = O.synth_rows(9, 0, 1, DIM)
    n = len(emb)
    periods = [f"Q{i % 4 + 1}" for i in range(n)]
    docs = [i // 6 for i in range(n)]
    allow = np.array([p in ("Q1", "Q3") for p in periods])
    rows, sc = want_groups(emb, q, docs, 5, allow)
    got = search(col, q, limit=5, expr='period in ["Q1", "Q3"]', group_by_field="doc", round_decimal=3)[0]
    assert got.ids == [f"c{r}" for r in rows] and got.distances == [round(s, 3) for s in sc]
    # delete each group's best row: the group is then represented by its next row
    top, _ = want_groups(emb, q, docs, 3)
    col.delete(f'id in [{", ".join(repr(f"c{r}") for r in top)}]')
    live = np.ones(n, bool)
    live[top] = False
    rows, sc = want_groups(emb, q, docs, 20, live)
    got = search(col, q, limit=20, group_by_field="doc")[0]
    assert got.ids == [f"c{r}" for r in rows] and got.distances == sc
    assert not set(top) & set(rows)
    # rows inserted after the codes were built extend them; compact() renumbers the rows and rebuilds them
    extra = O.synth_rows(11, 0, 12, DIM)
    col.insert([[f"d{i}" for i in range(12)], extra, ["Q9"] * 12, [100 + i // 3 for i in range(12)], [0.5] * 12, [{}] * 12])
    col.flush()
    all_emb = np.concatenate([emb, extra])
    all_docs = docs + [100 + i // 3 for i in range(12)]
    live = np.concatenate([live, np.ones(12, bool)])
    rows, sc = want_groups(all_emb, q, all_docs, 30, live)
    pks = [f"c{i}" for i in range(n)] + [f"d{i}" for i in range(12)]
    got = search(col, q, limit=30, group_by_field="doc")[0]
    assert got.ids == [pks[r] for r in rows] and got.distances == sc
    col.compact()
    assert col._st.group_codes == {}
    got = search(col, q, limit=30, group_by_field="doc", output_fields=["doc"])[0]
    assert got.ids == [pks[r] for r in rows] and got.distances == sc
    assert [h.entity.get("doc") for h in got] == [all_docs[r] for r in rows]


@pytest.mark.parametrize("kw, what", [
    (dict(group_by_field="nope"), "not exist"),
    (dict(group_by_field="embedding"), "not supported"),
    (dict(group_by_field="weight"), "not supported"),
    (dict(group_by_field="meta"), "not supported"),
    (dict(group_by_field=3), "field name"),
])
def test_bad_group_by_field_raises(kw, what):
    col, _ = make()
    with pytest.raises(mc.MilvusException, match=what):
        search(col, O.synth_rows(9, 0, 1, DIM), **kw)


def test_group_by_with_range_search_is_refused():
    col, _ = make()
    with pytest.raises(mc.MilvusException, match="range search"):
        col.search(O.synth_rows(9, 0, 1, DIM), "embedding", {"metric_type": "COSINE", "params": {"radius": 0.1}}, limit=5,
                   group_by_field="period")


def test_library_validates_the_group_arguments_without_a_device():
    """The codes are checked before the handle: NULL codes and n_groups < 1 fail with EINVAL and their own message; valid
    codes then reach the handle check."""
    from ragfin_b200 import _lib
    if not os.path.exists(_lib.SO_PATH):
        pytest.skip("library not built")
    L = _lib.load()
    q = (ctypes.c_float * DIM)()
    ids = (ctypes.c_int64 * 4)()
    sc = (ctypes.c_float * 4)()
    codes = (ctypes.c_int32 * 4)()
    for g, ng, msg in ((None, 4, "NULL group codes"), (codes, 0, "n_groups"), (codes, -1, "n_groups"), (codes, 4, "NULL handle")):
        assert L.ragfin_search_grouped(None, q, 1, 4, g, ng, None, 0, ids, sc, None) == _lib.EINVAL
        assert msg in L.ragfin_last_error().decode(), (ng, L.ragfin_last_error())
        assert L.ragfin_search_grouped_host(None, q, 1, 4, g, 0, ng, None, 0, ids, sc) == _lib.EINVAL
        assert msg in L.ragfin_last_error().decode(), (ng, L.ragfin_last_error())


def test_index_refuses_group_by_with_a_window():
    import ragfin_b200
    idx = ragfin_b200.Index.__new__(ragfin_b200.Index)
    with pytest.raises(ValueError, match="radius"):
        idx._check_groups(np.zeros(3, np.int32), 2, 0.1, None)
    with pytest.raises(ValueError, match="n_groups"):
        idx._check_groups(np.zeros(3, np.int32), 0, None, None)
    with pytest.raises(ValueError, match="needs group_by"):
        idx._check_groups(None, 3, None, None)
