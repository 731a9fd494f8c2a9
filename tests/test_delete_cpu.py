"""CPU suite for row deletion in the pymilvus-shaped shim: delete / upsert / compact, deleted rows absent from search and
query, num_entities, persistence.  The engine is replaced by an oracle-backed stand-in (tombstones kept as a live mask,
filtered searches over allow AND live, compaction that keeps the survivors' order) through the shim's index_factory hook,
so the host bookkeeping is what is under test; tests/test_delete_gpu.py checks the engine itself."""
import ctypes
import os

import numpy as np
import pytest

from oracle import ragfin_oracle as O
from ragfin_b200 import milvus_compat as mc

DIM = 64


class TombstoneIndex:
    """The `Index` surface the shim uses, with deletion: add / search / delete / live_mask / compact / save / load."""

    def __init__(self, dim, dtype, capacity, device):
        self.dim, self.dtype, self.capacity = dim, dtype, capacity
        self.rows = np.zeros((0, dim), np.float32)
        self.live = np.zeros(0, bool)

    def add(self, rows):
        rows = np.asarray(rows, np.float32)
        assert len(self.rows) + len(rows) <= self.capacity
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
        ids = np.asarray(ids, np.int64).reshape(-1)
        if ids.size and (ids.min() < 0 or ids.max() >= len(self.rows)):
            raise ValueError("id out of range")
        ids = np.unique(ids)
        n = int(self.live[ids].sum())
        self.live[ids] = False
        return n

    def live_mask(self):
        return self.live.copy()

    def compact(self):
        keep = np.flatnonzero(self.live)
        self.rows, self.live = self.rows[keep], np.ones(len(keep), bool)
        return keep

    def search(self, q, k, allow=None):
        mask = self.live if allow is None else (np.asarray(allow, bool) & self.live)
        rows = np.flatnonzero(mask)
        ids, sc = O.cosine_topk(np.asarray(q, np.float32), self.rows[rows], k)
        return np.where(ids >= 0, rows[np.clip(ids, 0, None)] if len(rows) else -1, -1), sc

    def save(self, path):
        np.savez(path + ".npz", rows=self.rows, live=self.live, dtype=self.dtype, dim=self.dim)
        os.replace(path + ".npz", path)

    @classmethod
    def load(cls, path, capacity, device):
        z = np.load(path, allow_pickle=False)
        self = cls(int(z["dim"]), str(z["dtype"]), max(capacity, len(z["rows"])), device)
        self.rows, self.live = z["rows"], z["live"]
        return self

    def close(self):
        pass


def fields():
    F, D = mc.FieldSchema, mc.DataType
    return [F("id", D.VARCHAR, max_length=32, is_primary=True), F("embedding", D.FLOAT_VECTOR, dim=DIM),
            F("period", D.VARCHAR, max_length=20), F("value", D.INT64)]


def rows(n, seed, first=0, period=None):
    emb = O.synth_rows(seed, 0, n, DIM)
    ids = [f"c{first + i}" for i in range(n)]
    periods = [period or f"Q{(first + i) % 4 + 1}" for i in range(n)]
    return [ids, emb, periods, [first + i for i in range(n)]], emb


def make(name="dele", n=40, seed=3):
    if mc.utility.has_collection(name):
        mc.utility.drop_collection(name)
    col = mc.Collection(name, mc.CollectionSchema(fields(), "deletion"), index_factory=TombstoneIndex, initial_capacity=16)
    col.create_index("embedding", {"metric_type": "COSINE"})
    data, emb = rows(n, seed)
    col.insert(data)
    col.flush()
    return col, emb


def expected(emb_live, pks_live, q, k):
    """Oracle answer over the live rows only -> list of pk lists."""
    ids, _ = O.cosine_topk(q, O.normalize_rows(emb_live, "f32"), k)
    return [[pks_live[i] for i in r if i >= 0] for r in ids]


def hit_ids(res):
    return [h.ids for h in res]


def test_delete_by_pk_and_by_field_counts_and_hides_rows():
    col, emb = make()
    r = col.delete('id in ["c1", "c3", "c3", "nope"]')
    assert r.delete_count == 2 and sorted(r.primary_keys) == ["c1", "c3"] and r.insert_count == 0
    assert col.delete('id in ["c1"]').delete_count == 0                     # already deleted: nothing to do
    r = col.delete('period == "Q1"')                                         # rows 0, 4, 8, ...
    assert r.delete_count == 10 and "c0" in r.primary_keys and "c1" not in r.primary_keys
    dead = {1, 3} | set(range(0, 40, 4))
    live = [i for i in range(40) if i not in dead]
    q = O.synth_rows(9, 0, 3, DIM)
    got = col.search(q, "embedding", {"metric_type": "COSINE"}, limit=50)
    assert hit_ids(got) == expected(emb[live], [f"c{i}" for i in live], q, 50)
    # filtered search: the filter selects deleted rows too, they never come back
    got = col.search(q, "embedding", {}, limit=50, expr='period in ["Q1", "Q2"]')
    keep = [i for i in live if i % 4 in (0, 1)]
    assert hit_ids(got) == expected(emb[keep], [f"c{i}" for i in keep], q, 50)
    # query never returns deleted rows
    assert [x["id"] for x in col.query('period == "Q1"')] == []
    assert [x["id"] for x in col.query('id in ["c1", "c2"]')] == ["c2"]
    assert len(col.query("", limit=100)) == len(live)


def test_num_entities_counts_stored_rows_until_compact():
    col, _ = make()
    col.delete('id in ["c0", "c5"]')
    assert col.num_entities == 40            # Milvus: deleted rows are counted until compaction
    col.compact()
    assert col.num_entities == 38
    assert col.get_compaction_state().state == "Completed"
    assert col.wait_for_compaction_completed().state == "Completed"


def test_upsert_replaces_rows_and_failed_validation_changes_nothing():
    col, emb = make()
    new_emb = O.synth_rows(21, 0, 2, DIM)
    r = col.upsert([["c2", "c99"], new_emb, ["Q9", "Q9"], [1002, 1099]])
    assert r.upsert_count == 2 and r.delete_count == 1 and r.insert_count == 2
    col.flush()
    assert col.num_entities == 42
    assert [x["value"] for x in col.query('id in ["c2"]', output_fields=["value"])] == [1002]
    live_emb = np.concatenate([np.delete(emb, 2, axis=0), new_emb])
    pks = [f"c{i}" for i in range(40) if i != 2] + ["c2", "c99"]
    q = np.concatenate([new_emb[:1], O.synth_rows(4, 0, 2, DIM)])
    got = col.search(q, "embedding", {}, limit=45)
    assert hit_ids(got) == expected(live_emb, pks, q, 45)
    assert got[0][0].id == "c2" and got[0][0].entity.get("value") is None
    # a failed validation leaves everything as it was
    before = (col.num_entities, dict(col._st.pk_to_row), set(col._st.dead))
    with pytest.raises(mc.MilvusException):
        col.upsert([["c4", "c5"], O.synth_rows(5, 0, 2, DIM), ["Q1", "x" * 21], [0, 0]])   # period too long
    with pytest.raises(mc.MilvusException):
        col.upsert([["c4", "c4"], O.synth_rows(5, 0, 2, DIM), ["Q1", "Q1"], [0, 0]])       # duplicate inside one call
    assert (col.num_entities, dict(col._st.pk_to_row), set(col._st.dead)) == before
    assert [x["id"] for x in col.query('id in ["c4", "c5"]')] == ["c4", "c5"]


def test_reinsert_of_a_deleted_pk():
    col, emb = make()
    with pytest.raises(mc.MilvusException):
        col.insert(rows(1, 30, first=7)[0])            # c7 is live: a duplicate
    col.delete('id == "c7"')
    data, e7 = rows(1, 30, first=7)
    assert col.insert(data).insert_count == 1
    got = col.search(e7, "embedding", {}, limit=1, output_fields=["value"])
    assert got[0][0].id == "c7" and got[0][0].distance == pytest.approx(1.0, abs=1e-6)
    assert len(col.query('id == "c7"')) == 1


def test_compact_remaps_pks_columns_and_scalar_filters():
    col, emb = make()
    col.search(emb[:1], "embedding", {}, limit=3, expr='period == "Q2"')   # builds the scalar index for `period`
    col.delete('id in ["c0", "c1", "c10", "c39"]')
    before = col.search(emb[:4], "embedding", {}, limit=10, expr='period == "Q2"', output_fields=["value"])
    col.compact()
    st = col._st
    live = [i for i in range(40) if i not in (0, 1, 10, 39)]
    assert st.columns["id"] == [f"c{i}" for i in live] and st.columns["value"] == live
    assert st.pk_to_row == {f"c{i}": j for j, i in enumerate(live)}
    assert st.scalar_index["period"]["Q2"] == [j for j, i in enumerate(live) if i % 4 == 1]
    after = col.search(emb[:4], "embedding", {}, limit=10, expr='period == "Q2"', output_fields=["value"])
    assert hit_ids(after) == hit_ids(before)
    assert [[h.entity.value for h in hs] for hs in after] == [[h.entity.value for h in hs] for hs in before]
    assert [x["value"] for x in col.query('id in ["c2", "c11"]', output_fields=["value"])] == [2, 11]
    # inserts after a compaction continue at the new row count
    col.insert(rows(2, 40, first=100)[0])
    col.flush()
    assert col.query('id in ["c101"]')[0]["id"] == "c101" and st.pk_to_row["c101"] == 37


def test_save_load_round_trip_keeps_deletions(tmp_path):
    col, emb = make("persist")
    col.delete('id in ["c3", "c4"]')
    q = O.synth_rows(8, 0, 2, DIM)
    want = hit_ids(col.search(q, "embedding", {}, limit=40))
    mc.save_collection("persist", str(tmp_path))
    col2 = mc.load_collection("persist", str(tmp_path), index_loader=TombstoneIndex.load)
    assert col2._st.dead == {3, 4} and "c3" not in col2._st.pk_to_row
    assert col2.num_entities == 40
    assert hit_ids(col2.search(q, "embedding", {}, limit=40)) == want
    assert col2.query('id == "c4"') == []
    # a matrix file whose live mask disagrees with the recorded deletions is refused
    import json
    meta_path = os.path.join(str(tmp_path), "persist.columns.json")
    meta = json.load(open(meta_path))
    meta["deleted"] = [3]
    json.dump(meta, open(meta_path, "w"))
    with pytest.raises(mc.MilvusException):
        mc.load_collection("persist", str(tmp_path), index_loader=TombstoneIndex.load)


def test_delete_validates_its_expression():
    col, _ = make()
    for bad in ("", "   ", 'id like "c%"'):
        with pytest.raises(mc.MilvusException):
            col.delete(bad)
    assert col.delete('id in ["zz"]').delete_count == 0


def test_new_symbols_validate_null_handles():
    import __graft_entry__ as ge
    from ragfin_b200 import _lib
    if not os.path.exists(_lib.SO_PATH):
        ge.build()
    L = _lib.load()
    n = ctypes.c_int64(-5)
    ids = (ctypes.c_int64 * 1)(0)
    assert L.ragfin_delete(None, ids, 1, ctypes.byref(n)) == _lib.EINVAL
    assert L.ragfin_live_count(None, ctypes.byref(n)) == _lib.EINVAL
    words = (ctypes.c_uint32 * 1)()
    assert L.ragfin_read_live_mask(None, words) == _lib.EINVAL
    assert L.ragfin_compact(None) == _lib.EINVAL
    assert b"NULL" in L.ragfin_last_error()
