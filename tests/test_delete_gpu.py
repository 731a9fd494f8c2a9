"""GPU suite for row deletion (include/ragfin.h ragfin_delete / ragfin_compact): every search path, forced with the tuning
knobs, returns exactly the oracle's top-k over the LIVE rows (ids and score bits); the tombstone mask survives add, reserve,
views and files; compaction moves the survivors bit for bit and answers like a collection built from them."""
import numpy as np
import pytest

from oracle import ragfin_oracle as O

pytestmark = pytest.mark.gpu

N, DIM = 40000, 256
DTYPES = ["f32", "bf16", "f16", "f32+f16"]


def _index(x, dtype, capacity=None):
    import ragfin_b200
    idx = ragfin_b200.Index(x.shape[1], dtype, capacity=capacity or max(len(x), 1), device=0)
    if len(x):
        idx.add(x)
    return idx


def _stored(coracle, x, dtype):
    return coracle.normalize_rows(x, "f32" if dtype == "f32+f16" else dtype)


def _oracle_live(coracle, q, stored, live, k):
    rows = np.flatnonzero(live)
    if not len(rows):
        return np.full((len(q), k), -1, np.int64), np.full((len(q), k), -np.inf, np.float32)
    ids, sc = coracle.cosine_topk(q, stored[rows], k)
    return np.where(ids >= 0, rows[np.clip(ids, 0, None)], -1), sc


def _same(got, want, what=""):
    gi, gs = (np.asarray(a.cpu()) if hasattr(a, "cpu") else a for a in got)
    wi, ws = want
    assert np.array_equal(gi, wi), f"{what}: ids differ\n{gi[:2]}\n{wi[:2]}"
    assert np.array_equal(np.ascontiguousarray(gs).view(np.uint32), np.ascontiguousarray(ws).view(np.uint32)), f"{what}: score bits differ"


def _reset(idx):
    idx.set_fused(True)
    idx.set_gemm_variant(0)
    idx.set_append_mode(True)
    idx.set_bound_pass(True)


def _delete_random(idx, n, frac, seed):
    rng = np.random.default_rng(seed)
    dead = rng.random(n) < frac
    ids = np.flatnonzero(dead)
    assert idx.delete(np.concatenate([ids, ids[:5]])) == len(ids)     # duplicates count once
    assert idx.delete(ids[:3]) == 0                                  # already deleted
    return ~dead


# (name, knobs, nq, k, expected stats path)
PATHS = [
    ("one-kernel b1", dict(), 1, 10, 3),
    ("one-kernel b16", dict(), 16, 10, 3),
    ("gemm_rows append", dict(fused=False), 8, 10, 1),
    ("pair append", dict(), 160, 10, 1),
    ("single-CTA MODE 3", dict(variant=1), 40, 10, 1),
    ("single-CTA MODE 3, 2 tiles", dict(variant=1), 160, 10, 1),
    ("list mode + bound pass", dict(fused=False, append=False), 40, 10, 1),
    ("batched large k", dict(), 2, 1000, 2),
]


def _apply(idx, knobs):
    _reset(idx)
    if knobs.get("fused") is False:
        idx.set_fused(False)
    if "variant" in knobs:
        idx.set_gemm_variant(knobs["variant"])
    if knobs.get("append") is False:
        idx.set_append_mode(False)


@pytest.mark.parametrize("dtype", DTYPES)
def test_every_path_returns_the_oracle_over_live_rows(coracle, dtype):
    import torch
    x = O.synth_rows(900, 0, N, DIM, dup_every=37)
    q = O.synth_rows(901, 0, 160, DIM)
    q[3] = x[1234]                          # a query whose exact match is deleted
    idx = _index(x, dtype)
    live = _delete_random(idx, N, 0.01, 1)
    assert idx.delete([1234]) == (1 if live[1234] else 0)
    live[1234] = False
    assert idx.live_count == live.sum() and len(idx) == N
    assert np.array_equal(idx.live_mask(), live)
    stored = _stored(coracle, x, dtype)
    want10 = _oracle_live(coracle, q, stored, live, 10)
    want1000 = _oracle_live(coracle, q[:2], stored, live, 1000)
    for name, knobs, nq, k, path in PATHS:
        _apply(idx, knobs)
        want = want1000 if k == 1000 else (want10[0][:nq], want10[1][:nq])
        _same(idx.search(q[:nq], k), want, f"{dtype} {name} host")
        assert idx.stats()["path"] == path, (name, idx.stats())
        if path != 2 and "list" not in name:     # append mode and the one-kernel search: no exact fallback
            assert idx.stats()["queries_rescanned"] == 0, (name, idx.stats())
        qd = torch.from_numpy(q[:nq]).cuda()
        got = idx.search_device(qd, k)
        torch.cuda.synchronize()
        _same(got, want, f"{dtype} {name} device")
    # the scan (small corpus, 1-2 queries) and the one-query large-k path
    small = _index(x[:5000], dtype)
    live_s = _delete_random(small, 5000, 0.05, 2)
    _same(small.search(q[:2], 10), _oracle_live(coracle, q[:2], stored[:5000], live_s, 10), f"{dtype} scan")
    assert small.stats()["path"] == 0


def test_one_query_large_k_path(coracle, monkeypatch):
    monkeypatch.setenv("RAGFIN_NO_BIGK_BATCHED", "1")
    x = O.synth_rows(910, 0, 20000, DIM)
    q = O.synth_rows(911, 0, 2, DIM)
    idx = _index(x, "bf16")
    live = _delete_random(idx, 20000, 0.3, 3)
    _same(idx.search(q, 1000), _oracle_live(coracle, q, _stored(coracle, x, "bf16"), live, 1000), "one-query large k")
    assert idx.stats()["path"] == 2


@pytest.mark.parametrize("pattern", ["90%", "fewer than k", "all"])
def test_deletion_patterns(coracle, pattern):
    x = O.synth_rows(920, 0, N, DIM)
    q = O.synth_rows(921, 0, 160, DIM)
    idx = _index(x, "bf16")
    if pattern == "90%":
        live = _delete_random(idx, N, 0.9, 4)
    else:
        keep = np.array([5, 777, 30001]) if pattern == "fewer than k" else np.array([], np.int64)
        live = np.zeros(N, bool)
        live[keep] = True
        assert idx.delete(np.flatnonzero(~live)) == N - len(keep)
    stored = _stored(coracle, x, "bf16")
    for name, knobs, nq, k, _ in PATHS:
        _apply(idx, knobs)
        got = idx.search(q[:nq], k)
        _same(got, _oracle_live(coracle, q[:nq], stored, live, k), f"{pattern} {name}")
        if pattern == "all":
            assert (got[0] == -1).all() and np.isneginf(got[1]).all()


def test_filter_plus_tombstones_host_and_device_masks(coracle):
    import torch
    from ragfin_b200 import _lib
    x = O.synth_rows(930, 0, N, DIM, dup_every=19)
    q = O.synth_rows(931, 0, 40, DIM)
    idx = _index(x, "f16")
    live = _delete_random(idx, N, 0.1, 5)
    allow = np.random.default_rng(6).random(N) < 0.4
    stored = _stored(coracle, x, "f16")
    packed = np.packbits(allow, bitorder="little").view(np.uint32)
    L = _lib.load()
    for nq, k in ((1, 10), (40, 10), (2, 300)):
        want = _oracle_live(coracle, q[:nq], stored, allow & live, k)
        _same(idx.search(q[:nq], k, allow=allow), want, f"host filter nq={nq} k={k}")
        qd = torch.from_numpy(q[:nq]).cuda()
        bits = torch.from_numpy(packed.view(np.int32).copy()).cuda()
        ids = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        sc = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        _lib.check(L.ragfin_search_filtered(idx._h, qd.data_ptr(), nq, k, bits.data_ptr(), int(allow.sum()), ids.data_ptr(),
                                            sc.data_ptr(), torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        _same((ids, sc), want, f"device filter nq={nq} k={k}")


def test_deleted_topic_runs_put_no_query_on_an_exact_fallback(coracle):
    """Templated corpus: the queries' own topic runs (16 384 near-duplicates each) are deleted.  No tombstoned row may take an
    append slot, so no query overflows to tier 2 or to the one-kernel search's in-kernel scan."""
    import ragfin_b200
    from ragfin_b200.synthetic import synth_topic_rows
    n, dim, topic_rows = 8 * 16384, 128, 16384
    rows_fn = lambda s, r0, m, d: coracle.synth_rows(s, r0, m, d)   # noqa: E731
    x = synth_topic_rows(700, 0, n, dim, topic_rows, 3, rows_fn)
    q = np.concatenate([synth_topic_rows(700, 3 * topic_rows + 11, 1, dim, topic_rows, 2, rows_fn),
                        synth_topic_rows(701, 5 * topic_rows, 1, dim, topic_rows, 3, rows_fn)])
    idx = ragfin_b200.Index(dim, "bf16", capacity=n, device=0)
    idx.add_synthetic_topics(700, 0, n, topic_rows, 3)
    live = np.ones(n, bool)
    for t in (3, 5):
        live[t * topic_rows:(t + 1) * topic_rows] = False
    assert idx.delete(np.flatnonzero(~live)) == 2 * topic_rows
    want = _oracle_live(coracle, q, coracle.normalize_rows(x, "bf16"), live, 10)
    idx.set_fused(True, 1)
    _same(idx.search(q, 10), want, "templated, one-kernel")
    assert idx.stats()["path"] == 3 and idx.stats()["queries_rescanned"] == 0
    appended, rescored = idx.fused_counts(2)
    assert (rescored >= 0).all(), rescored
    idx.set_fused(False)
    idx.set_gemm_min_batch(1)
    _same(idx.search(q, 10), want, "templated, gemm_rows append")
    assert idx.stats()["path"] == 1 and idx.stats()["queries_rescanned"] == 0


def test_delete_then_add_and_reserve(coracle):
    x = O.synth_rows(940, 0, 30000, DIM)
    q = O.synth_rows(941, 0, 20, DIM)
    idx = _index(x[:12000], "bf16", capacity=20000)
    live = np.ones(30000, bool)
    live[:12000] = _delete_random(idx, 12000, 0.2, 7)
    idx.add(x[12000:20000])                  # new rows are live
    idx.reserve(30000)                       # the mask grows with the matrix
    idx.add(x[20000:])
    assert idx.delete([25000, 12001]) == 2
    live[[25000, 12001]] = False
    assert np.array_equal(idx.live_mask(), live) and idx.live_count == live.sum()
    stored = _stored(coracle, x, "bf16")
    for nq in (1, 20):
        _same(idx.search(q[:nq], 10), _oracle_live(coracle, q[:nq], stored, live, 10), f"after add + reserve nq={nq}")


def test_save_load_round_trip_and_file_versions(coracle, tmp_path):
    import ragfin_b200
    x = O.synth_rows(950, 0, 20000, DIM)
    q = O.synth_rows(951, 0, 8, DIM)
    idx = _index(x, "f32+f16")
    p1 = str(tmp_path / "plain.ragfin")
    idx.save(p1)
    assert int.from_bytes(open(p1, "rb").read(12)[8:12], "little") == 1          # no deletions: today's version-1 file
    live = _delete_random(idx, 20000, 0.05, 8)
    p2 = str(tmp_path / "dead.ragfin")
    idx.save(p2)
    hd = open(p2, "rb").read(64)
    assert int.from_bytes(hd[8:12], "little") == 2 and int.from_bytes(hd[40:48], "little") == (~live).sum()
    back = ragfin_b200.Index.load(p2, device=0)
    assert np.array_equal(back.live_mask(), live) and back.live_count == live.sum() and len(back) == 20000
    assert np.array_equal(back.read_rows(0, 20000).view(np.uint32), idx.read_rows(0, 20000).view(np.uint32))
    for nq in (1, 8):
        _same(back.search(q[:nq], 10), idx.search(q[:nq], 10), f"reloaded nq={nq}")
        _same(back.search(q[:nq], 10), _oracle_live(coracle, q[:nq], _stored(coracle, x, "f32+f16"), live, 10), "oracle")


@pytest.mark.parametrize("dtype", ["bf16", "f32+f16"])
def test_compact_moves_survivors_and_answers_like_a_fresh_collection(coracle, dtype):
    x = O.synth_rows(960, 0, N, DIM, dup_every=23)
    q = O.synth_rows(961, 0, 40, DIM)
    idx = _index(x, dtype, capacity=N + 100)
    live = _delete_random(idx, N, 0.3, 9)
    before = [idx.search(q[:nq], 10) for nq in (1, 40)]
    survivors = idx.compact()
    assert np.array_equal(survivors, np.flatnonzero(live))
    assert len(idx) == live.sum() and idx.live_count == live.sum() and idx.live_mask().all()
    fresh = _index(x[survivors], dtype)
    m = len(survivors)
    assert np.array_equal(idx.read_rows(0, m).view(np.uint32), fresh.read_rows(0, m).view(np.uint32))
    assert np.array_equal(idx.read_sweep_rows(0, m).view(np.uint32), fresh.read_sweep_rows(0, m).view(np.uint32))
    for (bi, bs), nq in zip(before, (1, 40)):
        got = idx.search(q[:nq], 10)
        _same(got, fresh.search(q[:nq], 10), f"compacted vs fresh nq={nq}")
        _same((np.where(got[0] >= 0, survivors[np.clip(got[0], 0, None)], -1), got[1]), (bi, bs), f"ids map back nq={nq}")
    idx.add(x[:50])                                  # rows after a compaction append at the new count
    assert len(idx) == m + 50


def test_views_keep_their_snapshot_and_block_compaction(coracle):
    from ragfin_b200 import _lib
    x = O.synth_rows(970, 0, 20000, DIM)
    q = O.synth_rows(971, 0, 4, DIM)
    idx = _index(x, "bf16")
    first = np.arange(0, 20000, 7)
    idx.delete(first)
    v = idx.view()
    idx.delete(np.arange(1, 20000, 7))                # after the view was made: the view still sees these rows
    stored = _stored(coracle, x, "bf16")
    live_v = np.ones(20000, bool)
    live_v[first] = False
    live_p = live_v.copy()
    live_p[1::7] = False
    _same(v.search(q, 10), _oracle_live(coracle, q, stored, live_v, 10), "view snapshot")
    _same(idx.search(q, 10), _oracle_live(coracle, q, stored, live_p, 10), "parent")
    with pytest.raises(_lib.RagfinError) as e:
        idx.compact()
    assert e.value.code == _lib.EUNSUPPORTED
    with pytest.raises(_lib.RagfinError) as e:
        v.delete([3])
    assert e.value.code == _lib.EUNSUPPORTED
    v.close()
    assert np.array_equal(idx.compact(), np.flatnonzero(live_p))


def test_out_of_range_ids_change_nothing():
    from ragfin_b200 import _lib
    x = O.synth_rows(980, 0, 1000, 64)
    idx = _index(x, "f32")
    idx.delete([10])
    for bad in ([1000], [-1], [5, 6, 1000]):
        with pytest.raises(_lib.RagfinError) as e:
            idx.delete(bad)
        assert e.value.code == _lib.EINVAL
    assert idx.live_count == 999 and np.flatnonzero(~idx.live_mask()).tolist() == [10]
    idx.set_id_base(5000)                             # ids are id_base + row
    with pytest.raises(_lib.RagfinError):
        idx.delete([999])
    assert idx.delete([5011]) == 1 and idx.live_count == 998


def test_shim_delete_upsert_compact_save_load(tmp_path):
    from ragfin_b200 import milvus_compat as mc
    F, D = mc.FieldSchema, mc.DataType
    mc.utility.drop_collection("gdel")
    col = mc.Collection("gdel", mc.CollectionSchema([F("id", D.VARCHAR, max_length=100, is_primary=True),
                                                      F("embedding", D.FLOAT_VECTOR, dim=DIM), F("period", D.VARCHAR, max_length=20)]))
    x = O.synth_rows(990, 0, 3000, DIM)
    col.insert([[f"c{i}" for i in range(3000)], x, [f"Q{i % 4 + 1}" for i in range(3000)]])
    col.load()
    assert col.delete('id in ["c10", "c11"]').delete_count == 2
    assert col.delete('period == "Q2"').delete_count == 750             # c1, c5, ...: c10 and c11 are Q3 / Q4
    hits = col.search(x[10:12], "embedding", {"metric_type": "COSINE"}, 5)
    assert all(h.id not in ("c10", "c11") for hs in hits for h in hs)
    assert all(int(h.id[1:]) % 4 != 1 for hs in hits for h in hs)
    col.upsert([["c12"], x[10:11], ["Q1"]])
    col.flush()
    assert col.search(x[10:11], "embedding", {}, 1)[0][0].id == "c12"
    assert col.num_entities == 3001
    want = [h.id for h in col.search(x[:3], "embedding", {}, 5)[0]]
    mc.save_collection("gdel", str(tmp_path))
    back = mc.load_collection("gdel", str(tmp_path))          # replaces the open collection of that name
    assert [h.id for h in back.search(x[:3], "embedding", {}, 5)[0]] == want
    back.compact()
    assert back.num_entities == 3001 - 753                               # 752 deleted + c12 replaced
    assert back.search(x[10:11], "embedding", {}, 1)[0][0].id == "c12"
    mc.utility.drop_collection("gdel")
