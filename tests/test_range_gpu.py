"""GPU suite for range search (include/ragfin.h ragfin_search_range[_host]): every route - the three append epilogues, the
batched large-k pipeline and the one-query exact path - returns exactly the oracle's top-k over the rows with
radius < score <= range_filter (ids and score bits), on all four dtypes, through host and device entry points; the bounds
are fp32 compares on the returned score; windows compose with filters, tombstones and views; append overflow stays exact."""
import ctypes

import numpy as np
import pytest

from oracle import ragfin_oracle as O

pytestmark = pytest.mark.gpu

N, DIM = 40000, 256
DTYPES = ["f32", "bf16", "f16", "f32+f16"]


def _index(x, dtype):
    import ragfin_b200
    idx = ragfin_b200.Index(x.shape[1], dtype, capacity=len(x), device=0)
    idx.add(x)
    return idx


def _stored(coracle, x, dtype):
    return coracle.normalize_rows(x, "f32" if dtype == "f32+f16" else dtype)


def _scores(coracle, q, stored):
    qhat = coracle.normalize_rows(np.atleast_2d(q), "f32")
    return np.stack([coracle.exact_scores(stored, qhat[i]) for i in range(len(qhat))])


def _oracle(S, k, radius=-np.inf, range_filter=np.inf, allow=None):
    """Top k of exact scores S [nq, n] restricted to radius < s <= range_filter (fp32 compares), padded with (-1, -inf)."""
    lo, hi = np.float32(radius), np.float32(range_filter)
    ids = np.full((len(S), k), -1, np.int64)
    sc = np.full((len(S), k), -np.inf, np.float32)
    for i, s in enumerate(S):
        ok = (s > lo) & (s <= hi)
        if allow is not None:
            ok &= allow
        rows = np.flatnonzero(ok)
        order = rows[np.lexsort((rows, -s[rows].astype(np.float64)))][:k]
        ids[i, :len(order)], sc[i, :len(order)] = order, s[order]
    return ids, sc


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
    idx.set_gemm_min_batch(0)


# (name, knobs, nq, k, expected stats path)
ROUTES = [
    ("gemm_rows append", dict(), 8, 10, 1),
    ("single-CTA MODE 3", dict(variant=1), 40, 10, 1),
    ("pair append", dict(variant=4), 160, 10, 1),
    ("batched large k, append off", dict(append=False), 20, 10, 2),
    ("batched large k, k > 256", dict(), 3, 300, 2),
    ("batched large k, batch below the tensor-core minimum", dict(), 1, 10, 2),
]


def _apply(idx, knobs):
    _reset(idx)
    if "variant" in knobs:
        idx.set_gemm_variant(knobs["variant"])
    if knobs.get("append") is False:
        idx.set_append_mode(False)


def _windows(S):
    """(name, radius, range_filter) from the score distribution of the queries: a band, a floor, a ceiling."""
    flat = np.sort(S.ravel())
    q = lambda p: float(flat[int(p * (len(flat) - 1))])   # noqa: E731
    return [("band", q(0.95), q(0.999)), ("floor", q(0.9995), np.inf), ("ceiling", -np.inf, q(0.99))]


def _search(idx, q, k, radius, rf, device):
    import torch
    if device:
        got = idx.search_device(torch.from_numpy(q).cuda(), k, radius=radius, range_filter=rf)
        torch.cuda.synchronize()
        return got
    return idx.search(q, k, radius=radius, range_filter=rf)


@pytest.mark.parametrize("dtype", DTYPES)
def test_every_route_returns_the_oracle_over_the_window(coracle, dtype):
    x = O.synth_rows(1200, 0, N, DIM, dup_every=37)
    q = O.synth_rows(1201, 0, 160, DIM)
    idx = _index(x, dtype)
    S = _scores(coracle, q, _stored(coracle, x, dtype))
    for wname, radius, rf in _windows(S):
        for name, knobs, nq, k, path in ROUTES:
            _apply(idx, knobs)
            want = _oracle(S[:nq], k, radius, rf)
            for device in (False, True):
                _same(_search(idx, q[:nq], k, radius, rf, device), want, f"{dtype} {wname} {name} {'device' if device else 'host'}")
                st = idx.stats()
                assert st["path"] == path, (name, st)
                if path == 1:
                    assert st["queries_rescanned"] == 0, (name, st)
    # the one-query exact path: a corpus below 4 096 rows
    small = _index(x[:3000], dtype)
    Ss = _scores(coracle, q[:4], _stored(coracle, x[:3000], dtype))
    for wname, radius, rf in _windows(Ss):
        for device in (False, True):
            _same(_search(small, q[:4], 10, radius, rf, device), _oracle(Ss, 10, radius, rf), f"{dtype} {wname} search_bigk")
            assert small.stats()["path"] == 2


def test_bounds_are_fp32_compares_on_the_returned_score(coracle):
    x = O.synth_rows(1210, 0, N, DIM, dup_every=2)      # every odd row repeats its predecessor: every score is tied
    q = O.synth_rows(1211, 0, 8, DIM)
    idx = _index(x, "bf16")
    S = _scores(coracle, q, _stored(coracle, x, "bf16"))
    order = np.lexsort((np.arange(N), -S[0].astype(np.float64)))
    # the 7th-or-later best score whose fp32 successor no row scores (so that the window between them is empty)
    v = next(S[0, r] for r in order[6:] if not (S[0] == np.nextafter(S[0, r], np.float32(np.inf))).any())
    nxt = np.nextafter(v, np.float32(np.inf))
    tied = np.flatnonzero(S[0] == v)
    assert len(tied) >= 2
    for name, knobs, nq, k, _ in ROUTES:
        _apply(idx, knobs)
        qq, SS = q[:min(nq, 8)], S[:min(nq, 8)]
        got = idx.search(qq, k, radius=float(v))                       # radius == score: the row and its ties are out
        _same(got, _oracle(SS, k, v), f"radius tie {name}")
        assert not np.isin(tied, got[0][0]).any()
        got = idx.search(qq, k, radius=-1.0, range_filter=float(v))    # range_filter == score: they are in
        _same(got, _oracle(SS, k, -1.0, v), f"range_filter tie {name}")
        assert np.isin(tied, got[0][0]).all()
        got = idx.search(q[:1], k, radius=float(v), range_filter=float(nxt))   # between adjacent fp32 values: empty
        assert (got[0] == -1).all() and (got[1] == -np.inf).all(), name
        _same(idx.search(qq, k, radius=-np.inf, range_filter=np.inf), idx.search(qq, k), f"open bounds {name}")


def test_degenerate_windows(coracle):
    x = O.synth_rows(1220, 0, N, DIM)
    q = O.synth_rows(1221, 0, 40, DIM)
    idx = _index(x, "f16")
    S = _scores(coracle, q, _stored(coracle, x, "f16"))
    few = float(np.sort(S, axis=1)[:, -4].max())   # above it, every query keeps at most 3 rows
    for name, knobs, nq, k, _ in ROUTES:
        _apply(idx, knobs)
        qq, SS = q[:min(nq, 40)], S[:min(nq, 40)]
        got = idx.search(qq, k, radius=-3.0, range_filter=-2.0)
        assert (got[0] == -1).all() and (got[1] == -np.inf).all(), name
        _same(idx.search(qq, k, radius=few), _oracle(SS, k, few), f"fewer than k {name}")
        _same(idx.search(qq, k, radius=-2.0, range_filter=2.0), _oracle(SS, k), f"every row {name}")
        _same(idx.search(qq, k, radius=-2.0, range_filter=2.0), idx.search(qq, k), f"every row = plain {name}")


def test_window_composes_with_filters_tombstones_and_views(coracle):
    import torch
    x = O.synth_rows(1230, 0, N, DIM)
    q = O.synth_rows(1231, 0, 20, DIM)
    idx = _index(x, "bf16")
    S = _scores(coracle, q, _stored(coracle, x, "bf16"))
    radius, rf = _windows(S)[0][1:]
    rng = np.random.default_rng(5)
    allow = rng.random(N) < 0.5
    _reset(idx)
    want = _oracle(S, 10, radius, rf, allow)
    _same(idx.search(q, 10, allow=allow, radius=radius, range_filter=rf), want, "host mask")
    packed, n_allowed = idx._pack_allow(allow)
    mask_d = torch.from_numpy(packed.view(np.int32)).cuda()
    qd = torch.from_numpy(q).cuda()
    ids = torch.empty((20, 10), dtype=torch.int64, device="cuda")
    sc = torch.empty((20, 10), dtype=torch.float32, device="cuda")
    from ragfin_b200 import _lib
    window = (ctypes.c_float * 2)(radius, rf)
    _lib.check(idx._L.ragfin_search_range(idx._h, qd.data_ptr(), 20, 10, window, mask_d.data_ptr(), n_allowed, ids.data_ptr(),
                                          sc.data_ptr(), None))
    torch.cuda.synchronize()
    _same((ids, sc), want, "device mask")
    # tombstones: the append path keeps serving
    dead = rng.random(N) < 0.1
    idx.delete(np.flatnonzero(dead))
    for name, knobs, nq, k, path in ROUTES:
        _apply(idx, knobs)
        nq = min(nq, 20)
        _same(idx.search(q[:nq], k, radius=radius, range_filter=rf), _oracle(S[:nq], k, radius, rf, ~dead), f"tombstones {name}")
        assert idx.stats()["path"] == path
    _same(idx.search(q, 10, allow=allow, radius=radius, range_filter=rf), _oracle(S, 10, radius, rf, allow & ~dead), "mask + tombstones")
    v = idx.view()
    _same(v.search(q, 10, radius=radius, range_filter=rf), _oracle(S, 10, radius, rf, ~dead), "view")
    v.close()


def _topics(coracle):
    import ragfin_b200
    from ragfin_b200.synthetic import synth_topic_rows
    n, dim, topic_rows = 8 * 16384, 128, 16384
    rows_fn = lambda s, r0, m, d: coracle.synth_rows(s, r0, m, d)   # noqa: E731
    x = synth_topic_rows(700, 0, n, dim, topic_rows, 3, rows_fn)
    q = np.concatenate([synth_topic_rows(700, 3 * topic_rows + 11, 1, dim, topic_rows, 2, rows_fn),
                        synth_topic_rows(700, 5 * topic_rows + 99, 1, dim, topic_rows, 2, rows_fn)])
    idx = ragfin_b200.Index(dim, "bf16", capacity=n, device=0)
    idx.add_synthetic_topics(700, 0, n, topic_rows, 3)
    return idx, q, _scores(coracle, q, coracle.normalize_rows(x, "bf16")), topic_rows


def test_templated_ceiling_under_the_topic_run_needs_no_fallback(coracle):
    """A small templated corpus (8 runs of 16 384 rows, 512 tiles): the bound pass samples many tiles of every run, so the
    threshold comes from the best run below the ceiling and no query overflows.  It says nothing about corpora whose sample
    stride exceeds a run (10M rows: README, profiles/r04/range.json)."""
    idx, q, S, tr = _topics(coracle)
    runs = [S[0, 3 * tr:4 * tr], S[1, 5 * tr:6 * tr]]
    rf = float(min(r.min() for r in runs)) - 0.02
    outside = np.ones(S.shape[1], bool)
    outside[3 * tr:4 * tr] = outside[5 * tr:6 * tr] = False
    assert max(S[0, outside].max(), S[1, outside].max()) < rf     # the next-best rows lie outside the runs
    want = _oracle(S, 10, -np.inf, rf)
    _reset(idx)
    idx.set_gemm_min_batch(1)
    _same(idx.search(q, 10, range_filter=rf), want, "templated ceiling, append")
    assert idx.stats()["path"] == 1 and idx.stats()["queries_rescanned"] == 0, idx.stats()
    assert not np.isin(want[0][0], np.arange(3 * tr, 4 * tr)).any()


def test_overflow_stays_exact_and_is_counted(coracle):
    """Planted duplicates: every other row is all-zero, so 20 000 rows score exactly 0.  The window (-1e-3, 0] puts all of them
    into the append buffer (more than it holds) and into the large-k candidates: both routes fall back to their exact tier,
    count the queries in queries_rescanned and return the 10 lowest-id zero rows."""
    x = O.synth_rows(1240, 0, N, DIM, zero_every=2)
    q = O.synth_rows(1241, 0, 40, DIM)
    idx = _index(x, "bf16")
    S = _scores(coracle, q, _stored(coracle, x, "bf16"))
    assert (S[:, 1::2] == 0).all()
    for name, knobs, nq, k, path in ROUTES[:2] + ROUTES[3:4]:
        _apply(idx, knobs)
        want = _oracle(S[:nq], k, -1e-3, 0.0)
        assert (want[1] == 0).all()
        _same(idx.search(q[:nq], k, radius=-1e-3, range_filter=0.0), want, f"overflow {name}")
        st = idx.stats()
        assert st["path"] == path and st["queries_rescanned"] == nq, (name, st)


def test_shim_end_to_end(coracle):
    from ragfin_b200 import milvus_compat as mc
    F, D = mc.FieldSchema, mc.DataType
    if mc.utility.has_collection("range_gpu"):
        mc.utility.drop_collection("range_gpu")
    col = mc.Collection("range_gpu", mc.CollectionSchema([F("id", D.INT64, is_primary=True), F("embedding", D.FLOAT_VECTOR, dim=DIM)]))
    col.create_index("embedding", {"metric_type": "COSINE"})
    x = O.synth_rows(1250, 0, 20000, DIM)
    col.insert([list(range(20000)), x])
    col.flush()
    q = O.synth_rows(1251, 0, 4, DIM)
    S = _scores(coracle, q, coracle.normalize_rows(x, "f32"))
    radius, rf = 0.05, 0.15
    res = col.search(q, "embedding", {"metric_type": "COSINE", "params": {"radius": radius, "range_filter": rf}}, limit=10)
    ids, sc = _oracle(S, 10, radius, rf)
    for h, i, s in zip(res, ids, sc):
        assert h.ids == [int(r) for r in i if r >= 0]
        assert h.distances == [float(v) for v in s[i >= 0]]
    mc.utility.drop_collection("range_gpu")


def test_bad_windows_are_refused_by_the_library(coracle):
    import torch
    import ragfin_b200
    from ragfin_b200 import _lib
    x = O.synth_rows(1260, 0, 5000, DIM)
    q = O.synth_rows(1261, 0, 2, DIM)
    idx = _index(x, "bf16")
    qd = torch.from_numpy(q).cuda()
    for radius, rf, msg in ((0.5, 0.4, "greater than radius"), (0.5, 0.5, "greater than radius"), (np.nan, None, "NaN"),
                            (0.1, np.nan, "NaN"), (np.inf, None, "greater than radius")):
        with pytest.raises(ragfin_b200.RagfinError, match=msg) as e:
            idx.search(q, 5, radius=radius, range_filter=rf)
        assert e.value.code == _lib.EINVAL
        with pytest.raises(ragfin_b200.RagfinError, match=msg):
            idx.search_device(qd, 5, radius=radius, range_filter=rf)
    ids = torch.empty((2, 5), dtype=torch.int64, device="cuda")
    sc = torch.empty((2, 5), dtype=torch.float32, device="cuda")
    assert idx._L.ragfin_search_range(idx._h, qd.data_ptr(), 2, 5, None, None, 0, ids.data_ptr(), sc.data_ptr(), None) == _lib.EINVAL
    assert b"NULL range" in idx._L.ragfin_last_error()
    _same(idx.search(q, 5, radius=0.0), _oracle(_scores(coracle, q, _stored(coracle, x, "bf16")), 5, 0.0), "usable after errors")
