"""GPU suite for grouping search (include/ragfin.h ragfin_search_grouped[_host], DESIGN.md 7d): the batched large-k route
and the exact path return exactly the reference answer (tests/_grouping.py grouped_topk) over the C oracle's exact
scores (ids and score bits), on all four dtypes, through host and device entry points with host and device codes, over
every code layout; grouping composes with filters, tombstones and views; a templated corpus overflows the batched route
into the exact path and stays exact."""
import numpy as np
import pytest

import _edge_families as E
from _grouping import grouped_topk
from oracle import ragfin_oracle as O
from test_edges_gpu import _eps_approx, _eps_q

pytestmark = pytest.mark.gpu

N, DIM = 40000, 256
DTYPES = ["f32", "bf16", "f16", "f32+f16"]
NQS, KS = (1, 3, 20), (1, 10, 100, 300)


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


def _same(got, want, what=""):
    gi, gs = (np.asarray(a.cpu()) if hasattr(a, "cpu") else a for a in got)
    wi, ws = want
    assert np.array_equal(gi, wi), f"{what}: ids differ\n{gi[:2, :12]}\n{wi[:2, :12]}"
    assert np.array_equal(np.ascontiguousarray(gs).view(np.uint32), np.ascontiguousarray(ws).view(np.uint32)), f"{what}: score bits differ"


def _layouts(n):
    """(name, codes int32 [n], n_groups)."""
    rng = np.random.default_rng(7)
    return [
        ("runs of 16", np.arange(n, dtype=np.int32) // 16, (n + 15) // 16),
        ("1000 random groups", rng.integers(0, 1000, n).astype(np.int32), 1000),
        ("single group", np.zeros(n, np.int32), 1),
        ("one group per row", np.arange(n, dtype=np.int32), n),
        ("fewer groups than k", (np.arange(n) % 5).astype(np.int32), 5),
        ("unused codes", (rng.integers(0, 500, n) * 2).astype(np.int32), 1000),
        ("codes out of range", rng.integers(-50, 1050, n).astype(np.int32), 1000),
    ]


def _search(idx, q, k, codes, ng, mode, allow=None):
    """mode: "host" (numpy codes), "host+dev" (host queries, CUDA codes), "device" (search_device)."""
    import torch
    if mode == "host":
        return idx.search(q, k, group_by=codes, n_groups=ng, allow=allow)
    gd = torch.from_numpy(codes).cuda()
    if mode == "host+dev":
        return idx.search(q, k, group_by=gd, n_groups=ng, allow=allow)
    got = idx.search_device(torch.from_numpy(q).cuda(), k, group_by=gd, n_groups=ng)
    torch.cuda.synchronize()
    return got


@pytest.mark.parametrize("dtype", DTYPES)
def test_batched_route_every_layout(coracle, dtype):
    x = O.synth_rows(1300, 0, N, DIM, dup_every=37)   # exact duplicates inside and across groups: the tie-break is by row
    q = O.synth_rows(1301, 0, max(NQS), DIM)
    idx = _index(x, dtype)
    S = _scores(coracle, q, _stored(coracle, x, dtype))
    for name, codes, ng in _layouts(N):
        want = grouped_topk(S, codes, ng, max(KS))   # the top-k groups are a prefix of the top-300 groups
        if name == "codes out of range":
            ok = want[0] >= 0
            assert ((codes[want[0][ok]] >= 0) & (codes[want[0][ok]] < ng)).all()
        for nq in NQS:
            for k in KS:
                for mode in ("host", "host+dev", "device"):
                    got = _search(idx, q[:nq], k, codes, ng, mode)
                    _same(got, (want[0][:nq, :k], want[1][:nq, :k]), f"{dtype} {name} nq={nq} k={k} {mode}")
                    st = idx.stats()
                    assert st["path"] == 2 and st["queries_rescanned"] == 0, (name, nq, k, st)
        if name == "one group per row":
            for k in (10, 300):
                _same(idx.search(q, k, group_by=codes, n_groups=ng), idx.search(q, k), f"{dtype} identity k={k}")
        if name == "single group":
            plain = idx.search(q, 1)
            got = idx.search(q, 10, group_by=codes, n_groups=ng)
            assert np.array_equal(got[0][:, :1], plain[0]) and (got[0][:, 1:] == -1).all()
            assert np.array_equal(got[1][:, :1].view(np.uint32), plain[1].view(np.uint32)) and (got[1][:, 1:] == -np.inf).all()
    idx.close()


@pytest.mark.parametrize("dtype", DTYPES)
def test_exact_path_small_corpus_and_knob(coracle, dtype, monkeypatch):
    x = O.synth_rows(1310, 0, N, DIM, dup_every=23)
    q = O.synth_rows(1311, 0, 3, DIM)
    small = _index(x[:3000], dtype)
    Ss = _scores(coracle, q, _stored(coracle, x[:3000], dtype))
    for name, codes, ng in _layouts(3000):
        want = grouped_topk(Ss, codes, ng, 300)
        for k in (1, 10, 300):
            for mode in ("host", "device"):
                _same(_search(small, q, k, codes, ng, mode), (want[0][:, :k], want[1][:, :k]), f"{dtype} small {name} k={k} {mode}")
                st = small.stats()
                assert st["path"] == 2 and st["queries_rescanned"] == 0, st
    small.close()
    monkeypatch.setenv("RAGFIN_NO_BIGK_BATCHED", "1")   # read when the handle is created
    idx = _index(x, dtype)
    S = _scores(coracle, q, _stored(coracle, x, dtype))
    for name, codes, ng in _layouts(N):
        want = grouped_topk(S, codes, ng, 100)
        for k in (10, 100):
            _same(_search(idx, q, k, codes, ng, "host"), (want[0][:, :k], want[1][:, :k]), f"{dtype} knob {name} k={k}")
            assert idx.stats()["path"] == 2
    idx.close()


@pytest.mark.parametrize("n", [3000, N])
def test_filters_tombstones_and_views(coracle, n):
    x = O.synth_rows(1320, 0, n, DIM, dup_every=41)
    q = O.synth_rows(1321, 0, 4, DIM)
    idx = _index(x, "bf16")
    S = _scores(coracle, q, _stored(coracle, x, "bf16"))
    codes = np.arange(n, dtype=np.int32) // 16
    ng = (n + 15) // 16
    allow = np.random.default_rng(3).random(n) < 0.6
    for mode in ("host", "host+dev"):
        _same(_search(idx, q, 50, codes, ng, mode, allow=allow), grouped_topk(S, codes, ng, 50, allow=allow), f"filter {mode}")
    # deleting each query's best row promotes the next row of its group
    before = grouped_topk(S, codes, ng, 10)
    live = np.ones(n, bool)
    dead = np.unique(before[0][:, 0])
    assert idx.delete(dead) == len(dead)
    live[dead] = False
    want = grouped_topk(S, codes, ng, 10, allow=live)
    every = idx.search(q, ng, group_by=codes, n_groups=ng)   # every group: the deleted row's group is still there
    _same(every, grouped_topk(S, codes, ng, ng, allow=live), "tombstones, every group")
    for i in range(len(q)):
        g0 = codes[before[0][i, 0]]
        promoted = [r for r in every[0][i] if r >= 0 and codes[r] == g0]
        assert len(promoted) == 1 and live[promoted[0]], "the group of the deleted row is represented by its next row"
    for mode in ("host", "host+dev", "device"):
        _same(_search(idx, q, 10, codes, ng, mode), want, f"tombstones {mode}")
    _same(_search(idx, q, 30, codes, ng, "host", allow=allow), grouped_topk(S, codes, ng, 30, allow=allow & live), "filter + tombstones")
    v = idx.view()
    _same(_search(v, q, 10, codes, ng, "host"), want, "view")
    v.close()
    idx.close()


@pytest.mark.parametrize("family", ["negative", "zeros", "sub_eps_2000", "low_dim_3", "extreme", "non_finite"])
@pytest.mark.parametrize("dtype", DTYPES)
def test_edge_families(coracle, family, dtype):
    x, q = E.build(family, N, DIM, 4)
    idx = _index(x, dtype)
    S = _scores(coracle, q, _stored(coracle, x, dtype))
    codes = (np.arange(N) // 16).astype(np.int32)
    ng = N // 16
    for k in (10, 100):
        _same(_search(idx, q, k, codes, ng, "host"), grouped_topk(S, codes, ng, k), f"{family} {dtype} k={k}")
        assert idx.stats()["path"] == 2
    idx.close()


def test_templated_corpus_overflows_into_the_exact_path(coracle):
    """Runs of 16 384 near-duplicates (noise 2^-10) grouped by run: every row of a run lies within 2 eps of its run's maximum,
    far more than the batched route's cmax = keff + 4 096 candidates, so every query takes the exact path."""
    import ragfin_b200
    from ragfin_b200.synthetic import synth_topic_rows
    n, dim, topic_rows, shift = 4 * 16384, 128, 16384, 10
    rows_fn = lambda s, r0, m, d: coracle.synth_rows(s, r0, m, d)   # noqa: E731
    x = synth_topic_rows(700, 0, n, dim, topic_rows, shift, rows_fn)
    q = np.concatenate([synth_topic_rows(700, 2 * topic_rows + 11, 1, dim, topic_rows, 2, rows_fn),
                        synth_topic_rows(701, 1 * topic_rows, 1, dim, topic_rows, 3, rows_fn)])
    idx = ragfin_b200.Index(dim, "bf16", capacity=n, device=0)
    idx.add_synthetic_topics(700, 0, n, topic_rows, shift)
    stored = coracle.normalize_rows(x, "bf16")
    assert np.array_equal(idx.read_rows(0, n), stored)
    S = _scores(coracle, q, stored)
    codes = (np.arange(n) // topic_rows).astype(np.int32)
    e = _eps_approx("bf16", dim) + _eps_q(coracle.normalize_rows(q, "f32"), "bf16")
    for k in (1, 10):
        cmax = k + 4096
        for i in range(len(q)):
            near = sum(int((S[i][codes == g] >= S[i][codes == g].max() - 2 * e[i]).sum()) for g in range(4))
            assert near > cmax, (i, near, cmax)
        for mode in ("host", "device"):
            _same(_search(idx, q, k, codes, 4, mode), grouped_topk(S, codes, 4, k), f"templated k={k} {mode}")
            st = idx.stats()
            assert st["path"] == 2 and st["queries_rescanned"] == len(q), st
    idx.close()


def test_shim_group_by_period(coracle):
    import json
    import os
    from ragfin_b200 import milvus_compat as mc
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fin_chunks_collection.json")) as f:
        chunks = json.load(f)["chunks"]
    F, D = mc.FieldSchema, mc.DataType
    if mc.utility.has_collection("grouped_gpu"):
        mc.utility.drop_collection("grouped_gpu")
    col = mc.Collection("grouped_gpu", mc.CollectionSchema([F("id", D.VARCHAR, max_length=96, is_primary=True),
                                                            F("embedding", D.FLOAT_VECTOR, dim=DIM),
                                                            F("period", D.VARCHAR, max_length=20)]))
    col.create_index("embedding", {"metric_type": "COSINE"})
    n = 20000
    x = O.synth_rows(1330, 0, n, DIM, dup_every=13)
    periods = [chunks[i % len(chunks)]["period"] for i in range(n)]
    col.insert([[f"{chunks[i % len(chunks)]['id']}#{i}" for i in range(n)], x, periods])
    col.flush()
    q = O.synth_rows(1331, 0, 3, DIM)
    S = _scores(coracle, q, coracle.normalize_rows(x, "f32"))
    first = {}
    codes = np.array([first.setdefault(p, len(first)) for p in periods], np.int32)
    want = grouped_topk(S, codes, len(first), 10)
    res = col.search(q, "embedding", {"metric_type": "COSINE"}, limit=10, group_by_field="period", output_fields=["period"])
    for h, i, s in zip(res, *want):
        assert len(h) == len(first) == 4
        assert [x_.entity.get("period") for x_ in h] == [periods[r] for r in i if r >= 0]
        assert len({x_.entity.get("period") for x_ in h}) == len(h)
        assert h.ids == [f"{chunks[r % len(chunks)]['id']}#{r}" for r in i if r >= 0]
        assert h.distances == [float(v) for v in s[i >= 0]]
    mc.utility.drop_collection("grouped_gpu")
