"""GPU suite for the "f32+f16" storage type (include/ragfin.h RAGFIN_F32_F16): the fp32 rows are bit for bit those of an f32
collection, the fp16 copy bit for bit what an f16 collection stores, and every search path returns the ids, score bits and
padding of the f32 collection and of the f32 oracle."""
import numpy as np
import pytest

from oracle import ragfin_oracle as O

pytestmark = pytest.mark.gpu
DT = "f32+f16"


def _index(x, dtype, capacity=None, device_src=False):
    import ragfin_b200
    idx = ragfin_b200.Index(x.shape[1], dtype, capacity=capacity or max(len(x), 1), device=0)
    if len(x):
        if device_src:
            import torch
            idx.add(torch.from_numpy(x).cuda())
        else:
            idx.add(x)
    return idx


def _same(got, want, what=""):
    gi, gs = got
    wi, ws = want
    assert np.array_equal(gi, wi), f"{what}: ids differ\n{gi}\n{wi}"
    assert np.array_equal(gs.view(np.uint32), ws.view(np.uint32)), f"{what}: score bits differ\n{gs}\n{ws}"


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ------------------------------------------------------------------------------------------------
# 1. ingest: both copies, every source
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [8, 33, 100, 384, 768, 1024, 2048])
def test_ingest_writes_the_f32_rows_and_the_f16_copy(coracle, dim):
    import ragfin_b200
    x = O.synth_rows(3, 0, 777, dim, zero_every=17)
    x[5] *= 1000.0
    x[6] *= 1e-6
    for device_src in (False, True):
        both = _index(x, DT, device_src=device_src)
        f32, f16 = _index(x, "f32", device_src=device_src), _index(x, "f16", device_src=device_src)
        assert np.array_equal(_bits(both.read_rows(0, 777)), _bits(f32.read_rows(0, 777)))
        assert np.array_equal(_bits(both.read_rows(0, 777)), _bits(coracle.normalize_rows(x, "f32")))
        assert np.array_equal(_bits(both.read_sweep_rows(0, 777)), _bits(f16.read_rows(0, 777)))
        assert np.array_equal(_bits(f32.read_sweep_rows(0, 777)), _bits(f32.read_rows(0, 777)))   # no copy: the stored rows
        for i in (both, f32, f16):
            i.close()
    synth = {}
    for dtype in (DT, "f32", "f16"):
        idx = ragfin_b200.Index(dim, dtype, capacity=3000, device=0)
        idx.add_synthetic(1234, 0, 1000, dup_every=7, zero_every=11)
        idx.add_synthetic_topics(1234, 1000, 2000, topic_rows=300, noise_shift=3)
        synth[dtype] = (idx.read_rows(0, 3000), idx.read_sweep_rows(0, 3000))
        idx.close()
    assert np.array_equal(_bits(synth[DT][0]), _bits(synth["f32"][0]))
    assert np.array_equal(_bits(synth[DT][1]), _bits(synth["f16"][0]))


# ------------------------------------------------------------------------------------------------
# 2. results: every path equals the f32 collection and the f32 oracle
# ------------------------------------------------------------------------------------------------
def _check(coracle, both, f32, q, k, what, stored=None, x=None, allow=None):
    got = both.search(q, k, allow=allow)
    ref = f32.search(q, k, allow=allow)
    _same(got, ref, f"{what}: vs f32 collection")
    if stored is None:
        stored = coracle.normalize_rows(x, "f32")
    if allow is None:
        want = coracle.cosine_topk(q, stored, k)
    else:
        rows = np.flatnonzero(allow)
        wi, ws = coracle.cosine_topk(q, stored[rows], k)
        want = (np.where(wi >= 0, rows[np.clip(wi, 0, None)] if len(rows) else -1, -1), ws)
    _same(got, want, f"{what}: vs oracle")
    return got


def test_one_kernel_and_multi_kernel_searches(coracle):
    import torch
    n, dim = 20000, 768
    x = O.synth_rows(40, 0, n, dim, dup_every=97, zero_every=1013)
    q = O.synth_rows(41, 0, 16, dim)
    stored = coracle.normalize_rows(x, "f32")
    both, f32 = _index(x, DT), _index(x, "f32")
    want128 = coracle.cosine_topk(q, stored, 128)
    allow = np.random.default_rng(3).random(n) < 0.4
    qd = torch.from_numpy(q).cuda()
    for fused in (True, False):
        both.set_fused(fused)
        f32.set_fused(fused)
        for nq in (1, 2, 9, 16):
            for k in (1, 10, 100, 128):
                what = f"fused={fused} nq={nq} k={k}"
                got = both.search(q[:nq], k)
                _same(got, (want128[0][:nq, :k], want128[1][:nq, :k]), what)
                _same(got, f32.search(q[:nq], k), what + " vs f32")
                ids, sc = both.search_device(qd[:nq], k)
                _same((ids.cpu().numpy(), sc.cpu().numpy()), got, what + " device")
                _check(coracle, both, f32, q[:nq], k, what + " filtered", stored=stored, allow=allow)
                if fused and nq <= 2 and k <= 100:
                    assert both.stats()["path"] == 3
    both.set_fused(True)
    both.set_pipelined(True)
    outs = [(nq, k, both.search_device(qd[:nq], k)) for _ in range(5) for nq, k in ((1, 10), (2, 5), (16, 10), (1, 100))]
    torch.cuda.synchronize()
    for nq, k, (ids, sc) in outs:
        _same((ids.cpu().numpy(), sc.cpu().numpy()), (want128[0][:nq, :k], want128[1][:nq, :k]), f"pipelined nq={nq} k={k}")
    both.close()
    f32.close()


def test_tensor_core_modes_pairs_and_large_k(coracle):
    n, dim = 60000, 768
    x = O.synth_rows(45, 0, n, dim, dup_every=53, zero_every=509)
    stored = coracle.normalize_rows(x, "f32")
    both, f32 = _index(x, DT), _index(x, "f32")
    q = O.synth_rows(46, 0, 1030, dim)
    for append in (True, False):                          # append mode, or K' lists seeded by the bound pass
        both.set_append_mode(append)
        f32.set_append_mode(append)
        for nq, k in ((17, 10), (128, 100)):
            _check(coracle, both, f32, q[:nq], k, f"append={append} nq={nq} k={k}", stored=stored)
            assert both.stats()["path"] == 1
    both.set_append_mode(True)
    f32.set_append_mode(True)
    for nq in (129, 300, 1030):                           # 2-SM MMA pairs
        _check(coracle, both, f32, q[:nq], 10, f"pairs nq={nq}", stored=stored)
    for k, nq in ((300, 3), (1000, 17), (5000, 2)):       # batched large k: approximate dump, exact rescore from the fp32 rows
        _check(coracle, both, f32, q[:nq], k, f"large k={k}", stored=stored)
        assert both.stats()["path"] == 2
    both.close()
    f32.close()


def test_scan_small_corpora_empty_and_k_above_n(coracle):
    x = O.synth_rows(60, 0, 4096, 384, dup_every=31)
    q = O.synth_rows(61, 0, 2, 384)
    both, f32 = _index(x, DT), _index(x, "f32")
    for variant in (1, 2):                                # LDG scan and TMA-fed scan: they read the fp32 rows
        both.set_scan_variant(variant)
        f32.set_scan_variant(variant)
        for nq in (1, 2):
            _check(coracle, both, f32, q[:nq], 10, f"scan variant {variant} nq={nq}", x=x)
            assert both.stats()["path"] == 0
    for n in (1, 16, 33, 257):
        s, f = _index(x[:n], DT), _index(x[:n], "f32")
        for k in (3, 20, 300):
            got = _check(coracle, s, f, q, k, f"n={n} k={k}", x=x[:n])
            if k > n:
                assert (got[0][:, n:] == -1).all() and np.isneginf(got[1][:, n:]).all()
    import ragfin_b200
    empty = ragfin_b200.Index(384, DT, capacity=8, device=0)
    ids, sc = empty.search(np.ones((2, 384), np.float32), 3)
    assert (ids == -1).all() and np.isneginf(sc).all()


def test_duplicates_identical_rows_and_templated_corpus(coracle):
    import ragfin_b200
    from ragfin_b200.synthetic import synth_topic_rows
    x = O.synth_rows(70, 0, 20000, 768)
    q = O.synth_rows(71, 0, 2, 768)
    x[100:400] = q[0] * 3.0
    x[4000:4100] = q[1]
    both, f32 = _index(x, DT), _index(x, "f32")
    for fused in (True, False):
        both.set_fused(fused)
        f32.set_fused(fused)
        got = _check(coracle, both, f32, q, 10, f"duplicates fused={fused}", x=x)
        assert got[0][0].tolist() == list(range(100, 110))
    same = np.tile(O.synth_rows(80, 0, 1, 384), (9000, 1))
    qs = O.synth_rows(81, 0, 1, 384)
    got = _check(coracle, _index(same, DT), _index(same, "f32"), qs, 5, "identical rows", x=same)
    assert got[0][0].tolist() == [0, 1, 2, 3, 4]
    n, dim, topic_rows = 120000, 128, 6000
    rows_fn = lambda s, r0, m, d: coracle.synth_rows(s, r0, m, d)
    xt = synth_topic_rows(700, 0, n, dim, topic_rows, 3, rows_fn)
    qt = np.concatenate([synth_topic_rows(700, 7 * topic_rows + 11, 1, dim, topic_rows, 2, rows_fn), coracle.synth_rows(702, 0, 1, dim)])
    idx = {}
    for dtype in (DT, "f32"):
        idx[dtype] = ragfin_b200.Index(dim, dtype, capacity=n, device=0)
        idx[dtype].add_synthetic_topics(700, 0, n, topic_rows, 3)
        idx[dtype].set_fused(True, 1)
    _check(coracle, idx[DT], idx["f32"], qt, 10, "templated corpus", x=xt)
    assert idx[DT].stats()["path"] == 3 and idx[DT].stats()["queries_rescanned"] == 0


def test_view_reserve_save_load_and_merge(coracle, tmp_path):
    import torch
    import ragfin_b200
    n, dim = 30000, 768
    x = O.synth_rows(220, 0, n, dim, dup_every=17)
    q = O.synth_rows(221, 0, 12, dim)
    stored = coracle.normalize_rows(x, "f32")
    want = coracle.cosine_topk(q, stored, 10)
    both = _index(x[:20000], DT, capacity=20000)
    both.reserve(n)                                          # both matrices grow on the device
    both.add(x[20000:])
    _same(both.search(q, 10), want, "after reserve")
    _same(both.search(q[:1], 10), (want[0][:1], want[1][:1]), "after reserve, one query")
    v = both.view()
    _same(v.search(q, 10), want, "view")
    _same(v.search(q[:2], 10), (want[0][:2], want[1][:2]), "view, two queries")
    v.close()
    sweep = both.read_sweep_rows(0, n)
    path = str(tmp_path / "both.ragfin")
    both.save(path)
    both.close()
    with open(path, "rb") as f:
        assert int.from_bytes(f.read(64)[20:24], "little") == 3
    import os
    assert os.path.getsize(path) == 64 + n * dim * 4           # the fp32 rows only
    back = ragfin_b200.Index.load(path, device=0)
    assert back.dtype == DT and len(back) == n
    assert np.array_equal(_bits(back.read_sweep_rows(0, n)), _bits(sweep))   # the rebuilt copy is the ingested one
    assert np.array_equal(_bits(back.read_rows(0, n)), _bits(stored))
    _same(back.search(q, 10), want, "reloaded")
    _same(back.search(q[:1], 10), (want[0][:1], want[1][:1]), "reloaded, one query")
    back.close()
    qd = torch.from_numpy(q).cuda()
    shards, outs = [], []
    for a, b in ((0, 12000), (12000, n)):                     # two handles on one GPU, merged
        s = _index(x[a:b], DT)
        s.set_id_base(a)
        shards.append(s)
        outs.append(s.search_device(qd, 10))
    mi, ms = ragfin_b200.merge_topk(torch.cat([o[0] for o in outs], 1), torch.cat([o[1] for o in outs], 1), 2, 10)
    torch.cuda.synchronize()
    _same((mi.cpu().numpy(), ms.cpu().numpy()), want, "merged shards")


def test_shim_collection_with_the_fp16_copy(coracle, tmp_path):
    from ragfin_b200 import milvus_compat as mc
    F, D = mc.FieldSchema, mc.DataType
    fields = [F("id", D.INT64, is_primary=True), F("period", D.VARCHAR, max_length=20), F("embedding", D.FLOAT_VECTOR, dim=384)]
    mc.utility.drop_collection("copy")
    col = mc.Collection("copy", mc.CollectionSchema(fields, ""), storage_dtype=DT)
    x = O.synth_rows(230, 0, 10000, 384)
    col.insert([list(range(10000)), [f"Q{i % 4}" for i in range(10000)], x])
    col.flush()
    col.load()
    q = O.synth_rows(231, 0, 2, 384)
    stored = coracle.normalize_rows(x, "f32")
    wi, ws = coracle.cosine_topk(q, stored, 5)
    hits = col.search(q, "embedding", {"metric_type": "COSINE"}, limit=5)
    assert [h.id for h in hits[0]] == wi[0].tolist()
    rows = np.arange(10000)[np.arange(10000) % 4 == 1]
    fi, fs = coracle.cosine_topk(q, stored[rows], 5)
    hits = col.search(q, "embedding", {"metric_type": "COSINE"}, limit=5, expr='period == "Q1"')
    assert [h.id for h in hits[1]] == rows[fi[1]].tolist()
    mc.save_collection("copy", str(tmp_path))
    back = mc.load_collection("copy", str(tmp_path))
    hits = back.search(q, "embedding", {"metric_type": "COSINE"}, limit=5)
    assert [h.id for h in hits[0]] == wi[0].tolist()
    assert np.array_equal(np.array([h.score for h in hits[0]], np.float32).view(np.uint32), ws[0].view(np.uint32))
    mc.utility.drop_collection("copy")


# ------------------------------------------------------------------------------------------------
# 3. error bound of the sweep over the copy
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [384, 768, 2048])
def test_sweep_scores_equal_f16_and_stay_inside_the_bound(dim):
    """The raw tensor-core scores of an f32+f16 handle are those of an f16 collection (same operands, same kernel), and
    their error against the score of the fp32 rows stays inside eps_gemm_const(f16) + eps_sweep (csrc/ragfin_api.cu), on
    all-positive operands (largest partial sums, rounding errors of one sign) and random ones."""
    import math
    import torch
    ld = (dim + 7) // 8 * 8
    eps_gemm = (ld + 64) * 2.0 ** -22 * 1.0625 + 2.0 ** -21
    eps_sweep = (1 + 2.0 ** -22) * (2.0 ** -11 * (1 + 2.0 ** -20) + 2.0 ** -25 * math.sqrt(ld))
    worst = 0.0
    for positive in (True, False):
        x = O.synth_rows(510, 0, 4000, dim)
        q = O.synth_rows(511, 0, 130, dim)
        if positive:
            x, q = np.abs(x), np.abs(q)
        both, f16 = _index(x, DT), _index(x, "f16")
        qd = torch.from_numpy(q).cuda()
        got = both.debug_gemm_scores(qd).cpu().numpy()
        assert np.array_equal(_bits(got), _bits(f16.debug_gemm_scores(qd).cpu().numpy()))
        rows32 = both.read_rows(0, len(x)).astype(np.float64)
        q16 = O.round_to_storage(O.normalize_rows(q, "f32"), "f16").astype(np.float64)
        worst = max(worst, float(np.abs(got.astype(np.float64) - q16 @ rows32.T).max()))
        both.close()
        f16.close()
    assert worst <= eps_gemm + eps_sweep, (worst, eps_gemm, eps_sweep)


def test_host_calls_on_a_fresh_handle_wait_for_their_own_results(coracle):
    """A handle's first synchronous host call of the one-kernel search polls a completion word in mapped pinned memory; that
    memory may be what a destroyed handle left behind, still holding that handle's last sequence number.  Handles made and
    dropped one after the other, each searched once, must each return their own results."""
    for i, dtype in enumerate((DT, "f32", DT, "bf16", DT)):
        x = O.synth_rows(600 + i, 0, 9000, 128)
        q = O.synth_rows(700 + i, 0, 1 + i % 2, 128)
        idx = _index(x, dtype)
        idx.set_fused(True, 1)
        got = idx.search(q, 5 + i)
        assert idx.stats()["path"] == 3
        _same(got, coracle.cosine_topk(q, coracle.normalize_rows(x, "bf16" if dtype == "bf16" else "f32"), 5 + i), f"handle {i}")
        idx.close()
