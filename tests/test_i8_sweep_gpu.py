"""GPU suite of the one-kernel search's int8 tile filter (csrc/sweep_fused.cuh, DESIGN.md 2.5), forced on small corpora with
Index.set_sweep_copy(True): the int8 copy holds what a CPU quantization of read_rows gives, and every search returns the ids
and score bits of the same search with the copy off and of the C oracle - every entry point, filters, tombstones, views,
mutations after the copy exists, the edge families, a templated corpus and a corpus sorted by similarity."""
import os
import tempfile

import numpy as np
import pytest

from oracle import ragfin_oracle as O

from _edge_families import build as edge_family

pytestmark = pytest.mark.gpu
N, DIM = 150_000, 256       # ~4 tiles per CTA on 148 SMs: most tiles are screened


def _index(x, dtype, copy=True, capacity=None):
    import ragfin_b200
    idx = ragfin_b200.Index(x.shape[1], dtype, capacity=capacity or len(x), device=0)
    idx.add(x)
    idx.set_sweep_copy(copy)
    return idx


def _same(got, want, what=""):
    assert np.array_equal(got[0], want[0]), f"{what}: ids differ\n{got[0]}\n{want[0]}"
    assert np.array_equal(np.ascontiguousarray(got[1]).view(np.uint32), np.ascontiguousarray(want[1]).view(np.uint32)), f"{what}: score bits differ"


def _both(idx, q, k, **kw):
    """The search with the int8 filter, then with it off; both results must agree bit for bit."""
    idx.set_sweep_copy(True)
    a = idx.search(q, k, **kw)
    st = idx.stats()
    tiles = idx.fused_tiles()
    idx.set_sweep_copy(False)
    b = idx.search(q, k, **kw)
    idx.set_sweep_copy(True)
    _same(a, b, f"copy on vs off k={k}")
    return a, st, tiles


def _cpu_quantize(rows):
    """What quantize_i8_kernel stores, in numpy fp32 (same roundings), and the exact residual norm in fp64."""
    x = rows.astype(np.float32)
    mx = np.abs(x).max(axis=1)
    live = np.isfinite(x).all(axis=1) & (mx > 0)
    s = np.where(live, mx / np.float32(127), np.float32(0)).astype(np.float32)
    with np.errstate(divide="ignore"):
        rs = np.where(live, np.float32(127) / np.where(live, mx, np.float32(1)), np.float32(0)).astype(np.float32)
    q = np.clip(np.rint((x * rs[:, None]).astype(np.float32)), -127, 127)
    q[~live] = 0
    d = x.astype(np.float64) - s[:, None].astype(np.float64) * q
    d[~live] = 0
    return q.astype(np.int8), s, np.sqrt((d * d).sum(axis=1))


@pytest.mark.parametrize("dtype", ["bf16", "f16"])
def test_copy_matches_cpu_quantization(dtype):
    x = O.synth_rows(11, 0, 20_000, 200, zero_every=97)
    x[3] *= 1e-30                                  # subnormal-range components in the stored row (bf16)
    x[5] = 0.0; x[5, 7] = 3.0                      # one component
    x[9, ::2] *= 1e-6                              # components far below the maximum
    idx = _index(x, dtype)
    idx.search(O.synth_rows(12, 0, 1, 200), 10)
    rows = idx.read_rows(0, len(x))
    q8, side = idx.sweep_copy_rows(0, len(x))
    want_q, want_s, want_e = _cpu_quantize(rows)
    assert q8.shape[1] % 16 == 0 and q8.shape[1] >= 200 and not q8[:, 200:].any()
    assert np.array_equal(q8[:, :200], want_q)
    assert np.array_equal(side[:, 0].view(np.uint32), want_s.view(np.uint32))
    e = side[:, 1].astype(np.float64)
    assert (e >= want_e).all()                      # rounded up
    assert (e <= want_e * (1 + 2e-6) + 1e-44).all()
    idx.close()


@pytest.mark.parametrize("dtype", ["bf16", "f16"])
@pytest.mark.parametrize("nq", [1, 8, 16])
@pytest.mark.parametrize("k", [1, 10, 100])
def test_parity_with_oracle_and_copy_off(coracle, dtype, nq, k):
    x = O.synth_rows(21, 0, N, DIM, dup_every=13)
    q = O.synth_rows(22, 0, nq, DIM)
    idx = _index(x, dtype)
    got, st, (t16, t8) = _both(idx, q, k)
    _same(got, coracle.cosine_topk(q, coracle.normalize_rows(x, dtype), k), "oracle")
    if st["path"] == 3:
        assert t8 > 0 and t16 >= 148, (t16, t8)      # every CTA's first tile in 16 bits, the others screened
    idx.close()


@pytest.mark.parametrize("dtype", ["bf16", "f16"])
def test_entry_points_filters_tombstones_views(coracle, dtype):
    import torch
    x = O.synth_rows(31, 0, N, DIM)
    q = O.synth_rows(32, 0, 4, DIM)
    idx = _index(x, dtype)
    stored = coracle.normalize_rows(x, dtype)
    _same(idx.search(q, 10), coracle.cosine_topk(q, stored, 10), "host")
    ids, sc = idx.search_device(torch.from_numpy(q).cuda(), 10)
    torch.cuda.synchronize()
    _same((ids.cpu().numpy(), sc.cpu().numpy()), coracle.cosine_topk(q, stored, 10), "device")
    allow = np.zeros(N, bool)
    allow[::3] = True
    want = coracle.cosine_topk(q, stored[allow], 10)
    got, _, _ = _both(idx, q, 10, allow=allow)
    rows = np.flatnonzero(allow)
    assert np.array_equal(got[0], np.where(want[0] >= 0, rows[np.maximum(want[0], 0)], -1))
    # tombstones: the best rows of every query deleted
    idx.delete(np.unique(idx.search(q, 5)[0].ravel()))
    _both(idx, q, 10)
    v = idx.view()
    _same(v.search(q, 10), idx.search(q, 10), "view")
    v.close()
    idx.close()


@pytest.mark.parametrize("dtype", ["bf16", "f16"])
def test_mutations_after_the_copy_exists(coracle, dtype):
    x = O.synth_rows(41, 0, N, DIM)
    y = O.synth_rows(43, 0, 60_000, DIM)
    q = O.synth_rows(42, 0, 3, DIM)
    idx = _index(x, dtype, capacity=N + 20_000)
    idx.search(q, 10)
    idx.add(y[:20_000])                              # rows past the copy: the next search extends it
    _both(idx, q, 10)
    idx.reserve(N + 60_000)                          # capacity outgrows the copy: rebuilt
    idx.add(y[20_000:])
    got, _, _ = _both(idx, q, 10)
    allx = np.concatenate([x, y])
    _same(got, coracle.cosine_topk(q, coracle.normalize_rows(allx, dtype), 10), "after add / reserve")
    rows = idx.read_rows(0, len(allx))
    q8, _ = idx.sweep_copy_rows(0, len(allx))
    assert np.array_equal(q8[:, :DIM], _cpu_quantize(rows)[0])
    idx.delete(np.arange(0, len(allx), 2))
    idx.compact()                                    # rows move: the copy is rebuilt from the compacted rows
    got, _, _ = _both(idx, q, 10)
    _same(got, coracle.cosine_topk(q, coracle.normalize_rows(allx[1::2], dtype), 10), "after compact")
    with tempfile.TemporaryDirectory() as d:
        import ragfin_b200
        p = os.path.join(d, "c.rf")
        idx.save(p)
        back = ragfin_b200.Index.load(p)
        back.set_sweep_copy(True)
        _same(back.search(q, 10), got, "after load")
        back.close()
    idx.close()


@pytest.mark.parametrize("family", ["negative", "zeros", "sub_eps_64", "low_dim_3", "extreme", "non_finite"])
@pytest.mark.parametrize("dtype", ["bf16", "f16"])
def test_edge_families(coracle, family, dtype):
    x, q = edge_family(family, 60_000, DIM, 4)
    idx = _index(x, dtype)
    got, _, _ = _both(idx, q, 10)
    _same(got, coracle.cosine_topk(q, coracle.normalize_rows(x, dtype), 10), family)
    idx.close()


def test_templated_corpus_needs_no_exact_scan():
    import ragfin_b200
    n, topic = 600_000, 16_384
    idx = ragfin_b200.Index(DIM, "bf16", capacity=n, device=0)
    idx.add_synthetic_topics(51, 0, n, topic_rows=topic, noise_shift=3)
    idx.set_sweep_copy(True)
    rows = idx.read_rows(0, n)
    q = rows[[topic * 5 + 7, topic * 20 + 3]].astype(np.float32) + O.synth_rows(52, 0, 2, DIM) / 4
    got, st, (t16, t8) = _both(idx, q, 10)
    assert st["queries_rescanned"] == 0
    assert (idx.fused_counts(2)[1] >= 0).all()
    assert t8 > 0
    idx.close()


def test_sorted_corpus_refines_every_tile():
    """Rows sorted by similarity to the query, all within the int8 bound of each other: no tile can be skipped."""
    n = 100_000
    base = O.synth_rows(61, 0, 1, DIM)[0]
    noise = O.synth_rows(62, 0, n, DIM) * 1e-4
    x = (base[None, :] + noise).astype(np.float32)
    idx = _index(x, "bf16", copy=False)
    idx.search(base[None, :], 10)
    all_tiles, none = idx.fused_tiles()
    assert none == 0
    got, st, (t16, t8) = _both(idx, base[None, :], 10)
    assert st["path"] == 3
    assert t16 == all_tiles and t8 > 0, (t16, t8, all_tiles)
    idx.close()
