"""GPU suite at the numeric edges: every (family, path, dtype) cell returns the C oracle's ids and fp32 score bits, on the
path it was meant to take, with the exact fallbacks DESIGN.md 2.3-2.5 predict from the family's construction.

Families (tests/_edge_families.py): negative top-k scores, a block of ~35 000 rows scoring exactly 0 with the cut inside it,
clusters of 500 / 2 000 / 2 100 / 17 000 rows within ~1e-5 of each other (below and above the 2 048-row rescore cap and the
16 384-row append cap), dims 1-7 with components in {-1, 0, 1} (a handful of score values, +-1 included), extreme fp32
magnitudes, and NaN / Inf components (stored and searched as zero vectors).

Fallbacks are predicted per query from the oracle's exact scores S and each path's own eps, computed as the library computes
it (eps_gemm_const / eps_sweep_const / eps_fp32_accumulate in csrc/ragfin_api.cu; eps_q of prep_queries_kernel from the
oracle's normalised query; the one-kernel search's a-priori query term of the variant the cell runs, from
ragfin_debug_fused_plan).  The approximate error is taken as at most eps / 2:
test_tensor_core_error_stays_inside_the_allowance holds it below eps / 4.  With S_k the k-th exact score:
  * a cut T - 2 eps keeps every row with S >= S_k - eps for certain and no row below S_k - 3 eps;
  * the bound pass is simulated on the exact scores (bound_geometry: 256-row tiles, the rank-th largest sampled block maximum),
    which bounds the rows an append buffer can collect;
  * list mode's certificate over K' = 32 candidates holds for certain when S_k - S_K' > 1.5 eps and fails for certain when
    S_k - S_K' <= 0.5 eps.
Every cell asserts `queries_rescanned` (and, for the one-kernel search, `fused_counts`) unless one of its queries falls between
the certain cases.  Those cells are listed in UNPREDICTED with the reason, carry "-count_unpredicted" in their test id, and
assert that they still cannot be predicted (so the list cannot go stale).

Cells left out: k = 100 (needs 1 024 * k = 102 400 rows; the corpora have 40 000); filtered searches have no device entry
point in `Index`, so their device leg is not run."""
import os

import numpy as np
import pytest

import _edge_families as E
from oracle import ragfin_oracle as O
from test_delete_gpu import PATHS, _apply

pytestmark = pytest.mark.gpu

N, DIM, NQ = 40000, 256, 160
DTYPES = ["f32", "bf16", "f16", "f32+f16"]
FAMILIES = ["negative", "zeros", "sub_eps_500", "sub_eps_2000", "sub_eps_2100", "sub_eps_17000", "low_dim_1", "low_dim_2",
            "low_dim_3", "low_dim_4", "low_dim_7", "extreme", "non_finite"]
SMALL = 5000
KEEP = lambda n: np.arange(n) % 3 != 1          # noqa: E731  filter of the filtered cells

# (name, knobs, nq, k, stats path, fallback rule); knobs as test_delete_gpu._apply takes them, plus scan / filtered / range /
# one_query.  Rules: "fused" (one-kernel search: buffer cap 16 384 for k <= 16), "append" (rescore cap 2 048, buffer cap
# 16 384), "list" / "scan" (certificate over K' = 32 candidates), "bigk" (keff + max(keff, 4 096) compacted rows), None (the
# path counts no fallback: range and filtered searches, the one-query large-k path).
RULE = {"one-kernel b1": "fused", "one-kernel b16": "fused", "gemm_rows append": "append", "pair append": "append",
        "single-CTA MODE 3": "append", "single-CTA MODE 3, 2 tiles": "append", "list mode + bound pass": "list",
        "batched large k": "bigk"}
ALL_PATHS = [p + (RULE[p[0]],) for p in PATHS] + [
    ("scan v1", dict(scan=1), 2, 10, 0, "scan"),
    ("scan v2", dict(scan=2), 2, 10, 0, "scan"),
    ("one-query large k", dict(one_query=True), 2, 1000, 2, None),
    ("filtered one-kernel", dict(filtered=True), 1, 10, 3, None),
    ("filtered list mode", dict(filtered=True, fused=False, append=False), 40, 10, 1, None),
    ("range", dict(range=True), 40, 10, 1, None),
]
CELLS = [(f, d, p) for f in FAMILIES for d in DTYPES for p in ALL_PATHS]


def _same(got, want, what):
    gi, gs = (np.asarray(a.cpu()) if hasattr(a, "cpu") else np.asarray(a) for a in got)
    wi, ws = want
    assert np.array_equal(gi, wi), f"{what}: ids differ\n{gi[:3, :12]}\n{wi[:3, :12]}"
    assert np.array_equal(np.ascontiguousarray(gs).view(np.uint32), np.ascontiguousarray(ws, np.float32).view(np.uint32)), \
        f"{what}: score bits differ\n{gs[:3, :12]}\n{ws[:3, :12]}"


def _topk_from_scores(S, k, ok=None):
    """Oracle top-k from the oracle's exact scores S [nq, n]: (-score, id) order over the rows where ok holds."""
    nq, n = S.shape
    ids = np.full((nq, k), -1, np.int64)
    sc = np.full((nq, k), -np.inf, np.float32)
    for i in range(nq):
        rows = np.arange(n) if ok is None else np.flatnonzero(ok[i])
        order = rows[np.lexsort((rows, -S[i, rows].astype(np.float64)))][:k]
        ids[i, :len(order)], sc[i, :len(order)] = order, S[i, order]
    return ids, sc


class Cell:
    """Everything one (family, dtype) needs, built once: the index, the oracle's stored rows, exact scores and answers."""

    def __init__(self, coracle, family, dtype):
        self.x, self.q = E.build(family, N, DIM, NQ)
        self.dim = self.x.shape[1]
        self.dtype = dtype
        self.stored = coracle.normalize_rows(self.x, "f32" if dtype == "f32+f16" else dtype)
        qh = coracle.normalize_rows(self.q, "f32")
        self.eps_q = _eps_q(qh, dtype)
        self.S = np.stack([coracle.exact_scores(self.stored, v) for v in qh])
        self.want = {10: coracle.cosine_topk(self.q, self.stored, 10), 1000: coracle.cosine_topk(self.q[:2], self.stored, 1000)}
        _same(_topk_from_scores(self.S[:8], 10), (self.want[10][0][:8], self.want[10][1][:8]), "scores vs cosine_topk")
        self._full = self._small = self._one_query = None

    def full(self):
        import ragfin_b200
        if self._full is None:
            self._full = ragfin_b200.Index(self.dim, self.dtype, capacity=N, device=0)
            self._full.add(self.x)
        return self._full

    def small(self):
        import ragfin_b200
        if self._small is None:
            self._small = ragfin_b200.Index(self.dim, self.dtype, capacity=SMALL, device=0)
            self._small.add(self.x[:SMALL])
        return self._small

    def one_query(self):
        import ragfin_b200
        if self._one_query is None:
            old = os.environ.get("RAGFIN_NO_BIGK_BATCHED")
            os.environ["RAGFIN_NO_BIGK_BATCHED"] = "1"            # read when the handle is created
            try:
                self._one_query = ragfin_b200.Index(self.dim, self.dtype, capacity=N, device=0)
            finally:
                if old is None:
                    del os.environ["RAGFIN_NO_BIGK_BATCHED"]
                else:
                    os.environ["RAGFIN_NO_BIGK_BATCHED"] = old
            self._one_query.add(self.x)
        return self._one_query

    def close(self):
        for i in (self._full, self._small, self._one_query):
            if i is not None:
                i.close()


_cache = {}


def _drop_cache():
    for c in _cache.values():
        c.close()
    _cache.clear()


@pytest.fixture(scope="module", autouse=True)
def _release_indexes():
    """The last cell's indexes hold device memory until they are closed."""
    yield
    _drop_cache()


def _cell(coracle, family, dtype):
    key = (family, dtype)
    if key not in _cache:
        _drop_cache()
        _cache[key] = Cell(coracle, family, dtype)
    return _cache[key]


def _ld(dim):
    return (dim + 7) // 8 * 8


def _eps_approx(dtype, ld):
    """eps_approx: the tensor-core accumulation allowance (tf32 truncation for fp32 rows) + eps_sweep for the fp16 copy."""
    e = (ld + 64) * 2.0 ** -22 * 1.0625 + 2.0 ** -21
    if dtype == "f32":
        e += 2 * 2.0 ** -10 * 1.0625
    if dtype == "f32+f16":
        e += (1 + 2.0 ** -22) * (2.0 ** -11 * (1 + 2.0 ** -20) + 2.0 ** -25 * np.sqrt(ld))
    return e


def _eps_q(qh, dtype):
    """prep_queries_kernel: |qhat - round16(qhat)|_2 * 1.0078125 + 1e-9 for a 16-bit sweep, 0 for an fp32 one."""
    if dtype == "f32":
        return np.zeros(len(qh))
    d = qh.astype(np.float64) - O.round_to_storage(qh, "bf16" if dtype == "bf16" else "f16")
    return np.sqrt((d * d).sum(axis=1)) * 1.0078125 + 1e-9


def _eps_fused(dtype, dim, nq, k):
    """eps of the one-kernel search for the variant this shape takes (split: the query enters as hi + lo; plain: hi alone),
    as the library plans it (ragfin_debug_fused_plan)."""
    from ragfin_b200.engine import fused_plan
    p = fused_plan(dtype, dim, nq, k)
    assert p["ncol"], p
    return p["eps_approx"] + p["eps_query"]


def _bound_threshold(S, k, nq):
    """Exact-score counterpart of the bound pass (bound_geometry, append mode): rank-k largest maximum of the sampled blocks."""
    n = S.shape[1]
    n_tiles = (n + 255) // 256
    nblk = min(n_tiles // 2, min(max(16 * k, 256), 1024))
    qt0 = (nq + 127) // 128
    frac = max(k / 5000.0, 1 / 256 if qt0 == 1 else 1 / 96)
    if qt0 >= 2:
        frac = max(frac, 0.008 * np.sqrt(k))
    sample = min(max(int(frac * n_tiles), nblk), n_tiles // 2)
    g = max(int((sample + nblk // 2) // nblk), 1)
    while g > 1 and nblk * g > n_tiles // 2:
        g -= 1
    bstride = max((n_tiles - 1) // (nblk * g), 1)
    tiles = np.arange(nblk * g) * bstride
    tmax = np.stack([S[:, t * 256:(t + 1) * 256].max(axis=1) for t in tiles], axis=1)
    bmax = tmax.reshape(len(S), nblk, g).max(axis=2)
    return -np.sort(-bmax, axis=1)[:, k - 1]


def _predict(c, nq, k, rule, S=None):
    """Per query: True (falls back for certain), False (certainly does not) or None, from the exact scores."""
    S = c.S[:nq] if S is None else S
    ld = _ld(c.dim)
    Sk = -np.sort(-S, axis=1)[:, k - 1]
    u = 2.5e-7
    count = lambda t: (S >= t[:, None]).sum(axis=1)                 # noqa: E731
    if rule == "fused":
        eps = _eps_fused(c.dtype, c.dim, nq, k)
        c_in, c_poss = count(Sk - eps), count(Sk - 3 * eps - u)
        return [True if a > 16384 else False if b <= 8192 else None for a, b in zip(c_in, c_poss)], c_in
    eps = _eps_approx(c.dtype, ld) + c.eps_q[:nq] if rule != "scan" else np.full(nq, (ld + 64) * 2.0 ** -24 * 1.0625 + 2.0 ** -21)
    c_in, c_poss = count(Sk - eps), count(Sk - 3 * eps - u)
    if rule == "append":
        m_max = count(_bound_threshold(S, k, nq) - 4 * eps - u)
        return [True if a > 2048 else False if b <= 2048 and m <= 16384 else None for a, b, m in zip(c_in, c_poss, m_max)], c_in
    if rule == "bigk":
        cmax = k + max(k, 4096)
        return [True if a > cmax else False if b <= cmax else None for a, b in zip(c_in, c_poss)], c_in
    gap = Sk - (-np.sort(-S, axis=1)[:, 31])                       # list / scan certificate over K' = 32 candidates
    return [False if g > 1.5 * e else True if g <= 0.5 * e else None for g, e in zip(gap, eps)], c_in


def _cell_id(family, dtype, name):
    return f"{family}-{dtype}-{name.replace(' ', '_').replace(',', '')}"


# Cells in which at least one query lies between the certain cases of _predict: ids, score bits and the path are checked,
# the fallback count is not.
UNPREDICTED = {
    "negative-f32-gemm_rows_append": "8 of 8 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "negative-f32-pair_append": "160 of 160 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "negative-f32-single-CTA_MODE_3": "40 of 40 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "negative-f32-single-CTA_MODE_3_2_tiles": "160 of 160 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "negative-f32-list_mode_+_bound_pass": "19 of 40 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "negative-f32-batched_large_k": "2 of 2 queries: rows within the cut's reach straddle the 5 096-row candidate buffer",
    "negative-bf16-gemm_rows_append": "1 of 8 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "negative-bf16-pair_append": "16 of 160 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "negative-bf16-single-CTA_MODE_3": "3 of 40 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "negative-bf16-single-CTA_MODE_3_2_tiles": "16 of 160 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "negative-bf16-list_mode_+_bound_pass": "25 of 40 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "negative-bf16-batched_large_k": "2 of 2 queries: rows within the cut's reach straddle the 5 096-row candidate buffer",
    "negative-f32+f16-list_mode_+_bound_pass": "28 of 40 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "negative-f32+f16-batched_large_k": "1 of 2 queries: rows within the cut's reach straddle the 5 096-row candidate buffer",
    "sub_eps_500-f16-scan_v1": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_500-f16-scan_v2": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_2000-bf16-scan_v1": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_2000-bf16-scan_v2": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_2000-f16-scan_v1": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_2000-f16-scan_v2": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_2100-bf16-scan_v1": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_2100-bf16-scan_v2": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_2100-f16-scan_v1": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_2100-f16-scan_v2": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_17000-bf16-one-kernel_b1": "1 of 1 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "sub_eps_17000-bf16-one-kernel_b16": "16 of 16 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "sub_eps_17000-bf16-scan_v1": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_17000-bf16-scan_v2": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_17000-f16-one-kernel_b1": "1 of 1 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "sub_eps_17000-f16-one-kernel_b16": "16 of 16 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "sub_eps_17000-f16-scan_v1": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "sub_eps_17000-f16-scan_v2": "2 of 2 queries: k-th and 32nd exact scores 0.5-1.5 eps apart: the certificate may go either way",
    "low_dim_1-f32-one-kernel_b1": "1 of 1 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "low_dim_1-f32-one-kernel_b16": "16 of 16 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "low_dim_1-bf16-one-kernel_b1": "1 of 1 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "low_dim_1-bf16-one-kernel_b16": "16 of 16 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "low_dim_1-f16-one-kernel_b1": "1 of 1 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "low_dim_1-f16-one-kernel_b16": "16 of 16 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "low_dim_1-f32+f16-one-kernel_b1": "1 of 1 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "low_dim_1-f32+f16-one-kernel_b16": "16 of 16 queries: 8 192-16 384 rows within the cut's reach: the finalize may rescore them or take the exact scan",
    "extreme-bf16-gemm_rows_append": "1 of 8 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "extreme-bf16-pair_append": "3 of 160 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "extreme-bf16-single-CTA_MODE_3": "3 of 40 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "extreme-bf16-single-CTA_MODE_3_2_tiles": "3 of 160 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "extreme-f32+f16-pair_append": "3 of 160 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "extreme-f32+f16-single-CTA_MODE_3": "3 of 40 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
    "extreme-f32+f16-single-CTA_MODE_3_2_tiles": "3 of 160 queries: rows within the cut's reach straddle the 2 048-row rescore cap",
}


@pytest.mark.parametrize("family,dtype,path", [
    pytest.param(f, d, p, id=_cell_id(f, d, p[0]) + ("-count_unpredicted" if _cell_id(f, d, p[0]) in UNPREDICTED else ""))
    for f, d, p in CELLS])
def test_edge_family_on_every_path(coracle, family, dtype, path):
    import torch
    name, knobs, nq, k, want_path, rule = path
    c = _cell(coracle, family, dtype)
    q = c.q[:nq]
    idx = c.small() if "scan" in knobs else c.one_query() if knobs.get("one_query") else c.full()
    _apply(idx, knobs)
    if "scan" in knobs:
        idx.set_scan_variant(knobs["scan"])
    what = f"{family} {dtype} {name}"
    S = c.S[:nq, :SMALL] if "scan" in knobs else c.S[:nq]
    if knobs.get("filtered"):
        allow = KEEP(N)
        want = _topk_from_scores(S, k, np.broadcast_to(allow, S.shape))
        got = idx.search(q, k, allow=allow)
        _same(got, want, what)
        assert idx.stats()["path"] == want_path, (what, idx.stats())
        return
    if knobs.get("range"):
        radius = float(c.want[10][1][0, k - 1])           # cuts through the tie at query 0's k-th score (0 on "zeros")
        want = _topk_from_scores(S, k, S > np.float32(radius))
        _same(idx.search(q, k, radius=radius), want, what + " host")
        assert idx.stats()["path"] == want_path, (what, idx.stats())
        got = idx.search_device(torch.from_numpy(q).cuda(), k, radius=radius)
        torch.cuda.synchronize()
        _same(got, want, what + " device")
        return
    if "scan" in knobs:
        want = _topk_from_scores(S, k)
    else:
        want = c.want[k] if k == 1000 else (c.want[10][0][:nq], c.want[10][1][:nq])
    _same(idx.search(q, k), want, what + " host")
    st = idx.stats()
    assert st["path"] == want_path, (what, st)
    if rule is not None:
        pred, c_in = _predict(c, nq, k, rule, S)
        if _cell_id(family, dtype, name) in UNPREDICTED:
            assert None in pred, f"{what}: every query is predictable now; take the cell off UNPREDICTED"
        else:
            assert None not in pred, f"{what}: queries {[i for i, p in enumerate(pred) if p is None]} cannot be predicted"
            assert st["queries_rescanned"] == sum(pred), (what, st, pred)
        if rule == "fused":
            appended, rescored = idx.fused_counts(nq)
            for i, p in enumerate(pred):
                if p is True:
                    assert rescored[i] == -1, (what, i, rescored[i])
                elif p is False:
                    # every row certainly inside the cut was appended and rescored exactly
                    assert rescored[i] >= c_in[i] and appended[i] >= c_in[i], (what, i, appended[i], rescored[i], c_in[i])
    got = idx.search_device(torch.from_numpy(q).cuda(), k)
    torch.cuda.synchronize()
    _same(got, want, what + " device")
    assert idx.stats()["path"] == want_path, (what, idx.stats())


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("family", ["extreme", "non_finite"])
def test_every_normaliser_stores_and_searches_the_same_bits(coracle, family, dtype):
    """Host rows (ingest_vec_kernel), an aligned device tensor (ingest_vec_kernel) and a device tensor one fp32 off 16-byte
    alignment (ingest_kernel) store the oracle's bits, fp16 sweep copy included; queries one fp32 off alignment take the
    one-kernel search's scalar prologue and the tensor-core paths' prep_queries_kernel and give the oracle's answer."""
    import torch
    import ragfin_b200
    n = 20000
    x, q = E.build(family, n, DIM, 16)
    sdt = "f32" if dtype == "f32+f16" else dtype
    stored = coracle.normalize_rows(x, sdt)
    flat = torch.empty(n * DIM + 1, dtype=torch.float32, device="cuda")
    flat[1:] = torch.from_numpy(x.reshape(-1)).cuda()
    sources = {"host": x, "device": torch.from_numpy(x).cuda(), "device+4B": flat[1:].view(n, DIM)}
    assert sources["device+4B"].data_ptr() % 16 == 4
    want = coracle.cosine_topk(q, stored, 10)
    qflat = torch.empty(16 * DIM + 1, dtype=torch.float32, device="cuda")
    qflat[1:] = torch.from_numpy(q.reshape(-1)).cuda()
    q_mis = qflat[1:].view(16, DIM)
    for src_name, src in sources.items():
        idx = ragfin_b200.Index(DIM, dtype, capacity=n, device=0)
        idx.add(src)
        assert np.array_equal(idx.read_rows(0, n).view(np.uint32), stored.view(np.uint32)), (family, dtype, src_name)
        sweep = O.round_to_storage(stored, "f16") if dtype == "f32+f16" else stored
        assert np.array_equal(idx.read_sweep_rows(0, n).view(np.uint32), sweep.view(np.uint32)), (family, dtype, src_name)
        for nq, fused in ((1, True), (16, True), (16, False)):
            idx.set_fused(fused)
            _same(idx.search(q[:nq], 10), (want[0][:nq], want[1][:nq]), f"{family} {dtype} {src_name} host nq={nq}")
            got = idx.search_device(q_mis[:nq], 10)
            torch.cuda.synchronize()
            _same(got, (want[0][:nq], want[1][:nq]), f"{family} {dtype} {src_name} misaligned queries nq={nq}")
            assert idx.stats()["path"] == (3 if fused else 1), idx.stats()
        idx.close()


def _np_merge(ids, scores, k):
    """Reference merge of per-part lists [parts, nq, k]: (-score, id) order over the valid (id >= 0) entries."""
    return O.merge_topk(list(ids), list(scores), k)


def _parts(parts, nq, k, seed, negative=False, ties=False, pad=False):
    """Per-part exact hit lists (descending score, lower id first among equal scores), distinct ids across parts."""
    r = np.random.default_rng(seed)
    ids = np.full((parts, nq, k), -1, np.int64)
    sc = np.full((parts, nq, k), -np.inf, np.float32)
    for p in range(parts):
        for i in range(nq):
            m = k if not pad or p % 3 != 1 else int(r.integers(0, k))       # some parts hold fewer than k hits
            if ties:
                s = np.float32(-0.25 if negative else 0.5) - np.float32(2.0 ** -20) * r.integers(0, 3, m).astype(np.float32)
            else:
                s = (r.random(m) * 0.5 - (1.0 if negative else 0.0)).astype(np.float32)
            rows = r.choice(1000, m, replace=False) * parts + p               # distinct across parts
            o = np.lexsort((rows, -s.astype(np.float64)))
            ids[p, i, :m], sc[p, i, :m] = rows[o], s[o]
    return ids, sc


@pytest.mark.parametrize("parts", [1, 3, 8])
@pytest.mark.parametrize("data", ["plain", "ties", "negative", "negative_ties", "padded"])
def test_merge_topk_matches_numpy_in_all_three_layouts(parts, data):
    """ragfin_merge_topk against a numpy merge, with the part-major [parts, nq, k] layout, the concatenation [nq, parts * k]
    and the packed {ids | scores} record the NCCL all-gather moves (PackedHits): equal score bits across parts go to the
    lower id, all-negative scores, and -1 / -inf padding in some parts."""
    import torch
    from ragfin_b200.engine import PackedHits, merge_topk
    nq, k = 5, 24
    ids, sc = _parts(parts, nq, k, parts * 10 + len(data), negative="negative" in data, ties="ties" in data, pad=data == "padded")
    want = _np_merge(ids, sc, k)
    dev = torch.device("cuda", 0)
    t_ids, t_sc = torch.from_numpy(ids).to(dev), torch.from_numpy(sc).to(dev)
    got = merge_topk(t_ids, t_sc, parts, k)                                      # [parts, nq, k]
    torch.cuda.synchronize()
    _same(got, want, f"{data} part-major")
    got = merge_topk(t_ids.permute(1, 0, 2).reshape(nq, parts * k), t_sc.permute(1, 0, 2).reshape(nq, parts * k), parts, k)
    torch.cuda.synchronize()
    _same(got, want, f"{data} concatenated")
    ph = PackedHits(nq, k, parts, dev)
    for p in range(parts):                                                        # what the all-gather leaves in `gathered`
        ph.ids.copy_(t_ids[p])
        ph.scores.copy_(t_sc[p])
        ph.gathered[p * ph.record:(p + 1) * ph.record].copy_(ph.local)
    got = ph.merge()
    torch.cuda.synchronize()
    _same(got, want, f"{data} packed record")
    if data == "ties":
        gi, gs = (a.cpu().numpy() for a in got)
        same = gs[:, 1:] == gs[:, :-1]
        assert same.any() and (gi[:, 1:][same] > gi[:, :-1][same]).all()
