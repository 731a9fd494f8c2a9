"""GPU suite for the one-kernel search at wide embeddings (2 560-4 096-d), where 9-16 queries no longer fit the split operand
block and take the plain variant: the query enters the MMA as hi = RNE16(q) alone and its rounding costs up to a full unit
roundoff 2^-p |q|_2 of every approximate score (tests/_query_rounding.py, test_query_rounding_cpu.py).

* Wrong answer: bf16, adversarial queries, rows A and B tilted along the query's residual.  A eps that charged half that
  roundoff cut A (the exact best row) away and returned B; the search must return the oracle's ids and score bits.
* Parity: bf16, f16 and f32+f16 at 2 560 / 3 072 / 4 096-d, split (8 queries) and plain (16), adversarial and random
  queries, against the C oracle and the multi-kernel path; fp32 rows (no one-kernel search at these widths) against the
  oracle on the path they take.

Each (dtype, dim) builds one 16 384-row index for the module."""
import numpy as np
import pytest

import _query_rounding as R
from oracle import ragfin_oracle as O

pytestmark = pytest.mark.gpu

DIMS = R.WRONG_ANSWER_DIMS
NQ = 16


class Corpus:
    def __init__(self, coracle, dtype, dim):
        import ragfin_b200
        self.x, self.q, self.where = R.corpus(dim, "f16" if dtype in ("f16", "f32+f16") else "bf16", NQ)
        self.random = O.synth_rows(900 + dim, 0, NQ, dim)
        self.stored = coracle.normalize_rows(self.x, "f32" if dtype == "f32+f16" else dtype)
        self.want = {}
        self.idx = ragfin_b200.Index(dim, dtype, capacity=len(self.x), device=0)
        self.idx.add(self.x)

    def queries(self, kind, nq):
        return (self.q if kind == "adversarial" else self.random)[:nq]

    def oracle(self, coracle, kind, nq, k):
        if (kind, k) not in self.want:
            self.want[(kind, k)] = coracle.cosine_topk(self.queries(kind, NQ), self.stored, k)
        ids, sc = self.want[(kind, k)]
        return ids[:nq], sc[:nq]


_cache = {}


@pytest.fixture(scope="module", autouse=True)
def _release_indexes():
    yield
    for c in _cache.values():
        c.idx.close()
    _cache.clear()


def _corpus(coracle, dtype, dim):
    if (dtype, dim) not in _cache:
        _cache[(dtype, dim)] = Corpus(coracle, dtype, dim)
    return _cache[(dtype, dim)]


def _same(got, want, what):
    gi, gs = (np.asarray(a.cpu()) if hasattr(a, "cpu") else np.asarray(a) for a in got)
    assert np.array_equal(gi, want[0]), f"{what}: ids differ\n{gi}\n{want[0]}"
    assert np.array_equal(gs.view(np.uint32), want[1].view(np.uint32)), f"{what}: score bits differ\n{gs}\n{want[1]}"


@pytest.mark.parametrize("k", [1, 10])
@pytest.mark.parametrize("dim", DIMS)
def test_bf16_plain_variant_keeps_the_row_its_rounded_query_underrates(coracle, dim, k):
    from ragfin_b200.engine import fused_plan
    nq = R.WRONG_ANSWER_NQ[dim]
    plan = fused_plan("bf16", dim, nq, k)
    assert plan["ncol"] and not plan["split"], plan
    c = _corpus(coracle, "bf16", dim)
    want = c.oracle(coracle, "adversarial", nq, k)
    assert np.array_equal(want[0][:, 0], c.where[:nq]), want[0]            # A is every query's exact best row
    got = c.idx.search(c.q[:nq], k)
    st = c.idx.stats()
    assert st["path"] == 3 and st["queries_rescanned"] == 0, st
    lost = [j for j in range(nq) if c.where[j] not in got[0][j]]
    assert not lost, f"dim={dim} k={k}: row A cut for queries {lost}; returned {got[0][lost[0]][:3]} where the oracle has " \
                     f"{want[0][lost[0]][:3]} (B = A + 1)"
    _same(got, want, f"bf16 dim={dim} nq={nq} k={k}")


@pytest.mark.parametrize("kind", ["adversarial", "random"])
@pytest.mark.parametrize("nq", [8, 16])
@pytest.mark.parametrize("dim", DIMS)
@pytest.mark.parametrize("dtype", ["bf16", "f16", "f32+f16"])
def test_wide_embedding_parity_on_both_variants(coracle, dtype, dim, nq, kind):
    import torch
    from ragfin_b200.engine import fused_plan
    k = 10
    plan = fused_plan(dtype, dim, nq, k)
    assert plan["ncol"] and plan["split"] == int(nq <= 8), plan
    c = _corpus(coracle, dtype, dim)
    q = c.queries(kind, nq)
    want = c.oracle(coracle, kind, nq, k)
    what = f"{dtype} dim={dim} nq={nq} {kind}"
    c.idx.set_fused(True)
    _same(c.idx.search(q, k), want, what + " one-kernel, host")
    st = c.idx.stats()
    assert st["path"] == 3 and st["queries_rescanned"] == 0, (what, st)
    got = c.idx.search_device(torch.from_numpy(q).cuda(), k)
    torch.cuda.synchronize()
    _same(got, want, what + " one-kernel, device")
    c.idx.set_fused(False)
    _same(c.idx.search(q, k), want, what + " multi-kernel")
    assert c.idx.stats()["path"] == 1, (what, c.idx.stats())
    c.idx.set_fused(True)


@pytest.mark.parametrize("dim", DIMS)
def test_f32_rows_at_wide_embeddings_take_the_multi_kernel_paths(coracle, dim):
    """The fp32 operand block (kind::tf32, 32 elements per 128-byte k-block) of one query tile no longer fits in shared
    memory from 2 560-d: no shape takes the one-kernel search."""
    from ragfin_b200.engine import fused_plan
    c = _corpus(coracle, "f32", dim)
    for nq in (1, 8, 16):
        assert fused_plan("f32", dim, nq, 10)["ncol"] == 0
        assert not c.idx.fused_eligible(nq, 10)
        for kind in ("adversarial", "random"):
            _same(c.idx.search(c.queries(kind, nq), 10), c.oracle(coracle, kind, nq, 10), f"f32 dim={dim} nq={nq} {kind}")
            assert c.idx.stats()["path"] == (0 if nq < 3 else 1), c.idx.stats()
