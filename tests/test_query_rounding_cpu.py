"""CPU suite for the one-kernel search's query-rounding term (eps_fused_query in csrc/ragfin_api.cu, reported by
ragfin_debug_fused_plan): the per-element bound on every fp32 value where it could fail, the vector bound on adversarial
queries, the planner's choice of variant at wide embeddings, and the row pairs test_query_rounding_gpu.py searches for.

The kernel prologue computes hi = RNE16(y), rest = y - hi in fp32 and lo = RNE16(rest) (split variant) for every normalised
query component y; |y - hi (- lo)| <= rel |y| + sub must hold for every fp32 y.  A relative term of half the true worst case
(as the kernel once used) fails the exhaustive check, and one twice too large fails its tightness check."""
import numpy as np
import pytest

import _query_rounding as R
from oracle import ragfin_oracle as O


def _plan(dtype, dim, nq, k=10, max_nq=0, max_nqk=0):
    from ragfin_b200.engine import fused_plan
    return fused_plan(dtype, dim, nq, k, max_nq, max_nqk)


def _variant(dtype, dim, split):
    """The plan of a shape that takes the given variant: one query is split; plain needs more queries than the split
    operand block holds (9 from 2 560-d, 33 below)."""
    p = _plan(dtype, dim, 1 if split else 9 if dim >= 2560 else 33, 1, 64, 1 << 20)
    assert p["ncol"] and p["split"] == int(split), (dtype, dim, split, p)
    return p


def _fp32_range(lo_bits, hi_bits, chunk=1 << 23):
    """Every positive fp32 with bit pattern in [lo_bits, hi_bits), in chunks."""
    for b in range(lo_bits, hi_bits, chunk):
        yield np.arange(b, min(b + chunk, hi_bits), dtype=np.uint32).view(np.float32)


def _bits(x):
    return int(np.float32(x).view(np.uint32))


# bf16 has fp32's exponent range, so its relative error is the same in every normal binade once hi and lo are normal:
# one full binade, plus everything below 2^-112 (fp32 and bf16 subnormals; lo can turn subnormal below 2^-117).
# fp16 turns subnormal below 2^-14 (lo below 2^-3 for the split): everything in [2^-26, 1), where its components live.
RANGES = {"bf16": [(1, _bits(2.0 ** -112)), (_bits(0.5), _bits(1.0))], "f16": [(_bits(2.0 ** -26), _bits(1.0))]}


@pytest.mark.parametrize("split", [False, True], ids=["plain", "split"])
@pytest.mark.parametrize("store", ["bf16", "f16"])
def test_per_element_bound_holds_on_every_fp32_value_and_is_tight(store, split):
    p = _variant(store, 2560, split)
    rel, sub = p["rel"], p["sub"]
    worst = {}
    for region, (b0, b1) in enumerate(RANGES[store]):
        w = 0.0
        for y in _fp32_range(b0, b1):
            for sy in (y, -y):
                hi, lo = R.query_parts(sy, store, split)
                err = np.abs(sy.astype(np.float64) - hi.astype(np.float64) - lo.astype(np.float64))
                ratio = err / (rel * np.abs(sy.astype(np.float64)) + sub)
                i = int(np.argmax(ratio))
                assert ratio[i] <= 1.0, f"{store} split={split}: |y - hi - lo| = {err[i]:.6e} at y = {sy[i]!r} exceeds " \
                                        f"{rel!r} |y| + {sub!r}"
                w = max(w, float(ratio[i]))
        worst[region] = w
    # the normal binade reaches the relative term (a rel twice too large would leave the worst case at or below 1/2); the
    # subnormal range reaches sub
    assert worst[len(worst) - 1] > 0.5, (store, split, worst)
    assert worst[0] > 0.5, (store, split, worst)


@pytest.mark.parametrize("dim", [768, 2560, 3072, 4096])
@pytest.mark.parametrize("store", ["bf16", "f16"])
def test_adversarial_query_residual_stays_inside_the_query_term(store, dim):
    q = O.normalize_rows(R.adversarial_queries(4, dim, store, dim), "f32")
    for split in (False, True):
        p = _variant(store, dim, split)
        for y in q:
            hi, lo = R.query_parts(y, store, split)
            r = y.astype(np.float64) - hi.astype(np.float64) - lo.astype(np.float64)
            norm = np.sqrt(r @ r)
            assert norm * 1.0078125 <= p["eps_query"], (store, dim, split, norm, p["eps_query"])
            if not split:
                assert norm > 0.99 * p["rel"], (store, dim, norm)      # the generator reaches the bound it is meant to test


@pytest.mark.parametrize("dim", [2560, 3072, 4096])
@pytest.mark.parametrize("dtype", ["bf16", "f16", "f32+f16"])
def test_planner_takes_plain_from_9_queries_and_split_up_to_8_at_wide_embeddings(dtype, dim):
    """With the default limits a 16-bit sweep of 2 560-d rows or wider no longer fits the split operand block for 9-16
    queries (N = 32 columns) in 227 KB of shared memory: those batches take the plain variant, the one with the large
    query term.  test_query_rounding_gpu.py relies on which variant each shape takes."""
    for nq in range(1, 17):
        for k in (1, 10):
            p = _plan(dtype, dim, nq, k)
            assert p["ncol"] == 16 and p["split"] == int(nq <= 8), (dtype, dim, nq, k, p)
            if not p["split"]:
                assert p["rel"] == 2.0 ** -R.BITS[R.SWEEP[dtype]], p
    assert _plan("f32", dim, 1)["ncol"] == 0                         # the fp32 operand block does not fit at all


def test_plan_hook_rejects_bad_arguments():
    import ctypes
    from ragfin_b200 import _lib
    L = _lib.load()
    out, eps = (ctypes.c_int64 * 5)(), (ctypes.c_double * 4)()
    assert L.ragfin_debug_fused_plan(4, 768, 1, 10, 0, 0, out, eps) == _lib.EINVAL       # dtype
    assert L.ragfin_debug_fused_plan(1, 0, 1, 10, 0, 0, out, eps) == _lib.EINVAL         # dim
    assert L.ragfin_debug_fused_plan(1, 768, 0, 10, 0, 0, out, eps) == _lib.EINVAL       # nq
    assert L.ragfin_debug_fused_plan(1, 768, 1, 10, 65, 0, out, eps) == _lib.EINVAL      # max_nq
    assert L.ragfin_debug_fused_plan(1, 768, 1, 10, 0, 0, None, eps) == _lib.EINVAL
    assert L.ragfin_debug_fused_plan(1, 768, 1, 10, 0, 0, out, None) == _lib.EINVAL
    _lib.check(L.ragfin_debug_fused_plan(1, 768, 17, 10, 0, 0, out, eps))
    assert out[0] == 0                                                                    # 17 queries: over the default limit
    _lib.check(L.ragfin_debug_fused_plan(1, 768, 17, 10, 64, 0, out, eps))
    assert out[0] == 64                                                                   # split, 32 hi + 32 lo columns


@pytest.mark.parametrize("dim", R.WRONG_ANSWER_DIMS)
def test_pairs_break_the_old_bound_and_not_the_new_one(dim):
    """For every query and row pair test_query_rounding_gpu.py searches (bf16, plain variant), in fp64 emulation: the
    approximate scores differ by more than 2 eps_old + allowance / 2 (the kernel's real accumulation error stays below
    allowance / 4 per score, test_tensor_core_error_stays_inside_the_allowance), so a cut at T - 2 eps_old drops A for
    certain; by less than 2 eps - allowance / 2, so the corrected cut keeps it for certain; and A's exact score is the
    higher one."""
    nq = R.WRONG_ANSWER_NQ[dim]
    p = _plan("bf16", dim, nq)
    assert p["ncol"] and not p["split"], p
    low, high = R.wrong_answer_window(p, (dim + 7) // 8 * 8)
    x, q, where = R.corpus(dim, "bf16")
    qh = O.normalize_rows(q[:nq], "f32")
    for j in range(nq):
        a, b = where[j], where[j] + 1
        stored = O.normalize_rows(x[[a, b]], "bf16")
        exact, approx = R.emulate(stored, qh[j], "bf16", False)
        gap = approx[1] - approx[0]
        assert low < gap < high, (dim, j, low, gap, high)
        assert np.float32(exact[0]) > np.float32(exact[1]), (dim, j, exact)
        assert a // 256 == (b + R.B_COPIES - 1) // 256                   # A and all copies of B in one 256-row tile
