"""The reference at the numeric edges, without a GPU: the numpy and C oracles agree bit for bit on every edge family of
tests/_edge_families.py (normalised rows, ids and score bits of the top k), the extreme-magnitude rows are normalised and
scored to the rounding DESIGN.md 2 states (checked against exact rational arithmetic), and the non-finite rule holds in
both oracles and at the shim (include/ragfin.h: a vector with a NaN or +-Inf component is the zero vector)."""
from decimal import Decimal, getcontext
from fractions import Fraction

import numpy as np
import pytest

import _edge_families as E
from oracle import ragfin_oracle as O

FAMILIES = ["negative", "zeros", "sub_eps_500", "low_dim_1", "low_dim_2", "low_dim_3", "low_dim_4", "low_dim_7",
            "extreme", "non_finite"]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("dtype", O.DTYPES)
@pytest.mark.parametrize("family", FAMILIES)
def test_numpy_and_c_oracles_agree_on_the_edge_families(coracle, family, dtype):
    x, q = E.build(family, 3000, 64, 6)
    s_np, s_c = O.normalize_rows(x, dtype), coracle.normalize_rows(x, dtype)
    assert np.array_equal(_bits(s_np), _bits(s_c))
    assert np.isfinite(s_np).all()
    for k in (1, 10, 700):
        i_np, v_np = O.cosine_topk(q, s_np, k)
        i_c, v_c = coracle.cosine_topk(q, s_c, k)
        assert np.array_equal(i_np, i_c), (k, i_np[:, :12], i_c[:, :12])
        assert np.array_equal(_bits(v_np), _bits(v_c)), k
        assert np.isfinite(v_np).all()
        assert (np.diff(v_np.astype(np.float64), axis=1) <= 0).all()           # descending
        # ties go to the lower id
        same = v_np[:, 1:] == v_np[:, :-1]
        assert (i_np[:, 1:][same] > i_np[:, :-1][same]).all()


def test_families_have_the_shape_they_claim(coracle):
    """The scores the GPU matrix relies on: negative top-k, thousands of exact zeros, a sub-eps cluster, few score levels."""
    def scores(fam, n=20000, dim=256, nq=4, dtype="bf16"):
        x, q = E.build(fam, n, dim, nq)
        st = coracle.normalize_rows(x, dtype)
        qh = coracle.normalize_rows(q, "f32")
        return np.stack([coracle.exact_scores(st, qq) for qq in qh])
    s = np.sort(scores("negative"), axis=1)[:, ::-1]
    assert (s[:, :100] < -0.9).all() and (s[:, :100] > -1.0).all()
    s = scores("zeros")
    assert ((s > 0).sum(axis=1) == 5).all() and ((s == 0).sum(axis=1) == 20000 - 5005).all()
    s = scores("sub_eps_2100", dtype="f32")
    top = np.sort(s, axis=1)[:, ::-1]
    assert (top[:, 0] - top[:, 2099] < 2e-5).all() and (top[:, 2099] - top[:, 2100] > 0.5).all()
    assert all(len(np.unique(r[:2100])) > 20 for r in top)                     # not one tie: distinct scores too
    s = scores("low_dim_2")
    assert all(len(np.unique(r)) <= 9 for r in s)


def _ulp32(v):
    return Decimal(float(np.spacing(np.float32(abs(v)))))


def _exact_normalised(row):
    """x / |x| per element, 60 significant digits (the square root is irrational in general)."""
    getcontext().prec = 60
    s = sum(Fraction(float(v)) ** 2 for v in row)
    root = (Decimal(s.numerator) / Decimal(s.denominator)).sqrt()
    return [Decimal(float(v)) / root for v in row]


@pytest.mark.parametrize("oracle", ["numpy", "c"])
def test_extreme_rows_normalise_to_the_correctly_rounded_fp32(coracle, oracle):
    """stored = RNE_f32(x * (1 / sqrt(n2))) with n2 and 1/sqrt in fp64: within half an fp32 ulp of the exact x / |x| (plus
    the fp64 steps' 2^-50 relative), and exactly 0 where the exact value is below half of 2^-149."""
    dim = 64
    rows = E.extreme_rows(dim)
    norm = O.normalize_rows if oracle == "numpy" else coracle.normalize_rows
    got = norm(rows, "f32")
    for row, y in zip(rows, got):
        z = _exact_normalised(row)
        for zi, yi in zip(z, y):
            tol = _ulp32(yi) / 2 + abs(zi) * Decimal(2) ** -50
            assert abs(Decimal(float(yi)) - zi) <= tol, (row[:4], float(zi), float(yi))
    # the 1e30 / 1e-30 rows: the small parts underflow to +-0 in fp32 and in every storage type
    mixed = rows[5:7]
    for dtype in O.DTYPES:
        y = norm(mixed, dtype)
        assert (y[np.abs(mixed) < 1e-20] == 0).all() and (np.abs(y[np.abs(mixed) > 1e20]) > 0).all()
    # a lone 2^-149 normalises to exactly 1
    assert (norm(rows[2:5], "f32").max(axis=1) == 1.0).all()


@pytest.mark.parametrize("oracle", ["numpy", "c"])
def test_rounding_midpoints_tie_to_even_in_bf16_and_fp16(coracle, oracle):
    """Unit rows whose first component is 1 - 2^-9 (a bf16 midpoint: ties to 1.0) or 1 - 2^-12 (an fp16 midpoint: ties to
    1.0), at scales 1, 2^100 and 2^-100: inv is a power of two, so the fp32 row is the input exactly."""
    norm = O.normalize_rows if oracle == "numpy" else coracle.normalize_rows
    mid = E.midpoint_rows(16)
    for s in (1.0, 2.0 ** 100, 2.0 ** -100):
        x = mid * np.float32(s)
        assert np.array_equal(_bits(norm(x, "f32")), _bits(mid))
        b, h = norm(x, "bf16"), norm(x, "f16")
        assert b[0, 0] == 1.0 and b[1, 0] == 1.0                                  # 1 - 2^-9 and 1 - 2^-12 -> 1 in bf16
        assert h[0, 0] == np.float32(1 - 2.0 ** -9) and h[1, 0] == 1.0            # fp16 holds 1 - 2^-9; 1 - 2^-12 ties up
        assert b[0, 1] == np.float32(31 * 2.0 ** -9) and h[1, 1] == np.float32(90 * 2.0 ** -12)
        # one fp32 ulp off the midpoint decides the direction
        for sign, want in ((1, 1.0), (-1, np.float32(1 - 2.0 ** -8))):
            y = np.float32(1 - 2.0 ** -9) + sign * np.spacing(np.float32(1 - 2.0 ** -9))
            assert O.round_to_storage(np.array([y], np.float32), "bf16")[0] == want


@pytest.mark.parametrize("oracle", ["numpy", "c"])
def test_canonical_dot_of_extreme_rows_is_the_rounded_exact_dot(coracle, oracle):
    """score = RNE_f32(canonical fp64 dot) + 0: within half an fp32 ulp of the exact rational dot of the stored operands, plus
    the fp64 accumulation (dim * 2^-53 * sum |products|)."""
    dim = 64
    rows = E.extreme_rows(dim)
    norm = O.normalize_rows if oracle == "numpy" else coracle.normalize_rows
    score = O.exact_scores if oracle == "numpy" else coracle.exact_scores
    for dtype in O.DTYPES:
        st = norm(rows, dtype)
        for qi in range(len(rows)):
            qh = norm(rows[qi], "f32")[0]
            s = score(st, qh)
            for r in range(len(rows)):
                prods = [Fraction(float(a)) * Fraction(float(b)) for a, b in zip(st[r], qh)]
                exact = sum(prods)
                slack = Fraction(dim) * Fraction(2) ** -53 * sum(abs(p) for p in prods)
                tol = Fraction(float(np.spacing(np.float32(abs(s[r]))))) / 2 + slack
                assert abs(Fraction(float(s[r])) - exact) <= tol, (dtype, qi, r, float(exact), s[r])
                assert _bits(s[r:r + 1])[0] != 0x80000000                        # -0 is canonicalised


def _nonfinite_corpus():
    x = O.synth_rows(77, 0, 50, 16)
    x[7, 3] = np.inf
    x[19, 0] = np.nan
    x[23, [1, 2]] = [-np.inf, np.nan]
    return x


@pytest.mark.parametrize("dtype", O.DTYPES)
def test_non_finite_rows_are_stored_as_zero_rows_by_both_oracles(coracle, dtype):
    x = _nonfinite_corpus()
    for norm in (O.normalize_rows, coracle.normalize_rows):
        st = norm(x, dtype)
        assert np.isfinite(st).all()
        assert not st[[7, 19, 23]].any()
        keep = np.setdiff1d(np.arange(50), [7, 19, 23])
        assert np.array_equal(_bits(st[keep]), _bits(norm(x[keep], dtype)))      # the other rows are untouched
    assert np.array_equal(_bits(O.normalize_rows(x, dtype)), _bits(coracle.normalize_rows(x, dtype)))


def test_non_finite_rows_and_queries_give_one_answer_in_both_oracles(coracle):
    """The case that used to split the oracles: numpy dropped the NaN rows, the C insertion sort returned a misordered list."""
    x = _nonfinite_corpus()
    st = O.normalize_rows(x, "bf16")
    q = O.synth_rows(78, 0, 4, 16)
    q[1, 2], q[2, 0], q[3, 15] = np.nan, np.inf, -np.inf
    for k in (5, 30, 50):
        i_np, v_np = O.cosine_topk(q, st, k)
        i_c, v_c = coracle.cosine_topk(q, coracle.normalize_rows(x, "bf16"), k)
        assert np.array_equal(i_np, i_c) and np.array_equal(_bits(v_np), _bits(v_c))
        assert np.isfinite(v_np).all() and (np.diff(v_np[0].astype(np.float64)) <= 0).all()
        # the zero rows score exactly 0 and rank among the other zeros by id
        s0 = O.exact_scores(st, O.normalize_rows(q[0])[0])
        assert (s0[[7, 19, 23]] == 0).all()
        # a non-finite query is the zero query: every row scores 0, the answer is rows 0 .. k-1
        for j in (1, 2, 3):
            assert i_np[j].tolist() == list(range(k)) and not v_np[j].any()
    assert (v_np[0] > -1).all()


def test_shim_refuses_non_finite_vectors_on_insert_and_search():
    from ragfin_b200 import milvus_compat as mc
    from test_shim_cpu import OracleIndex
    F, D = mc.FieldSchema, mc.DataType
    mc.utility.drop_collection("edges_nf")
    col = mc.Collection("edges_nf", mc.CollectionSchema([F("id", D.INT64, is_primary=True), F("embedding", D.FLOAT_VECTOR, dim=8)]),
                        index_factory=OracleIndex)
    x = O.synth_rows(79, 0, 6, 8)
    col.insert([list(range(6)), x])
    col.flush()
    for bad in (np.nan, np.inf, -np.inf):
        y = O.synth_rows(80, 0, 3, 8)
        y[1, 4] = bad
        with pytest.raises(mc.MilvusException, match="NaN or Inf"):
            col.insert([[10, 11, 12], y])
        with pytest.raises(mc.MilvusException, match="NaN or Inf"):
            col.upsert([[0, 11, 12], y])
        with pytest.raises(mc.MilvusException, match="NaN or Inf"):
            col.search(y, "embedding", {"metric_type": "COSINE"}, 3)
    assert col.num_entities == 6                                  # nothing of a refused insert or upsert was kept
    hits = col.search(x[2:3], "embedding", {"metric_type": "COSINE"}, 6)[0]
    assert [h.id for h in hits][0] == 2 and len(hits) == 6
    mc.utility.drop_collection("edges_nf")
