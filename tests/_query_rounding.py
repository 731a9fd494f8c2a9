"""Adversarial queries for the one-kernel search's query-rounding bound, and row pairs that turn a too-small bound into a
wrong answer.  Shared by test_query_rounding_cpu.py (fp64 emulation) and test_query_rounding_gpu.py (the kernel).

The one-kernel search scores rows against hi = RNE16(q) (plain) or hi + lo with lo = RNE16(q - hi) (split), so its
approximate score of a stored row x is x.q - x.r with the residual r = q - hi (- lo).  A query whose every component sits just
beside a 16-bit rounding midpoint right above a power of two has |r|_2 close to a full unit roundoff 2^-p.  Rows A and B tilted
in opposite directions along r (and A a little towards q, so that A's exact score is the higher one) then have approximate
scores whose difference is close to 2 |r|_2: a cut of T - 2 eps with an eps that charges only half of |r|_2 drops A."""
import math

import numpy as np

from oracle import ragfin_oracle as O

SWEEP = {"bf16": "bf16", "f16": "f16", "f32+f16": "f16"}   # the 16-bit type the tensor-core sweep reads
BITS = {"bf16": 8, "f16": 11}                               # significant bits (p): unit roundoff 2^-p


def query_parts(y, store, split):
    """The one-kernel search's prologue on normalised fp32 queries y: hi = RNE(y), rest = y - hi in fp32 (exact),
    lo = RNE(rest) for the split variant, else 0.  Returns (hi, lo) as fp32 values."""
    y = np.ascontiguousarray(y, np.float32)
    hi = O.round_to_storage(y, store)
    if not split:
        return hi, np.zeros_like(hi)
    return hi, O.round_to_storage(y - hi, store)


def adversarial_queries(n, dim, store, seed):
    """n fp32 queries [n, dim] of unit norm whose components are 2^e (1 + 2^-p +- 2^-20): 2^-20 beside the midpoint between
    2^e and the next 16-bit value, rounding down or up at random (so r stays nearly orthogonal to q), random signs.  The
    exponents are chosen greedily so that the squares sum to just below 1; the last component makes up the rest.  2^-20 is
    sixteen fp32 ulps: normalisation (a scale within a few ulps of 1) cannot move a component across its midpoint."""
    rng = np.random.default_rng(seed)
    u = 2.0 ** -BITS[store]
    out = np.empty((n, dim), np.float32)
    for j in range(n):
        m = 1 + u + np.where(rng.random(dim) < 0.5, -2.0 ** -20, 2.0 ** -20)
        sign = np.where(rng.random(dim) < 0.5, -1.0, 1.0)
        rest = 1.0
        for i in range(dim - 1):
            v = 2.0 ** math.floor(math.log2(math.sqrt(rest / (dim - i)) / (1 + u))) * m[i]
            out[j, i] = sign[i] * v
            rest -= v * v
        out[j, -1] = sign[-1] * math.sqrt(rest)
    return out


def pair_rows(qhat, store, seed):
    """Rows A and B (raw fp32) for one normalised query qhat and the plain variant's residual r = qhat - hi:
    A = (1 + 2^-10) qhat + s r_perp + w, B = qhat - s r_perp + w, with r_perp the unit part of r orthogonal to qhat and w a
    random unit vector orthogonal to both (it decorrelates the rows' own storage rounding from the query's mantissa pattern).
    s = 4.9 puts the approximate scores 98 % of the way to their largest difference, 2 |r_perp|; the 2^-10 makes A's exact
    score the higher one by a few 1e-4, well above what the rows' storage rounding moves it."""
    q = qhat.astype(np.float64)
    r = q - query_parts(qhat, store, False)[0].astype(np.float64)
    rp = r - (r @ q) / (q @ q) * q
    rp /= np.sqrt(rp @ rp)
    s = 0.98 / np.sqrt(1 - 0.98 ** 2)
    w = np.random.default_rng(seed).standard_normal(len(q))
    w -= (w @ q) / (q @ q) * q + (w @ rp) * rp
    w /= np.sqrt(w @ w)
    return np.stack([(1 + 2.0 ** -10) * q + s * rp + w, q - s * rp + w]).astype(np.float32)


def emulate(stored, qhat, store, split):
    """(exact, approx) scores of stored rows [n, dim] against one query: exact = the oracle's canonical fp32 score, approx =
    the tensor-core score without its accumulation error (fp64 dot with hi + lo)."""
    hi, lo = query_parts(qhat, store, split)
    exact = O.exact_scores(stored, qhat).astype(np.float64)
    return exact, stored.astype(np.float64) @ (hi.astype(np.float64) + lo.astype(np.float64))


def old_eps(plan, ld):
    """eps of the one-kernel search before its query term was corrected: the same bound with half the relative term."""
    return plan["eps_approx"] + (plan["rel"] / 2 + plan["sub"] * np.sqrt(ld)) * 1.0078125


# The wrong-answer searches: bf16 rows, 9-16 queries at 2 560-4 096-d (the plain variant, test_query_rounding_cpu.py).
WRONG_ANSWER_DIMS = (2560, 3072, 4096)
WRONG_ANSWER_NQ = {2560: 9, 3072: 12, 4096: 16}
N_ROWS = 16384              # >= 8 192 random filler rows: the one-kernel search's smallest corpus
B_COPIES = 10               # k = 10: the exact top-10 is A and nine copies of B, a cut that drops A returns ten copies of B


def corpus(dim, store, nq=16, seed=0):
    """(raw rows [N_ROWS, dim], raw queries [nq, dim], where[nq]): random filler rows and nq adversarial queries; query j's
    row A sits at where[j] and B_COPIES copies of its row B right behind it, all in one 256-row tile (tile 4 j)."""
    q = adversarial_queries(nq, dim, store, seed + dim)
    qh = O.normalize_rows(q, "f32")
    x = np.random.default_rng(seed + dim + 1).standard_normal((N_ROWS, dim)).astype(np.float32)
    where = np.arange(nq) * 4 * 256 + 7
    for j in range(nq):
        a, b = pair_rows(qh[j], store, seed + j)
        x[where[j]] = a
        x[where[j] + 1:where[j] + 1 + B_COPIES] = b
    return x, q, where


def wrong_answer_window(plan, ld):
    """(low, high): approx(B) - approx(A) above low drops A under the old eps for certain, below high keeps it under the
    corrected one for certain (an accumulation error below allowance / 4 per score on either side)."""
    allowance = plan["eps_approx"]
    return 2 * old_eps(plan, ld) + allowance / 2, 2 * (allowance + plan["eps_query"]) - allowance / 2
