"""Edge-case data families for the numeric-edge suites (test_edges_cpu.py, test_edges_gpu.py).

Every family is built from fixed seeds, in fp32, and returns (rows [n, dim], queries [nq, dim]).  `synth_rows` only ever
gives positive, well-spread top-k scores (about 0.1-0.2 against a random query); these families put the top-k where
kernels go wrong: below zero, on thousands of exact ties, within a few fp32 ulps of each other, on a handful of score
values, at the ends of the fp32 range, and on NaN / Inf components (which the library stores as zero vectors)."""
import numpy as np

from oracle import ragfin_oracle as O

FMAX = float(np.finfo(np.float32).max)
TINY = 2.0 ** -149                      # smallest fp32 subnormal


def _rng(seed):
    return np.random.default_rng(seed)


def negative(n, dim, nq, seed=1):
    """Rows in a cone around c (4c + noise), queries near -c: every top-k score is about -0.95."""
    c = O.synth_rows(seed, 0, 1, dim)[0]
    x = np.float32(4.0) * c[None, :] + O.synth_rows(seed + 1, 0, n, dim)
    q = -c[None, :] + O.synth_rows(seed + 2, 0, nq, dim) * np.float32(1 / 16)
    return x.astype(np.float32), q.astype(np.float32)


def zeros(n, dim, nq, seed=2):
    """Queries live on the first half of the coordinates.  5 rows score above 0, 5 000 below, and every other row lives on
    the second half only, so it scores exactly 0: a top-k with k > 5 cuts through ~n - 5 000 tied keys."""
    h = dim // 2
    p = O.synth_rows(seed, 0, 1, h)[0]
    noise = O.synth_rows(seed + 1, 0, n, dim)
    x = noise.copy()
    x[:, :h] = 0.0                                              # the tie block
    kind = _rng(seed).permutation(n)
    above, below = kind[:5], kind[5:5005]
    x[above, :h] = p + noise[above, :h] * np.float32(0.25)
    x[below, :h] = -p + noise[below, :h] * np.float32(0.25)
    q = np.zeros((nq, dim), np.float32)
    q[:, :h] = p + O.synth_rows(seed + 2, 0, nq, h) * np.float32(0.25)
    return x, q


def _orthonormal(dim, seed, m):
    v = O.synth_rows(seed, 0, m, dim).astype(np.float64)
    out = []
    for r in v:
        for o in out:
            r = r - (r @ o) * o
        out.append(r / np.linalg.norm(r))
    return out


def sub_eps(n, dim, nq, m, seed=3):
    """m rows u + t w (w orthogonal to u, 0 <= t <= 4e-3) at random positions among synthetic rows; queries u + s w2
    (s <= 1e-3).  Stored in fp32 (f32, f32+f16) the m rows' exact scores all lie within ~1e-5 of each other - a tenth of
    the smallest 2 eps of any path - so which of them make the top k is decided by the exact rescore alone.  16-bit
    storage rounds each row by up to 2^-9 (bf16) or 2^-12 (fp16) per element, which spreads the cluster to ~5e-4 / ~6e-5."""
    u, w, w2 = _orthonormal(dim, seed, 3)
    r = _rng(seed)
    x = O.synth_rows(seed + 1, 0, n, dim)
    pos = r.choice(n, m, replace=False)
    t = r.random(m) * 4e-3
    x[pos] = (u[None, :] + t[:, None] * w[None, :]).astype(np.float32)
    s = r.random(nq) * 1e-3
    q = (u[None, :] + s[:, None] * w2[None, :]).astype(np.float32)
    return x, q


def low_dim(n, dim, nq, seed=4):
    """Components in {-1, 0, 1}: every score is one of a few values (+-1 included), with massive exact ties at the top."""
    r = _rng(seed + dim)
    x = r.integers(-1, 2, size=(n, dim)).astype(np.float32)
    q = r.integers(-1, 2, size=(nq, dim)).astype(np.float32)
    q[~q.any(axis=1), 0] = 1.0                                  # no zero query (those are covered elsewhere)
    return x, q


def midpoint_rows(dim):
    """Rows of unit norm EXACTLY (so 1/sqrt(n2) = 1 and the normalised row is the input) whose first component lies on a
    bf16 (1 - 2^-9) or fp16 (1 - 2^-12) rounding midpoint: 1023 = 31^2 + 7^2 + 3^2 + 2^2, 8191 = 90^2 + 9^2 + 3^2 + 1^2."""
    a = np.zeros((2, dim), np.float32)
    a[0, :5] = np.array([512 - 1, 31, 7, 3, 2], np.float32) * np.float32(2.0 ** -9)
    a[1, :5] = np.array([4096 - 1, 90, 9, 3, 1], np.float32) * np.float32(2.0 ** -12)
    assert (a.astype(np.float64) ** 2).sum(axis=1).tolist() == [1.0, 1.0]
    return a


def extreme_rows(dim, seed=5):
    """Rows at the ends of the fp32 range: largest finite components, a lone 2^-149, 1e30 mixed with 1e-30 (whose
    normalised parts underflow in every storage type), and the midpoint rows scaled by 2^100 and 2^-100."""
    r = _rng(seed)
    out = []
    a = np.zeros(dim, np.float32)
    a[r.choice(dim, 3, replace=False)] = [FMAX, -FMAX, FMAX]
    out.append(a)
    a = np.full(dim, FMAX, np.float32) * np.where(r.random(dim) < 0.5, -1, 1).astype(np.float32)
    out.append(a)
    for j in (0, dim // 2, dim - 1):
        a = np.zeros(dim, np.float32)
        a[j] = TINY
        out.append(a)
    a = np.where(r.random(dim) < 0.1, 1e30, 1e-30).astype(np.float32) * np.where(r.random(dim) < 0.5, -1, 1).astype(np.float32)
    out.append(a)
    a = np.full(dim, 1e-30, np.float32)
    a[dim // 3] = -1e30
    out.append(a)
    mid = midpoint_rows(dim)
    for s in (1.0, 2.0 ** 100, 2.0 ** -100):
        out.extend(mid * np.float32(s))
        out.extend(-mid[:, ::-1] * np.float32(s))
    return np.stack(out).astype(np.float32)


def extreme(n, dim, nq, seed=5):
    """Synthetic rows with every 7th row replaced by one of `extreme_rows` (in turn); queries the same kinds of rows and
    synthetic queries scaled by 2^100, 2^-120 and to the largest finite fp32."""
    x = O.synth_rows(seed, 0, n, dim)
    e = extreme_rows(dim, seed)
    idx = np.arange(0, n, 7)
    x[idx] = e[np.arange(len(idx)) % len(e)]
    q = O.synth_rows(seed + 1, 0, nq, dim)
    q[: len(e)] = e[: nq]
    scale = np.array([2.0 ** 100, 2.0 ** -120, FMAX / 2.0], np.float64)
    for i in range(len(e), nq):
        if i % 4 < 3:
            q[i] = (q[i].astype(np.float64) * scale[i % 4] / (1 if i % 4 < 2 else np.abs(q[i]).max())).astype(np.float32)
    return x, q


def non_finite(n, dim, nq, seed=6):
    """NaN, +Inf, -Inf components in rows (every 97th row, 4 kinds) and in queries 1-3."""
    x = O.synth_rows(seed, 0, n, dim)
    for j, vals in enumerate(([np.nan], [np.inf], [-np.inf], [np.nan, np.inf, -np.inf])):
        for r in range(j, n, 97):
            x[r, [(r * 7 + t) % dim for t in range(len(vals))]] = vals
    q = O.synth_rows(seed + 1, 0, nq, dim)
    q[1, 5], q[2, 0], q[3, dim - 1] = np.nan, np.inf, -np.inf
    return x, q


def build(name, n, dim, nq):
    """Family by name: negative, zeros, sub_eps_<m>, low_dim_<d> (the dim argument is ignored), extreme, non_finite."""
    if name.startswith("sub_eps_"):
        return sub_eps(n, dim, nq, int(name[8:]))
    if name.startswith("low_dim_"):
        return low_dim(n, int(name[8:]), nq)
    return {"negative": negative, "zeros": zeros, "extreme": extreme, "non_finite": non_finite}[name](n, dim, nq)
