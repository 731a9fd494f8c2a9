"""CPU checks of the one-kernel search's int8 tile filter (csrc/sweep_fused.cuh, DESIGN.md 2.5), no GPU: the screen value
u = approx8 + c1 e + c0 bounds the exact score from above on adversarial rows and queries, with the quantizers and the fp32
evaluation restated in numpy as the kernels round them; and the argument checks of the new ABI symbols."""
import ctypes

import numpy as np
import pytest

from oracle import ragfin_oracle as O

F = np.float32


def quantize_rows(x):
    """quantize_i8_kernel: s = max|x| / 127, x8 = clamp(rint(x * (127 / max))), e = |x - s x8|_2 (exact, fp64)."""
    mx = np.abs(x).max(axis=1)
    live = np.isfinite(x).all(axis=1) & (mx > 0)
    s = np.where(live, mx / F(127), F(0)).astype(F)
    rs = np.where(live, F(127) / np.where(live, mx, F(1)), F(0)).astype(F)
    q = np.clip(np.rint((x * rs[:, None]).astype(F)), -127, 127)
    q[~live] = 0
    d = x.astype(np.float64) - s[:, None].astype(np.float64) * q
    d[~live] = 0
    return q, s, np.sqrt((d * d).sum(axis=1)) * (1 + 1e-15)


def quantize_query(y):
    """The kernel's prologue: y ~ sq (hi + lo / 256), |d|_2 of the exact residual."""
    mx = F(np.abs(y).max())
    sq = F(mx / F(127))
    rsq = F(F(127) / mx) if mx > 0 else F(0)
    hi = np.clip(np.rint((y * rsq).astype(F)), -127, 127)
    lo = np.clip(np.rint(((y - (sq * hi).astype(F)).astype(F) * rsq * F(256)).astype(F)), -127, 127)
    d = (y.astype(np.float64) - np.float64(sq) * hi) - np.float64(sq) * lo / 256
    return hi, lo, sq, np.sqrt((d * d).sum()) * (1 + 1e-15)


def eps_i8_conv(ld):
    r = np.sqrt(ld)
    return 5.01 * 2.0 ** -24 * 1.0078125 * (1 + r / 250) * (1.00001 + r / 125)


def screen_bound(x, y):
    """(exact q.x, approx8 as the kernel evaluates it, E) for every row of x."""
    x8, s, e = quantize_rows(x)
    hi, lo, sq, dq = quantize_query(y)
    H = (x8 * hi).sum(axis=1)
    L = (x8 * lo).sum(axis=1)
    w = ((s * sq).astype(F) * (H.astype(F) + L.astype(F) * F(1 / 256)).astype(F)).astype(F)
    E = (1 + 2.0 ** -20 + dq) * e + 1.0078125 * dq + eps_i8_conv(x.shape[1])
    exact = x.astype(np.float64) @ y.astype(np.float64)
    return exact, w.astype(np.float64), E


def _unit(v):
    v = v.astype(np.float64)
    n = np.linalg.norm(v, axis=-1, keepdims=True)
    return (v / np.where(n > 0, n, 1)).astype(F)


def _bf16(v):
    u = np.ascontiguousarray(v, dtype=F).view(np.uint32)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.view(F)


@pytest.mark.parametrize("dim", [8, 100, 768, 1024])
def test_screen_value_bounds_the_exact_score(dim):
    rng = np.random.default_rng(dim)
    rows = [O.synth_rows(1, 0, 200, dim)]
    spiky = rng.standard_normal((100, dim)) * 1e-4
    spiky[np.arange(100), rng.integers(0, dim, 100)] = 1.0           # one large component, the rest far below it
    rows.append(spiky)
    half = np.zeros((50, dim)); half[:, : max(1, dim // 2)] = 1.0      # many components at exactly the maximum
    rows.append(half)
    mid = rng.standard_normal((50, dim)); mid *= (np.rint(mid * 127) + 0.5) / 127 / np.where(mid == 0, 1, mid)   # midpoints
    rows.append(mid)
    x = _bf16(_unit(np.concatenate(rows)))
    x[5, :] = 0.0
    x[6, ::3] = 1e-30                                                  # subnormal-range components (bf16)
    queries = [O.synth_rows(2, 0, 8, dim), rng.standard_normal((4, dim)) ** 3, np.eye(dim)[:2] + 1e-7]
    for y in _unit(np.concatenate(queries)):
        exact, w, E = screen_bound(x, y)
        assert (np.abs(exact - w) <= E).all(), np.max(np.abs(exact - w) - E)


def test_query_residual_is_small():
    """The query term: |d|_2 <= sqrt(dim) * sq / 512 (hi and lo each within half a step), far below the row residual."""
    for dim in (8, 768, 4096):
        for y in _unit(O.synth_rows(3, 0, 16, dim)):
            _, _, sq, dq = quantize_query(y)
            assert dq <= np.sqrt(dim) * float(sq) / 512 * 1.0001 + 1e-30


def test_abi_argument_checks():
    from ragfin_b200 import _lib
    L = _lib.load()
    ld8 = ctypes.c_int32(0)
    out = (ctypes.c_int64 * 2)()
    assert L.ragfin_set_sweep_copy(None, 1) == _lib.EINVAL
    assert L.ragfin_debug_sweep_copy(None, 0, 0, None, None, ctypes.byref(ld8)) == _lib.EINVAL
    assert L.ragfin_debug_fused_tiles(None, out) == _lib.EINVAL
