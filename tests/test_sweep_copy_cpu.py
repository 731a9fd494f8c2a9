"""CPU suite for the "f32+f16" storage type (include/ragfin.h RAGFIN_F32_F16): fp32 rows for every exact step plus an fp16
copy the tensor-core sweeps stream.  No device needed: argument handling, the Python names, the shim's pass-through and the
error bound of DESIGN.md 2 (|q.x - q.RNE_f16(x)| <= |q| (2^-11 |x| + 2^-25 sqrt(ld))) on adversarial rows."""
import ctypes
import math

import numpy as np
import pytest

from oracle import ragfin_oracle as O


@pytest.fixture(scope="module")
def lib():
    import os
    import __graft_entry__ as ge
    from ragfin_b200 import _lib
    if not os.path.exists(_lib.SO_PATH):
        ge.build()
    return _lib.load()


def test_create_without_a_device_fails_with_ecuda_not_einval(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    h = ctypes.c_void_p()
    assert lib.ragfin_create(ctypes.byref(h), 8, 3, 10, 0) == -2     # dtype 3 is valid: only the missing device fails
    assert lib.ragfin_create(ctypes.byref(h), 8, 4, 10, 0) == -1     # EINVAL: no dtype 4
    assert h.value is None


def test_names_and_abi_version(lib):
    from ragfin_b200 import engine, _lib
    assert engine.DTYPE_CODE["f32+f16"] == 3
    assert "ragfin_read_sweep_rows" in _lib.SYMBOLS
    assert lib.ragfin_abi_version() == 4
    assert "f32+f16" not in O.DTYPES                                  # existing parametrisations are not widened


def eps_sweep_const(ld):
    """csrc/ragfin_api.cu eps_sweep_const: |q|_2 <= 1 + 2^-22, |x|_2 <= 1 + 2^-20."""
    return (1 + 2.0 ** -22) * (2.0 ** -11 * (1 + 2.0 ** -20) + 2.0 ** -25 * math.sqrt(ld))


def _check_bound(x, tight_rel=None):
    """q = x / |x| (the query aligned with the row: the error terms add up instead of cancelling)."""
    x = np.asarray(x, np.float32)
    ld = x.shape[1]
    xd = x.astype(np.float64)
    err_rows = xd - x.astype(np.float16).astype(np.float64)          # numpy's float16 cast rounds to nearest even
    norms = np.linalg.norm(xd, axis=1)
    assert (norms <= 1 + 2.0 ** -20).all()
    q = xd / norms[:, None]
    err = np.abs(np.einsum("ij,ij->i", q, err_rows))
    bound = np.linalg.norm(q, axis=1) * (2.0 ** -11 * norms + 2.0 ** -25 * math.sqrt(ld))
    assert (err <= bound).all(), float((err / bound).max())
    assert (bound <= eps_sweep_const(ld)).all()
    if tight_rel is not None:                                         # the rows really are adversarial
        assert (err >= tight_rel * 2.0 ** -11 * norms).all(), float((err / (2.0 ** -11 * norms)).min())
    return err


@pytest.mark.parametrize("dim", [8, 100, 768, 2048])
def test_bound_on_random_rows(dim):
    x = O.normalize_rows(O.synth_rows(90 + dim, 0, 400, dim), "f32")
    _check_bound(x)


@pytest.mark.parametrize("dim", [64, 768, 1024])
def test_bound_on_rows_next_to_fp16_rounding_midpoints(dim):
    """All-positive rows whose every component sits one fp32 ulp below the midpoint of two fp16 neighbours at the bottom of
    a binade, where the relative rounding error is largest (just under 2^-11): q . (x - x16) is a sum of same-sign terms."""
    rng = np.random.default_rng(dim)
    e = math.floor(math.log2(0.99 / math.sqrt(dim)))                  # the bottom of binade [2^e, 2^(e+1)) keeps |x| < 1
    ulp16 = 2.0 ** (e - 10)
    m = rng.integers(0, 8, size=(200, dim))                           # first few fp16 values of the binade
    mid = (2.0 ** e + (m + 0.5) * ulp16).astype(np.float32)
    x = np.nextafter(mid, np.float32(0))                              # just below the midpoint: rounds down by ~ulp16 / 2
    _check_bound(x, tight_rel=0.99)


@pytest.mark.parametrize("dim", [64, 768])
def test_bound_on_rows_with_subnormal_range_components(dim):
    """Rows whose components are mostly below fp16's normal range (|x_i| < 2^-14, spacing 2^-24), each one fp32 ulp below a
    subnormal rounding midpoint, plus a few large ones that carry the norm."""
    rng = np.random.default_rng(7 + dim)
    j = rng.integers(1, 200, size=(200, dim))
    x = np.nextafter(((j + 0.5) * 2.0 ** -24).astype(np.float32), np.float32(0))
    x[:, :4] = np.float32(0.45)
    err = _check_bound(x)
    assert err.max() > 0


def test_shim_passes_the_storage_type_to_its_index_factory():
    from ragfin_b200 import milvus_compat as mc
    seen = []

    class Fake:
        def __init__(self, dim, dtype, capacity, device):
            seen.append(dtype)
            self.rows = np.zeros((0, dim), np.float32)

        def add(self, rows):
            self.rows = np.concatenate([self.rows, O.normalize_rows(rows, "f32")])

        def reserve(self, capacity):
            pass

        def search(self, q, k, allow=None):
            return O.cosine_topk(q, self.rows, k)

        def close(self):
            pass

    F, D = mc.FieldSchema, mc.DataType
    fields = [F("id", D.INT64, is_primary=True), F("embedding", D.FLOAT_VECTOR, dim=16)]
    mc.connections.connect("default")
    if mc.utility.has_collection("sweep_copy"):
        mc.utility.drop_collection("sweep_copy")
    col = mc.Collection("sweep_copy", mc.CollectionSchema(fields, ""), index_factory=Fake, storage_dtype="f32+f16")
    x = O.synth_rows(5, 0, 20, 16)
    col.insert([list(range(20)), x.tolist()])
    col.flush()
    col.load()
    res = col.search(x[:1].tolist(), "embedding", {"metric_type": "COSINE"}, limit=3)
    assert seen == ["f32+f16"] and res[0].ids[0] == 0
    assert mc.DEFAULTS["storage_dtype"] == "f32"
    mc.utility.drop_collection("sweep_copy")
