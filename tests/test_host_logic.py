"""CPU-only checks of the host side of legate.sparse_b200: the C-ABI library loads and exports every
symbol include/b200sparse.h declares, argument validation returns error codes, constructors / mmread /
diags agree with scipy, and compute entry points fail loudly without a GPU (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest
import scipy.io as sio
import scipy.sparse as sp
import torch

from conftest import MTX_FILES, ROOT, mtx_path

import legate.sparse_b200 as sparse
from legate.sparse_b200 import _lib


@pytest.fixture(autouse=True)
def _host_tensors(monkeypatch):
    """Host-side checks: keep the package on host tensors where a GPU is visible too (it would place them there)."""
    from legate.sparse_b200.runtime import Runtime

    monkeypatch.setattr(Runtime, "has_cuda", property(lambda self: False))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "b200sparse.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b2s_[a-z0-9_]+)\s*\(", text)))


def test_abi_exports_every_declared_symbol():
    names = _declared_symbols()
    assert len(names) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/b200sparse.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature in _lib.py"


def test_abi_signature_arity_matches_header():
    """Every prototype in include/b200sparse.h has as many parameters as its ctypes signature in _lib.py."""
    text = open(os.path.join(ROOT, "include", "b200sparse.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    protos = re.findall(r"\b(b2s_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", text, flags=re.S)
    assert len(protos) >= 30
    for name, params in protos:
        params = params.strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        assert len(_lib.SIGNATURES[name][1]) == n, f"{name}: header has {n} parameters, ctypes {len(_lib.SIGNATURES[name][1])}"


def test_reference_package_alias():
    """`import sparse` (the reference's package name) resolves to this implementation."""
    import sparse as ref_name
    import sparse.io
    import sparse.linalg

    assert ref_name.csr_array is sparse.csr_array and ref_name.linalg.cg is sparse.linalg.cg
    assert ref_name.io.mmread is sparse.io.mmread


def test_abi_version_and_sizes():
    assert _lib.lib.b2s_version() == 1
    assert _lib.lib.b2s_ws_bytes() >= 16 + 8 * 1024
    assert _lib.lib.b2s_spmv_plan_tiles(1, 0, 0) == 0
    t = _lib.lib.b2s_spmv_plan_tiles(1, 1000, 5000)
    assert t >= 1 and t == -(-6000 // 1020)  # default config: CAP 1024 for fp64
    assert _lib.lib.b2s_spmv_plan_bytes(1, 1000, 5000) == (t + 2) * 16


def test_abi_argument_validation_without_gpu():
    L = _lib.lib
    # bad type code / NULL pointers are rejected before any CUDA call
    rc = L.b2s_spmv_csr(7, 0, 0, 4, 4, 4, None, None, None, None, None, None, None)
    assert rc == _lib.EINVAL and "type code" in _lib.last_error()
    rc = L.b2s_spmv_csr(1, 0, 0, 4, 4, 4, None, None, None, None, None, None, None)
    assert rc == _lib.EINVAL and "NULL" in _lib.last_error()
    rc = L.b2s_axpby(1, -3, None, None, None, None, 1, 0, None)
    assert rc == _lib.EINVAL
    rc = L.b2s_spmv_set_config(99, 0)
    assert rc == _lib.EINVAL
    with pytest.raises(_lib.B200SparseError):
        _lib.check(rc, "b2s_spmv_set_config")


@pytest.mark.parametrize("name", MTX_FILES)
def test_mmread(name):
    arr = sparse.io.mmread(mtx_path(name))
    s = sio.mmread(mtx_path(name), spmatrix=False)
    assert np.array_equal(arr.todense(), s.toarray())          # reference tests/integration/test_io.py:23-28
    csr = arr.tocsr()
    sc = s.tocsr()
    sc.sort_indices()
    assert np.array_equal(csr.indptr.numpy(), sc.indptr)
    assert np.array_equal(csr.indices.numpy(), sc.indices)
    assert np.array_equal(csr.data.numpy(), sc.data)
    assert csr.dtype == np.float64 and csr.indices.dtype == torch.int32


def test_constructors_match_scipy():
    rng = np.random.default_rng(5)
    D = rng.standard_normal((13, 9)) * (rng.random((13, 9)) < 0.3)
    S = sp.csr_array(D)
    for A in (sparse.csr_array(D), sparse.csr_array(S), sparse.csr_matrix(sp.csr_matrix(D)),
              sparse.csr_array((S.data, S.indices, S.indptr), shape=S.shape),
              sparse.csr_array((S.tocoo().data, (S.tocoo().row, S.tocoo().col)), shape=S.shape)):
        assert A.shape == (13, 9) and A.nnz == S.nnz
        assert np.array_equal(A.todense(), D)
        assert np.array_equal(A.indptr.numpy(), S.indptr)
    A = sparse.csr_array(D)
    assert A.astype(np.float32).dtype == np.float32
    assert np.array_equal(A.copy().todense(), D)
    assert np.array_equal(A.T.todense(), D.T)
    assert np.array_equal(A.tocoo().todense(), D)
    back = A.to_scipy_sparse_csr()
    assert (back != S).nnz == 0
    with pytest.raises(AssertionError):
        sparse.csr_array((S.data, S.indices, S.indptr))          # shape required (reference csr.py:171)


@pytest.mark.parametrize("name", MTX_FILES)
def test_conversions_on_the_reference_fixtures(name):
    """reference tests/integration/test_csr_conversion.py:26-83 and test_csr_misc.py:39-55 (format logic only)."""
    s = sio.mmread(mtx_path(name), spmatrix=False)
    coo = sparse.io.mmread(mtx_path(name))
    arr = coo.tocsr()
    dense = s.toarray()
    assert np.array_equal(sparse.csr_array(coo.todense()).todense(), dense)                 # from dense
    assert np.array_equal(arr.todense(), arr.tocoo().todense())                             # to COO
    c = arr.tocoo()
    assert np.array_equal(sparse.csr_array((c.data, (c.row, c.col)), dtype=c.dtype, shape=c.shape).todense(), dense)
    assert np.array_equal(sparse.csr_array(sp.csr_array(dense).astype(np.float64)).todense(), dense)   # from scipy
    assert np.array_equal(arr.conj(copy=False).todense(), s.tocsr().conj(copy=False).toarray())
    assert np.array_equal(arr.to_scipy_sparse_csr().toarray(), dense)
    for dt in (np.float32, np.float64):
        assert np.array_equal(arr.astype(dt).todense(), s.tocsr().astype(dt).toarray())
    assert np.array_equal(arr.T.todense(), np.ascontiguousarray(dense.T))                   # transpose
    assert np.array_equal(np.asarray(arr.diagonal(k=0)), s.tocsr().diagonal(k=0))           # diagonal


def test_diags_and_eye_match_scipy():
    n = 50
    for nnz_per_row in (1, 5, 11):
        offs = [x - (nnz_per_row // 2) for x in range(nnz_per_row)]
        ours = sparse.diags([1] * nnz_per_row, offs, shape=(n, n), format="csr", dtype=np.float64)
        ref = sp.diags([1] * nnz_per_row, offs, shape=(n, n), format="csr", dtype=np.float64)
        assert np.array_equal(ours.todense(), ref.toarray())
        assert np.array_equal(ours.indptr.numpy(), ref.indptr)
    # pde.py:124-163 construction: diags(...).tocsc().T with explicit zeros on the +-1 diagonals
    nx = ny = 9
    a, g = 64.0, 64.0
    diag_a = a * np.ones((nx - 2) * (ny - 2) - 1)
    diag_a[nx - 3 :: nx - 2] = 0.0
    diag_g = g * np.ones((nx - 2) * (ny - 3))
    diag_c = (-2 * a - 2 * g) * np.ones((nx - 2) * (ny - 2))
    args = ([diag_g, diag_a, diag_c, diag_a, diag_g], [-(nx - 2), -1, 0, 1, nx - 2])
    ours = sparse.diags(*args, dtype=np.float64).tocsc().T
    ref = sp.diags(*args, dtype=np.float64).tocsr()
    assert isinstance(ours, sparse.csr_array)
    assert np.array_equal(ours.todense(), ref.toarray())
    N = (nx - 2) * (ny - 2)
    assert ours.nnz == 5 * N - 4 * (nx - 2)                       # explicit zeros dropped (dia.py:236)
    assert np.array_equal(sparse.eye(7).todense(), np.eye(7))
    assert sparse.is_sparse_matrix(ours) and not sparse.is_sparse_matrix(np.eye(3))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    A = sparse.io.mmread(mtx_path("test.mtx")).tocsr()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        A @ np.ones(5)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        A @ A
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        sparse.linalg.cg(A, np.ones(5))


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under legate/sparse_b200 may reference it."""
    pkg = os.path.join(ROOT, "legate", "sparse_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower().replace("test oracle", ""), f"{f} mentions the oracle"
