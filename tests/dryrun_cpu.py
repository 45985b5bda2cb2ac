"""Developer aid (NOT part of either test suite, never imported by the package): runs `-m gpu` test files in this
GPU-less container with every tensor pretending to be a CUDA tensor and the leaf launchers of `_ops` swapped for
the CPU oracle.  It checks the Python side of a new GPU test (shapes, dtypes, dispatch, return conventions) before
GPU minutes are spent on it; it says nothing about the kernels.

    python tests/dryrun_cpu.py tests/test_gpu_zspmm.py [-k expr]
"""
import os
import sys

os.environ["CUDA_VISIBLE_DEVICES"] = ""   # a host run by design: where a GPU is visible, keep the package off it

import numpy as np  # noqa: E402
import pytest  # noqa: E402
import torch  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def install():
    from legate.sparse_b200 import _ops
    from legate.sparse_b200.runtime import runtime
    from oracle import oracle as orc

    torch.Tensor.is_cuda = property(lambda self: True)
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.cuda.synchronize = lambda *a, **k: None
    real_to = torch.Tensor.to

    def to(self, *a, **k):
        a = tuple("cpu" if (isinstance(v, (str, torch.device)) and str(v).startswith("cuda")) else v for v in a)
        if str(k.get("device", "cpu")).startswith("cuda"):
            k["device"] = "cpu"
        return real_to(self, *a, **k)

    torch.Tensor.to = to
    for name in ("zeros", "empty", "ones", "full", "rand", "randn", "arange", "tensor"):
        orig = getattr(torch, name)

        def wrapped(*a, __orig=orig, **k):
            if str(k.get("device", "cpu")).startswith("cuda"):
                k["device"] = "cpu"
            return __orig(*a, **k)

        setattr(torch, name, wrapped)

    class FakePlan:
        chunks = []
        config = rowgroup = uniform = scattered = tiles = short_rows = tma = 0
        kernel_name = "oracle"

    def spmv_plan(indptr, indices, shape, nnz, vdtype, tma_only=False):
        return FakePlan()

    def spmv(indptr, indices, data, x, y, shape, plan=None):
        y[:] = torch.from_numpy(orc.spmv(indptr.numpy(), indices.numpy(), data.numpy(), x.numpy()))
        return y

    def spmv_add(indptr, indices, data, x, y, shape, plan):
        y += torch.from_numpy(orc.spmv(indptr.numpy(), indices.numpy(), data.numpy(), x.numpy()))
        return y

    def spmm(indptr, indices, data, X, Y, shape):
        Y[:] = torch.from_numpy(orc.spmm(indptr.numpy(), indices.numpy(), data.numpy(), X.contiguous().numpy()))
        return Y

    def dot(x, y, out=None):
        r = torch.from_numpy(orc.dot(x.numpy(), y.numpy()))
        if out is not None:
            out[:] = r
            return out
        return r

    def nrm2(x, out=None):
        return torch.from_numpy(orc.nrm2(x.numpy()))

    def axpby(y, x, a, b, isalpha=True, negate=False):
        yy = y.numpy().copy()
        orc.axpby(yy, x.numpy(), a.numpy(), b.numpy(), isalpha=isalpha, negate=negate)
        y[:] = torch.from_numpy(yy)
        return y

    def spmv_dot(indptr, indices, data, x, y, w, out, shape, plan):
        spmv(indptr, indices, data, x, y, shape)
        out[:] = torch.from_numpy(orc.dot(w.numpy(), y.numpy()))
        return y

    def cg_update_xr(x, r, p, q, rho, pq, rr_out):
        axpby(x, p, rho, pq, True, False)
        axpby(r, q, rho, pq, True, True)
        rr_out[:] = torch.from_numpy(orc.dot(r.numpy(), r.numpy()))
        return rr_out

    def csr_diagonal(indptr, indices, data, nrows):
        import scipy.sparse as sp

        n = int(indices.max()) + 1 if indices.numel() else 0
        S = sp.csr_array((data.numpy(), indices.numpy(), indptr.numpy()), shape=(nrows, max(n, nrows)))
        return torch.from_numpy(np.ascontiguousarray(S.diagonal()[:nrows]))

    def spgemm(a_ptr, a_idx, a_val, b_ptr, b_idx, b_val, shape_a, shape_b):
        cp, ci, cv = orc.spgemm((a_ptr.numpy(), a_idx.numpy(), a_val.numpy()), (b_ptr.numpy(), b_idx.numpy(), b_val.numpy()),
                                shape_a, shape_b, sort_rows=True)
        return (torch.from_numpy(cp), torch.from_numpy(ci.astype(np.int32)), torch.from_numpy(cv),
                {"nnz": int(cp[-1]), "products": 0, "dense_rows": 0})

    def coo_to_csr(rows, cols, vals, nrows, ptr_dtype, idx_dtype):
        import scipy.sparse as sp

        r, c = rows.numpy().astype(np.int64), cols.numpy().astype(np.int64)
        if r.size and (r.min() < 0 or r.max() >= nrows):
            raise ValueError(f"{int(((r < 0) | (r >= nrows)).sum())} triplets have a row index outside [0, {nrows})")
        ncols = int(c.max()) + 1 if c.size else 1
        S = sp.coo_array((vals.numpy(), (r, c)), shape=(nrows, ncols)).tocsr()
        S.sort_indices()
        return (torch.from_numpy(S.indptr.astype(np.int64)).to(ptr_dtype), torch.from_numpy(S.indices.astype(np.int64)).to(idx_dtype),
                torch.from_numpy(S.data))

    def csr_transpose(indptr, indices, data, shape):
        import scipy.sparse as sp

        S = sp.csr_array((data.numpy(), indices.numpy(), indptr.numpy()), shape=shape).T.tocsr()
        S.sort_indices()
        return (torch.from_numpy(S.indptr.astype(np.int64)).to(indptr.dtype),
                torch.from_numpy(S.indices.astype(np.int64)).to(indices.dtype), torch.from_numpy(S.data))

    _ops.coo_to_csr, _ops.csr_transpose = coo_to_csr, csr_transpose
    _ops.spmv_plan, _ops.spmv, _ops.spmm, _ops.dot, _ops.nrm2 = spmv_plan, spmv, spmm, dot, nrm2
    _ops.spmv_add = spmv_add
    _ops.axpby, _ops.spmv_dot, _ops.cg_update_xr, _ops.csr_diagonal, _ops.spgemm = (axpby, spmv_dot, cg_update_xr,
                                                                                      csr_diagonal, spgemm)
    runtime.require_cuda = lambda what: None
    os.environ["B2S_CG_GRAPH"] = "0"


if __name__ == "__main__":
    install()
    sys.exit(pytest.main(["-m", "gpu", "-q", "-p", "no:cacheprovider"] + sys.argv[1:]))
