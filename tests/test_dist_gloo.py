"""world_size-2 (and 3) CPU tests of the multi-GPU host logic over the gloo backend: row-block plan,
column windows, the all-gather and point-to-point x exchanges, all-reduced CG scalars.  The per-shard
compute is swapped for the CPU oracle here (tests only) -- on the GPU box the same code drives the CUDA
kernels (tests/test_gpu_dist.py)."""
import os
import socket
import sys

import numpy as np
import pytest
import scipy.io as sio
import scipy.sparse as sp
import torch
import torch.multiprocessing as mp

from conftest import ROOT, mtx_path, sample_spd


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _patch_ops_with_oracle():
    """Route the leaf launchers to the CPU oracle (CPU tensors in, CPU tensors out)."""
    from legate.sparse_b200 import _ops, csr as csr_mod
    from oracle import oracle as orc

    def spmv(indptr, indices, data, x, y, shape, plan=None):
        y[:] = torch.from_numpy(orc.spmv(indptr.numpy(), indices.numpy(), data.numpy(), x.numpy()[: shape[1]]))
        return y

    def spmm(indptr, indices, data, X, Y, shape):
        Y[:] = torch.from_numpy(orc.spmm(indptr.numpy(), indices.numpy(), data.numpy(), X.numpy()[: shape[1]]))
        return Y

    def spmv_dot(indptr, indices, data, x, y, w, out, shape, plan):
        spmv(indptr, indices, data, x, y, shape)
        out[:] = torch.from_numpy(orc.dot(w.numpy(), y.numpy()))
        return y

    def axpby(y, x, a, b, isalpha=True, negate=False):
        yy = y.numpy().copy()
        orc.axpby(yy, x.numpy(), a.numpy(), b.numpy(), isalpha=isalpha, negate=negate)
        y[:] = torch.from_numpy(yy)
        return y

    def dot(x, y, out=None):
        r = torch.from_numpy(orc.dot(x.numpy(), y.numpy()))
        if out is not None:
            out[:] = r
            return out
        return r

    def nrm2(x, out=None):
        return torch.from_numpy(orc.nrm2(x.numpy()))

    def cg_update_xr(x, r, p, q, rho, pq, rr_out):
        axpby(x, p, rho, pq, True, False)
        axpby(r, q, rho, pq, True, True)
        rr_out[:] = torch.from_numpy(orc.dot(r.numpy(), r.numpy()))
        return rr_out

    def spgemm(a_ptr, a_idx, a_val, b_ptr, b_idx, b_val, shape_a, shape_b):
        cp, ci, cv = orc.spgemm((a_ptr.numpy(), a_idx.numpy(), a_val.numpy()), (b_ptr.numpy(), b_idx.numpy(), b_val.numpy()),
                                shape_a, shape_b, sort_rows=True)
        return (torch.from_numpy(cp), torch.from_numpy(ci.astype(np.int32)), torch.from_numpy(cv),
                {"nnz": int(cp[-1]), "products": 0, "dense_rows": 0})

    _ops.spmv, _ops.spmv_dot, _ops.axpby, _ops.dot, _ops.cg_update_xr = spmv, spmv_dot, axpby, dot, cg_update_xr
    _ops.spgemm = spgemm
    _ops.spmm = spmm
    _ops.nrm2 = nrm2
    csr_mod.csr_array._get_plan = lambda self: None
    csr_mod.runtime.require_cuda = lambda what: None


def _worker(rank, world, port, case, q):
    # host process by design (gloo, oracle leaf ops): where GPUs are visible, init_process_group would bind each rank
    # to GPU `rank` and the package would place shards on it, so hide them before anything initialises CUDA
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    try:
        sys.path.insert(0, ROOT)
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                          LOCAL_RANK=str(rank))
        import torch.distributed as dist
        from legate.sparse_b200 import dist as bd

        bd.init_process_group("gloo")
        _patch_ops_with_oracle()
        out = {}
        if case == "spmv":
            for name in ("karate.mtx", "GlossGT.mtx", "cage4.mtx"):
                S = sio.mmread(mtx_path(name), spmatrix=False).tocsr().astype(np.float64)
                x = np.random.default_rng(3).random(S.shape[1])
                for mode in ("allgather", "p2p"):
                    os.environ["B2S_EXCHANGE"] = mode
                    A = bd.dist_csr_array.from_global(S)
                    assert A.exchange_mode == mode
                    y = A.matvec_global(x)
                    assert np.allclose(y, S @ x, rtol=1e-13), (name, mode)
                    lo, hi = A.row_plan.rows(rank)
                    if hi > lo and S.indptr[hi] > S.indptr[lo]:
                        seg = S.indices[S.indptr[lo] : S.indptr[hi]]
                        assert A.window == (seg.min(), seg.max() + 1)
            # banded matrix: the auto heuristic must choose the p2p halo exchange and move only the halo
            os.environ["B2S_EXCHANGE"] = "auto"
            n = 4000
            S = sp.diags([1.0, 2.0, 3.0], [-37, 0, 37], shape=(n, n), format="csr")
            A = bd.dist_csr_array.from_global(S)
            assert A.exchange_mode == "p2p"
            assert A.recv_elems <= 2 * 37
            x = np.random.default_rng(4).random(n)
            assert np.allclose(A.matvec_global(x), S @ x, rtol=1e-13)
            # dense-ish random matrix: windows span everything -> all-gather
            S = sp.random(300, 300, density=0.2, random_state=np.random.default_rng(9), format="csr")
            A = bd.dist_csr_array.from_global(S)
            assert A.exchange_mode == "allgather"
            assert np.allclose(A.matvec_global(x[:300]), S @ x[:300], rtol=1e-12)
            # nnz-balanced row cuts (reference csr_array.balance(), tests/integration/test_csr_misc.py:26-37)
            rng = np.random.default_rng(12)
            lens = np.minimum((rng.pareto(1.1, 600) * 3).astype(np.int64), 400)
            rows = np.repeat(np.arange(600), lens)
            cols = rng.integers(0, 600, rows.shape[0])
            S = sp.coo_array((rng.standard_normal(rows.shape[0]), (rows, cols)), shape=(600, 600)).tocsr()
            S.sum_duplicates()
            A = bd.dist_csr_array.from_global(S, balanced=True)
            nnzs = [None] * world
            dist.all_gather_object(nnzs, A.local.nnz)
            assert sum(nnzs) == S.nnz and max(nnzs) <= S.nnz / world + lens.max() + 1
            assert not A.row_plan.uniform or world == 1
            xs = rng.standard_normal(600)
            assert np.allclose(A.matvec_global(xs), S @ xs, rtol=1e-12, atol=1e-12)
            out["ok"] = True
        elif case == "spmm":
            rng = np.random.default_rng(21)
            for name in ("karate.mtx", "cage4.mtx"):
                S = sio.mmread(mtx_path(name), spmatrix=False).tocsr().astype(np.float64)
                X = rng.random((S.shape[1], 6))
                for mode in ("allgather", "p2p"):
                    os.environ["B2S_EXCHANGE"] = mode
                    A = bd.dist_csr_array.from_global(S)
                    assert np.allclose(A.matmat_global(X), S @ X, rtol=1e-13), (name, mode)
            # banded: only halo ROWS of the dense operand travel; rectangular: x sharded by its own plan
            os.environ["B2S_EXCHANGE"] = "auto"
            S = sp.diags([1.0, 2.0, 3.0], [-37, 0, 37], shape=(4000, 4000), format="csr")
            A = bd.dist_csr_array.from_global(S)
            assert A.exchange_mode == "p2p"
            X = rng.random((4000, 3))
            assert np.allclose(A.matmat_global(X), S @ X, rtol=1e-13)
            S = sp.random(130, 90, density=0.05, random_state=rng, format="csr", dtype=np.float64)
            A = bd.dist_csr_array.from_global(S)
            X = rng.random((90, 4))
            assert np.allclose(A.matmat_global(X), S @ X, rtol=1e-12, atol=1e-13)
            lo, hi = A.row_plan.rows(rank)
            full = A.new_full_matrix(4)
            clo, chi = A.my_cols
            full[clo:chi] = torch.from_numpy(X[clo:chi])
            Yl = A.spmm(full)
            assert tuple(Yl.shape) == (hi - lo, 4) and np.allclose(Yl.numpy(), (S @ X)[lo:hi], rtol=1e-12, atol=1e-13)
            out["ok"] = True
        elif case == "krylov":
            import scipy.sparse.linalg as spla
            from legate.sparse_b200 import linalg

            # non-symmetric, diagonally dominant system sharded by rows: every vector of the solvers is a shard,
            # inner products are all-reduced (krylov._Space), the operator exchanges x per product
            rng = np.random.default_rng(33)
            n = 240
            S = sp.csr_array(sp.random(n, n, density=0.05, random_state=rng, format="csr", dtype=np.float64)
                             + 10.0 * sp.eye(n))
            xs = rng.standard_normal(n)
            y = S @ xs
            for mode in ("allgather", "p2p"):
                os.environ["B2S_EXCHANGE"] = mode
                A = bd.dist_csr_array.from_global(S)
                lo, hi = A.row_plan.rows(rank)
                bl = torch.from_numpy(y[lo:hi].copy())
                for solver in (linalg.cgs, linalg.bicgstab):
                    xl = solver(A, bl, tol=1e-9)
                    xg = bd.gather_vector(xl if isinstance(xl, torch.Tensor) else torch.from_numpy(xl), A.row_plan, rank)
                    assert np.linalg.norm(S @ xg - y) < 1e-8, (solver.__name__, mode)
                xl, info = linalg.gmres(A, bl, tol=1e-10, restart=25)
                xg = bd.gather_vector(xl if isinstance(xl, torch.Tensor) else torch.from_numpy(xl), A.row_plan, rank)
                assert info == 0 and np.linalg.norm(S @ xg - y) <= 1.01e-10 * np.linalg.norm(y)
                ref = spla.gmres(S, y, rtol=1e-10, atol=0.0, restart=25)[0]
                assert np.allclose(xg, ref, atol=1e-7)
                for solver in (linalg.bicg, linalg.lsqr):      # need A^T: not available on a row shard
                    try:
                        solver(A, bl)
                        raise AssertionError("expected NotImplementedError")
                    except NotImplementedError:
                        pass
            # symmetric eigenproblem, sharded Lanczos
            Sym = sp.csr_array(0.5 * (S + S.T))
            A = bd.dist_csr_array.from_global(Sym)
            lo, hi = A.row_plan.rows(rank)
            np.random.seed(5)
            w, Vl = linalg.eigsh(A, k=4, tol=1e-10)
            exact = np.linalg.eigvalsh(Sym.toarray())
            assert np.allclose(w, np.sort(exact[np.argsort(np.abs(exact))[-4:]]), atol=1e-8)
            assert Vl.shape == (hi - lo, 4)
            for i in range(4):
                vg = bd.gather_vector(torch.from_numpy(np.ascontiguousarray(Vl[:, i])), A.row_plan, rank)
                assert np.allclose(Sym @ vg, w[i] * vg, atol=1e-6)
            out["ok"] = True
        elif case == "assemble":
            # triplets dealt to the ranks at random -> row shards identical to slicing the global CSR
            rng = np.random.default_rng(77)
            for (m, n, nnz) in ((500, 300, 4000), (7, 900, 600), (901, 40, 3000)):
                flat = np.random.default_rng(m).choice(m * n, size=nnz, replace=False)      # same on every rank
                r, c = flat // n, flat % n
                v = np.random.default_rng(n).standard_normal(nnz)
                S = sp.coo_array((v, (r, c)), shape=(m, n)).tocsr()
                S.sort_indices()
                holder = np.random.default_rng(nnz).integers(0, world, nnz)              # who holds which triplet
                mine = holder == rank
                if m == 7:            # the last rank holds nothing: rank 0 also passes what it would have held
                    mine = np.zeros(nnz, dtype=bool) if rank == world - 1 else (mine | ((holder == world - 1) & (rank == 0)))
                A = bd.dist_csr_array.from_triplets(torch.from_numpy(v[mine]), torch.from_numpy(r[mine]),
                                                    torch.from_numpy(c[mine]), (m, n))
                lo, hi = A.row_plan.rows(rank)
                loc = A.local.to_scipy_sparse_csr()
                assert np.array_equal(loc.indptr, S.indptr[lo : hi + 1] - S.indptr[lo]), (m, n)
                assert np.array_equal(loc.indices, S.indices[S.indptr[lo] : S.indptr[hi]])
                assert np.array_equal(loc.data, S.data[S.indptr[lo] : S.indptr[hi]])
                x = np.random.default_rng(1).random(n)
                assert np.allclose(A.matvec_global(x), S @ x, rtol=1e-12, atol=1e-12)
            out["ok"] = True
        elif case == "spgemm":
            rng = np.random.default_rng(5)
            SA = sp.random(130, 90, density=0.05, random_state=rng, format="csr", dtype=np.float64)
            SB = sp.random(90, 110, density=0.06, random_state=rng, format="csr", dtype=np.float64)
            A, B = bd.dist_csr_array.from_global(SA), bd.dist_csr_array.from_global(SB)
            C = bd.spgemm(A, B)
            ref = (SA @ SB).tocsr()
            ref.sort_indices()
            lo, hi = C.row_plan.rows(rank)
            loc = C.local.to_scipy_sparse_csr()
            assert np.array_equal(loc.indptr, ref.indptr[lo : hi + 1] - ref.indptr[lo])
            assert np.array_equal(loc.indices, ref.indices[ref.indptr[lo] : ref.indptr[hi]])
            assert np.allclose(loc.data, ref.data[ref.indptr[lo] : ref.indptr[hi]], rtol=1e-12)
            assert C.nnz_offset == ref.indptr[lo] and C.global_nnz == ref.nnz
            G = bd.gather_matrix(C).to_scipy_sparse_csr()
            assert (G != ref).nnz == 0
            # nnz-balanced row cuts of A (uneven shards): C keeps A's row plan (it used to fall back to equal tiles)
            skew = SA.tolil()
            skew[:20, :] = 1.0                       # heavy leading rows -> very uneven balanced cuts
            SK = skew.tocsr()
            Ab = bd.dist_csr_array.from_global(SK, balanced=True)
            assert not Ab.row_plan.uniform
            Cb = bd.spgemm(Ab, B)
            assert Cb.row_plan.bounds == Ab.row_plan.bounds
            refb = (SK @ SB).tocsr()
            refb.sort_indices()
            lob, hib = Cb.row_plan.rows(rank)
            locb = Cb.local.to_scipy_sparse_csr()
            assert locb.shape[0] == hib - lob
            assert np.array_equal(locb.indptr, refb.indptr[lob : hib + 1] - refb.indptr[lob])
            assert np.array_equal(locb.indices, refb.indices[refb.indptr[lob] : refb.indptr[hib]])
            assert Cb.nnz_offset == refb.indptr[lob] and Cb.global_nnz == refb.nnz
            out["ok"] = True
        elif case == "cg":
            from oracle import oracle as orc

            Ad, xs = sample_spd(200, 0.1, 471014)
            S = sp.csr_array(Ad)
            y = S @ xs
            for mode in ("allgather", "p2p"):
                os.environ["B2S_EXCHANGE"] = mode
                A = bd.dist_csr_array.from_global(S)
                lo, hi = A.row_plan.rows(rank)
                xl, iters = bd.cg(A, y[lo:hi], tol=1e-8)
                xg = bd.gather_vector(xl, A.row_plan, rank)
                xo, io = orc.cg(lambda v: orc.spmv(S.indptr, S.indices, S.data, v), y, tol=1e-8)
                assert iters == io, (iters, io)
                assert np.allclose(xg, xo, rtol=1e-9, atol=1e-13)
                assert np.allclose(S @ xg, y)
            out["ok"] = True
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, out))
    except Exception as exc:  # pragma: no cover
        import traceback

        q.put((rank, {"error": f"{exc}\n{traceback.format_exc()}"}))


def _run(world, case):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, case, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = []
    try:
        while len(results) < world and not (results and "error" in results[-1][1]):
            results.append(q.get(timeout=240))
    finally:
        for p in procs:   # after a failure the other ranks wait in a collective: do not leave them running
            p.join(timeout=60 if len(results) == world else 0)
            if p.is_alive():
                p.kill()
                p.join()
    for rank, out in results:
        assert "error" not in out, f"rank {rank}: {out.get('error')}"
        assert out.get("ok")


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_spmv_gloo(world):
    _run(world, "spmv")


def test_sharded_cg_gloo():
    _run(2, "cg")


def test_sharded_spgemm_gloo():
    _run(3, "spgemm")


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_spmm_gloo(world):
    _run(world, "spmm")


def test_sharded_krylov_gloo():
    _run(2, "krylov")


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_assembly_from_scattered_triplets_gloo(world):
    _run(world, "assemble")


def test_row_block_plan_matches_oracle(oracle, golden):
    from legate.sparse_b200.dist import RowBlockPlan

    indptr = golden["GlossGT_indptr"]
    n = indptr.shape[0] - 1
    for P in (1, 2, 3, 5, 8, 100):
        plan = RowBlockPlan(n, P)
        for r in range(P):
            lo, hi, _, _ = oracle.row_block(indptr, r, P)
            assert plan.rows(r) == (lo, hi)
