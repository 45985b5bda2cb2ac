"""Host logic of the Krylov solvers next to cg (legate/sparse_b200/krylov.py) on CPU tensors: the operator
applies the matrix with the CPU oracle and the reductions are the oracle's dot / nrm2 (tests only), so what is
exercised here is the recurrences, the stopping rules and the return conventions, against scipy on the seeded
systems of the reference tests (tests/integration/test_cgs_solve.py, test_bicg_solve.py, test_gmres_solve.py,
test_lsqr_solve.py, test_eigsh.py).  The same code drives the CUDA kernels in tests/test_gpu_zy_krylov.py."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla
import torch

from conftest import sample, sample_spd


@pytest.fixture()
def cpu_ops(monkeypatch, oracle):
    from legate.sparse_b200 import _ops
    from legate.sparse_b200.runtime import runtime

    def dot(x, y, out=None):
        return torch.from_numpy(oracle.dot(x.numpy(), y.numpy()))

    def nrm2(x, out=None):
        return torch.from_numpy(oracle.nrm2(x.numpy()))

    monkeypatch.setattr(_ops, "dot", dot)
    monkeypatch.setattr(_ops, "nrm2", nrm2)
    monkeypatch.setattr(runtime, "require_cuda", lambda what: None)
    monkeypatch.setattr(type(runtime), "has_cuda", property(lambda self: False))   # host tensors where a GPU is visible too
    return oracle


def _operator(S, oracle, with_transpose=True):
    from legate.sparse_b200 import linalg

    S = sp.csr_array(S)
    St = sp.csr_array(S.T)

    def mv(M):
        def f(x):
            return torch.from_numpy(oracle.spmv(M.indptr, M.indices, M.data, x.numpy()))
        return f

    return linalg.LinearOperator(S.shape, matvec=mv(S), rmatvec=mv(St) if with_transpose else None, dtype=S.dtype)


def test_cgs_bicg_bicgstab_on_reference_system(cpu_ops):
    from legate.sparse_b200 import linalg

    S, x = sample(100, 100, 0.1, 471014)
    y = S @ x
    A = _operator(S, cpu_ops)
    xp = linalg.bicg(A, y, tol=1e-8)
    assert isinstance(xp, np.ndarray) and xp.dtype == np.float64
    assert np.allclose(S @ xp, y, rtol=1e-5, atol=1e-6)
    # CGS and BiCGSTAB are not robust on that indefinite system: whether CGS gets below 1e-8 within 10 n iterations
    # depends on the rounding of the inner products (scipy's cgs stalls at 6e-5 after 1000 iterations, its bicgstab
    # diverges; the reference skips its BiCGSTAB test, test_bicg_solve.py:35).  Same matrix shifted to be
    # diagonally dominant, still non-symmetric:
    S2 = sp.csr_array(S + 12.0 * sp.eye(100))
    y2 = S2 @ x
    for solver, ref_solver in ((linalg.cgs, spla.cgs), (linalg.bicgstab, spla.bicgstab)):
        xp = solver(_operator(S2, cpu_ops), y2, tol=1e-8)
        assert np.allclose(S2 @ xp, y2, rtol=1e-5, atol=1e-6), solver.__name__
        ref, info = ref_solver(S2, y2, rtol=0, atol=1e-8)
        assert info == 0 and np.allclose(xp, ref, atol=1e-6)


def test_false_convergence_is_caught(cpu_ops, monkeypatch):
    """The recurrence residual of CGS drifts from b - A x; a solver may only return once the recomputed residual
    is below tol.  Forced here by an operator that is slightly perturbed inside the recurrences' products."""
    from legate.sparse_b200 import krylov, linalg

    Ad, xs = sample_spd(60, 0.1, 7)
    S = sp.csr_array(Ad)
    y = S @ xs
    A = _operator(S, cpu_ops)
    calls = []
    real = krylov._confirm

    def spy(op, sp_, b, x, tol):
        r, ok = real(op, sp_, b, x, tol)
        calls.append(ok)
        return r, ok

    monkeypatch.setattr(krylov, "_confirm", spy)
    for solver in (linalg.cgs, linalg.bicg, linalg.bicgstab):
        calls.clear()
        xp = solver(A, y, tol=1e-9)
        assert calls and calls[-1] is True
        assert np.linalg.norm(S @ xp - y) < 1e-9


def test_plain_solvers_honour_x0_maxiter_and_reject_M(cpu_ops):
    from legate.sparse_b200 import linalg

    Ad, xs = sample_spd(60, 0.1, 7)
    S = sp.csr_array(Ad)
    y = S @ xs
    A = _operator(S, cpu_ops)
    for solver in (linalg.cgs, linalg.bicg, linalg.bicgstab):
        exact = solver(A, y, x0=xs.copy(), tol=1e-8)          # already converged: returned untouched
        assert np.array_equal(exact, xs)
        rough = solver(A, y, tol=1e-30, maxiter=3)            # cannot reach the tolerance: stops at maxiter
        good = solver(A, y, tol=1e-10)
        assert np.linalg.norm(S @ good - y) < 1e-9 < np.linalg.norm(S @ rough - y)
        with pytest.raises(AssertionError):
            solver(A, y, M=A)
        with pytest.raises(NotImplementedError):
            solver(A, y, callback=lambda x: None)
    xin = torch.from_numpy(xs.copy())
    linalg.cgs(A, y, x0=xin, tol=1e-8)
    assert torch.equal(xin, torch.from_numpy(xs))                # x0 is never modified in place


def test_gmres_matches_scipy(cpu_ops):
    from legate.sparse_b200 import linalg

    S, x = sample(100, 100, 0.1, 471014)
    y = S @ x
    A = _operator(S, cpu_ops)
    ref = spla.gmres(S, y, atol=1e-5, rtol=1e-5, maxiter=300, restart=20)[0]
    got, info = linalg.gmres(A, y, atol=1e-5, tol=1e-5, maxiter=300)
    assert np.allclose(ref, got, atol=1e-1)                   # the reference test's bar (test_gmres_solve.py:43)
    # a well-conditioned system converges: info == 0 and the residual meets atol
    Ad, xs = sample_spd(80, 0.1, 3)
    P = sp.csr_array(Ad)
    yp = P @ xs
    seen = []
    got, info = linalg.gmres(_operator(P, cpu_ops), yp, tol=1e-10, restart=30, callback=seen.append)
    assert info == 0 and np.linalg.norm(P @ got - yp) <= 1e-10 * np.linalg.norm(yp) * 1.01
    assert seen and all(isinstance(v, float) for v in seen) and seen[-1] <= 1e-10
    # preconditioned with the exact inverse it converges within the first cycle
    Minv = sp.csr_array(np.linalg.inv(Ad))
    got, info = linalg.gmres(_operator(P, cpu_ops), yp, tol=1e-10, M=_operator(Minv, cpu_ops), restart=5)
    assert info == 0 and np.allclose(got, xs, atol=1e-8)
    # zero right-hand side, iteration cap, callback_type validation
    z, info = linalg.gmres(A, np.zeros(100))
    assert info == 0 and not z.any()
    _, info = linalg.gmres(A, y, tol=1e-14, maxiter=40, restart=20)
    assert info == 40
    with pytest.raises(ValueError):
        linalg.gmres(A, y, callback=print, callback_type="bogus")


@pytest.mark.parametrize("shape", [(1000, 500), (300, 300), (200, 400)])
def test_lsqr_matches_scipy(cpu_ops, shape):
    from legate.sparse_b200 import linalg

    N, D = shape
    S, x = sample(N, D, 0.1, 471014)
    y = S @ x
    A = _operator(S, cpu_ops)
    got = linalg.lsqr(A, y, atol=1e-10, btol=1e-10)
    ref = spla.lsqr(S, y, atol=1e-10, btol=1e-10)
    assert len(got) == 10
    assert np.allclose(S @ got[0], y, atol=1e-6)
    assert got[1] == ref[1]                                    # istop
    assert abs(got[2] - ref[2]) <= 2                           # iterations (rounding may move the stop by one)
    # anorm / xnorm estimates: the Lanczos coefficients drift apart in the last digits between two
    # implementations once orthogonality is lost, so these agree to a few digits only on the long runs
    assert np.isclose(got[5], ref[5], rtol=1e-2) and np.isclose(got[8], ref[8], rtol=1e-6)
    assert np.allclose(got[0], ref[0], atol=1e-6)


def test_lsqr_damped_warm_start_and_variances(cpu_ops):
    from legate.sparse_b200 import linalg

    S, x = sample(120, 60, 0.2, 5)
    y = S @ x + 0.01 * np.random.default_rng(0).standard_normal(120)
    A = _operator(S, cpu_ops)
    got = linalg.lsqr(A, y, damp=0.5, atol=1e-12, btol=1e-12, calc_var=True)
    ref = spla.lsqr(S, y, damp=0.5, atol=1e-12, btol=1e-12, calc_var=True)
    assert np.allclose(got[0], ref[0], atol=1e-8)
    assert np.isclose(got[3], ref[3], rtol=1e-6) and np.isclose(got[4], ref[4], rtol=1e-6)   # r1norm, r2norm
    # var = sum of the squared search directions: sensitive to the loss of orthogonality, compare on a short run
    got6 = linalg.lsqr(A, y, damp=0.5, atol=1e-6, btol=1e-6, calc_var=True)
    ref6 = spla.lsqr(S, y, damp=0.5, atol=1e-6, btol=1e-6, calc_var=True)
    assert got6[2] == ref6[2] and np.allclose(got6[9], ref6[9], rtol=1e-2)
    assert not linalg.lsqr(A, y, damp=0.5)[9].any()                                            # calc_var off -> zeros
    x0 = ref[0] + 1e-3
    got = linalg.lsqr(A, y, atol=1e-12, btol=1e-12, x0=x0)
    ref = spla.lsqr(S, y, atol=1e-12, btol=1e-12, x0=x0)
    assert np.allclose(got[0], ref[0], atol=1e-8)
    # b = 0: immediate return with x = 0
    got = linalg.lsqr(A, np.zeros(120))
    assert got[1] == 0 and got[2] == 0 and not got[0].any()


def test_eigsh_eigenpairs(cpu_ops):
    from legate.sparse_b200 import linalg

    S, _ = sample(100, 100, 0.1, 471014)
    Sd = np.asarray(S.todense())
    Sym = sp.csr_array(0.5 * (Sd + Sd.T))
    A = _operator(Sym, cpu_ops)
    np.random.seed(0)
    w, V = linalg.eigsh(A)
    assert w.shape == (6,) and V.shape == (100, 6) and np.all(np.diff(w) >= 0)
    for i, lam in enumerate(w):
        assert np.allclose(Sym @ V[:, i], lam * V[:, i], atol=1e-3)      # the reference test's bar (test_eigsh.py:37)
    exact = np.linalg.eigvalsh(Sym.toarray())
    want = np.sort(exact[np.argsort(np.abs(exact))[-6:]])
    assert np.allclose(w, want, atol=1e-8)
    wa = linalg.eigsh(A, k=3, which="LA", return_eigenvectors=False)
    assert np.allclose(wa, exact[-3:], atol=1e-8)
    # a small ncv forces thick restarts
    wr, Vr = linalg.eigsh(A, k=4, ncv=10, tol=1e-10)
    assert np.allclose(wr, np.sort(exact[np.argsort(np.abs(exact))[-4:]]), atol=1e-7)
    assert np.allclose(Vr.T @ Vr, np.eye(4), atol=1e-7)
    for bad in (dict(k=0), dict(k=100), dict(which="SM")):
        with pytest.raises(ValueError):
            linalg.eigsh(A, **bad)


def test_eigsh_and_gmres_keep_their_basis_orthogonal(cpu_ops):
    """10 I + E: ||A v|| is ~7x the new Lanczos direction, so ONE Gram-Schmidt pass (the reference's and CuPy's
    recurrence) loses a digit of orthogonality per step and returns Ritz values in the hundreds after ~18 steps;
    the projection is applied twice here."""
    from legate.sparse_b200 import linalg

    rng = np.random.default_rng(33)
    n = 240
    S = sp.csr_array(sp.random(n, n, density=0.05, random_state=rng, format="csr", dtype=np.float64) + 10.0 * sp.eye(n))
    Sym = sp.csr_array(0.5 * (S + S.T))
    exact = np.linalg.eigvalsh(Sym.toarray())
    np.random.seed(5)
    w, V = linalg.eigsh(_operator(Sym, cpu_ops), k=4, tol=1e-10)
    assert np.allclose(w, np.sort(exact[np.argsort(np.abs(exact))[-4:]]), atol=1e-8)
    assert np.allclose(V.T @ V, np.eye(4), atol=1e-8)
    xs = rng.standard_normal(n)
    got, info = linalg.gmres(_operator(S, cpu_ops), S @ xs, tol=1e-12, restart=60)
    assert info == 0 and np.allclose(got, xs, atol=1e-9)
