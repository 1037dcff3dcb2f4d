"""Pins the QP half of the oracle (the reference's OWN vendored OSQP C code in oracle/_ref + the restated QDLDL 0.1.6)
against every known-answer vector the reference's tests hold at this boundary (SURVEY.md §8(c)):

  3rd/osqp/tests/basic_qp/generate_problem.py:21-24, basic_lp :21-24, basic_qp2 :21-30, unconstrained :12-14,
  primal_infeasibility (status), solve_linsys/generate_problem.py:9-31 (KKT solve vs SciPy splu, PCG64(1)),
  3rd/osqp-eigen/tests/QPTest.cpp:12-92.            Tolerance: the reference's TESTS_TOL = 1e-4 (tests/osqp_tester.h:13).

oracle/_ref is built where the reference's sources exist; elsewhere the recorded results of that build answer (tests/ref_record.py).
"""
import numpy as np
import pytest
from scipy import sparse
import scipy.sparse.linalg as spla

import oracle_lib

TOL = 1e-4
INF = 1e30  # OSQP_INFTY


def solve(P, q, A, l, u, **kw):
    st = oracle_lib.osqp_settings(eps_prim_inf=1e-4, max_iter=4000, eps_abs=1e-5, eps_rel=1e-5, **kw)
    l = np.clip(np.asarray(l, float), -INF, INF)
    u = np.clip(np.asarray(u, float), -INF, INF)
    return oracle_lib.osqp_solve(sparse.csc_matrix(P), q, sparse.csc_matrix(A), l, u, st)


def test_basic_qp():
    P = sparse.csc_matrix(np.triu([[4., 1.], [1., 2.]]))
    A = np.array([[1., 1.], [1., 0.], [0., 1.], [0., 1.]])
    x, y, info = solve(P, np.ones(2), A, [1., 0., 0., -np.inf], [1., 0.7, 0.7, np.inf])
    assert info["status_val"] == 1
    assert np.allclose(x, [0.3, 0.7], atol=TOL)
    assert np.allclose(y, [-2.9, 0.0, 0.2, 0.0], atol=TOL * 10)
    assert abs(info["obj_val"] - 1.88) < TOL * 10


def test_basic_lp():
    P = sparse.csc_matrix((2, 2))
    A = np.array([[1., 1.], [1., 0.], [0., 1.], [0., 1.]])
    x, y, info = solve(P, [1.1, 0.95], A, [1., 0., 0., -np.inf], [1., 0.7, 0.7, np.inf])
    assert info["status_val"] == 1
    assert np.allclose(x, [0.3, 0.7], atol=TOL)
    assert abs(info["obj_val"] - 0.995) < TOL * 10


def test_basic_qp2_and_update():
    P = sparse.csc_matrix(np.triu([[11., 0.], [0., 0.]]))
    A = np.array([[-1., 0.], [0., -1.], [-1., 3.], [2., 5.], [3., 4.]])
    l = -np.inf * np.ones(5)
    x, y, info = solve(P, [3., 4.], A, l, [0., 0., -15., 100., 80.])
    assert info["status_val"] == 1
    assert np.allclose(x, [15., 0.], atol=1e-3)
    assert np.allclose(y, [0., 508., 168., 0., 0.], atol=1e-1)
    assert abs(info["obj_val"] - 1282.5) < TOL * 1282.5  # relative, like the reference tester
    x, y, info = solve(P, [1., 1.], A, l, [-2., 0., -20., 100., 80.])
    assert np.allclose(x, [20., 0.], atol=1e-3)
    assert abs(info["obj_val"] - 2220.0) < TOL * 2220.0


def test_unconstrained():
    P = sparse.diags([0.617022, 0.92032449, 0.20011437, 0.50233257, 0.34675589], format="csc")
    q = np.array([-1.10593508, -1.65451545, -2.3634686, 1.13534535, -1.01701414])
    x, y, info = solve(P, q, sparse.csc_matrix((0, 5)), [], [])
    assert info["status_val"] == 1
    assert np.allclose(x, [1.79237542, 1.79775228, 11.81058885, -2.26014678, 2.93293975], atol=TOL * 10)
    assert abs(info["obj_val"] - (-19.209752026813277)) < 1e-3


def test_osqp_eigen_qptest():
    # QPTest.cpp "QPProblem - Unconstrained": alpha = 1.0
    x, _, info = solve(sparse.csc_matrix(np.triu([[3., 2.], [2., 4.]])), [3., 1.], sparse.csc_matrix((0, 2)), [], [],
                       alpha=1.0)
    assert np.allclose(x, [-1.25, 0.375], atol=TOL)
    # QPTest.cpp "QPProblem"
    A = np.array([[1., 1.], [1., 0.], [0., 1.]])
    x, _, info = solve(sparse.csc_matrix(np.triu([[4., 1.], [1., 2.]])), [1., 1.], A, [1., 0., 0.], [1., 0.7, 0.7])
    assert np.allclose(x, [0.3, 0.7], atol=TOL)


def test_primal_infeasible_status():
    # x >= 1 and x <= 0 cannot both hold: OSQP_PRIMAL_INFEASIBLE (status_val 3)
    A = np.array([[1.], [1.]])
    x, _, info = solve(sparse.csc_matrix([[1.0]]), [0.0], A, [1., -np.inf], [np.inf, 0.])
    assert info["status_val"] == 3


def test_kkt_solve_vs_scipy_splu():
    # 3rd/osqp/tests/solve_linsys/generate_problem.py:9-31 — same generator, same seed
    from numpy.random import Generator, PCG64
    rg = Generator(PCG64(1))
    n, m = 3, 4
    P = sparse.random(n, n, density=0.4, format="csc", random_state=rg)
    P = (P @ P.T).tocsc()
    A = sparse.random(m, n, density=0.4, format="csc", random_state=rg)
    Pu = sparse.triu(P, format="csc")
    rho, sigma = 4.0, 1.0
    KKT = sparse.bmat([[P + sigma * sparse.eye(n), A.T], [A, -1. / rho * sparse.eye(m)]], format="csc")
    rhs = rg.standard_normal(m + n)
    x = spla.splu(KKT).solve(rhs)
    x[n:] = rhs[n:] + x[n:] / rho  # the z-tilde fix-up of qdldl_interface.c:447-450
    sol = oracle_lib.kkt_solve(Pu, A, sigma, rho, rhs)
    assert np.allclose(sol, x, atol=TOL)


@pytest.mark.parametrize("n,m,seed", [(6, 4, 0), (24, 18, 1), (64, 43, 2)])
def test_restated_qdldl_on_random_quasidefinite(n, m, seed):
    """The restated QDLDL (oracle/qdldl/qdldl.c; source un-vendored, SURVEY.md §9.4) against a dense solve."""
    rng = np.random.default_rng(seed)
    M = sparse.random(n, n, density=0.3, random_state=rng, format="csc")
    P = (M @ M.T + 0.1 * sparse.eye(n)).tocsc()
    A = sparse.random(m, n, density=0.3, random_state=rng, format="csc")
    rho, sigma = 0.7, 1e-6
    K = np.block([[P.toarray() + sigma * np.eye(n), A.toarray().T], [A.toarray(), -np.eye(m) / rho]])
    rhs = rng.standard_normal(n + m)
    x = np.linalg.solve(K, rhs)
    x[n:] = rhs[n:] + x[n:] / rho
    sol = oracle_lib.kkt_solve(sparse.triu(P, format="csc"), A, sigma, rho, rhs)
    assert np.allclose(sol, x, rtol=1e-7, atol=1e-7)
