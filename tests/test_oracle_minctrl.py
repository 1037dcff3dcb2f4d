"""Pins the restated MinimumControl assembly (oracle/minctrl_ref.cpp) against the literal numbers in the reference
source and against the committed golden vectors (tests/golden/minctrl_golden.json, made by tests/golden/make_golden.py
with the reference's own OSQP)."""
import hashlib
import json
import os

import numpy as np
import pytest
from scipy import sparse

import oracle_lib

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "minctrl_golden.json")))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def dense(asm):
    n, m = asm["n"], asm["m"]
    P = sparse.csc_matrix((asm["Px"], asm["Pi"], asm["Pp"]), shape=(n, n)).toarray()
    A = sparse.csc_matrix((asm["Ax"], asm["Ai"], asm["Ap"]), shape=(m, n)).toarray()
    return P, A


def test_hessian_block_is_minimum_control_cpp_5_19():
    T = np.array([1.0, 0.7, 1.9])
    asm = oracle_lib.minctrl_assemble(5, 3, [1, 2, 3, 4], [0, 0], [0, 0], T)
    P, _ = dense(asm)
    for i, t in enumerate(T):
        blk = np.array([[36 * t, 72 * t**2, 120 * t**3], [72 * t**2, 192 * t**3, 360 * t**4],
                        [120 * t**3, 360 * t**4, 720 * t**5]])
        got = P[6 * i + 3:6 * i + 6, 6 * i + 3:6 * i + 6]
        assert np.allclose(np.triu(got), np.triu(blk), rtol=1e-14)       # OsqpEigen keeps the upper triangle (Data.tpp:42)
        assert np.all(np.tril(got, -1) == 0)
        assert np.all(P[6 * i:6 * i + 3, :] == 0)
    assert len(asm["Px"]) == 6 * 3


@pytest.mark.parametrize("S", [1, 2, 3, 4, 8])
def test_constraint_rows_min_jerk(S):
    rng = np.random.default_rng(S)
    T = rng.uniform(0.5, 2.0, S)
    pos = rng.normal(size=S + 1)
    bv, ba = rng.normal(size=2), rng.normal(size=2)
    asm = oracle_lib.minctrl_assemble(5, S, pos, bv, ba, T)
    _, A = dense(asm)
    n, m = 6 * S, 4 * S + 2
    assert (asm["n"], asm["m"]) == (n, m)
    assert len(asm["Ax"]) == 30 * S - 9          # explicit zeros are stored (minimum_control.cpp:55-91, SURVEY §8 b2)
    assert np.array_equal(asm["l"], asm["u"])    # equality constraints only (:98-125)
    # any polynomial set that satisfies A c = l interpolates the waypoints and is C2 at the knots
    c, *_ = np.linalg.lstsq(A, asm["l"], rcond=None)
    c = c.reshape(S, 6)
    ev = lambda i, t, d: sum(np.prod(np.arange(j, j - d, -1)) * c[i, j] * t ** (j - d) for j in range(d, 6))
    assert abs(ev(0, 0.0, 0) - pos[0]) < 1e-8 and abs(ev(0, 0.0, 1) - bv[0]) < 1e-8 and abs(ev(0, 0.0, 2) - ba[0]) < 1e-8
    assert abs(ev(S - 1, T[-1], 0) - pos[S]) < 1e-7 and abs(ev(S - 1, T[-1], 1) - bv[1]) < 1e-7
    assert abs(ev(S - 1, T[-1], 2) - ba[1]) < 1e-7
    for i in range(S - 1):
        assert abs(ev(i, T[i], 0) - pos[i + 1]) < 1e-7
        for d in range(3):
            assert abs(ev(i, T[i], d) - ev(i + 1, 0.0, d)) < 1e-7


@pytest.mark.parametrize("S", [2, 8, 16])
def test_snap_extension_dimensions(S):
    asm = oracle_lib.minctrl_assemble(7, S, np.arange(S + 1.0), [0, 0], [0, 0], np.ones(S), bound_jerk=[0, 0])
    assert (asm["n"], asm["m"]) == (8 * S, 5 * S + 3)   # SURVEY.md §9.3
    P, A = dense(asm)
    # 4x4 snap block, first entry (4!)^2 T
    assert P[4, 4] == 576.0
    assert np.linalg.matrix_rank(A) == asm["m"]


@pytest.mark.parametrize("case", GOLD, ids=lambda c: f"order{c['order']}_S{c['S']}")
def test_golden_coefficients(case):
    st = oracle_lib.osqp_settings(**case["settings"])
    for p in case["problems"]:
        asm = oracle_lib.minctrl_assemble(case["order"], case["S"], p["pos"], p["bound_vel"], p["bound_acc"], p["T"],
                                          bound_jerk=p["bound_jerk"])
        assert sha(asm["Px"]) == p["P_sha256"] and sha(asm["Ax"]) == p["A_sha256"]
        ok, coef, info = oracle_lib.minctrl_solve(case["order"], case["S"], p["pos"], p["bound_vel"], p["bound_acc"],
                                                  p["T"], bound_jerk=p["bound_jerk"], settings=st, like=np.array(p["coef"]))
        assert (ok, info["status_val"], info["iter"], info["rho_updates"]) == (p["solved"], p["status_val"], p["iter"],
                                                                               p["rho_updates"])
        assert np.array_equal(coef, np.array(p["coef"]))   # same machine code, same inputs: bit-identical


def test_qpsolve_fixture_is_a_min_jerk_trajectory():
    # test_qpsolve.cpp:10-18 — inputs only (the reference records no outputs); check optimality conditions instead
    ok, coef, info = oracle_lib.minctrl_solve(5, 3, [1, 2, 3, 4], [0, 0], [0, 0], [1, 1, 1])
    assert ok == 1 and info["iter"] % 25 == 0   # termination is only tested every 25 iterations (osqp_api.c:560)
    asm = oracle_lib.minctrl_assemble(5, 3, [1, 2, 3, 4], [0, 0], [0, 0], [1, 1, 1])
    P, A = dense(asm)
    P = P + np.triu(P, 1).T
    assert np.abs(A @ coef - asm["l"]).max() < 5e-3
    # exact KKT solution of the equality-constrained QP
    K = np.block([[P, A.T], [A, np.zeros((asm["m"],) * 2)]])
    sol = np.linalg.lstsq(K, np.concatenate([np.zeros(asm["n"]), asm["l"]]), rcond=None)[0][:asm["n"]]
    assert np.abs(sol - coef).max() < 5e-2
    # symmetry of the problem: p(t) - 2.5 is odd about the midpoint t = 1.5
    t = np.linspace(0, 1, 11)
    seg = lambda i, tt: sum(coef[6 * i + j] * tt ** j for j in range(6))
    assert np.allclose(seg(0, t) - 2.5, -(seg(2, 1 - t) - 2.5), atol=5e-3)


def test_libm_mode_only_changes_rounding():
    T = np.array([0.73, 1.31, 1.9, 0.55])
    a = oracle_lib.minctrl_assemble(5, 4, np.arange(5.0), [0, 0], [0, 0], T, libm_mode=0)
    b = oracle_lib.minctrl_assemble(5, 4, np.arange(5.0), [0, 0], [0, 0], T, libm_mode=1)
    assert np.allclose(a["Px"], b["Px"], rtol=4e-16) and np.allclose(a["Ax"], b["Ax"], rtol=4e-16)
