"""CPU: the schedule of the grouped warp-per-problem QP kernel (uavmp_minctrl_solve_ragged_batch) run on the host
(tests/host/qp_ragged_host.cpp).  One shared-memory arena is reused by chunks of different S, longest first, and poisoned with NaN
between chunks; every problem must come out bit for bit as when it is solved alone.  This is the failure mode the grouped kernel adds
(a plan reading what the previous chunk's plan left in shared memory), caught without a GPU."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CS = os.path.join(ROOT, "uav_motion_planning_b200", "csrc")
SRC = os.path.join(ROOT, "tests", "host", "qp_ragged_host.cpp")


class OsqpSettings(C.Structure):  # include/uavmp.h uavmp_osqp_settings
    _fields_ = [("rho", C.c_double), ("sigma", C.c_double), ("alpha", C.c_double), ("eps_abs", C.c_double),
                ("eps_rel", C.c_double), ("eps_prim_inf", C.c_double), ("eps_dual_inf", C.c_double),
                ("max_iter", C.c_int), ("check_termination", C.c_int), ("scaling", C.c_int),
                ("adaptive_rho", C.c_int), ("adaptive_rho_interval", C.c_int), ("adaptive_rho_tolerance", C.c_double)]


def default_settings(**kw):
    s = OsqpSettings(rho=0.1, sigma=1e-6, alpha=1.6, eps_abs=1e-3, eps_rel=1e-3, eps_prim_inf=1e-3, eps_dual_inf=1e-4, max_iter=1000,
                     check_termination=25, scaling=10, adaptive_rho=1, adaptive_rho_interval=0, adaptive_rho_tolerance=5.0)
    for k, v in kw.items():
        setattr(s, k, v)
    return s


@pytest.fixture(scope="module")
def lib():
    out = os.path.join(tempfile.mkdtemp(prefix="qp_ragged_host_"), "libqp_ragged_host.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared", "-I" + os.path.join(ROOT, "include"),
                    "-I" + CS, "-o", out, SRC, os.path.join(CS, "qp_symbolic.cpp")], check=True)
    return C.CDLL(out)


def problems(order, S_list, seed):
    """ragged batch: random waypoints, non-unit segment times, non-zero boundary velocities"""
    rng = np.random.default_rng(seed)
    S = np.array(S_list, np.int32)
    pos = [np.cumsum(rng.normal(size=s + 1)) for s in S]
    T = [rng.uniform(0.5, 1.8, size=s) for s in S]
    B = len(S)
    bv = rng.normal(size=(B, 2))
    ba = np.zeros((B, 2))
    ba[:, 0] = 0.3 * rng.normal(size=B)
    bj = np.zeros((B, 2)) if order == 7 else None
    return S, pos, T, bv, ba, bj


def p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def solve_grouped(lib, order, S, pos, T, bv, ba, bj, st):
    B = len(S)
    pos_p, T_p = np.ascontiguousarray(np.concatenate(pos)), np.ascontiguousarray(np.concatenate(T))
    coef = np.full(int(S.sum()) * (order + 1), np.nan)
    solved, status, iters = (np.full(B, -7, np.int32) for _ in range(3))
    chunks = lib.host_qp_solve_grouped(order, B, p(S), p(pos_p), p(bv), p(ba), p(bj), p(T_p), C.byref(st), p(coef), p(solved), p(status),
                                       p(iters))
    return chunks, coef, solved, status, iters


def solve_single(lib, order, s, pos, T, bv, ba, bj, st):
    coef = np.full(s * (order + 1), np.nan)
    out = [np.zeros(1, np.int32) for _ in range(3)]
    lib.host_qp_solve_single(order, int(s), p(np.ascontiguousarray(pos)), p(np.ascontiguousarray(bv)), p(np.ascontiguousarray(ba)),
                             p(None if bj is None else np.ascontiguousarray(bj)), p(np.ascontiguousarray(T)), C.byref(st), p(coef), *map(p, out))
    return coef, [int(o[0]) for o in out]


def check_against_single(lib, order, S_list, seed, st):
    S, pos, T, bv, ba, bj = problems(order, S_list, seed)
    chunks, coef, solved, status, iters = solve_grouped(lib, order, S, pos, T, bv, ba, bj, st)
    assert chunks >= len(set(S_list)) > 1, "one arena, reused by chunks of different plans"
    off = 0
    for b, s in enumerate(S):
        n = (order + 1) * s
        ref, (r_solved, r_status, r_iters) = solve_single(lib, order, s, pos[b], T[b], bv[b], ba[b], None if bj is None else bj[b], st)
        got = coef[off:off + n]
        assert np.array_equal(got.view(np.uint64), ref.view(np.uint64)), (order, b, s)
        assert (solved[b], status[b], iters[b]) == (r_solved, r_status, r_iters), (order, b, s)
        off += n
    assert off == coef.size
    return solved


def test_shared_memory_limits_of_the_grouped_kernel(lib):
    """the S ranges the grouped launch takes (DESIGN.md §4): order 5 up to S = 103, order 7 up to S = 70"""
    assert lib.host_qp_chunk_warps(5, 103) >= 1 and lib.host_qp_chunk_warps(5, 104) == 0
    assert lib.host_qp_chunk_warps(7, 70) >= 1 and lib.host_qp_chunk_warps(7, 71) == 0
    assert lib.host_qp_chunk_warps(5, 1) == 16


def test_order5_mixed_plans_in_one_arena(lib):
    # interleaved S, both AMD regimes (tabulated S <= 80, minimum degree beyond), one arena for all of them
    S_list = [7, 1, 41, 2, 20, 3, 81, 7, 1, 64, 2, 20, 3, 7, 1, 2, 3, 80, 1, 2, 3, 7, 20, 41, 1, 2, 3, 1, 2, 3, 1, 2, 3, 1, 2, 3, 1, 2, 3]
    solved = check_against_single(lib, 5, S_list, seed=11, st=default_settings())
    assert solved.mean() > 0.8


def test_order5_largest_group_and_tight_eps(lib):
    check_against_single(lib, 5, [103, 2, 97, 1, 3], seed=12, st=default_settings(eps_abs=1e-6, eps_rel=1e-6, max_iter=4000))


def test_order7_mixed_plans_in_one_arena(lib):
    check_against_single(lib, 7, [8, 1, 40, 1, 8, 2, 1, 70, 2, 1, 8, 1, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1], seed=13,
                         st=default_settings())
