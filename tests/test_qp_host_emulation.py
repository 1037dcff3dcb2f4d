"""CPU test of the product's QP kernel BODY: uav_motion_planning_b200/csrc/qp_body.h is compiled for the host by
tests/host/qp_host.cpp (identical statements to the device instantiation, workspace poisoned with NaN) and compared with
the committed golden vectors and with the reference's own OSQP (or its recorded results, tests/ref_record.py).  This covers the host logic
(qp_symbolic.cpp: pattern, ordering, etree, reach lists) and the OSQP restatement without a GPU; the GPU run of the same
source is checked by tests/test_qp_parity.py (-m gpu)."""
import json
import os

import numpy as np
import pytest

import host_qp
import oracle_lib
from uav_motion_planning_b200.minimum_control import default_settings

RTOL = 1e-5
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "minctrl_golden.json")))


@pytest.mark.parametrize("case", GOLD, ids=lambda c: f"order{c['order']}_S{c['S']}")
def test_against_golden(case):
    pr = case["problems"]
    arr = lambda k: np.array([p[k] for p in pr])
    got = host_qp.solve_batch(case["order"], arr("pos"), arr("bound_vel"), arr("bound_acc"), arr("T"), arr("bound_jerk"),
                              settings=default_settings(**case["settings"]))
    for b, p in enumerate(pr):
        assert (got["solved"][b], got["status"][b], got["iters"][b]) == (p["solved"], p["status_val"], p["iter"])
        ref = np.array(p["coef"])
        assert np.abs(ref - got["coef"][b]).max() / np.abs(ref).max() < RTOL
        # with the tabulated AMD order the restated OSQP follows the reference operation for operation
        assert np.array_equal(ref, got["coef"][b])


@pytest.mark.parametrize("order,S,eps", [(5, 1, 1e-3), (5, 2, 1e-3), (5, 6, 1e-4), (7, 2, 1e-3), (7, 16, 1e-4),
                                         (7, 16, 1e-6)])
def test_against_reference_osqp(order, S, eps):
    rng = np.random.default_rng(order * 100 + S)
    B = 6
    pos = np.cumsum(rng.normal(size=(B, S + 1)), axis=1)
    bv, ba, bj = rng.normal(size=(B, 2)) * 0.5, rng.normal(size=(B, 2)) * 0.2, np.zeros((B, 2))
    T = rng.uniform(0.5, 2.0, size=(B, S))
    kw = dict(eps_abs=eps, eps_rel=eps, max_iter=4000)
    got = host_qp.solve_batch(order, pos, bv, ba, T, bj, settings=default_settings(**kw))
    for b in range(B):
        ok, coef, info = oracle_lib.minctrl_solve(order, S, pos[b], bv[b], ba[b], T[b], bound_jerk=bj[b],
                                                  settings=oracle_lib.osqp_settings(**kw), like=got["coef"][b])
        assert (ok, info["status_val"], info["iter"]) == (got["solved"][b], got["status"][b], got["iters"][b])
        assert np.abs(coef - got["coef"][b]).max() / np.abs(coef).max() < RTOL
        assert np.array_equal(coef, got["coef"][b])


def test_fallback_ordering_outside_the_table():
    """Order 7, S = 41 is not tabulated: the plan falls back to its own minimum-degree order; agreement is then to rounding."""
    S, rng = 41, np.random.default_rng(41)
    pos = np.cumsum(rng.normal(size=(2, S + 1)), axis=1)
    z = np.zeros((2, 2))
    got = host_qp.solve_batch(7, pos, z, z, np.ones((2, S)), bj=z)
    for b in range(2):
        ok, coef, info = oracle_lib.minctrl_solve(7, S, pos[b], z[b], z[b], np.ones(S), bound_jerk=z[b], like=got["coef"][b])
        assert ok == got["solved"][b]
        assert np.abs(coef - got["coef"][b]).max() / np.abs(coef).max() < 1e-4


@pytest.mark.parametrize("S", [41, 56, 64, 80])
def test_long_minimum_jerk_chains_like_the_rrt_star_front_end(S):
    """The reference's own flow makes every RRT* optimal-path point a waypoint (test_minimum_jerk.cpp:44-71): 20 - 70 segments of order 5.
    AMD orders are tabulated up to S = 80 for order 5, so thread body, warp body (both loop orders) and the reference's OSQP agree bit
    for bit there too, adaptive-rho updates included."""
    rng = np.random.default_rng(S)
    B = 2
    pos = np.cumsum(rng.normal(0, 0.5, (B, S + 1)), axis=1)
    bv = np.zeros((B, 2)); bv[:, 0] = rng.normal(0, 1, B)
    ba = np.zeros((B, 2))
    T = np.ones((B, S)) if S != 64 else rng.uniform(0.5, 2.0, (B, S))
    r = host_qp.solve_batch(5, pos, bv, ba, T)
    rw = host_qp.solve_batch_warp(5, pos, bv, ba, T)
    rr = host_qp.solve_batch_warp(5, pos, bv, ba, T, reversed_loops=True)
    assert np.array_equal(r["coef"].view(np.uint64), rw["coef"].view(np.uint64)) and np.array_equal(rw["coef"].view(np.uint64), rr["coef"].view(np.uint64))
    for b in range(B):
        ok, coef, info = oracle_lib.minctrl_solve(5, S, pos[b], bv[b], ba[b], T[b], like=r["coef"][b])
        assert ok == r["solved"][b] and info["iter"] == r["iters"][b] == rw["iters"][b]
        assert np.array_equal(coef.view(np.uint64), r["coef"][b].view(np.uint64))


def test_max_iter_status():
    # max_iter below the first termination check: OSQP reports MAX_ITER_REACHED (7) or SOLVED_INACCURATE (2); solve() -> false
    pos = np.array([[0.0, 1.0, -1.0, 2.0]])
    z = np.zeros((1, 2))
    got = host_qp.solve_batch(5, pos, z, z, np.ones((1, 3)), settings=default_settings(max_iter=10))
    assert got["solved"][0] == 0 and got["status"][0] in (2, 7) and got["iters"][0] == 10
    ok, coef, info = oracle_lib.minctrl_solve(5, 3, pos[0], z[0], z[0], np.ones(3), settings=oracle_lib.osqp_settings(max_iter=10),
                                              like=got["coef"][0])
    assert (ok, info["status_val"], info["iter"]) == (0, got["status"][0], 10)
    assert np.abs(coef - got["coef"][0]).max() / np.abs(coef).max() < RTOL


@pytest.mark.parametrize("case", GOLD, ids=lambda c: f"warp_order{c['order']}_S{c['S']}")
def test_warp_body_against_golden_in_both_loop_orders(case):
    """qp_body_warp.h (one warp per problem on the GPU) run as a single lane, with every parallel loop executed forwards and then
    BACKWARDS: both must reproduce the reference OSQP bit for bit, so no parallel loop depends on its iteration order."""
    pr = case["problems"]
    arr = lambda k: np.array([p[k] for p in pr])
    for rev in (False, True):
        got = host_qp.solve_batch_warp(case["order"], arr("pos"), arr("bound_vel"), arr("bound_acc"), arr("T"), arr("bound_jerk"),
                                       settings=default_settings(**case["settings"]), reversed_loops=rev)
        for b, p in enumerate(pr):
            assert (got["solved"][b], got["status"][b], got["iters"][b]) == (p["solved"], p["status_val"], p["iter"])
            assert np.array_equal(np.array(p["coef"]), got["coef"][b])


def test_warp_body_equals_thread_body_on_random_problems():
    rng = np.random.default_rng(77)
    for order, S in [(5, 1), (5, 6), (7, 2), (7, 12)]:
        B = 5
        pos = np.cumsum(rng.normal(size=(B, S + 1)), axis=1)
        bv, ba, bj = rng.normal(size=(B, 2)) * 0.5, rng.normal(size=(B, 2)) * 0.2, np.zeros((B, 2))
        T = rng.uniform(0.5, 2.0, size=(B, S))
        a = host_qp.solve_batch(order, pos, bv, ba, T, bj)
        for rev in (False, True):
            w = host_qp.solve_batch_warp(order, pos, bv, ba, T, bj, reversed_loops=rev)
            assert np.array_equal(a["coef"], w["coef"]) and np.array_equal(a["iters"], w["iters"]) and np.array_equal(a["status"], w["status"])
    # max_iter below the first check and the fallback ordering (order 7, S = 41 is not tabulated)
    pos = np.cumsum(rng.normal(size=(2, 42)), axis=1)
    z = np.zeros((2, 2))
    a = host_qp.solve_batch(7, pos, z, z, np.ones((2, 41)), z, settings=default_settings(max_iter=10))
    w = host_qp.solve_batch_warp(7, pos, z, z, np.ones((2, 41)), z, settings=default_settings(max_iter=10), reversed_loops=True)
    assert np.array_equal(a["coef"], w["coef"]) and np.array_equal(a["status"], w["status"])


def corridor_problems(order, S, B, seed, margin=0.05):
    rng = np.random.default_rng(seed)
    pos = np.cumsum(rng.normal(size=(B, S + 1)), axis=1)
    bv, ba, bj = rng.normal(size=(B, 2)) * 0.2, np.zeros((B, 2)), np.zeros((B, 2))
    T = rng.uniform(0.5, 2.0, size=(B, S))
    lo = np.minimum(pos[:, :-1], pos[:, 1:]) - margin
    hi = np.maximum(pos[:, :-1], pos[:, 1:]) + margin
    return pos, bv, ba, bj, T, lo, hi


@pytest.mark.parametrize("order,S,Kc,eps", [(7, 12, 2, 1e-3), (7, 8, 3, 1e-5), (5, 4, 1, 1e-3), (5, 6, 2, 1e-4), (7, 16, 4, 1e-3)])
def test_corridor_rows_against_reference_osqp(order, S, Kc, eps):
    """Corridor (inequality) rows — the SURVEY.md §9.3 extension — through the reference's own OSQP: rho = 0.1 on those rows
    (1e3 x on the equality rows, auxil.c:75-104), the z-projection of update_z (auxil.c:188-203) clips, adaptive rho refactors.
    Same status, same iteration count, coefficients bit-identical (tabulated AMD order of the corridor pattern) for the
    thread body and for the warp body in both loop orders."""
    B = 6
    pos, bv, ba, bj, T, lo, hi = corridor_problems(order, S, B, seed=order * 1000 + S * 10 + Kc)
    kw = dict(eps_abs=eps, eps_rel=eps)
    st = default_settings(**kw)
    got = host_qp.solve_batch(order, pos, bv, ba, T, bj, settings=st, lo=lo, hi=hi, n_corridor=Kc)
    gw = host_qp.solve_batch_warp(order, pos, bv, ba, T, bj, settings=st, lo=lo, hi=hi, n_corridor=Kc)
    gr = host_qp.solve_batch_warp(order, pos, bv, ba, T, bj, settings=st, lo=lo, hi=hi, n_corridor=Kc, reversed_loops=True)
    free = host_qp.solve_batch(order, pos, bv, ba, T, bj, settings=st)
    n_rho, n_active = 0, 0
    for b in range(B):
        ok, coef, info = oracle_lib.minctrl_solve(order, S, pos[b], bv[b], ba[b], T[b], bound_jerk=bj[b],
                                                  settings=oracle_lib.osqp_settings(**kw), corridor_lo=lo[b], corridor_hi=hi[b],
                                                  n_corridor=Kc, like=got["coef"][b])
        for g in (got, gw, gr):
            assert (ok, info["status_val"], info["iter"]) == (g["solved"][b], g["status"][b], g["iters"][b])
        n_rho += info["rho_updates"] > 0
        if ok:
            assert np.abs(coef - got["coef"][b]).max() / np.abs(coef).max() < RTOL
            for g in (got, gw, gr):
                assert np.array_equal(coef, g["coef"][b])
            n_active += np.abs(coef - free["coef"][b]).max() > 1e-6   # the box changed the trajectory: rows are active
    assert n_rho > 0 and n_active > 0


def test_corridor_row_values_and_feasibility():
    """The solved polynomial respects its boxes at the sample times (to the ADMM tolerance) and lo > hi is refused upstream."""
    order, S, Kc = 7, 6, 3
    pos, bv, ba, bj, T, lo, hi = corridor_problems(order, S, 4, seed=3, margin=0.1)
    got = host_qp.solve_batch(order, pos, bv, ba, T, bj, settings=default_settings(eps_abs=1e-6, eps_rel=1e-6, max_iter=4000),
                              lo=lo, hi=hi, n_corridor=Kc)
    nc = order + 1
    for b in range(4):
        if not got["solved"][b]:
            continue
        for s in range(S):
            c = got["coef"][b][nc * s: nc * (s + 1)]
            for j in range(Kc):
                t = (j + 1) / (Kc + 1) * T[b, s]
                p = np.polyval(c[::-1], t)
                assert lo[b, s] - 1e-3 <= p <= hi[b, s] + 1e-3
