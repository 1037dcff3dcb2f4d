"""GPU parity: batched CUDA MinimumControl::solve vs the reference's own OSQP (oracle/_ref, or its recorded results) on the same inputs.

Gate (BASELINE.json north_star): segment coefficients within 1e-5 relative of the OSQP solution at the same ADMM
tolerance; we also require identical OSQP status and iteration count for every problem.
"""
import numpy as np
import pytest

import oracle_lib
import uav_motion_planning_b200 as u
from uav_motion_planning_b200.minimum_control import MinimumControl, default_settings

pytestmark = pytest.mark.gpu
RTOL = 1e-5


def make_problems(B, S, seed, unit_time=True):
    rng = np.random.default_rng(seed)
    pos = np.cumsum(rng.normal(size=(B, S + 1)), axis=1)
    bv = rng.normal(size=(B, 2)) * 0.5
    ba = rng.normal(size=(B, 2)) * 0.2
    bj = np.zeros((B, 2))
    T = np.ones((B, S)) if unit_time else rng.uniform(0.5, 2.0, size=(B, S))
    return pos, bv, ba, bj, T


def compare(ctx, order, S, B, seed, unit_time=True, **st_kw):
    pos, bv, ba, bj, T = make_problems(B, S, seed, unit_time)
    mc = MinimumControl(ctx, order=order)
    got = mc.solve_batch(pos, bv, ba, T, bound_jerk=bj, settings=default_settings(**st_kw))
    worst = 0.0
    for b in range(B):
        ok, coef, info = oracle_lib.minctrl_solve(order, S, pos[b], bv[b], ba[b], T[b], bound_jerk=bj[b],
                                                  settings=oracle_lib.osqp_settings(**st_kw), like=got["coef"][b])
        assert info["status_val"] == got["status"][b], (b, info, got["status"][b], got["iters"][b])
        assert info["iter"] == got["iters"][b], (b, info, got["iters"][b])
        assert ok == got["solved"][b]
        if ok:
            scale = np.abs(coef).max()
            err = np.abs(coef - got["coef"][b]).max() / scale
            worst = max(worst, err)
            assert err < RTOL, (b, err)
            if S <= 40:  # tabulated AMD order: bit-identical to the reference's OSQP
                assert np.array_equal(coef, got["coef"][b]), (b, err)
    return worst


def test_reference_fixture_qpsolve(gpu_ctx):
    # src/planner/test/src/test_qpsolve.cpp:10-18: waypoints 1,2,3,4, v = a = 0, T = 1,1,1
    mc = MinimumControl(gpu_ctx, order=5)
    assert mc.solve(np.array([1.0, 2.0, 3.0, 4.0]), np.zeros(2), np.zeros(2), np.ones(3))
    ok, coef, info = oracle_lib.minctrl_solve(5, 3, [1, 2, 3, 4], [0, 0], [0, 0], [1, 1, 1], like=mc.getCoef1d())
    assert ok == 1 and mc.last["iters"][0] == info["iter"]
    assert np.abs(mc.getCoef1d() - coef).max() / np.abs(coef).max() < RTOL


@pytest.mark.parametrize("S", [1, 2, 4, 8])
def test_min_jerk(gpu_ctx, S):
    compare(gpu_ctx, 5, S, 64, seed=S)


@pytest.mark.parametrize("S", [2, 8, 12, 16])
def test_min_snap_extension(gpu_ctx, S):
    compare(gpu_ctx, 7, S, 48, seed=100 + S)


def test_nonuniform_times(gpu_ctx):
    compare(gpu_ctx, 5, 4, 64, seed=7, unit_time=False)
    compare(gpu_ctx, 7, 8, 64, seed=8, unit_time=False)


@pytest.mark.parametrize("eps", [1e-3, 1e-4, 1e-5, 1e-6])
def test_eps_sweep_config5(gpu_ctx, eps):
    # BASELINE.json configs[4] in miniature: 16-segment snap, eps_abs = eps_rel swept, adaptive rho active
    compare(gpu_ctx, 7, 16, 24, seed=int(-np.log10(eps)), unit_time=False, eps_abs=eps, eps_rel=eps, max_iter=4000)


def test_ragged_batch_sizes(gpu_ctx):
    for B in (1, 31, 33, 257):
        compare(gpu_ctx, 5, 3, B, seed=B)


def test_both_kernels_agree_bitwise(gpu_ctx, monkeypatch):
    """The warp-per-problem kernel (default for small batches / the pipeline) and the thread-per-problem kernel (large batches)
    are two schedules of the same arithmetic: identical bits, both identical to the reference OSQP."""
    pos, bv, ba, bj, T = make_problems(96, 8, 5, unit_time=False)
    mc = MinimumControl(gpu_ctx, order=7)
    monkeypatch.setenv("UAVMP_QP_THREAD", "1")
    a = {k: v.copy() for k, v in mc.solve_batch(pos, bv, ba, T, bound_jerk=bj).items()}
    monkeypatch.delenv("UAVMP_QP_THREAD")
    monkeypatch.setenv("UAVMP_QP_WARP", "1")
    b = mc.solve_batch(pos, bv, ba, T, bound_jerk=bj)
    for k in ("coef", "iters", "status", "solved"):
        assert np.array_equal(a[k], b[k]), k
    ok, coef, info = oracle_lib.minctrl_solve(7, 8, pos[0], bv[0], ba[0], T[0], bound_jerk=bj[0], like=b["coef"][0])
    assert np.array_equal(coef, b["coef"][0]) and info["iter"] == b["iters"][0]


@pytest.mark.parametrize("order,S,Kc,eps", [(7, 12, 2, 1e-3), (7, 8, 3, 1e-5), (5, 4, 1, 1e-3), (7, 16, 4, 1e-4)])
def test_corridor_rows(gpu_ctx, monkeypatch, order, S, Kc, eps):
    """Corridor (inequality) rows, the §9.3 extension of configs[3]: ACTIVE z-projection (auxil.c:188-203), rho classes
    (auxil.c:75-104) and adaptive-rho refactorisations, on both CUDA kernels, against the reference's own OSQP: identical
    status and iteration count, coefficients within 1e-5 relative (and bit-identical: the corridor patterns' AMD orders are
    tabulated)."""
    from test_qp_host_emulation import corridor_problems
    B = 40
    pos, bv, ba, bj, T, lo, hi = corridor_problems(order, S, B, seed=order * 1000 + S * 10 + Kc)
    kw = dict(eps_abs=eps, eps_rel=eps)
    mc = MinimumControl(gpu_ctx, order=order)
    res = []
    for env in ("UAVMP_QP_THREAD", "UAVMP_QP_WARP"):
        monkeypatch.setenv(env, "1")
        r = mc.solve_batch(pos, bv, ba, T, bound_jerk=bj, settings=default_settings(**kw), corridor_lo=lo, corridor_hi=hi,
                           n_corridor=Kc)
        res.append({k: v.copy() for k, v in r.items()})
        monkeypatch.delenv(env)
    free = mc.solve_batch(pos, bv, ba, T, bound_jerk=bj, settings=default_settings(**kw))
    n_rho = n_active = n_ok = 0
    for b in range(B):
        ok, coef, info = oracle_lib.minctrl_solve(order, S, pos[b], bv[b], ba[b], T[b], bound_jerk=bj[b],
                                                  settings=oracle_lib.osqp_settings(**kw), corridor_lo=lo[b], corridor_hi=hi[b],
                                                  n_corridor=Kc, like=res[0]["coef"][b])
        for g in res:
            assert (ok, info["status_val"], info["iter"]) == (g["solved"][b], g["status"][b], g["iters"][b]), (b, info)
        n_rho += info["rho_updates"] > 0
        if ok:
            n_ok += 1
            for g in res:
                assert np.abs(coef - g["coef"][b]).max() / np.abs(coef).max() < RTOL
                assert np.array_equal(coef, g["coef"][b]), b
            n_active += np.abs(coef - free["coef"][b]).max() > 1e-6
    assert n_ok >= B // 4 and n_rho > 0 and n_active >= B // 8


def test_corridor_argument_checks(gpu_ctx):
    mc = MinimumControl(gpu_ctx, order=7)
    pos, z, T = np.zeros((2, 5)), np.zeros((2, 2)), np.ones((2, 4))
    with pytest.raises(u.UavmpError):  # lo > hi: osqp_setup would refuse the problem (auxil.c:856-921)
        mc.solve_batch(pos, z, z, T, bound_jerk=z, corridor_lo=np.ones((2, 4)), corridor_hi=np.zeros((2, 4)), n_corridor=2)
    with pytest.raises(u.UavmpError):
        mc.solve_batch(pos, z, z, T, bound_jerk=z, corridor_lo=np.zeros((2, 4)), corridor_hi=np.ones((2, 4)), n_corridor=9)
