"""GPU: ragged QP batches (uavmp_minctrl_solve_ragged_batch) and the batched RRT* -> minimum-jerk flow of the reference node
(uavmp_rrt_plan_batch, test_minimum_jerk.cpp:40-75).  Every ragged result must be bit-identical to a per-S uavmp_minctrl_solve_batch
call, and the pipeline must reproduce planner.rrt_minimum_jerk_batch (the per-S Python loop) and the reference build's golden vectors."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import uav_motion_planning_b200 as u
from uav_motion_planning_b200 import _lib, planner
from uav_motion_planning_b200.minimum_control import default_settings

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def ragged_problems(order, S_list, seed):
    rng = np.random.default_rng(seed)
    S = np.array(S_list, np.int32)
    pos = [np.cumsum(rng.normal(size=s + 1)) for s in S]
    T = [rng.uniform(0.5, 1.8, size=s) for s in S]
    bv = rng.normal(size=(len(S), 2))
    ba = np.zeros((len(S), 2))
    ba[:, 0] = 0.3 * rng.normal(size=len(S))
    bj = np.zeros((len(S), 2)) if order == 7 else None
    return S, pos, T, bv, ba, bj


def per_s(mc, order, S, pos, T, bv, ba, bj, settings):
    """the baseline: one uavmp_minctrl_solve_batch call per distinct S"""
    out = [None] * len(S)
    for s in sorted(set(S.tolist())):
        idx = np.nonzero(S == s)[0]
        r = mc.solve_batch(np.stack([pos[i] for i in idx]), bv[idx], ba[idx], np.stack([T[i] for i in idx]),
                           bound_jerk=None if bj is None else bj[idx], order=order, settings=settings)
        for k, i in enumerate(idx):
            out[i] = (r["coef"][k], r["solved"][k], r["status"][k], r["iters"][k])
    return out


def check_ragged(ctx, order, S_list, seed, settings=None):
    mc = u.MinimumControl(ctx, order=order)
    st = settings or default_settings()
    S, pos, T, bv, ba, bj = ragged_problems(order, S_list, seed)
    got = mc.solve_batch_ragged(pos, bv, ba, T, bound_jerk=bj, settings=st)
    tm = ctx.timings()
    ref = per_s(mc, order, S, pos, T, bv, ba, bj, st)
    off = got["coef_offsets"]
    for b in range(len(S)):
        c, so, stt, it = ref[b]
        assert np.array_equal(bits(got["coef"][off[b]:off[b + 1]]), bits(c)), (order, b, S[b])
        assert (got["solved"][b], got["status"][b], got["iters"][b]) == (so, stt, it), (order, b, S[b])
    # the packed form gives the same bits
    again = mc.solve_batch_ragged(np.concatenate(pos), bv, ba, np.concatenate(T), S=S, bound_jerk=bj, settings=st)
    assert np.array_equal(bits(again["coef"]), bits(got["coef"])) and np.array_equal(again["iters"], got["iters"])
    return got, tm


ORDER5_S = [1, 2, 3, 7, 20, 41, 64, 80, 81, 97, 103, 104, 130]
ORDER7_S = [1, 8, 40, 70, 71]


def test_ragged_equals_per_s_order5(gpu_ctx):
    """both sides of the shared-memory limit (103 / 104: grouped kernel / thread kernel) and of the AMD table (80 / 81)"""
    S_list = list(np.random.default_rng(1).permutation(np.repeat(ORDER5_S, 3)))
    got, tm = check_ragged(gpu_ctx, 5, S_list, seed=2)
    assert got["solved"].mean() > 0.5
    assert tm["qp_launches"] == 1 + 2  # one grouped launch + one thread-kernel launch each for S = 104, 130


def test_ragged_equals_per_s_order7(gpu_ctx):
    S_list = list(np.random.default_rng(3).permutation(np.repeat(ORDER7_S, 4)))
    _, tm = check_ragged(gpu_ctx, 7, S_list, seed=4)
    assert tm["qp_launches"] == 1 + 1  # S = 71 does not fit


def test_ragged_many_problems_per_group_and_eps_sweep(gpu_ctx):
    S_list = list(np.random.default_rng(5).integers(1, 60, size=400))
    for eps in (1e-3, 1e-6):
        check_ragged(gpu_ctx, 5, S_list, seed=6, settings=default_settings(eps_abs=eps, eps_rel=eps, max_iter=4000))


def test_ragged_single_problem(gpu_ctx):
    for s in (1, 41, 104):
        check_ragged(gpu_ctx, 5, [s], seed=7)


def test_ragged_argument_errors_leave_the_context_usable(gpu_ctx):
    lib, h = gpu_ctx.lib, gpu_ctx.h
    S = np.array([2, 0, 3], np.int32)
    pos, T = np.zeros(int(S.sum()) + 3), np.ones(int(S.sum()))
    b2 = np.zeros((3, 2))
    coef = np.zeros(8 * 5)
    st = default_settings()
    call = lambda order, B, S_, bj: lib.uavmp_minctrl_solve_ragged_batch(h, order, B, _lib.ptr(S_), _lib.ptr(pos), _lib.ptr(b2), _lib.ptr(b2),
                                                                        _lib.ptr(bj), _lib.ptr(T), C.byref(st), _lib.ptr(coef), None, None, None)
    ok_S = np.array([2, 1, 3], np.int32)
    assert call(5, 3, S, None) == -1           # UAVMP_EINVAL: S[1] = 0
    assert call(6, 3, ok_S, None) == -1
    assert call(7, 3, ok_S, None) == -1        # order 7 without bound_jerk
    assert call(5, 0, ok_S, None) == -1
    bad = default_settings(max_iter=0)
    assert lib.uavmp_minctrl_solve_ragged_batch(h, 5, 3, _lib.ptr(ok_S), _lib.ptr(pos), _lib.ptr(b2), _lib.ptr(b2), None, _lib.ptr(T),
                                                C.byref(bad), _lib.ptr(coef), None, None, None) == -1
    check_ragged(gpu_ctx, 5, [2, 1, 3], seed=8)


# ---- RRT* -> minimum jerk -------------------------------------------------------------------------------------------------
def small_setup(ctx, n=64):
    world = u.make_world(20, 20, 5, seed=1)
    rrt = u.RRTStar(ctx)
    rrt.setParam(max_tree_node_num=6000, sample_budget=6000)
    rrt.setGridMap(world)
    sp, _, ep, _ = u.sample_queries(world, n, seed=8, min_dist=4.0)
    seeds = np.arange(n, dtype=np.uint64) + np.uint64(123)
    return world, rrt, sp, ep, seeds


def same_plans(a, b):
    assert len(a) == len(b)
    for q, (x, y) in enumerate(zip(a, b)):
        assert (x is None) == (y is None), q
        if x is None:
            continue
        assert x["S"] == y["S"] and np.array_equal(x["solved"], y["solved"]) and np.array_equal(x["iters"], y["iters"]), q
        assert np.array_equal(bits(x["coef"]), bits(y["coef"])), q


def test_pipeline_equals_the_python_flow(gpu_ctx):
    _, rrt, sp, ep, seeds = small_setup(gpu_ctx)
    mc = u.MinimumControl(gpu_ctx)
    r, ref = planner.rrt_minimum_jerk_batch(rrt, mc, sp, ep, seeds)
    raw, plans = planner.rrt_plan_batch(rrt, sp, ep, seeds)
    tm = gpu_ctx.timings()
    assert np.array_equal(raw["search_status"], r["status"])
    same_plans(plans, ref)
    assert sum(p is not None for p in plans) >= 8
    # the waypoints: uavmp_rrt_get_paths after the call returns the optimal paths of the search
    off = r["path_offsets"]
    paths = np.zeros((int(off[-1]), 3))
    gpu_ctx.check(gpu_ctx.lib.uavmp_rrt_get_paths(gpu_ctx.h, _lib.ptr(paths), int(off[-1])))
    assert np.array_equal(bits(paths), bits(r["paths"]))
    # REACH_END with an empty optimal path: no QP posed (the node would reuse a stale path)
    empty = [q for q in range(len(sp)) if r["status"][q] == 1 and off[q + 1] - off[q] < 2]
    assert empty, "the batch must contain a REACH_END query without an optimal path"
    for q in empty:
        assert raw["n_segments"][q] == 0 and raw["qp_solved"][q] == 0 and raw["coef_offsets"][q + 1] == raw["coef_offsets"][q]
        assert (raw["iters"][q] == 0).all() and (raw["osqp_status"][q] == 0).all()
    # offsets, S and flags consistent
    assert np.array_equal(np.diff(raw["coef_offsets"]), 3 * 6 * raw["n_segments"].astype(np.int64))
    assert raw["coef_offsets"][-1] == len(raw["coef"])
    for q in range(len(sp)):
        n = int(off[q + 1] - off[q])
        assert raw["n_segments"][q] == (n - 1 if (r["status"][q] == 1 and n >= 2) else 0)
        assert raw["qp_solved"][q] == int(raw["n_segments"][q] > 0 and (raw["osqp_status"][q] == 1).all())
    assert tm["qp_launches"] == 1 and tm["search_ms"] > 0 and tm["qp_ms"] > 0


def test_pipeline_start_velocity_and_order7(gpu_ctx):
    _, rrt, sp, ep, seeds = small_setup(gpu_ctx, 32)
    sv = np.random.default_rng(9).normal(size=(32, 3))
    mc = u.MinimumControl(gpu_ctx)
    _, ref = planner.rrt_minimum_jerk_batch(rrt, mc, sp, ep, seeds, start_vel=sv)
    raw, plans = planner.rrt_plan_batch(rrt, sp, ep, seeds, start_vel=sv)
    same_plans(plans, ref)
    zero, _ = planner.rrt_plan_batch(rrt, sp, ep, seeds)
    assert not np.array_equal(bits(zero["coef"]), bits(raw["coef"]))
    # order 7 (bound_jerk = 0) against per-S minimum-snap solves of the same waypoints
    raw7, plans7 = planner.rrt_plan_batch(rrt, sp, ep, seeds, start_vel=sv, order=7, seg_time=0.8)
    r = rrt.search_batch(sp, ep, seeds)
    off = r["path_offsets"]
    for q in [q for q in range(32) if plans7[q] is not None][:6]:
        S = plans7[q]["S"]
        path = r["paths"][off[q]:off[q + 1]]
        bv = np.zeros((3, 2))
        bv[:, 0] = sv[q]
        g = mc.solve_batch(path.T.copy(), bv, np.zeros((3, 2)), np.full((3, S), 0.8), bound_jerk=np.zeros((3, 2)), order=7)
        assert np.array_equal(bits(plans7[q]["coef"]), bits(g["coef"])) and np.array_equal(plans7[q]["iters"], g["iters"]), q


def test_golden_vectors_of_the_reference_build(gpu_ctx):
    """tests/golden/rrt_plan_golden.json: the node flow with the reference's own RRT* and OSQP (make_rrt_plan_golden.py)"""
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "rrt_plan_golden.json")))
    world = u.make_world(*g["dims"], seed=g["map_seed"])
    assert hashlib.sha256(np.ascontiguousarray(world.occ).tobytes()).hexdigest() == g["occ_sha256"]
    rrt = u.RRTStar(gpu_ctx)
    rrt.setParam(**g["params"])
    rrt.setGridMap(world)
    qs = g["queries"]
    sp, ep = np.array([q["start_pt"] for q in qs]), np.array([q["end_pt"] for q in qs])
    raw, plans = planner.rrt_plan_batch(rrt, sp, ep, np.array([q["query_seed"] for q in qs], np.uint64))
    assert any(q["status"] == 1 and q["S"] == 0 for q in qs) and sum(q["S"] > 0 for q in qs) >= 8
    for i, q in enumerate(qs):
        assert (raw["search_status"][i], raw["n_segments"][i]) == (q["status"], q["S"]), i
        for ax, a in enumerate(q["axes"]):
            assert (raw["osqp_status"][i, ax], raw["iters"][i, ax], plans[i]["solved"][ax]) == (a["osqp_status"], a["iters"], a["solved"]), (i, ax)
            c = plans[i]["coef"][ax]
            if q["S"] <= 80:
                assert hashlib.sha256(np.ascontiguousarray(c).tobytes()).hexdigest() == a["coef_sha256"], (i, ax)
            else:
                ref = np.array(a["coef"])
                assert np.abs(c - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max()), (i, ax)


def test_scale_and_determinism_on_the_large_map(gpu_ctx):
    world = u.make_world(50, 50, 10, seed=1)
    rrt = u.RRTStar(gpu_ctx)
    rrt.setParam(max_tree_node_num=20000, sample_budget=20000)
    rrt.setGridMap(world)
    B = 4096
    sp, _, ep, _ = u.sample_queries(world, B, seed=8)
    seeds = np.arange(B, dtype=np.uint64) + np.uint64(1)
    a, _ = planner.rrt_plan_batch(rrt, sp, ep, seeds)
    b, plans = planner.rrt_plan_batch(rrt, sp, ep, seeds)
    for k in a:
        assert np.array_equal(np.asarray(a[k]).view(np.uint8), np.asarray(b[k]).view(np.uint8)), k
    S = a["n_segments"][a["n_segments"] > 0]
    assert len(np.unique(S)) >= 20
    # a random sample against per-S solves of the returned paths
    r = rrt.search_batch(sp, ep, seeds)
    off = r["path_offsets"]
    assert np.array_equal(r["status"], a["search_status"])
    mc = u.MinimumControl(gpu_ctx)
    done = np.nonzero(a["n_segments"] > 0)[0]
    for q in np.random.default_rng(10).choice(done, size=min(64, len(done)), replace=False):
        s = int(a["n_segments"][q])
        path = r["paths"][off[q]:off[q + 1]]
        g = mc.solve_batch(path.T.copy(), np.zeros((3, 2)), np.zeros((3, 2)), np.ones((3, s)), order=5)
        assert np.array_equal(bits(plans[q]["coef"]), bits(g["coef"])) and np.array_equal(plans[q]["iters"], g["iters"]), q


def test_path_capacity_error(gpu_ctx):
    _, rrt, sp, ep, seeds = small_setup(gpu_ctx, 16)
    rrt.setParam(path_cap=4)
    try:
        with pytest.raises(_lib.UavmpError, match="uavmp error -5"):
            planner.rrt_plan_batch(rrt, sp, ep, seeds)
        with pytest.raises(_lib.UavmpError, match="uavmp error -5"):
            rrt.search_batch(sp, ep, seeds)
    finally:
        rrt.setParam(path_cap=4096)
    raw, _ = planner.rrt_plan_batch(rrt, sp, ep, seeds)
    assert (raw["search_status"] > 0).all()
