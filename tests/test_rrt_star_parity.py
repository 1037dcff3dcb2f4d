"""GPU parity: batched CUDA RRTStar::search (uavmp_rrt_search_batch) vs the CPU oracle (oracle/rrt_star_ref.cpp, itself pinned to the
reference's rrt_star.cpp + kdtree.cpp): status, use_node_num, samples drawn, the goal's g_cost bits, the digest over position / parent /
g_cost of EVERY tree node, and getOptimalPath() bit for bit."""
import numpy as np
import pytest

import oracle_lib
import uav_motion_planning_b200 as u

pytestmark = pytest.mark.gpu


def compare(ctx, world, n, seed, min_dist, **kw):
    r = u.RRTStar(ctx)
    r.setParam(**kw)
    r.setGridMap(world)
    sp, _, ep, _ = u.sample_queries(world, n, seed=seed, min_dist=min_dist)
    seeds = np.arange(n, dtype=np.uint64) * np.uint64(7919) + np.uint64(seed)
    got = r.search_batch(sp, ep, seeds)
    okw = {k: v for k, v in kw.items() if k != "path_cap"}
    for q in range(n):
        ref = oracle_lib.rrt_search(world, sp[q], ep[q], int(seeds[q]), **okw)
        o0, o1 = got["path_offsets"][q], got["path_offsets"][q + 1]
        assert (ref["status"], ref["use_node_num"], ref["n_samples"], ref["tree_digest"]) == \
            (got["status"][q], got["use_node_num"][q], got["n_samples"][q], int(got["tree_digest"][q])), q
        assert np.float64(ref["goal_g_cost"]).view(np.uint64) == got["goal_g_cost"][q:q + 1].view(np.uint64)[0], q
        assert ref["n_opt_path"] == o1 - o0 and np.array_equal(ref["opt_path"].view(np.uint64), got["paths"][o0:o1].view(np.uint64)), q
    return got


def test_sample_stream_matches_libstdcxx(gpu_ctx):
    """uavmp_rrt_sample_seed is the documented counter hash (host side of the same function the kernel uses)"""
    r = u.RRTStar(gpu_ctx)
    def seed32(qs, i):
        m = (1 << 64) - 1
        z = (qs + 0x9E3779B97F4A7C15 * (i + 1)) & m
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & m
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & m
        return ((z ^ (z >> 31)) >> 32) & 0xffffffff
    for qs, i in ((0, 0), (77, 5), (2**63 + 11, 99999)):
        assert r.sample_seed(qs, i) == seed32(qs, i)


def test_whole_sample_loop_with_rewiring_and_goal_improvements(gpu_ctx):
    world = u.make_world(20, 20, 5, seed=1)
    got = compare(gpu_ctx, world, 24, seed=3, min_dist=5.0, max_tree_node_num=8000, sample_budget=8000)
    assert (got["status"] == 1).mean() > 0.5 and (np.diff(got["path_offsets"]) > 0).sum() >= 8


def test_sample_budget_tree_limit_and_other_parameters(gpu_ctx):
    world = u.make_world(20, 20, 5, seed=1)
    got = compare(gpu_ctx, world, 16, seed=4, min_dist=4.0, max_tree_node_num=20000, sample_budget=3000)
    assert ((got["status"] == 1) & (got["n_samples"] < 20000)).sum() >= 8
    got = compare(gpu_ctx, world, 8, seed=5, min_dist=8.0, max_tree_node_num=300, sample_budget=300)
    assert (got["n_samples"] == 300).all()
    compare(gpu_ctx, world, 8, seed=9, min_dist=5.0, max_tree_node_num=4000, sample_budget=4000, step_length=0.4, search_radius=0.9,
            collision_check_resolution=0.01)


def test_reference_class_call_and_batch_properties(gpu_ctx):
    world = u.make_world(20, 20, 5, seed=1)
    r = u.RRTStar(gpu_ctx)
    r.setParam(max_tree_node_num=6000, sample_budget=6000)
    r.setGridMap(world)
    r.init()
    sp, _, ep, _ = u.sample_queries(world, 256, seed=8, min_dist=4.0)
    seeds = np.arange(256, dtype=np.uint64) + np.uint64(123)
    got = r.search_batch(sp, ep, seeds)
    again = r.search_batch(sp, ep, seeds, want_paths=False)
    assert np.array_equal(got["tree_digest"], again["tree_digest"]) and np.array_equal(got["use_node_num"], again["use_node_num"])
    other = r.search_batch(sp, ep, seeds + np.uint64(1), want_paths=False)
    assert (other["tree_digest"] != got["tree_digest"]).all()
    off = got["path_offsets"]
    has = np.nonzero(np.diff(off) > 0)[0]
    assert len(has) > 20
    assert np.array_equal(got["paths"][off[has]], sp[has]) and np.array_equal(got["paths"][off[has + 1] - 1], ep[has])
    for q in has[:8]:   # a polyline of edges no longer than the search radius / step, not shorter than the straight line
        seg = np.linalg.norm(np.diff(got["paths"][off[q]:off[q + 1]], axis=0), axis=1)
        assert seg.max() <= 0.5 + 1e-9 and seg.sum() >= np.linalg.norm(ep[q] - sp[q]) - 1e-9
    for q in range(0, 256, 64):
        ref = oracle_lib.rrt_search(world, sp[q], ep[q], int(seeds[q]), max_tree_node_num=6000, sample_budget=6000)
        assert (ref["status"], ref["use_node_num"], ref["tree_digest"]) == (got["status"][q], got["use_node_num"][q], int(got["tree_digest"][q]))
    path = []
    st = r.search(sp[has[0]], ep[has[0]], path, query_seed=int(seeds[has[0]]))
    assert st == 1 and not path and np.array_equal(np.array(r.getOptimalPath()), got["paths"][off[has[0]]:off[has[0] + 1]])


def test_rrt_star_to_minimum_jerk_like_the_reference_node(gpu_ctx):
    """test_minimum_jerk.cpp:40-75: RRT* -> every optimal-path point a waypoint, T = 1 -> MinimumControl::solve per axis.  The QPs are
    bit-identical to the reference's OSQP while S <= 80 (AMD order tabulated for order 5) and within 1e-5 beyond (DESIGN.md §4)."""
    from uav_motion_planning_b200 import planner
    world = u.make_world(20, 20, 5, seed=1)
    rrt, mc = u.RRTStar(gpu_ctx), u.MinimumControl(gpu_ctx)
    rrt.setParam(max_tree_node_num=6000, sample_budget=6000)
    rrt.setGridMap(world)
    sp, _, ep, _ = u.sample_queries(world, 64, seed=8, min_dist=4.0)
    seeds = np.arange(64, dtype=np.uint64) + np.uint64(123)
    r, plans = planner.rrt_minimum_jerk_batch(rrt, mc, sp, ep, seeds)
    done = [q for q in range(64) if plans[q] is not None]
    assert len(done) >= 8 and all((r["status"][q] == 1) for q in done)
    n_exact = 0
    for q in done[:10]:
        S = plans[q]["S"]
        path = r["paths"][r["path_offsets"][q]:r["path_offsets"][q + 1]]
        assert len(path) == S + 1
        for ax in range(3):
            ok, coef, info = oracle_lib.minctrl_solve(5, S, path[:, ax], np.zeros(2), np.zeros(2), np.ones(S), like=plans[q]["coef"][ax])
            assert bool(plans[q]["solved"][ax]) == bool(ok)
            if not ok:
                continue
            got = plans[q]["coef"][ax]
            if S <= 80:
                assert np.array_equal(got.view(np.uint64), coef.view(np.uint64)) and plans[q]["iters"][ax] == info["iter"]
                n_exact += 1
            else:
                assert np.abs(got - coef).max() <= 1e-5 * max(1.0, np.abs(coef).max())
            # the spline interpolates the waypoints (position continuity rows of getConstraintMatrix)
            assert abs(got[0] - path[0, ax]) < 2e-2 and abs(got[6 * (S - 1):].sum() - path[-1, ax]) < 2e-2   # eps_abs = eps_rel = 1e-3
    assert n_exact >= 3


def test_golden_vectors_of_the_reference_build(gpu_ctx):
    """tests/golden/rrt_star_golden.json: outputs of the reference's own rrt_star.cpp + kdtree.cpp build (make_f4_golden.py)"""
    import hashlib
    import json
    import os
    cases = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "rrt_star_golden.json")))["cases"]
    for case in cases:
        world = u.make_world(*case["dims"], seed=case["map_seed"])
        r = u.RRTStar(gpu_ctx)
        r.setParam(**case["params"])
        r.setGridMap(world)
        sp = np.array([q["start_pt"] for q in case["queries"]])
        ep = np.array([q["end_pt"] for q in case["queries"]])
        seeds = np.array([q["query_seed"] for q in case["queries"]], np.uint64)
        got = r.search_batch(sp, ep, seeds)
        for i, q in enumerate(case["queries"]):
            o0, o1 = got["path_offsets"][i], got["path_offsets"][i + 1]
            assert (q["status"], q["use_node_num"], q["n_samples"], q["tree_digest"], q["n_opt_path"]) == \
                (got["status"][i], got["use_node_num"][i], got["n_samples"][i], str(int(got["tree_digest"][i])), o1 - o0), (case["name"], i)
            assert q["goal_g_cost_bits"] == str(got["goal_g_cost"][i:i + 1].view(np.uint64)[0]), (case["name"], i)
            assert hashlib.sha256(np.ascontiguousarray(got["paths"][o0:o1]).tobytes()).hexdigest() == q["opt_path_sha256"], (case["name"], i)
