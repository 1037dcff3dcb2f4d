"""The RRT* oracle (oracle/rrt_star_ref.cpp, a restatement incl. its own kd-tree) against the reference ITSELF:
/root/reference/src/planner/path_searching/src/rrt_star.cpp and src/kdtree/kdtree.cpp compiled unmodified against the header shims
(oracle/_ref/librrt_ref.so, recipe in oracle/Makefile; its recorded results where it is not built, tests/ref_record.py).  The reference draws every sample from a fresh std::random_device and stops on
wall-clock time; the shims pin both without touching the sources (shim/rrt_seeded_random.h, ros::time_hook), see
oracle/rrt_ref_driver.cpp.  Compared: status, use_node_num_, samples drawn, reach_goal_, the goal's g_cost, getOptimalPath() bit for
bit, and a digest over position / parent / g_cost of every tree node."""
import numpy as np

import oracle_lib
import uav_motion_planning_b200 as u

KEYS = ("status", "use_node_num", "n_opt_path", "reach_goal", "n_samples", "tree_digest", "goal_g_cost")


def same(a, b):
    return all(a[k] == b[k] for k in KEYS) and np.array_equal(a["opt_path"].view(np.uint64), b["opt_path"].view(np.uint64))


def test_restatement_matches_the_reference_build():
    world = u.make_world(20, 20, 5, seed=1)
    sp, _, ep, _ = u.sample_queries(world, 10, seed=3, min_dist=5.0)
    improved = 0
    for q in range(10):  # the whole sample loop: rewiring, goal improvements through stale links, getOptimalPath() rewritten
        kw = dict(query_seed=77 + q, max_tree_node_num=12000, sample_budget=12000)
        a = oracle_lib.rrt_search(world, sp[q], ep[q], **kw)
        b = oracle_lib.rrt_search_reference(world, sp[q], ep[q], **kw, like=a)
        assert same(a, b), q
        assert a["n_samples"] == 12000
        improved += a["n_opt_path"] > 0
    assert improved >= 5


def test_sample_budget_small_pool_and_parameters():
    world = u.make_world(20, 20, 5, seed=1)
    sp, _, ep, _ = u.sample_queries(world, 8, seed=4, min_dist=4.0)
    n_early = 0
    for q in range(8):   # budget reached before / after the first feasible path (rrt_star.cpp:413-418)
        kw = dict(query_seed=1000 + q, max_tree_node_num=20000, sample_budget=3000)
        a = oracle_lib.rrt_search(world, sp[q], ep[q], **kw)
        b = oracle_lib.rrt_search_reference(world, sp[q], ep[q], **kw, like=a)
        assert same(a, b), q
        n_early += a["status"] == 1 and a["n_samples"] < 20000
    assert n_early >= 4
    for q in range(4):   # tree limit before the goal: NO_PATH_FOUND
        kw = dict(query_seed=5 + q, max_tree_node_num=300, sample_budget=300)
        a = oracle_lib.rrt_search(world, sp[q], ep[q], **kw)
        b = oracle_lib.rrt_search_reference(world, sp[q], ep[q], **kw, like=a)
        assert same(a, b) and a["n_samples"] == 300
    for q in range(4):   # other step / radius / check resolution (more neighbours per range query, 100 lookups per edge)
        kw = dict(query_seed=9 + q, max_tree_node_num=4000, sample_budget=4000, step_length=0.4, search_radius=0.9,
                  collision_check_resolution=0.01)
        a = oracle_lib.rrt_search(world, sp[q], ep[q], **kw)
        b = oracle_lib.rrt_search_reference(world, sp[q], ep[q], **kw, like=a)
        assert same(a, b), q
