"""The grid A* oracle (oracle/astar_ref.cpp, a restatement) against the reference ITSELF: /root/reference/src/planner/path_searching/
src/a_star.cpp compiled unmodified against the header shims (oracle/_ref/libastar_ref.so, recipe in oracle/Makefile; its recorded results
where it is not built, tests/ref_record.py).
Status, use_node_num_, every path point bit for bit, and the digest of every position the search passes to GridMap::isInMap in call
order (= the ordered sequence of neighbour evaluations, hence of expansions) must be identical."""
import numpy as np

import oracle_lib
import uav_motion_planning_b200 as u

def same(a, b):
    return ((a["status"], a["use_node_num"], a["n_path"], a["lookup_digest"], a["n_in_map_calls"]) ==
            (b["status"], b["use_node_num"], b["n_path"], b["lookup_digest"], b["n_in_map_calls"]) and
            np.array_equal(a["path"].view(np.uint64), b["path"].view(np.uint64)))


def test_restatement_matches_the_reference_build():
    world = u.make_world(20, 20, 5, seed=1)
    sp, _, ep, _ = u.sample_queries(world, 40, seed=3, min_dist=5.0)
    n_reach = 0
    for q in range(40):
        a = oracle_lib.astar_search(world, sp[q], ep[q])
        b = oracle_lib.astar_search_reference(world, sp[q], ep[q], like=a)
        assert same(a, b), q
        n_reach += a["status"] == 1
    assert n_reach >= 30


def test_pool_exhaustion_weighted_heuristic_and_outside_goal():
    world = u.make_world(20, 20, 5, seed=1)
    sp, _, ep, _ = u.sample_queries(world, 12, seed=4, min_dist=8.0)
    for q in range(12):  # tiny pool: "allocated_node_num is too small" in the middle of an expansion (a_star.cpp:134-138)
        a = oracle_lib.astar_search(world, sp[q], ep[q], allocated_node_num=500)
        b = oracle_lib.astar_search_reference(world, sp[q], ep[q], allocated_node_num=500, like=a)
        assert same(a, b) and a["status"] == 2 and a["use_node_num"] == 500
    for q in range(6):   # lambda_heu 2.5: the in-place g updates reorder the open list differently
        a = oracle_lib.astar_search(world, sp[q], ep[q], lambda_heu=2.5)
        b = oracle_lib.astar_search_reference(world, sp[q], ep[q], lambda_heu=2.5, like=a)
        assert same(a, b)
    out = np.array([100.0, 0.0, 1.0])  # end point outside the map: returns at once (:52-56)
    a = oracle_lib.astar_search(world, sp[0], out)
    b = oracle_lib.astar_search_reference(world, sp[0], out, like=a)
    assert same(a, b) and a["status"] == 2 and a["use_node_num"] == 0
