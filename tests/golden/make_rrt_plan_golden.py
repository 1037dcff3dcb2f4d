"""Generates tests/golden/rrt_plan_golden.json from the REFERENCE ITSELF: the node flow of test_minimum_jerk.cpp:40-75 with the
reference's rrt_star.cpp + kdtree.cpp (oracle/_ref/librrt_ref.so) and its OSQP (oracle/_ref/libosqp_ref.so), run where oracle/_ref is
built.  Committed together with its output; tests never regenerate it.  tests/test_rrt_plan.py checks uavmp_rrt_plan_batch against it.

Per query: RRTStar::search; if REACH_END with an optimal path of n >= 2 points, S = n - 1, every point a waypoint, T_s = 1.0, zero
start velocity, and MinimumControl::solve per axis.  Recorded: status, n_opt, S (0: no QP posed) and per axis OSQP status, iterations
and the SHA-256 of the coefficient bits (plus the values where S > 80).

  python tests/golden/make_rrt_plan_golden.py
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle_lib  # noqa: E402
import uav_motion_planning_b200 as u  # noqa: E402

PARAMS = dict(max_tree_node_num=8000, sample_budget=8000)
N_QUERIES, QUERY_SEED, MIN_DIST = 24, 21, 5.0


def query_seeds(n):
    return [1000 + 17 * q for q in range(n)]


def main():
    assert oracle_lib.have_rrt_ref() and oracle_lib.have_ref(), "build oracle/_ref first (make -C oracle)"
    world = u.make_world(20, 20, 5, seed=1)
    sp, _, ep, _ = u.sample_queries(world, N_QUERIES, seed=QUERY_SEED, min_dist=MIN_DIST)
    qs = []
    for q, seed in enumerate(query_seeds(N_QUERIES)):
        r = oracle_lib.rrt_search_reference(world, sp[q], ep[q], seed, **PARAMS)
        n = int(r["n_opt_path"])
        S = n - 1 if (r["status"] == 1 and n >= 2) else 0
        axes = []
        for ax in range(3 if S else 0):
            ok, coef, info = oracle_lib.minctrl_solve(5, S, r["opt_path"][:, ax], np.zeros(2), np.zeros(2), np.ones(S))
            axes.append(dict(solved=int(bool(ok)), osqp_status=int(info["status_val"]), iters=int(info["iter"]),
                             coef_sha256=hashlib.sha256(np.ascontiguousarray(coef).tobytes()).hexdigest()))
            if S > 80:  # minimum-degree order here: the check is 1e-5 relative (DESIGN.md §4), so keep the values
                axes[-1]["coef"] = coef.tolist()
        qs.append(dict(start_pt=sp[q].tolist(), end_pt=ep[q].tolist(), query_seed=seed, status=int(r["status"]), n_opt=n, S=S, axes=axes))
    json.dump(dict(source="oracle/_ref/librrt_ref.so + libosqp_ref.so = the reference's rrt_star.cpp + kdtree.cpp and OSQP compiled "
                          "unmodified; the node flow of test_minimum_jerk.cpp:40-75 (T = 1, zero start velocity)",
                   dims=[20, 20, 5], map_seed=1, params=PARAMS, occ_sha256=hashlib.sha256(np.ascontiguousarray(world.occ).tobytes()).hexdigest(),
                   queries=qs), open(os.path.join(HERE, "rrt_plan_golden.json"), "w"), indent=1)
    print("written:", sum(1 for q in qs if q["S"]), "queries with a QP, S =", sorted(q["S"] for q in qs if q["S"]),
          "; REACH_END without an optimal path:", sum(1 for q in qs if q["status"] == 1 and not q["S"]))


if __name__ == "__main__":
    main()
