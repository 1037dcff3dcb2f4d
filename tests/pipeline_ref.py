"""CPU restatement of the search -> waypoints -> 3 x QP pipeline (TEST INFRASTRUCTURE; uses the oracle).

The chaining itself is an extension (uav_motion_planning_b200/planner.py states the rule); each half is the oracle:
KinoOracle.search (oracle/kino_ref.cpp) and oracle_lib.minctrl_solve (restated MinimumControl assembly -> the reference's
own OSQP in oracle/_ref, or its recorded results).
"""
import numpy as np

import oracle_lib


def waypoints_from_path(path, S):
    n = len(path)
    idx = (np.arange(S + 1, dtype=np.int64) * (n - 1)) // S
    return path[idx]


def segment_data(path, S, seg_time, time_alloc=0, step=0.075, n_corridor=0, margin=0.0):
    """The rule of uavmp_plan_options (include/uavmp.h): waypoints, segment times and corridor boxes from the sampled path."""
    n = len(path)
    idx = (np.arange(S + 1, dtype=np.int64) * (n - 1)) // S
    T = np.maximum(idx[1:] - idx[:-1], 1) * float(step) if time_alloc else np.full(S, float(seg_time))
    lo = hi = None
    if n_corridor > 0:
        lo = np.stack([path[idx[s]:idx[s + 1] + 1].min(axis=0) - margin for s in range(S)])
        hi = np.stack([path[idx[s]:idx[s + 1] + 1].max(axis=0) + margin for s in range(S)])
    return path[idx], T, lo, hi


def plan_one(orc, sp, sv, ep, ev, order, S, seg_time, settings=None, time_alloc=0, step=0.075, n_corridor=0, margin=0.0, like=None):
    """Returns (search_status, qp_solved, coef[3, (order+1)*S], search_result); like: the coef[3, ...] the caller compares with."""
    if time_alloc or n_corridor:
        r = orc.search(sp, sv, ep, ev)
        coef = np.zeros((3, (order + 1) * S))
        if r["status"] != 1 or r["n_path"] < 1:
            return r["status"], 0, coef, r
        wp, T, lo, hi = segment_data(r["path"], S, seg_time, time_alloc, step, n_corridor, margin)
        solved = 1
        for ax in range(3):
            ok, c, info = oracle_lib.minctrl_solve(order, S, wp[:, ax], [sv[ax], ev[ax]], [0.0, 0.0], T,
                                                   bound_jerk=[0.0, 0.0] if order == 7 else None, settings=settings,
                                                   corridor_lo=None if lo is None else lo[:, ax],
                                                   corridor_hi=None if hi is None else hi[:, ax], n_corridor=n_corridor,
                                                   like=None if like is None else like[ax])
            solved &= int(ok)
            coef[ax] = c
        return r["status"], solved, coef, r
    r = orc.search(sp, sv, ep, ev)
    n = (order + 1) * S
    coef = np.zeros((3, n))
    if r["status"] != 1 or r["n_path"] < 1:
        return r["status"], 0, coef, r
    wp = waypoints_from_path(r["path"], S)
    T = np.full(S, float(seg_time))
    solved = 1
    for ax in range(3):
        ok, c, info = oracle_lib.minctrl_solve(order, S, wp[:, ax], [sv[ax], ev[ax]], [0.0, 0.0], T,
                                               bound_jerk=[0.0, 0.0] if order == 7 else None, settings=settings,
                                               like=None if like is None else like[ax])
        solved &= int(ok)
        coef[ax] = c
    return r["status"], solved, coef, r
