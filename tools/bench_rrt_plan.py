"""Timing of the batched RRT* -> minimum-jerk flow (uavmp_rrt_plan_batch) on the 50 x 50 x 10 m map, and of the same QP problems
solved the old way: one uavmp_minctrl_solve_batch call per distinct S (what planner.rrt_minimum_jerk_batch does).  Not the bench line
(bench.py is the kino-A* + QP pipeline); prints one JSON line.

  python tools/bench_rrt_plan.py [B=4096] [nodes=20000] [reps=3]

Reported: search / QP-input packing / QP-stage / total device time of uavmp_rrt_plan_batch (uavmp_get_timings); for the per-S loop the
summed device time of its calls (H2D + QP + D2H) and the wall time of the host loop around them; the grouped kernel alone on the same
problems (uavmp_minctrl_solve_ragged_batch, host arrays in / out as the loop has); the histogram of S, groups, thread-kernel groups,
problems/s.  Variants of the grouped kernel (env knobs of qp_kernel.cu): chunks by increasing S instead of longest first, and two
112 KB CTAs per SM instead of one 226 KB CTA on the problems with S <= 50.  Medians over `reps` runs."""
import json
import os
import sys
import time

import numpy as np

sys.path[:0] = [os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")]
import uav_motion_planning_b200 as u  # noqa: E402
from uav_motion_planning_b200 import planner  # noqa: E402


def med(xs):
    return float(np.median(xs))


def per_s_loop(ctx, mc, probs):
    """the old way: group by S on the host, one synchronous uavmp_minctrl_solve_batch per group"""
    t0 = time.perf_counter()
    dev, qp = 0.0, 0.0
    groups = {}
    for i, (s, _, _) in enumerate(probs):
        groups.setdefault(s, []).append(i)
    for s, idx in sorted(groups.items()):
        pos = np.stack([probs[i][1] for i in idx])
        bv = np.stack([probs[i][2] for i in idx])
        mc.solve_batch(pos, bv, np.zeros_like(bv), np.ones((len(idx), s)), order=5)
        t = ctx.timings()
        dev += t["total_ms"]
        qp += t["qp_ms"]
    return (time.perf_counter() - t0) * 1e3, dev, qp, len(groups)


def ragged(ctx, mc, probs):
    S = np.array([p[0] for p in probs], np.int32)
    pos = np.concatenate([p[1] for p in probs])
    bv = np.stack([p[2] for p in probs])
    t0 = time.perf_counter()
    mc.solve_batch_ragged(pos, bv, np.zeros_like(bv), np.ones(int(S.sum())), S=S, order=5)
    wall = (time.perf_counter() - t0) * 1e3
    return wall, ctx.timings()


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
    nodes = int(sys.argv[2]) if len(sys.argv) > 2 else 20000
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
    ctx = u.Context(0)
    world = u.make_world(50, 50, 10, seed=1)
    rrt = u.RRTStar(ctx)
    rrt.setParam(max_tree_node_num=nodes, sample_budget=nodes)
    rrt.setGridMap(world)
    mc = u.MinimumControl(ctx)
    sp, _, ep, _ = u.sample_queries(world, B, seed=8)
    seeds = np.arange(B, dtype=np.uint64) + np.uint64(1)

    planner.rrt_plan_batch(rrt, sp, ep, seeds)  # warm-up: arenas, QP plans of every S in the batch
    runs = []
    for _ in range(reps):
        t0 = time.perf_counter()
        raw, _ = planner.rrt_plan_batch(rrt, sp, ep, seeds)
        wall = (time.perf_counter() - t0) * 1e3
        runs.append((wall, ctx.timings()))
    tm = [t for _, t in runs]
    nseg = raw["n_segments"]
    S_q = nseg[nseg > 0]
    hist = {int(s): int(c) for s, c in zip(*np.unique(S_q, return_counts=True))}
    P = 3 * len(S_q)

    # the same QP problems (waypoints = the optimal paths), problem 3 k + axis as in the pipeline
    r = rrt.search_batch(sp, ep, seeds)
    off = r["path_offsets"]
    probs = []
    for q in np.nonzero(nseg > 0)[0]:
        path = r["paths"][off[q]:off[q + 1]]
        for ax in range(3):
            probs.append((int(nseg[q]), np.ascontiguousarray(path[:, ax]), np.zeros(2)))
    loop = [per_s_loop(ctx, mc, probs) for _ in range(reps)]
    rag = [ragged(ctx, mc, probs) for _ in range(reps)]

    def variant(env, subset):
        os.environ.update(env)
        try:
            return [ragged(ctx, mc, subset)[1]["qp_ms"] for _ in range(reps)]
        finally:
            for k in env:
                os.environ.pop(k)

    small = [p for p in probs if p[0] <= 50]
    out = dict(
        workload=f"{B} RRT* queries x {nodes} samples, 50x50x10 m map, then 3 min-jerk QPs per query with S = optimal-path points - 1",
        queries=B, qp_queries=int(len(S_q)), qp_problems=P, distinct_S=len(hist), thread_kernel_groups=int(tm[-1]["qp_launches"] - 1),
        S_min=int(S_q.min()) if len(S_q) else 0, S_median=float(np.median(S_q)) if len(S_q) else 0, S_max=int(S_q.max()) if len(S_q) else 0,
        S_hist=hist,
        plan_batch=dict(search_ms=med([t["search_ms"] for t in tm]), path_ms=med([t["path_ms"] for t in tm]),
                        qp_ms=med([t["qp_ms"] for t in tm]), d2h_ms=med([t["d2h_ms"] for t in tm]), total_ms=med([t["total_ms"] for t in tm]),
                        wall_ms=med([w for w, _ in runs]), qp_launches=int(tm[-1]["qp_launches"]),
                        qp_problems_per_s=P / (med([t["qp_ms"] for t in tm]) * 1e-3) if P else 0.0),
        per_s_loop=dict(calls=loop[0][3], wall_ms=med([x[0] for x in loop]), device_ms=med([x[1] for x in loop]),
                        qp_ms=med([x[2] for x in loop]), host_ms=med([x[0] - x[1] for x in loop]),
                        qp_problems_per_s=P / (med([x[0] for x in loop]) * 1e-3) if P else 0.0),
        ragged_call=dict(wall_ms=med([w for w, _ in rag]), device_ms=med([t["total_ms"] for _, t in rag]),
                         qp_ms=med([t["qp_ms"] for _, t in rag]), qp_launches=int(rag[-1][1]["qp_launches"])),
        variants=dict(
            ascending_S_qp_ms=med(variant({"UAVMP_QP_RAGGED_ASC": "1"}, probs)),
            longest_first_qp_ms=med([t["qp_ms"] for _, t in rag]),
            S_le_50_problems=len(small),
            S_le_50_one_226KB_cta_qp_ms=med(variant({}, small)) if small else 0.0,
            S_le_50_two_112KB_ctas_qp_ms=med(variant({"UAVMP_QP_RAGGED_CTAS": "2"}, small)) if small else 0.0),
    )
    out["qp_stage_speedup_vs_per_s_loop_wall"] = out["per_s_loop"]["wall_ms"] / out["plan_batch"]["qp_ms"] if P else 0.0
    out["qp_kernel_speedup_vs_per_s_loop_device_qp"] = out["per_s_loop"]["qp_ms"] / out["ragged_call"]["qp_ms"] if P else 0.0
    print(json.dumps(out))


if __name__ == "__main__":
    main()
