"""search -> waypoints -> 3 x QP pipeline over the C-ABI (uavmp_plan_batch / uavmp_plan_batch_dev).

This chaining is an EXTENSION: the reference never feeds KinoAstar's path into MinimumControl (its QP front-end is
RRT*, src/planner/test/src/test_minimum_jerk.cpp:40-75).  The rule used here (and restated for the oracle in
tests/pipeline_ref.py): for a query that reaches the goal with n sampled path points, waypoint k = path[floor(k*(n-1)/S)],
T_i = seg_time (1.0 is the reference's convention, test_minimum_jerk.cpp:66-71), boundary velocity = start/end velocity,
boundary acceleration (and jerk) = 0.
"""
import ctypes as C

import numpy as np

from . import _lib


def plan_batch(ctx, start_pt, start_vel, end_pt, end_vel, order=7, S=8, seg_time=1.0, settings=None):
    """Host buffers in, host buffers out (copies are inside the call)."""
    sp, sv, ep, ev = (_lib.as_f64(a).reshape(-1, 3) for a in (start_pt, start_vel, end_pt, end_vel))
    B = sp.shape[0]
    n = (order + 1) * S
    status = np.zeros(B, np.int32)
    solved = np.zeros(B, np.int32)
    coef = np.zeros((B, 3, n))
    ctx.check(ctx.lib.uavmp_plan_batch(ctx.h, B, _lib.ptr(sp), _lib.ptr(sv), _lib.ptr(ep), _lib.ptr(ev), order, S,
                                       float(seg_time), C.byref(settings) if settings is not None else None,
                                       _lib.ptr(status), _lib.ptr(solved), _lib.ptr(coef)))
    return dict(search_status=status, qp_solved=solved, coef=coef)


PLAN_DEVICE_IO = 1


def _info_dict(info):
    return dict(error_flags=info.error_flags,
                counters={k: getattr(info.counters, k) for k, _ in _lib.KinoCounters._fields_},
                timings={k: getattr(info.timings, k) for k, _ in _lib.Timings._fields_})


def plan_options(order=7, S=8, seg_time=1.0, time_alloc=0, corridor_samples=0, corridor_margin=0.0):
    """uavmp_plan_options (include/uavmp.h): time_alloc 1 = the searched trajectory's own timing per segment; corridor_samples
    > 0 = box constraints around each segment's path points (+- corridor_margin) at that many interior times."""
    return _lib.PlanOptions(order, S, float(seg_time), int(time_alloc), int(corridor_samples), float(corridor_margin))


def plan_submit(ctx, B, sp, sv, ep, ev, status, solved, coef, order=7, S=8, seg_time=1.0, settings=None, device_io=False,
                options=None):
    """uavmp_plan_submit(_opt): asynchronous, returns a ticket.  Every argument is a raw pointer (int): page-locked host memory,
    or device memory with device_io=True.  The buffers must stay alive until plan_wait(ticket) has returned."""
    vp = C.c_void_p
    t = C.c_longlong(-1)
    st = C.byref(settings) if settings is not None else None
    fl = PLAN_DEVICE_IO if device_io else 0
    if options is not None:
        ctx.check(ctx.lib.uavmp_plan_submit_opt(ctx.h, B, vp(sp), vp(sv), vp(ep), vp(ev), C.byref(options), st, fl, vp(status),
                                                vp(solved), vp(coef), C.byref(t)))
    else:
        ctx.check(ctx.lib.uavmp_plan_submit(ctx.h, B, vp(sp), vp(sv), vp(ep), vp(ev), order, S, float(seg_time), st, fl,
                                            vp(status), vp(solved), vp(coef), C.byref(t)))
    return t.value


def plan_wait(ctx, ticket):
    """uavmp_plan_wait: blocks until the batch is complete; returns its error flags / counters / timings."""
    info = _lib.PlanInfo()
    ctx.check(ctx.lib.uavmp_plan_wait(ctx.h, ticket, C.byref(info)))
    return _info_dict(info)


def plan_stream_wait(ctx, ticket, cuda_stream):
    """Make a CUDA stream of the caller (raw handle) wait for the batch; the host does not block."""
    ctx.check(ctx.lib.uavmp_plan_stream_wait(ctx.h, ticket, C.c_void_p(cuda_stream)))


def max_in_flight(ctx):
    return ctx.lib.uavmp_plan_max_in_flight()


def plan_batches_pipelined(ctx, batches, order=7, S=8, seg_time=1.0, settings=None, options=None):
    """Host arrays in, host arrays out, every batch through uavmp_plan_submit / uavmp_plan_wait with as many batches in flight
    as the library allows (cross-batch pipelining).  `batches`: iterable of (start_pt, start_vel, end_pt, end_vel)."""
    if options is not None:
        order, S = options.order, options.S
    n = (order + 1) * S
    depth = max_in_flight(ctx)
    live, out = [], []

    def collect():
        t, bufs, res = live.pop(0)
        res["info"] = plan_wait(ctx, t)
        out.append(res)

    for bt in batches:
        sp, sv, ep, ev = (_lib.as_f64(a).reshape(-1, 3) for a in bt)
        B = sp.shape[0]
        res = dict(search_status=np.zeros(B, np.int32), qp_solved=np.zeros(B, np.int32), coef=np.zeros((B, 3, n)))
        if len(live) == depth:
            collect()
        t = plan_submit(ctx, B, sp.ctypes.data, sv.ctypes.data, ep.ctypes.data, ev.ctypes.data,
                        res["search_status"].ctypes.data, res["qp_solved"].ctypes.data, res["coef"].ctypes.data,
                        order=order, S=S, seg_time=seg_time, settings=settings, options=options)
        live.append((t, (sp, sv, ep, ev), res))
    while live:
        collect()
    return out


def plan_batch_dev(ctx, B, d_sp, d_sv, d_ep, d_ev, d_status, d_solved, d_coef, order=7, S=8, seg_time=1.0,
                   settings=None):
    """Every argument is a raw device pointer (int); asynchronous on the context's stream."""
    vp = C.c_void_p
    ctx.check(ctx.lib.uavmp_plan_batch_dev(ctx.h, B, vp(d_sp), vp(d_sv), vp(d_ep), vp(d_ev), order, S, float(seg_time),
                                           C.byref(settings) if settings is not None else None, vp(d_status),
                                           vp(d_solved), vp(d_coef)))


def rrt_minimum_jerk_batch(rrt, optimizer, start_pt, end_pt, query_seed, start_vel=None, seg_time=1.0):
    """The reference's own front-end → optimiser flow (test_minimum_jerk.cpp:40-75 GoalCallback), batched: RRTStar::search, then — for
    every query that returned REACH_END with a non-empty getOptimalPath() — EVERY point of the optimal path is a waypoint,
    `time_vec(i) = 1.0` for every segment (:65-71), end velocity / both accelerations zero (:31-37), and MinimumControl::solve runs once
    per axis.  The number of segments differs per query, so the QPs are solved in groups of equal S (one uavmp_minctrl_solve_batch
    call per group, 3 problems per query).  Returns a list with one entry per query: None, or dict(S, coef[3, 6 S], solved[3], iters[3])."""
    sp, ep = (_lib.as_f64(a).reshape(-1, 3) for a in (start_pt, end_pt))
    B = sp.shape[0]
    sv = np.zeros((B, 3)) if start_vel is None else _lib.as_f64(start_vel).reshape(B, 3)
    r = rrt.search_batch(sp, ep, query_seed)
    off = r["path_offsets"]
    groups = {}
    for q in range(B):
        n = int(off[q + 1] - off[q])
        if r["status"][q] == 1 and n >= 2:
            groups.setdefault(n - 1, []).append(q)
    out = [None] * B
    for S, qs in sorted(groups.items()):
        pos = np.stack([r["paths"][off[q]:off[q + 1]] for q in qs])            # [nq, S + 1, 3]
        pos_1d = np.ascontiguousarray(pos.transpose(0, 2, 1)).reshape(-1, S + 1)  # problem 3 i + axis
        bv = np.zeros((len(qs) * 3, 2))
        bv[:, 0] = sv[qs].reshape(-1)
        res = optimizer.solve_batch(pos_1d, bv, np.zeros_like(bv), np.full((len(qs) * 3, S), float(seg_time)), order=5)
        for i, q in enumerate(qs):
            out[q] = dict(S=S, coef=res["coef"][3 * i:3 * i + 3].copy(), solved=res["solved"][3 * i:3 * i + 3].copy(),
                          iters=res["iters"][3 * i:3 * i + 3].copy())
    return r, out


def rrt_plan_batch(rrt, start_pt, end_pt, query_seed, start_vel=None, order=5, seg_time=1.0, settings=None):
    """The same flow as rrt_minimum_jerk_batch in ONE call (uavmp_rrt_plan_batch): the search, the QP inputs written on the device from
    the optimal paths, and every query's three QPs in one ragged batch whatever their S.  Returns (raw, plans): raw = the packed
    arrays (search_status, n_segments, qp_solved, coef_offsets, osqp_status[B, 3], iters[B, 3], coef); plans = one entry per query as
    rrt_minimum_jerk_batch returns them, None or dict(S, coef[3, (order+1) S], solved[3], iters[3]).  rrt.search_batch-style paths
    stay available through uavmp_rrt_get_paths."""
    ctx = rrt.ctx
    sp, ep = (_lib.as_f64(a).reshape(-1, 3) for a in (start_pt, end_pt))
    B = sp.shape[0]
    sv = None if start_vel is None else _lib.as_f64(start_vel).reshape(B, 3)
    seeds = np.ascontiguousarray(np.broadcast_to(np.asarray(query_seed, np.uint64), (B,)))
    status, nseg, solved = np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32)
    offs = np.zeros(B + 1, np.int64)
    ost, its = np.zeros((B, 3), np.int32), np.zeros((B, 3), np.int32)
    total = ctx.check(ctx.lib.uavmp_rrt_plan_batch(ctx.h, B, _lib.ptr(sp), _lib.ptr(sv), _lib.ptr(ep), _lib.ptr(seeds), int(order),
                                                   float(seg_time), C.byref(settings) if settings is not None else None,
                                                   _lib.ptr(status), _lib.ptr(nseg), _lib.ptr(solved), _lib.ptr(offs), _lib.ptr(ost),
                                                   _lib.ptr(its)))
    coef = np.zeros(max(total, 1))
    ctx.check(ctx.lib.uavmp_rrt_plan_get_coef(ctx.h, _lib.ptr(coef), max(total, 1)))
    coef = coef[:total]
    raw = dict(search_status=status, n_segments=nseg, qp_solved=solved, coef_offsets=offs, osqp_status=ost, iters=its, coef=coef)
    n1 = order + 1
    plans = [None if nseg[q] == 0 else
             dict(S=int(nseg[q]), coef=coef[offs[q]:offs[q + 1]].reshape(3, n1 * nseg[q]).copy(),
                  solved=(ost[q] == 1).astype(np.int32), iters=its[q].copy())
             for q in range(B)]
    return raw, plans
