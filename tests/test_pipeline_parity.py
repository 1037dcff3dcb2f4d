"""GPU parity of the chained pipeline (uavmp_plan_batch): search -> waypoints -> 3 x QP vs the same chain on the oracle."""
import numpy as np
import pytest

import oracle_lib
import uav_motion_planning_b200 as u
from pipeline_ref import plan_one
from uav_motion_planning_b200.planner import plan_batch

pytestmark = pytest.mark.gpu
RTOL = 1e-5


@pytest.mark.parametrize("order,S", [(5, 4), (7, 8)])
def test_plan_batch_matches_oracle(gpu_ctx, order, S):
    world = u.make_world(20, 20, 5, seed=1)
    ka = u.KinoAstar(gpu_ctx)
    ka.setLaunchParams()
    ka.setGridMap(world)
    sp, sv, ep, ev = u.sample_queries(world, 24, seed=21, min_dist=8.0)
    sv[:, 0] = 0.5  # non-zero boundary velocity reaches the QP's start row
    got = plan_batch(gpu_ctx, sp, sv, ep, ev, order=order, S=S)
    orc = oracle_lib.KinoOracle(world, ka.params)
    n_checked = 0
    for q in range(24):
        st, solved, coef, _ = plan_one(orc, sp[q], sv[q], ep[q], ev[q], order, S, 1.0, like=got["coef"][q])
        assert st == got["search_status"][q]
        assert solved == got["qp_solved"][q]
        if solved:
            for ax in range(3):
                scale = max(np.abs(coef[ax]).max(), 1e-12)
                assert np.abs(coef[ax] - got["coef"][q, ax]).max() / scale < RTOL
            n_checked += 1
    assert n_checked >= 8


def test_full_batch_properties(gpu_ctx):
    """BASELINE.json configs[1] at full size (4096 queries, 50x50x10 m map): size-independent properties.

    * every solved trajectory interpolates its boundary conditions: segment 0 starts at the query's start point with
      the start velocity, the last segment ends at the last sampled path point;
    * C0..C3 continuity at every interior knot (the equality rows of the QP), to the OSQP tolerance;
    * idempotence: running the same batch twice gives bit-identical coefficients.
    """
    world = u.make_world(50, 50, 10, seed=1)
    ka = u.KinoAstar(gpu_ctx)
    ka.setLaunchParams()
    ka.setGridMap(world)
    B, S, order = 4096, 8, 7
    sp, sv, ep, ev = u.sample_queries(world, B, seed=11)
    a = plan_batch(gpu_ctx, sp, sv, ep, ev, order=order, S=S)
    b = plan_batch(gpu_ctx, sp, sv, ep, ev, order=order, S=S)
    assert np.array_equal(a["search_status"], b["search_status"])
    assert np.array_equal(a["coef"].view(np.uint64), b["coef"].view(np.uint64))
    ok = a["qp_solved"] == 1
    assert ok.mean() > 0.5
    c = a["coef"][ok].reshape(-1, 3, S, order + 1)
    # start position / velocity (local time 0 of segment 0)
    assert np.abs(c[:, :, 0, 0] - sp[ok]).max() < 5e-2   # eps_abs + eps_rel * |x|, |x| <= 25 m
    assert np.abs(c[:, :, 0, 1] - sv[ok]).max() < 5e-2
    # continuity of derivatives 0..3 at interior knots, T = 1: sum_j j!/(j-r)! c_j  ==  r! c'_r
    from math import factorial
    for r in range(4):
        lhs = sum(factorial(j) / factorial(j - r) * c[:, :, :-1, j] for j in range(r, order + 1))
        rhs = factorial(r) * c[:, :, 1:, r]
        scale = max(1.0, np.abs(rhs).max())
        assert np.abs(lhs - rhs).max() / scale < 5e-2, r


def test_fused_and_sequential_pipelines_agree_bitwise(gpu_ctx, monkeypatch):
    """Default: the CTA that finishes a query solves its three QPs inside the search kernel (qp_round, the warp body).
    UAVMP_NO_FUSE=1 runs search -> k_waypoints -> stand-alone QP kernel -> k_scatter_plan back to back.  Same bits either way,
    with the warp-per-problem and with the thread-per-problem stand-alone kernel."""
    world = u.make_world(20, 20, 5, seed=1)
    ka = u.KinoAstar(gpu_ctx)
    ka.setLaunchParams()
    ka.setGridMap(world)
    sp, sv, ep, ev = u.sample_queries(world, 200, seed=51, min_dist=8.0)
    a = plan_batch(gpu_ctx, sp, sv, ep, ev, order=7, S=8)
    monkeypatch.setenv("UAVMP_NO_FUSE", "1")
    b = plan_batch(gpu_ctx, sp, sv, ep, ev, order=7, S=8)
    monkeypatch.setenv("UAVMP_QP_THREAD", "1")   # and with the thread-per-problem QP kernel
    c = plan_batch(gpu_ctx, sp, sv, ep, ev, order=7, S=8)
    assert (a["qp_solved"] == 1).sum() > 50
    for other in (b, c):
        assert np.array_equal(a["search_status"], other["search_status"]) and np.array_equal(a["qp_solved"], other["qp_solved"])
        assert np.array_equal(a["coef"].view(np.uint64), other["coef"].view(np.uint64))


def test_batches_in_flight_match_synchronous_calls(gpu_ctx):
    """uavmp_plan_submit / uavmp_plan_wait with 6 batches in flight (their search kernels overlap and share the arena pool)
    give bit-identical results to one synchronous uavmp_plan_batch per batch, and the per-batch counters are those of the
    synchronous call."""
    from uav_motion_planning_b200.planner import plan_batches_pipelined
    world = u.make_world(50, 50, 10, seed=1)
    ka = u.KinoAstar(gpu_ctx)
    ka.setLaunchParams()
    ka.setGridMap(world)
    batches = [u.sample_queries(world, 700, seed=300 + i) for i in range(9)]
    ref, ref_cnt = [], []
    for bt in batches:
        ref.append(plan_batch(gpu_ctx, *bt, order=7, S=8))
        ref_cnt.append(ka.counters())
    got = plan_batches_pipelined(gpu_ctx, batches, order=7, S=8)
    assert len(got) == len(ref)
    for r, c, g in zip(ref, ref_cnt, got):
        assert g["info"]["error_flags"] == 0
        assert np.array_equal(r["search_status"], g["search_status"]) and np.array_equal(r["qp_solved"], g["qp_solved"])
        assert np.array_equal(r["coef"].view(np.uint64), g["coef"].view(np.uint64))
        # n_cloud_pts_tested is a diagnostic whose value depends on thread timing (a centre another lane has already rejected
        # is dropped from the sweep); every other counter is a function of the expansion sequence
        for k in ("n_pop", "n_occ_lookup", "n_hash_probe", "n_insert", "n_update", "n_heuristic", "n_shot"):
            assert c[k] == g["info"]["counters"][k], k
    assert sum(int((g["qp_solved"] == 1).sum()) for g in got) > 3000


def test_device_io_tickets_and_stream_wait(gpu_ctx):
    """Device pointers through uavmp_plan_submit(UAVMP_PLAN_DEVICE_IO): a torch side stream is made to wait for each ticket
    (uavmp_plan_stream_wait) and copies the result out without the host ever blocking until the end."""
    import torch
    from uav_motion_planning_b200.planner import plan_submit, plan_wait, plan_stream_wait
    world = u.make_world(20, 20, 5, seed=1)
    ka = u.KinoAstar(gpu_ctx)
    ka.setLaunchParams()
    ka.setGridMap(world)
    dev = torch.device("cuda", 0)
    n, B = 64, 96
    side = torch.cuda.Stream(device=dev)
    batches = [u.sample_queries(world, B, seed=400 + i, min_dist=8.0) for i in range(4)]
    ref = [plan_batch(gpu_ctx, *bt, order=7, S=8) for bt in batches]
    d_in = [[torch.from_numpy(a).to(dev) for a in bt] for bt in batches]
    d_out = [(torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros(B, dtype=torch.int32, device=dev),
              torch.zeros(B, 3 * n, dtype=torch.float64, device=dev)) for _ in batches]
    copies = [torch.zeros(B, 3 * n, dtype=torch.float64, device=dev) for _ in batches]
    torch.cuda.synchronize()
    tickets = []
    for (sp, sv, ep, ev), (st, so, co), cp in zip(d_in, d_out, copies):
        t = plan_submit(gpu_ctx, B, sp.data_ptr(), sv.data_ptr(), ep.data_ptr(), ev.data_ptr(), st.data_ptr(), so.data_ptr(),
                        co.data_ptr(), order=7, S=8, device_io=True)
        plan_stream_wait(gpu_ctx, t, side.cuda_stream)
        with torch.cuda.stream(side):
            cp.copy_(co, non_blocking=True)
        tickets.append(t)
    for t in tickets:
        assert plan_wait(gpu_ctx, t)["error_flags"] == 0
    side.synchronize()
    for r, (st, so, co), cp in zip(ref, d_out, copies):
        assert np.array_equal(r["search_status"], st.cpu().numpy()) and np.array_equal(r["qp_solved"], so.cpu().numpy())
        assert np.array_equal(r["coef"].reshape(B, -1).view(np.uint64), cp.cpu().numpy().view(np.uint64))
    with pytest.raises(u.UavmpError, match="ticket"):
        plan_wait(gpu_ctx, tickets[0])


@pytest.mark.parametrize("order,S,Kc,time_alloc", [(7, 12, 2, 0), (7, 8, 2, 1), (5, 4, 0, 1)])
def test_plan_options_time_allocation_and_corridor(gpu_ctx, monkeypatch, order, S, Kc, time_alloc):
    """uavmp_plan_submit_opt: segment times from the searched trajectory's own timing (time_alloc 1) and corridor boxes around
    each segment's path points (corridor rows active in the QP), against the same chain on the oracle (tests/pipeline_ref.py):
    identical search status / qp_solved, coefficients bit-identical; the in-kernel QP (default) and the sequential pipeline
    (UAVMP_NO_FUSE) give the same bits."""
    from uav_motion_planning_b200.planner import plan_batches_pipelined, plan_options
    world = u.make_world(20, 20, 5, seed=1)
    ka = u.KinoAstar(gpu_ctx)
    ka.setLaunchParams()
    ka.setGridMap(world)
    margin = 0.15
    sp, sv, ep, ev = u.sample_queries(world, 40, seed=61, min_dist=8.0)
    opt = plan_options(order=order, S=S, seg_time=1.0, time_alloc=time_alloc, corridor_samples=Kc, corridor_margin=margin)
    a = plan_batches_pipelined(gpu_ctx, [(sp, sv, ep, ev)], options=opt)[0]
    monkeypatch.setenv("UAVMP_NO_FUSE", "1")
    b = plan_batches_pipelined(gpu_ctx, [(sp, sv, ep, ev)], options=opt)[0]
    monkeypatch.delenv("UAVMP_NO_FUSE")
    assert a["info"]["error_flags"] == 0
    assert np.array_equal(a["search_status"], b["search_status"]) and np.array_equal(a["qp_solved"], b["qp_solved"])
    assert np.array_equal(a["coef"].view(np.uint64), b["coef"].view(np.uint64))
    plain = plan_batch(gpu_ctx, sp, sv, ep, ev, order=order, S=S)
    orc = oracle_lib.KinoOracle(world, ka.params)
    n_ok = n_diff = 0
    for q in range(40):
        st, solved, coef, _ = plan_one(orc, sp[q], sv[q], ep[q], ev[q], order, S, 1.0, time_alloc=time_alloc,
                                       step=ka.params.time_step_size, n_corridor=Kc, margin=margin, like=a["coef"][q])
        assert (st, solved) == (a["search_status"][q], a["qp_solved"][q]), q
        if solved:
            assert np.array_equal(coef, a["coef"][q]), q
            n_ok += 1
            n_diff += np.abs(coef - plain["coef"][q]).max() > 1e-6
    assert n_ok >= 10 and n_diff >= 5   # the options change the trajectories (they are not silently ignored)
