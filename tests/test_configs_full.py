"""BASELINE.json configs[2] and configs[3] at (near) full size on the GPU: size-independent properties over the whole batch
plus bit-exact oracle parity on a seeded subset (the oracle needs ~0.1 s per query, so it cannot cover 32 768)."""
import numpy as np
import pytest

import oracle_lib
import uav_motion_planning_b200 as u
from pipeline_ref import plan_one
from uav_motion_planning_b200.planner import plan_batch

pytestmark = pytest.mark.gpu


def check_subset(ka, world, qs, got, idx):
    sp, sv, ep, ev = qs
    orc = oracle_lib.KinoOracle(world, ka.params)
    for q in idx:
        ref = orc.search(sp[q], sv[q], ep[q], ev[q])
        o0, o1 = got["path_offsets"][q], got["path_offsets"][q + 1]
        assert (ref["status"], ref["use_node_num"], ref["n_pop"], ref["pop_hash"]) == \
            (got["status"][q], got["use_node_num"][q], got["n_pop"][q], int(got["pop_hash"][q])), q
        assert np.array_equal(ref["path"].view(np.uint64), got["paths"][o0:o1].view(np.uint64))


def test_config2_ellipsoid_only_32768(gpu_ctx):
    """configs[2]: batch 32 768, 50x50x10 m map, collision_check_type 2 (SE(3) ellipsoid only, r = 0.4, h = 0.1)."""
    world = u.make_world(50, 50, 10, seed=1)
    ka = u.KinoAstar(gpu_ctx)
    ka.setLaunchParams()
    ka.setParam(collision_check_type=2)
    ka.setGridMap(world)
    B = 32768
    qs = u.sample_queries(world, B, seed=23)
    a = {k: (v.copy() if v is not None else None) for k, v in ka.search_batch(*qs).items()}
    b = ka.search_batch(*qs, want_paths=False)
    assert set(np.unique(a["status"])) <= {1, 2}
    assert (a["status"] == 1).mean() > 0.9
    assert np.array_equal(a["pop_hash"], b["pop_hash"]) and np.array_equal(a["use_node_num"], b["use_node_num"])   # idempotent
    # every path starts at its query's start point and ends within the shot's reach of the goal
    off = a["path_offsets"]
    ok = np.nonzero(a["status"] == 1)[0]
    assert np.array_equal(a["paths"][off[ok]], qs[0][ok])
    assert np.linalg.norm(a["paths"][off[ok + 1] - 1] - qs[2][ok], axis=1).max() < 1.0
    # failures exhausted the pool or the open list; nobody overran the pool
    assert a["use_node_num"].max() <= ka.params.allocated_node_num
    check_subset(ka, world, qs, a, list(range(0, B, B // 24)))


def test_config3_wall_map_12_segments_with_corridor(gpu_ctx):
    """configs[3]: two-slab wall map, search + 12-segment minimum snap WITH corridor box constraints (2 samples per segment, boxes
    = the segment's path extent +- 0.2 m; uavmp_plan_options), through uavmp_plan_submit_opt; oracle chain on a subset."""
    from uav_motion_planning_b200.planner import plan_batches_pipelined, plan_options
    world = u.make_world(50, 50, 10, seed=1, map_type=2)
    ka = u.KinoAstar(gpu_ctx)
    ka.setLaunchParams()
    ka.setGridMap(world)
    B = 2048
    sp, sv, ep, ev = u.sample_queries(world, B, seed=29)
    # half of the queries must cross the wall plane x = 0 (through the 0.5 m gap or around)
    sp[: B // 2, 0] = -np.abs(sp[: B // 2, 0]) - 1.0
    ep[: B // 2, 0] = np.abs(ep[: B // 2, 0]) + 1.0
    opt = plan_options(order=7, S=12, seg_time=1.0, corridor_samples=2, corridor_margin=0.2)
    got = plan_batches_pipelined(gpu_ctx, [(sp, sv, ep, ev)], options=opt)[0]
    assert got["info"]["error_flags"] == 0
    assert set(np.unique(got["search_status"])) <= {1, 2}
    plain = plan_batch(gpu_ctx, sp, sv, ep, ev, order=7, S=12)
    assert np.array_equal(plain["search_status"], got["search_status"])
    orc = oracle_lib.KinoOracle(world, ka.params)
    n_ok = n_active = 0
    for q in list(range(0, 8)) + list(range(B // 2, B // 2 + 8)):
        st, solved, coef, _ = plan_one(orc, sp[q], sv[q], ep[q], ev[q], 7, 12, 1.0, n_corridor=2, margin=0.2, like=got["coef"][q])
        assert (st, solved) == (got["search_status"][q], got["qp_solved"][q])
        if solved:
            assert np.array_equal(coef, got["coef"][q])   # tabulated AMD order: bit-identical to the reference's OSQP
            n_ok += 1
            n_active += np.abs(coef - plain["coef"][q]).max() > 1e-6
    assert n_ok >= 4 and n_active >= 2
