"""world_size-2 gloo test (CPU) of the multi-GPU host logic: slicing + the all-gather of solved trajectories.
The per-rank compute is a stand-in (the oracle pipeline on a tiny map) because there is no GPU here; on the GPU box the
same function is driven by the CUDA pipeline (bench.py --gpus N)."""
import os
import socket
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ctypes as C
    import torch.distributed as dist
    import oracle_lib
    import uav_motion_planning_b200 as u
    from pipeline_ref import plan_one
    from uav_motion_planning_b200 import _lib
    from uav_motion_planning_b200.sharding import plan_sharded
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    world_map = u.make_world(20, 20, 5, seed=1)
    p = _lib.KinoParams()
    u.load().uavmp_kino_params_launch(C.byref(p))
    orc = oracle_lib.KinoOracle(world_map, p)
    sp, sv, ep, ev = u.sample_queries(world_map, 5, seed=31, min_dist=8.0)   # 5 queries on 2 ranks: ragged split 3 + 2

    def solve_local(a, b, c, d):
        res = [plan_one(orc, a[i], b[i], c[i], d[i], 5, 4, 1.0) for i in range(len(a))]
        return dict(search_status=[r[0] for r in res], qp_solved=[r[1] for r in res], coef=np.stack([r[2] for r in res]))

    got = plan_sharded(solve_local, sp, sv, ep, ev, n_coef=24)
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **got)
    if rank == 0:
        full = solve_local(sp, sv, ep, ev)
        np.savez(os.path.join(out_dir, "full.npz"), search_status=np.array(full["search_status"]),
                 qp_solved=np.array(full["qp_solved"]), coef=full["coef"])
    dist.destroy_process_group()


def test_shard_ranges():
    from uav_motion_planning_b200.sharding import shard_range
    assert [shard_range(5, r, 2) for r in range(2)] == [(0, 3), (3, 5)]
    assert [shard_range(4096, r, 8) for r in range(8)][-1] == (3584, 4096)
    assert [shard_range(3, r, 4) for r in range(4)] == [(0, 1), (1, 2), (2, 3), (3, 3)]   # more ranks than work
    assert shard_range(0, 0, 2) == (0, 0)


def test_all_gather_of_solved_trajectories_world2(tmp_path):
    import torch.multiprocessing as mp
    port = free_port()
    mp.spawn(worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    full = np.load(tmp_path / "full.npz")
    for r in range(2):
        got = np.load(tmp_path / f"rank{r}.npz")
        assert np.array_equal(got["search_status"], full["search_status"])
        assert np.array_equal(got["qp_solved"], full["qp_solved"])
        assert np.array_equal(got["coef"], full["coef"])          # every rank ends up with every trajectory, bit for bit
