#!/usr/bin/env python
"""bench.py — plans/sec of the batched kino-A* + minimum-snap QP hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W [--config C]   one rank per GPU (under torchrun for N > 1)
  python bench.py --impl reference [...]                       the CPU path (oracle restatement of KinoAstar::search + the
                                                               reference's own OSQP C code), all host threads, rank 0 only

--config 1 (default, BASELINE.json configs[1] — the configuration the metric is quoted on): a "step" = one pass of the hot path
over one batch of B = 4096 synthetic start->goal queries on the 50 x 50 x 10 m random-obstacle map @ 0.1 m: KinoAstar::search
(launch-file parameters, collision_check_type 1) -> S+1 waypoints -> three 8-segment 7th-order minimum-snap QPs per query.
--config 2: configs[2], 32 768 queries per step with collision_check_type 2 (ellipsoid only), same map.
--config 3: configs[3], 65 536 queries per step in TOTAL (strong scaling: each of the N ranks takes 65 536 / N), fix-wall map,
12-segment minimum snap with corridor box constraints (2 samples per segment, box = the segment's path extent +- 0.2 m).
--config 4: configs[4], QP only: 16 384 16-segment minimum-snap problems per step, eps_abs = eps_rel swept 1e-3 .. 1e-6.

Every step uses a different seeded batch.  The K timed steps are issued through the library's asynchronous entry point
(uavmp_plan_submit / uavmp_plan_wait) with up to uavmp_plan_max_in_flight() batches in flight: a batch is ONE kernel, and the
CTAs of batch k + 1 take the SM slots the long tail of batch k leaves idle (cross-batch pipelining), so the timed region is
K complete batches, first submit to last result, and nothing is skipped.  Weak scaling: every rank processes its own B
queries per step, the map is replicated, and (N > 1) the solved trajectories of every step are all-gathered with NCCL on a
side stream inside the timed region.

--dump-outputs DIR writes the last timed step's results (what uavmp_plan_submit returns to its caller) as DIR/<name>.npy, a fixed
seeded sample of the queries when they exceed 64 MB, so that two builds can be compared output for output.

Keys beyond the base contract: `roofline` (the search kernel: algorithmic bytes of SURVEY.md §8(d) over the timed region),
`cpu_baseline` (bounded sample of the same workload on the host cores), `e2e` (pinned host buffers through
uavmp_plan_submit / uavmp_plan_wait, copies inside the timed region), `clocks`, `gpu_launches`.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "plans/sec (kino-A* + min-snap QP) batched queries"
NODE_BYTES, HASH_SLOT, HEAP_SLOT = 72, 16, 4  # DESIGN.md "algorithmic bytes"

WORKLOADS = {
    1: dict(tag="configs[1]", batch=4096, map=(50.0, 50.0, 10.0), map_type=0, ctype=1, order=7, S=8, seg_time=1.0,
            text="batch 4096 queries, 50x50x10 m random map @0.1 m, kino-A* + 8-seg 7th-order min-snap, per GPU",
            kino="launch-file params, collision_check_type 1 (grid + ellipsoid)"),
    3: dict(tag="configs[3]", batch=65536, map=(50.0, 50.0, 10.0), map_type=2, ctype=1, order=7, S=12, seg_time=1.0, Kc=2, margin=0.2,
            strong=True, warm_batch=4096,
            text="batch 65536 queries, fix-wall map (two slabs, 0.5 m gap), kino-A* + 12-seg 7th-order min-snap with corridor box "
                 "constraints (2 samples per segment, box = segment path extent +- 0.2 m), sharded over the GPUs (strong scaling)",
            kino="launch-file params, collision_check_type 1 (grid + ellipsoid)"),
    2: dict(tag="configs[2]", batch=32768, map=(50.0, 50.0, 10.0), map_type=0, ctype=2, order=7, S=8, seg_time=1.0,
            text="batch 32768 queries, 50x50x10 m random map @0.1 m, SE(3) ellipsoid collision (r=0.4 h=0.1), kino-A* + 8-seg "
                 "7th-order min-snap, per GPU",
            kino="launch-file params, collision_check_type 2 (ellipsoid only)"),
}


def workload_config(wl, B, n_gpus):
    """identical on both arms (the driver compares them)"""
    corr = f", corridor rows: {wl['Kc']} samples / segment, margin {wl['margin']} m" if wl.get("Kc") else ""
    return {"workload": f"{wl['tag']}: {wl['text']}", "batch_per_gpu": B, "global_batch": B * n_gpus,
            "map": "500x500x100 int8, " + ("fix_map_type 2 (wall)" if wl["map_type"] == 2 else "random_forest seed 1"), "kino": wl["kino"],
            "qp": f"order {wl['order']}, S {wl['S']}, T_i {wl['seg_time']}, OSQP eps 1e-3, 3 axes per plan{corr}",
            "warmup_batch": wl.get("warm_batch"),
            "batches": "a different seeded query batch every step; steps may overlap in time (GPU: up to 6 batches in flight, "
                       "CPU: one work queue over all steps), every step's results are complete inside the timed region",
            "l2": "256 MiB flush write before every step; the per-step working set (>= 5 GB of search arenas + a different "
                  "query batch) exceeds the 126 MB L2",
            "parallelism": f"queries sharded x{n_gpus}, map replicated"}


def make_batches(world, B, n, rank):
    import uav_motion_planning_b200 as u
    return [u.sample_queries(world, B, seed=1000 * rank + 11 + i) for i in range(n)]


def search_bytes(c):
    """SURVEY.md §8(d) bytes_a from the search counters (summed over the batch)."""
    return (1 * c["n_occ_lookup"] + 12 * c["n_cloud_pts_tested"] + HASH_SLOT * c["n_hash_probe"] +
            (NODE_BYTES + HASH_SLOT + HEAP_SLOT) * c["n_insert"] + NODE_BYTES * c["n_update"] +
            (HEAP_SLOT + NODE_BYTES) * c["n_pop"])


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except Exception:
                continue
            for nme, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        # median over the upper half = the samples taken under load
        under = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": under[len(under) // 2] if under else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """arrays: {name: array with one row per query}; ints are written as float32, floats as float64.  Above DUMP_BYTES in all, a
    fixed seeded sample of the rows is written, with the sampled query indices as query_index.npy."""
    n = len(next(iter(arrays.values())))
    row = sum(a[0].nbytes if a.dtype.kind == "f" else 4 * a[0].size for a in arrays.values())
    if n * row > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // row, replace=False))
        arrays = dict({k: a[idx] for k, a in arrays.items()}, query_index=idx.astype(np.float64))
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(dirname, k + ".npy"), a.astype(np.float64 if a.dtype.kind == "f" else np.float32))


# ---------------------------------------------------------------------------------------------------------------
# CPU path (oracle): used ONLY by the cpu_baseline leg and by --impl reference
# ---------------------------------------------------------------------------------------------------------------
def have_cpu_path():
    """The CPU path solves its QPs with the reference's own OSQP (oracle/_ref), built only where the reference's sources exist."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    return oracle_lib.have_ref()


def cpu_plans(world, params, wl, jobs, threads):
    """Run the CPU pipeline for `jobs` = [(queries, index), ...] on `threads` host threads that pull from ONE queue in the given
    order (no barrier between steps: a long query does not idle the other threads).  Returns (wall seconds, sum of the threads'
    busy seconds, n_reached, n_solved)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    from pipeline_ref import plan_one
    order, S, seg = wl["order"], wl["S"], wl["seg_time"]
    oracles = [oracle_lib.KinoOracle(world, params) for _ in range(threads)]
    oracle_lib.minctrl_solve(order, S, np.arange(S + 1.0), [0, 0], [0, 0], np.ones(S), bound_jerk=[0, 0])  # dlopen
    nxt, lock, res, busy = [0], threading.Lock(), [], [0.0] * threads

    def work(t):
        o = oracles[t]
        while True:
            with lock:
                k = nxt[0]
                nxt[0] += 1
            if k >= len(jobs):
                return
            (sp, sv, ep, ev), q = jobs[k]
            t0 = time.perf_counter()
            r = plan_one(o, sp[q], sv[q], ep[q], ev[q], order, S, seg, n_corridor=wl.get("Kc", 0), margin=wl.get("margin", 0.0))[:2]
            busy[t] += time.perf_counter() - t0
            res.append(r)

    t0 = time.perf_counter()
    ts = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    dt = time.perf_counter() - t0
    for o in oracles:
        o.close()
    return dt, sum(busy), sum(1 for s, _ in res if s == 1), sum(1 for _, k in res if k)


def lpt_jobs(batches, n_s):
    """The first n_s queries of every batch, longest straight-line distance first within a batch (the order the GPU path uses)."""
    jobs = []
    for bt in batches:
        d = np.linalg.norm(bt[0][:n_s] - bt[2][:n_s], axis=1)
        jobs += [(bt, int(q)) for q in np.argsort(-d, kind="stable")]
    return jobs


def kind_of_cpu_path():
    return ("port", "search: oracle/kino_ref.cpp (restatement, pinned against the reference's kino_astar.cpp compiled in "
            "oracle/_ref when that is built); QP: the reference's vendored OSQP C core compiled unmodified (oracle/_ref) + "
            "restated QDLDL")


def cpu_summary(n, wall, busy, threads):
    return {"plans_per_s_makespan": n / wall, "plans_per_s_busy": n * threads / busy if busy > 0 else None,
            "thread_busy_frac": busy / (wall * threads), "cpu_model": cpu_model()}


def run_reference(args, rank, world_size, wl):
    if rank != 0:
        return
    if not have_cpu_path():
        raise SystemExit("bench.py --impl reference: oracle/_ref/libosqp_ref.so (the reference's OSQP) is not built")
    import uav_motion_planning_b200 as u
    from uav_motion_planning_b200 import _lib
    world = u.make_world(*wl["map"], seed=1, map_type=wl["map_type"])  # host-only input generator (libuavmp_worldgen.so)
    params = _lib.launch_params(collision_check_type=wl["ctype"])
    threads = os.cpu_count() or 1
    # bounded sample: n_s queries of every step's batch, sized so that K steps are ~2-3 minutes of wall time on the host
    # (mean cost ~0.9 core-seconds per query, p99.9 ~60 core-seconds: one queue over all steps keeps the tail amortised)
    n_s = args.cpu_sample or int(min(wl["batch"], max(2 * threads, (150.0 * threads / 0.9) // max(args.steps, 1))))
    batches = make_batches(world, wl["batch"], args.steps + args.warmup, 0)
    if args.warmup:
        cpu_plans(world, params, wl, lpt_jobs(batches[:1], min(n_s, 2 * threads)), threads)
    jobs = lpt_jobs(batches[args.warmup:], n_s)
    wall, busy, reached, _ = cpu_plans(world, params, wl, jobs, threads)
    cnt = len(jobs)
    val = cnt / wall
    kind, how = kind_of_cpu_path()
    sample = (f"first {n_s} queries of each step's {wl['batch']}-query batch ({args.steps} steps = {cnt} plans), {threads} "
              f"threads pulling from one queue (longest straight-line distance first within a step); {how}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "plans/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / max(args.steps, 1) * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(wl, wl["batch"], args.gpus),
        "cpu_baseline": dict({"value": val, "unit": "plans/s", "cores": threads, "kind": kind, "sample": sample,
                              "reach_end_frac": reached / cnt}, **cpu_summary(cnt, wall, busy, threads)),
        "e2e": {"value": val, "unit": "plans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ---------------------------------------------------------------------------------------------------------------
def run_gpu(args, rank, world_size, local_rank, wl):
    import torch
    import torch.distributed as dist
    import uav_motion_planning_b200 as u
    from uav_motion_planning_b200 import planner

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference "
                         "for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world_size > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = u.Context(local_rank)
    strong = bool(wl.get("strong")) and not args.batch
    B, K, W = args.batch or (wl["batch"] // world_size if strong else wl["batch"]), args.steps, args.warmup
    order, S, seg = wl["order"], wl["S"], wl["seg_time"]
    n = (order + 1) * S
    opts = planner.plan_options(order=order, S=S, seg_time=seg, corridor_samples=wl.get("Kc", 0), corridor_margin=wl.get("margin", 0.0))
    world = u.make_world(*wl["map"], seed=1, map_type=wl["map_type"])
    ka = u.KinoAstar(ctx)
    ka.setLaunchParams()
    ka.setParam(collision_check_type=wl["ctype"])
    ka.setGridMap(world)
    if strong:  # one global batch per step, cut into contiguous shards (sharding.shard_range): rank r works on its own slice
        from uav_motion_planning_b200.sharding import shard_range
        lo_q, hi_q = shard_range(wl["batch"], rank, world_size)
        batches = [tuple(a[lo_q:hi_q] for a in bt) for bt in make_batches(world, wl["batch"], K + W, 0)]
    else:
        batches = make_batches(world, B, K + W, rank)
    if wl.get("warm_batch") and not args.batch:
        # the W warm-up steps of this configuration use a smaller batch (its full batch is minutes of work: wall-crossing queries
        # exhaust the 100 000-node pool); the K timed steps are full size
        wb = max(1, wl["warm_batch"] // world_size)
        batches = [tuple(a[:wb] for a in bt) if i < W else bt for i, bt in enumerate(batches)]
    depth = planner.max_in_flight(ctx)
    lib_stream = torch.cuda.ExternalStream(ctx.stream, device=dev)  # the context's stream: device inputs are ordered after it
    side = torch.cuda.Stream(device=dev)                            # all-gathers run here, behind each batch's completion

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # every tensor is allocated on torch's default stream (nothing the caching allocator tracks lives on the library's streams)
    d_in = [[torch.from_numpy(a).to(dev) for a in bt] for bt in batches]  # resident in HBM before timing
    ring = [dict(status=torch.zeros(B, dtype=torch.int32, device=dev), solved=torch.zeros(B, dtype=torch.int32, device=dev),
                 coef=torch.zeros(B, 3 * n, dtype=torch.float64, device=dev)) for _ in range(depth)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    if world_size > 1:
        for r in ring:
            r["g_coef"] = torch.empty(world_size * B, 3 * n, dtype=torch.float64, device=dev)
            r["g_solved"] = torch.empty(world_size * B, dtype=torch.int32, device=dev)
            r["gathered"] = torch.cuda.Event()
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h_in = [[pin(a) for a in bt] for bt in batches]
    h_ring = [dict(status=torch.zeros(B, dtype=torch.int32).pin_memory(), solved=torch.zeros(B, dtype=torch.int32).pin_memory(),
                   coef=torch.zeros(B, 3 * n, dtype=torch.float64).pin_memory()) for _ in range(depth)]
    torch.cuda.synchronize()

    def gather(r, src_coef, src_solved):
        """"all-gather of solved trajectories only", on the side stream, ordered behind the batch that produced them"""
        with torch.cuda.stream(side):
            dist.all_gather_into_tensor(r["g_coef"], src_coef)
            dist.all_gather_into_tensor(r["g_solved"], src_solved)
            r["gathered"].record(side)

    def run_steps(first, count, host_io):
        """`count` batches through submit / wait with `depth` in flight; returns the uavmp_plan_info of every batch"""
        live, infos = [], []
        for i in range(first, first + count):
            slot = (i - first) % depth
            if len(live) == depth:
                infos.append(planner.plan_wait(ctx, live.pop(0)))
            with torch.cuda.stream(lib_stream):
                flush.fill_(i & 0xff)  # evict the previous steps' working set from L2 (ordered before this batch)
                if world_size > 1 and i - first >= depth:
                    lib_stream.wait_event(ring[slot]["gathered"])  # the ring entry is free once its gather has read it
            if host_io:
                sp, sv, ep, ev = h_in[i]
                o = h_ring[slot]
            else:
                sp, sv, ep, ev = d_in[i]
                o = ring[slot]
            t = planner.plan_submit(ctx, int(sp.shape[0]), sp.data_ptr(), sv.data_ptr(), ep.data_ptr(), ev.data_ptr(), o["status"].data_ptr(),
                                    o["solved"].data_ptr(), o["coef"].data_ptr(), device_io=not host_io, options=opts)
            live.append(t)
            if world_size > 1:
                if host_io:  # results land in pinned host memory: they go back up for the gather once the batch is complete
                    planner.plan_stream_wait(ctx, t, side.cuda_stream)
                    with torch.cuda.stream(side):
                        ring[slot]["coef"].copy_(o["coef"], non_blocking=True)
                        ring[slot]["solved"].copy_(o["solved"], non_blocking=True)
                else:
                    planner.plan_stream_wait(ctx, t, side.cuda_stream)
                gather(ring[slot], ring[slot]["coef"], ring[slot]["solved"])
        while live:
            infos.append(planner.plan_wait(ctx, live.pop(0)))
        side.synchronize()
        return infos

    # ---- value: inputs resident in HBM --------------------------------------------------------------------------
    run_steps(0, W, False)
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(lib_stream)          # the first batch is ordered after this event
    t0 = time.perf_counter()
    infos = run_steps(W, K, False)  # returns when every batch (and gather) of the K steps is complete
    e1.record(lib_stream)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    ms = e0.elapsed_time(e1)
    last = ring[(K - 1) % depth]
    reached = int((last["status"] == 1).sum().item())
    solved = int(last["solved"].sum().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"plan_status": last["status"].cpu().numpy(), "qp_solved": last["solved"].cpu().numpy(),
                                         "coef": last["coef"].cpu().numpy()})
    bytes_a = [search_bytes(i["counters"]) for i in infos]
    pops = [i["counters"]["n_pop"] for i in infos]
    launch_ms = [i["timings"]["search_ms"] for i in infos]
    launches = sum(i["timings"]["search_launches"] + i["timings"]["qp_launches"] + i["timings"]["aux_launches"] for i in infos)
    flags = [i["error_flags"] for i in infos]

    # ---- e2e: pinned host buffers through uavmp_plan_submit / wait, copies inside the timed region ----------------
    run_steps(0, min(W, 2), True)
    barrier()
    t0 = time.perf_counter()
    run_steps(W, K, True)
    barrier()
    e2e_s = time.perf_counter() - t0
    clk = clocks.stop() if rank == 0 else None

    t_ms = torch.tensor([ms, e2e_s * 1e3, wall_ms], dtype=torch.float64, device=dev)
    if world_size > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms, e2e_ms, wall_ms = t_ms.tolist()
    total_q = B * world_size * K
    value = total_q / (ms / 1e3)
    e2e_val = total_q / (e2e_ms / 1e3)

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        # the K launches overlap each other (that is the point): the kernel's achieved rate is all their algorithmic bytes over
        # the timed region; `launch_ms_mean` is the CUDA-event duration of one launch on its own stream, neighbours included
        achieved = float(np.sum(bytes_a)) / (ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("kino_search_kernel_dram_bytes_per_launch")
        out = {
            "metric": METRIC, "value": value, "unit": "plans/s", "n_gpus": world_size, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(wl, B, world_size),
            "execution": f"uavmp_plan_submit / uavmp_plan_wait, {depth} batches in flight; the QP of a query is solved inside the search "
                         "kernel by the CTA that finished it (one warp per 1-D problem)",
            "e2e": {"value": e2e_val, "unit": "plans/s", "h2d_bytes_per_step": B * 12 * 8,
                    "d2h_bytes_per_step": B * (3 * n * 8 + 8), "ms_per_step": e2e_ms / K},
            "gpu_launches": int(launches),
            "roofline": {"kernel": "kino_search_kernel (search + in-kernel QP)", "bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "kernel_ms": ms / K, "launch_ms_mean": float(np.mean(launch_ms)),
                         "launches_overlapping": float(np.mean(launch_ms)) / (ms / K),
                         "kernel_share_of_step": 1.0,
                         "algorithmic_bytes_per_launch": float(np.mean(bytes_a)),
                         "expansions_per_s": float(np.sum(pops)) / (ms * 1e-3),
                         "qp": {"problems_per_s": 3.0 * solved / B * total_q / world_size / (ms * 1e-3),
                                "algorithmic_bytes_per_problem": 8 * ((S + 1) + 6 + S) + 8 * n,
                                "note": "on-chip (one warp per problem, workspace in shared memory): the QP's HBM traffic is its "
                                        "inputs and outputs only"}},
            "clocks": clk, "wall_ms_per_step": wall_ms / K,
            "result_check": {"reach_end_frac_last_step": reached / B, "qp_solved_frac_last_step": solved / B,
                             "error_flags": int(np.bitwise_or.reduce(flags))},
        }
        if world_size == 1 and not args.no_cpu and not have_cpu_path():
            out["cpu_baseline"] = {"unavailable": "oracle/_ref/libosqp_ref.so (the reference's OSQP) is not built"}
        elif world_size == 1 and not args.no_cpu:
            threads = os.cpu_count() or 1
            n_s = args.cpu_sample or min(B, 16 * threads)  # ~15 s of host time at ~0.9 core-seconds per query
            jobs = lpt_jobs([batches[W]], n_s)
            wall, busy, _, _ = cpu_plans(world, ka.params, wl, jobs, threads)
            kind, how = kind_of_cpu_path()
            out["cpu_baseline"] = dict({"value": len(jobs) / wall, "unit": "plans/s", "cores": threads, "kind": kind,
                                        "sample": f"first {n_s} queries of the first timed batch, {threads} threads pulling "
                                                  f"from one queue; {how}"}, **cpu_summary(len(jobs), wall, busy, threads))
        print(json.dumps(out), flush=True)
    # Orderly teardown: tensors first, then NCCL, then the library context (its streams die with it).
    del d_in, ring, flush, h_in, h_ring
    torch.cuda.synchronize()
    if world_size > 1:
        dist.barrier()
        dist.destroy_process_group()
    del lib_stream
    ka = None
    ctx.sync()
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------
def run_qp_sweep(args, rank, world_size, local_rank):
    """configs[4]: the solver-bound regime.  16 384 one-dimensional 16-segment minimum-snap QPs per step, random-walk waypoints,
    T_i ~ U(0.5, 2), eps_abs = eps_rel in {1e-3, 1e-4, 1e-5, 1e-6}, adaptive_rho_interval 100 (SURVEY.md §8(d) config 5)."""
    import torch
    import uav_motion_planning_b200 as u
    from uav_motion_planning_b200.minimum_control import MinimumControl, default_settings
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device")
    if rank != 0:
        return
    torch.cuda.set_device(local_rank)
    ctx = u.Context(local_rank)
    B, S, order = args.batch or 16384, 16, 7
    K, W = args.steps, args.warmup
    mc = MinimumControl(ctx, order=order)
    rng = np.random.default_rng(5)
    z = np.zeros((B, 2))
    sweep = []
    clocks = ClockSampler(local_rank)
    clocks.start()
    for eps in (1e-3, 1e-4, 1e-5, 1e-6):
        st = default_settings(eps_abs=eps, eps_rel=eps, adaptive_rho_interval=100)
        ms, iters, solved = [], [], []
        for i in range(W + K):
            pos = np.cumsum(rng.normal(size=(B, S + 1)), axis=1)
            T = rng.uniform(0.5, 2.0, size=(B, S))
            r = mc.solve_batch(pos, z, z, T, bound_jerk=z, settings=st)
            if i >= W:
                ms.append(ctx.timings()["qp_ms"]); iters.append(float(r["iters"].mean())); solved.append(float(r["solved"].mean()))
        sweep.append({"eps": eps, "kernel_ms": float(np.mean(ms)), "problems_per_s": B / (np.mean(ms) * 1e-3),
                      "iters_mean": float(np.mean(iters)), "qp_iters_per_s": B * np.mean(iters) / (np.mean(ms) * 1e-3),
                      "solved_frac": float(np.mean(solved))})
    clk = clocks.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: r[k] for k in ("coef", "iters", "status", "solved")})
    base = sweep[0]
    # SURVEY.md §8(d): flops per ADMM iteration ~ 4 nnz(L) + 2 nnz(A) + 12 (n + m); order 7, S 16: nnzL 1201, nnzA 786, n 128, m 83
    nnzL, nnzA, nq, mq = 1201, 786, 128, 83
    flops_iter = 4 * nnzL + 2 * nnzA + 12 * (nq + mq)
    smem_iter = 2 * nnzL * 16 + 12 * (nq + mq) * 8  # bytes the two triangular solves and the vector passes move per iteration
    peak_hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
    io_bytes = 8 * ((S + 1) + 6 + S) + 8 * (order + 1) * S
    out = {"metric": "QP problems/sec (16-seg min-snap, one axis), ADMM sweep", "value": base["problems_per_s"], "unit": "problems/s",
           "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": base["kernel_ms"], "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": "configs[4]: ADMM iteration sweep, 16-seg 7th-order min-snap, eps_abs = eps_rel 1e-3 -> 1e-6, batch "
                                  f"{B}, 1xB200 (solver-bound regime); random-walk waypoints N(0,1), T_i U(0.5,2), adaptive_rho_interval 100",
                      "batch_per_gpu": B}, "sweep": sweep,
           "roofline": {"kernel": "qp_solve_warp_kernel (one warp per problem, whole workspace in shared memory; UAVMP_QP_THREAD=1 selects "
                                  "the thread-per-problem kernel)", "bound": "hbm",
                        "achieved": B * io_bytes / (base["kernel_ms"] * 1e-3) / 1e9, "peak": peak_hbm, "unit": "GB/s", "traffic": None,
                        "algorithmic_bytes_per_problem": io_bytes,
                        "note": "on-chip kernel: HBM carries inputs and outputs only, so the HBM fraction says nothing about it; it is bound "
                                "by the latency of the dependent chains of the sparse triangular solves (2 x ~100 elimination-tree levels "
                                "per ADMM iteration), see fp64 / smem below",
                        "fp64": {"achieved_gflops": [s_["qp_iters_per_s"] * flops_iter / 1e9 for s_ in sweep],
                                 "flops_per_iteration": flops_iter, "peak_gflops_nominal": 37000.0,
                                 "frac": [s_["qp_iters_per_s"] * flops_iter / 1e9 / 37000.0 for s_ in sweep]},
                        "smem": {"achieved_gbs": [s_["qp_iters_per_s"] * smem_iter / 1e9 for s_ in sweep], "bytes_per_iteration": smem_iter,
                                 "peak_gbs_nominal": 148 * 128 * 1.965, "frac": [s_["qp_iters_per_s"] * smem_iter / 1e9 / (148 * 128 * 1.965) for s_ in sweep]}},
           "clocks": clk, "gpu_launches": 4 * (K + W)}
    out["roofline"]["frac"] = out["roofline"]["achieved"] / out["roofline"]["peak"]
    print(json.dumps(out), flush=True)
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 3, 4], help="BASELINE.json configs[N] (default 1: the metric's)")
    ap.add_argument("--batch", type=int, default=0, help="queries per GPU per step (0: the configuration's own)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="queries per step in the CPU sample (0: auto)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.config == 4:
        if args.impl == "reference":
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "configs[4] is a kernel sweep; the reference arm times configs[1]"}))
            return
        return run_qp_sweep(args, rank, world_size, local_rank)
    wl = WORKLOADS[args.config]
    if args.impl == "reference":
        run_reference(args, rank, world_size, wl)
    else:
        run_gpu(args, rank, world_size, local_rank, wl)


if __name__ == "__main__":
    main()
