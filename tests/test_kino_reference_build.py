"""Pins the search oracle to the reference itself: oracle/_ref/libkino_ref.so is /root/reference's own
src/planner/path_searching/src/kino_astar.cpp compiled UNMODIFIED (against the header shims in oracle/shim/, recipe in
oracle/Makefile), driven through oracle/kino_ref_driver.cpp.  The restatement oracle/kino_ref.cpp (glibc libm mode, like a
reference build) must agree with it on

  * the return code and KinoAstar::use_node_num_,
  * every point search() appended to `path`, bit for bit,
  * a digest of every position the search passed to GridMap::isInMap, in call order — every expansion tests the popped node's
    own position first (t = 0) and then every checkpoint of every primitive, so equal digests mean equal ordered expansion
    sequences with bit-identical states,

for the golden queries (whose expected values tests/golden/kino_golden.json holds) and for > 150 random queries on both
collision types, the code-default parameters, a pool small enough to hit "reach max node num", and the wall map.  Where
oracle/_ref is not built, the recorded results of that build stand in for it (tests/ref_record.py).
What stays restated (oracle/shim/Eigen/Eigen) is Eigen's floating-point association (SURVEY.md §9.1's contract).
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

import oracle_lib
import ref_record
import uav_motion_planning_b200 as u
from uav_motion_planning_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "libkino_ref.so")
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "kino_golden.json")))


class RefParams(C.Structure):
    _fields_ = [("allocated_node_num", C.c_int), ("collision_check_type", C.c_int)] + \
        [(n, C.c_double) for n in ("rou_time", "lambda_heu", "goal_tolerance", "time_step_size", "max_velocity",
                                   "max_acceleration", "acc_resolution", "sample_tau", "robot_r", "robot_h")]


class RefResult(C.Structure):
    _fields_ = [("status", C.c_int), ("use_node_num", C.c_int), ("n_path", C.c_int), ("pad", C.c_int),
                ("lookup_digest", C.c_uint64), ("n_in_map_calls", C.c_longlong), ("n_occ_lookup", C.c_longlong)]


class ReferenceKino:
    def __init__(self, world, p):
        rp = RefParams(p.allocated_node_num, p.collision_check_type, p.rou_time, p.lambda_heu, p.goal_tolerance, p.time_step_size,
                       p.max_velocity, p.max_accelration, p.acc_resolution, p.sample_tau, p.robot_r, p.robot_h)
        self.occ = np.ascontiguousarray(world.occ, np.int8)
        self.cloud = np.ascontiguousarray(world.cloud, np.float32)
        origin, msz = np.ascontiguousarray(world.origin, np.float64), np.ascontiguousarray(world.map_size, np.float64)
        self.key = ref_record.digest(rp, self.occ, self.cloud, world.dims, origin, msz, world.resolution)
        self.lib = self.h = None
        if os.path.exists(LIB):
            self.lib = C.CDLL(LIB)
            self.lib.refkino_create.restype = C.c_void_p
            self.lib.refkino_create.argtypes = [C.POINTER(RefParams), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                                C.c_double, C.c_void_p, C.c_int]
            self.lib.refkino_search.argtypes = [C.c_void_p] + [C.c_void_p] * 4 + [C.POINTER(RefResult), C.c_void_p, C.c_int]
            self.lib.refkino_destroy.argtypes = [C.c_void_p]
            self.h = self.lib.refkino_create(C.byref(rp), self.occ.ctypes.data, *world.dims, origin.ctypes.data, msz.ctypes.data,
                                             world.resolution, self.cloud.ctypes.data, len(self.cloud))

    def search(self, sp, sv, ep, ev, path_cap=4096, like=None):
        sp, sv, ep, ev = (np.ascontiguousarray(a, np.float64) for a in (sp, sv, ep, ev))

        def live():
            res = RefResult()
            path = np.zeros((path_cap, 3))
            self.lib.refkino_search(self.h, sp.ctypes.data, sv.ctypes.data, ep.ctypes.data, ev.ctypes.data, C.byref(res),
                                    path.ctypes.data, path_cap)
            return dict(status=res.status, use_node_num=res.use_node_num, n_path=res.n_path, path=path[:res.n_path].copy(),
                        lookup_digest=res.lookup_digest, n_in_map_calls=res.n_in_map_calls)

        return ref_record.call("refkino_search", live if self.lib else None, (self.key, sp, sv, ep, ev, path_cap),
                               like=None if like is None else {"path": like["path"]})

    def close(self):
        if self.lib:
            self.lib.refkino_destroy(self.h)


def params(launch=True, **kw):
    p = _lib.KinoParams(**(_lib.LAUNCH_PARAMS if launch else _lib.DEFAULT_PARAMS))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def agree(ref, orc, q):
    b = orc.search(*q)
    a = ref.search(*q, like=b)
    assert (a["status"], a["use_node_num"], a["n_path"]) == (b["status"], b["use_node_num"], b["n_path"]), (a, b)
    assert a["n_in_map_calls"] == b["n_in_map_calls"] and a["lookup_digest"] == b["lookup_digest"]
    assert np.array_equal(a["path"].view(np.uint64), b["path"].view(np.uint64))
    return b


@pytest.mark.parametrize("case", GOLD[:5], ids=lambda c: c["name"])
def test_reference_build_reproduces_the_golden_vectors(case):
    """The goldens were generated by the restatement in fpmath mode; the reference build (glibc libm) must give the same
    status / use_node_num / path length on them and agree with the restatement in glibc mode bit for bit."""
    world = u.make_world(*case["dims"], seed=case["map_seed"], map_type=case["map_type"])
    p = params(case["launch_params"], collision_check_type=case["collision_check_type"])
    if case["allocated_node_num"]:
        p.allocated_node_num = case["allocated_node_num"]
    ref, orc = ReferenceKino(world, p), oracle_lib.KinoOracle(world, p, libm_mode=1)
    same = 0
    queries = case["queries"][:2] if case["name"].startswith("wall") else case["queries"]   # wall searches exhaust the pool: ~15 s each
    for q in queries:
        b = agree(ref, orc, (q["start_pt"], q["start_vel"], q["end_pt"], q["end_vel"]))
        assert b["status"] == q["status"]
        same += int((b["use_node_num"], b["n_pop"], b["n_path"]) == (q["use_node_num"], q["n_pop"], q["n_path"]))
    assert same >= len(queries) - 1   # glibc vs fpmath: <= 1 ulp in cbrt / acos / cos may move one search (documented)
    ref.close()


@pytest.mark.parametrize("name,dims,map_type,launch,kw,n,seed", [
    ("type1", (20, 20, 5), 0, True, dict(collision_check_type=1), 80, 101),
    ("type2", (20, 20, 5), 0, True, dict(collision_check_type=2), 40, 102),
    ("defaults", (20, 20, 5), 0, False, dict(), 20, 103),
    ("pool3000", (20, 20, 5), 0, True, dict(allocated_node_num=3000), 12, 104),
    ("wall", (20, 20, 5), 2, True, dict(allocated_node_num=20000), 6, 105),
])
def test_reference_build_agrees_with_the_restatement(name, dims, map_type, launch, kw, n, seed):
    world = u.make_world(*dims, seed=1, map_type=map_type)
    p = params(launch, **kw)
    ref, orc = ReferenceKino(world, p), oracle_lib.KinoOracle(world, p, libm_mode=1)
    sp, sv, ep, ev = u.sample_queries(world, n, seed=seed, min_dist=8.0)
    sv[::3, 0] = 0.7   # some non-zero start velocities
    st = [agree(ref, orc, (sp[q], sv[q], ep[q], ev[q]))["status"] for q in range(n)]
    assert 1 in st
    if name == "pool3000":
        assert 2 in st
    ref.close()
