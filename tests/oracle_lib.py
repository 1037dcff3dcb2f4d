"""ctypes binding of oracle/liboracle.so — the CPU checker.  Imported by tests/, smoke() and bench.py's CPU legs only."""
import ctypes as C
import os
import subprocess

import numpy as np

import ref_record

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB = os.path.join(ORACLE_DIR, "liboracle.so")


class KinoParams(C.Structure):
    _fields_ = [("allocated_node_num", C.c_int), ("collision_check_type", C.c_int)] + \
        [(n, C.c_double) for n in ("rou_time", "lambda_heu", "goal_tolerance", "time_step_size", "max_velocity",
                                   "max_acceleration", "acc_resolution", "sample_tau", "robot_r", "robot_h")] + \
        [("libm_mode", C.c_int)]


class Counters(C.Structure):
    _fields_ = [(n, C.c_longlong) for n in ("n_pop", "n_occ_lookup", "n_cloud_pts_tested", "n_hash_probe", "n_insert",
                                            "n_update", "n_heuristic", "n_shot", "heap_len_sum")]


class Result(C.Structure):
    _fields_ = [("status", C.c_int), ("use_node_num", C.c_int), ("n_pop", C.c_int), ("n_path", C.c_int),
                ("n_path_nodes", C.c_int), ("shot_duration", C.c_double), ("pop_hash", C.c_uint64),
                ("counters", Counters), ("lookup_digest", C.c_uint64), ("n_in_map_calls", C.c_longlong)]


_lib = None


def build():
    subprocess.run(["make", "-C", ORACLE_DIR], check=True, capture_output=True)


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            build()
        lib = C.CDLL(LIB)
        lib.oracle_kino_create.restype = C.c_void_p
        lib.oracle_kino_create.argtypes = [C.POINTER(KinoParams), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_double, C.c_void_p, C.c_int]
        lib.oracle_kino_destroy.argtypes = [C.c_void_p]
        lib.oracle_kino_search.argtypes = [C.c_void_p] + [C.c_void_p] * 4 + [C.POINTER(Result), C.c_void_p, C.c_int,
                                                                            C.c_void_p, C.c_int]
        lib.oracle_fp_eval_n.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_longlong]
        _lib = lib
    return _lib


def params_from(p, libm_mode=0):
    """uav_motion_planning_b200.KinoParams (or any object with the same fields) -> oracle params."""
    return KinoParams(p.allocated_node_num, p.collision_check_type, p.rou_time, p.lambda_heu, p.goal_tolerance,
                      p.time_step_size, p.max_velocity, p.max_accelration, p.acc_resolution, p.sample_tau, p.robot_r,
                      p.robot_h, libm_mode)


class KinoOracle:
    def __init__(self, world, params, libm_mode=0):
        self.lib = load()
        kp = params_from(params, libm_mode)
        self.occ = np.ascontiguousarray(world.occ, np.int8)
        self.cloud = np.ascontiguousarray(world.cloud, np.float32)
        origin = np.ascontiguousarray(world.origin, np.float64)
        msz = np.ascontiguousarray(world.map_size, np.float64)
        self.h = self.lib.oracle_kino_create(C.byref(kp), self.occ.ctypes.data, *world.dims, origin.ctypes.data,
                                             msz.ctypes.data, world.resolution, self.cloud.ctypes.data,
                                             len(self.cloud))

    def search(self, sp, sv, ep, ev, path_cap=4096, pop_cap=0):
        sp, sv, ep, ev = (np.ascontiguousarray(a, np.float64) for a in (sp, sv, ep, ev))
        res = Result()
        path = np.zeros((path_cap, 3))
        trace = np.zeros((max(pop_cap, 1), 3), np.int32)
        self.lib.oracle_kino_search(self.h, sp.ctypes.data, sv.ctypes.data, ep.ctypes.data, ev.ctypes.data,
                                    C.byref(res), path.ctypes.data, path_cap, trace.ctypes.data if pop_cap else None,
                                    pop_cap)
        c = res.counters
        return dict(status=res.status, use_node_num=res.use_node_num, n_pop=res.n_pop, pop_hash=res.pop_hash,
                    path=path[:min(res.n_path, path_cap)].copy(), n_path=res.n_path,
                    trace=trace[:min(res.n_pop, pop_cap)].copy(), lookup_digest=res.lookup_digest,
                    n_in_map_calls=res.n_in_map_calls,
                    counters={k: getattr(c, k) for k, _ in Counters._fields_})

    def close(self):
        if self.h:
            self.lib.oracle_kino_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def fp_eval(op, x, n_pow=0):
    lib = load()
    x = np.ascontiguousarray(x, np.float64)
    y = np.zeros_like(x)
    lib.oracle_fp_eval_n(op, x.ctypes.data, n_pow, y.ctypes.data, x.size)
    return y


# ---- QP side ---------------------------------------------------------------------------------------------------
class OsqpSettings(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("rho", "sigma", "alpha", "eps_abs", "eps_rel", "eps_prim_inf",
                                          "eps_dual_inf")] + \
        [(n, C.c_int) for n in ("max_iter", "check_termination", "scaling", "adaptive_rho", "adaptive_rho_interval")] + \
        [("adaptive_rho_tolerance", C.c_double), ("want_scaling_dump", C.c_int), ("dump_D", C.c_void_p),
         ("dump_E", C.c_void_p)]


class OsqpInfo(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("setup_flag", "solve_flag", "status_val", "iter", "rho_updates",
                                       "adaptive_rho_interval_used")] + \
        [(n, C.c_double) for n in ("rho_final", "prim_res", "dual_res", "obj_val", "scaling_c")]


def osqp_settings(**kw):
    """What MinimumControl::solve runs OSQP with (minimum_control.cpp:160-162 over osqp_api_constants.h:96-153)."""
    s = OsqpSettings(0.1, 1e-6, 1.6, 1e-3, 1e-3, 1e-3, 1e-4, 1000, 25, 10, 1, 0, 5.0, 0, None, None)
    for k, v in kw.items():
        setattr(s, k, v)
    return s


_have_ref = None


def have_ref():
    """True when oracle/_ref/libosqp_ref.so (the reference's OSQP) is built; otherwise the QP calls below answer from the record
    (tests/ref_record.py)."""
    global _have_ref
    if _have_ref is None:
        _have_ref = bool(load().oracle_have_ref())
    return _have_ref


def info_dict(info):
    return {k: getattr(info, k) for k, _ in OsqpInfo._fields_}


def _f(a):
    return None if a is None else np.ascontiguousarray(a, np.float64)


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def minctrl_solve(order, S, pos_1d, bound_vel, bound_acc, T, bound_jerk=None, settings=None, libm_mode=0,
                  corridor_lo=None, corridor_hi=None, n_corridor=0, like=None):
    """n_corridor > 0: the corridor extension (SURVEY.md §9.3) — corridor_lo / corridor_hi hold one box per segment.
    like: the coefficients the caller compares the result with (ref_record.call)."""
    lib = load()
    st = settings or osqp_settings()
    pos_1d, bound_vel, bound_acc, bound_jerk, T = _f(pos_1d), _f(bound_vel), _f(bound_acc), _f(bound_jerk), _f(T)
    lo, hi = _f(corridor_lo), _f(corridor_hi)

    def live():
        coef = np.zeros((order + 1) * S)
        info = OsqpInfo()
        lib.oracle_minctrl_solve_c.argtypes = [C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 7 + [C.POINTER(OsqpSettings), C.c_int,
                                                                                              C.c_void_p, C.POINTER(OsqpInfo)]
        ok = lib.oracle_minctrl_solve_c(order, S, n_corridor, _p(pos_1d), _p(bound_vel), _p(bound_acc), _p(bound_jerk), _p(T),
                                        _p(lo), _p(hi), C.byref(st), libm_mode, _p(coef), C.byref(info))
        if ok < 0:
            raise RuntimeError("oracle/_ref/libosqp_ref.so is not available")
        return dict(ok=ok, coef=coef, info=info_dict(info))

    r = ref_record.call("minctrl_solve", live if have_ref() else None,
                        (order, S, n_corridor, pos_1d, bound_vel, bound_acc, bound_jerk, T, lo, hi, st, libm_mode),
                        like=None if like is None else {"coef": like})
    return r["ok"], r["coef"], r["info"]


def minctrl_assemble(order, S, pos_1d, bound_vel, bound_acc, T, bound_jerk=None, libm_mode=0):
    lib = load()
    n, m, nnzP, nnzA = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    lib.oracle_minctrl_dims(order, S, C.byref(n), C.byref(m), C.byref(nnzP), C.byref(nnzA))
    n, m, nnzP, nnzA = n.value, m.value, nnzP.value, nnzA.value
    pos_1d, bound_vel, bound_acc, bound_jerk, T = _f(pos_1d), _f(bound_vel), _f(bound_acc), _f(bound_jerk), _f(T)
    Pp, Pi, Px = np.zeros(n + 1, np.int64), np.zeros(nnzP, np.int64), np.zeros(nnzP)
    Ap, Ai, Ax = np.zeros(n + 1, np.int64), np.zeros(nnzA, np.int64), np.zeros(nnzA)
    q, l, u = np.zeros(n), np.zeros(m), np.zeros(m)
    lib.oracle_minctrl_assemble.argtypes = [C.c_int, C.c_int] + [C.c_void_p] * 5 + [C.c_int] + [C.c_void_p] * 9
    lib.oracle_minctrl_assemble(order, S, _p(pos_1d), _p(bound_vel), _p(bound_acc), _p(bound_jerk), _p(T), libm_mode,
                                _p(Pp), _p(Pi), _p(Px), _p(q), _p(Ap), _p(Ai), _p(Ax), _p(l), _p(u))
    return dict(n=n, m=m, Pp=Pp, Pi=Pi, Px=Px, q=q, Ap=Ap, Ai=Ai, Ax=Ax, l=l, u=u)


def _csc(M):
    i64 = lambda a: np.ascontiguousarray(a, np.int64)
    return i64(M.indptr), i64(M.indices), np.ascontiguousarray(M.data, np.float64)


def osqp_solve(P_triu_csc, q, A_csc, l, u, settings=None):
    """Generic QP through the reference's OSQP (scipy CSC inputs)."""
    lib = load()
    st = settings or osqp_settings(eps_prim_inf=1e-4, max_iter=4000)
    n, m = P_triu_csc.shape[0], A_csc.shape[0]
    Pp, Pi, Px = _csc(P_triu_csc)
    Ap, Ai, Ax = _csc(A_csc)
    q, l, u = _f(q), _f(l), _f(u)

    def live():
        x, y = np.zeros(n), np.zeros(max(m, 1))
        info = OsqpInfo()
        lib.oracle_osqp_solve.argtypes = [C.c_longlong, C.c_longlong] + [C.c_void_p] * 9 + \
            [C.POINTER(OsqpSettings), C.c_void_p, C.c_void_p, C.POINTER(OsqpInfo)]
        rc = lib.oracle_osqp_solve(n, m, _p(Pp), _p(Pi), _p(Px), _p(q), _p(Ap), _p(Ai), _p(Ax), _p(l), _p(u),
                                   C.byref(st), _p(x), _p(y), C.byref(info))
        if rc < 0:
            raise RuntimeError("oracle/_ref/libosqp_ref.so is not available")
        return dict(x=x, y=y[:m], info=info_dict(info))

    r = ref_record.call("osqp_solve", live if have_ref() else None, (n, m, Pp, Pi, Px, q, Ap, Ai, Ax, l, u, st))
    return r["x"], r["y"], r["info"]


def kkt_solve(P_triu_csc, A_csc, sigma, rho, rhs):
    lib = load()
    n, m = P_triu_csc.shape[0], A_csc.shape[0]
    Pp, Pi, Px = _csc(P_triu_csc)
    Ap, Ai, Ax = _csc(A_csc)
    rhs = _f(rhs)

    def live():
        sol = np.zeros(n + m)
        lib.oracle_osqp_kkt_solve.argtypes = [C.c_longlong, C.c_longlong] + [C.c_void_p] * 6 + \
            [C.c_double, C.c_double, C.c_void_p, C.c_void_p]
        rc = lib.oracle_osqp_kkt_solve(n, m, _p(Pp), _p(Pi), _p(Px), _p(Ap), _p(Ai), _p(Ax), sigma, rho, _p(rhs), _p(sol))
        if rc:
            raise RuntimeError(f"kkt solve failed ({rc})")
        return dict(sol=sol)

    return ref_record.call("kkt_solve", live if have_ref() else None, (n, m, Pp, Pi, Px, Ap, Ai, Ax, sigma, rho, rhs))["sol"]


# ---- grid A* ---------------------------------------------------------------------------------------------------------
class AstarResult(C.Structure):
    _fields_ = [("status", C.c_int), ("use_node_num", C.c_int), ("n_pop", C.c_int), ("n_path", C.c_int),
                ("pop_hash", C.c_uint64), ("lookup_digest", C.c_uint64), ("n_in_map_calls", C.c_longlong)]


class RefAstarResult(C.Structure):
    _fields_ = [("status", C.c_int), ("use_node_num", C.c_int), ("n_path", C.c_int), ("pad", C.c_int),
                ("lookup_digest", C.c_uint64), ("n_in_map_calls", C.c_longlong)]


def astar_search(world, start_pt, end_pt, lambda_heu=1.0, allocated_node_num=100000, path_cap=8192):
    """oracle/astar_ref.cpp: the restated path_searching::Astar, a fresh object per query."""
    lib = load()
    occ = np.ascontiguousarray(world.occ, np.int8)
    origin, msz = _f(world.origin), _f(world.map_size)
    sp, ep = _f(start_pt), _f(end_pt)
    res = AstarResult()
    path = np.zeros((path_cap, 3))
    lib.oracle_astar_search.argtypes = [C.c_double, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_double,
                                        C.c_void_p, C.c_void_p, C.POINTER(AstarResult), C.c_void_p, C.c_int]
    lib.oracle_astar_search(lambda_heu, allocated_node_num, occ.ctypes.data, *world.dims, _p(origin), _p(msz), world.resolution, _p(sp),
                            _p(ep), C.byref(res), path.ctypes.data, path_cap)
    return dict(status=res.status, use_node_num=res.use_node_num, n_pop=res.n_pop, n_path=res.n_path, pop_hash=res.pop_hash,
                lookup_digest=res.lookup_digest, n_in_map_calls=res.n_in_map_calls, path=path[:min(res.n_path, path_cap)].copy())


_astar_ref = None


def have_astar_ref():
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", "libastar_ref.so"))


def astar_search_reference(world, start_pt, end_pt, lambda_heu=1.0, allocated_node_num=100000, path_cap=8192, like=None):
    """oracle/_ref/libastar_ref.so: the reference's a_star.cpp compiled unmodified against the header shims (recorded result where it
    is not built; like: a result whose path the caller compares with, see ref_record.call)."""
    occ = np.ascontiguousarray(world.occ, np.int8)
    origin, msz = _f(world.origin), _f(world.map_size)
    sp, ep = _f(start_pt), _f(end_pt)

    def live():
        global _astar_ref
        if _astar_ref is None:
            _astar_ref = C.CDLL(os.path.join(ORACLE_DIR, "_ref", "libastar_ref.so"))
            _astar_ref.refastar_search.argtypes = [C.c_double, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                                   C.c_double, C.c_void_p, C.c_void_p, C.POINTER(RefAstarResult), C.c_void_p, C.c_int]
        res = RefAstarResult()
        path = np.zeros((path_cap, 3))
        _astar_ref.refastar_search(lambda_heu, allocated_node_num, occ.ctypes.data, *world.dims, _p(origin), _p(msz), world.resolution,
                                   _p(sp), _p(ep), C.byref(res), path.ctypes.data, path_cap)
        return dict(status=res.status, use_node_num=res.use_node_num, n_path=res.n_path, lookup_digest=res.lookup_digest,
                    n_in_map_calls=res.n_in_map_calls, path=path[:min(res.n_path, path_cap)].copy())

    return ref_record.call("astar_search_reference", live if have_astar_ref() else None,
                           (lambda_heu, allocated_node_num, occ, world.dims, origin, msz, world.resolution, sp, ep, path_cap),
                           like=None if like is None else {"path": like["path"]})


# ---- RRT* (SURVEY.md §8(f) row 4, second half) ----------------------------------------------------------------------------------
class RrtResult(C.Structure):
    _fields_ = [("status", C.c_int), ("use_node_num", C.c_int), ("n_opt_path", C.c_int), ("reach_goal", C.c_int),
                ("n_samples", C.c_longlong), ("tree_digest", C.c_uint64), ("goal_g_cost", C.c_double), ("n_kd_visits", C.c_longlong)]


_RRT_ARGS = [C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_uint64, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
             C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.POINTER(RrtResult), C.c_void_p, C.c_int]
_rrt_ref = None


def have_rrt_ref():
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", "librrt_ref.so"))


def _rrt_call(fn, world, start_pt, end_pt, query_seed, max_tree_node_num, step_length, search_radius, collision_check_resolution,
              sample_budget, path_cap):
    occ = np.ascontiguousarray(world.occ, np.int8)
    origin, msz = _f(world.origin), _f(world.map_size)
    sp, ep = _f(start_pt), _f(end_pt)
    res = RrtResult()
    path = np.zeros((path_cap, 3))
    fn.argtypes = _RRT_ARGS
    fn(max_tree_node_num, step_length, search_radius, collision_check_resolution, float(sample_budget), int(query_seed), occ.ctypes.data,
       *world.dims, _p(origin), _p(msz), world.resolution, _p(sp), _p(ep), C.byref(res), path.ctypes.data, path_cap)
    return dict(status=res.status, use_node_num=res.use_node_num, n_opt_path=res.n_opt_path, reach_goal=res.reach_goal,
                n_samples=res.n_samples, tree_digest=res.tree_digest, goal_g_cost=res.goal_g_cost,
                opt_path=path[:min(res.n_opt_path, path_cap)].copy())


def rrt_search(world, start_pt, end_pt, query_seed, max_tree_node_num=100000, step_length=0.5, search_radius=0.5,
               collision_check_resolution=0.05, sample_budget=2.0, path_cap=8192):
    """oracle/rrt_star_ref.cpp: the restated path_searching::RRTStar with the seeded sample stream and a sample budget for
    `max_tolerance_time`; defaults = rrt_star.cpp:7-11."""
    return _rrt_call(load().oracle_rrt_search, world, start_pt, end_pt, query_seed, max_tree_node_num, step_length, search_radius,
                     collision_check_resolution, sample_budget, path_cap)


def rrt_search_reference(world, start_pt, end_pt, query_seed, max_tree_node_num=100000, step_length=0.5, search_radius=0.5,
                         collision_check_resolution=0.05, sample_budget=2.0, path_cap=8192, like=None):
    """oracle/_ref/librrt_ref.so: the reference's rrt_star.cpp + kdtree.cpp compiled unmodified (shims pin the RNG and the clock);
    recorded result where it is not built (like: a result whose path the caller compares with, see ref_record.call)."""
    def live():
        global _rrt_ref
        if _rrt_ref is None:
            _rrt_ref = C.CDLL(os.path.join(ORACLE_DIR, "_ref", "librrt_ref.so"))
        return _rrt_call(_rrt_ref.refrrt_search, world, start_pt, end_pt, query_seed, max_tree_node_num, step_length, search_radius,
                         collision_check_resolution, sample_budget, path_cap)

    key = (np.ascontiguousarray(world.occ, np.int8), world.dims, _f(world.origin), _f(world.map_size), world.resolution, _f(start_pt),
           _f(end_pt), int(query_seed), max_tree_node_num, step_length, search_radius, collision_check_resolution, float(sample_budget),
           path_cap)
    return ref_record.call("rrt_search_reference", live if have_rrt_ref() else None, key,
                           like=None if like is None else {"opt_path": like["opt_path"]})
