"""ctypes binding of libuavmp.so (the C-ABI in include/uavmp.h).

There is no CPU fallback: if the CUDA library is missing or no GPU is present, loading / creating a context raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libuavmp.so")
WORLDGEN_PATH = os.path.join(_HERE, "libuavmp_worldgen.so")  # host-only input generator (include/uavmp_worldgen.h)


class KinoParams(C.Structure):
    """uavmp_kino_params == the ROS parameters of KinoAstar::setParam (kino_astar.cpp:8-19)."""
    _fields_ = [("allocated_node_num", C.c_int), ("collision_check_type", C.c_int), ("rou_time", C.c_double),
                ("lambda_heu", C.c_double), ("goal_tolerance", C.c_double), ("time_step_size", C.c_double),
                ("max_velocity", C.c_double), ("max_accelration", C.c_double), ("acc_resolution", C.c_double),
                ("sample_tau", C.c_double), ("robot_r", C.c_double), ("robot_h", C.c_double)]


class OsqpSettings(C.Structure):
    _fields_ = [("rho", C.c_double), ("sigma", C.c_double), ("alpha", C.c_double), ("eps_abs", C.c_double),
                ("eps_rel", C.c_double), ("eps_prim_inf", C.c_double), ("eps_dual_inf", C.c_double),
                ("max_iter", C.c_int), ("check_termination", C.c_int), ("scaling", C.c_int),
                ("adaptive_rho", C.c_int), ("adaptive_rho_interval", C.c_int),
                ("adaptive_rho_tolerance", C.c_double)]


class MapgenParams(C.Structure):
    _fields_ = [("map_type", C.c_int), ("seed", C.c_uint32), ("x_size", C.c_double), ("y_size", C.c_double),
                ("resolution", C.c_double), ("init_x", C.c_double), ("init_y", C.c_double),
                ("init_radius", C.c_double), ("polar_num", C.c_int), ("circle_num", C.c_int), ("w_l", C.c_double),
                ("w_h", C.c_double), ("h_l", C.c_double), ("h_h", C.c_double), ("radius_l", C.c_double),
                ("radius_h", C.c_double), ("z_l", C.c_double), ("z_h", C.c_double), ("theta", C.c_double),
                ("wall_x", C.c_double), ("wall_y", C.c_double), ("wall_w", C.c_double)]


class Timings(C.Structure):
    _fields_ = [("h2d_ms", C.c_float), ("search_ms", C.c_float), ("path_ms", C.c_float), ("qp_ms", C.c_float),
                ("d2h_ms", C.c_float), ("total_ms", C.c_float), ("search_launches", C.c_int),
                ("qp_launches", C.c_int), ("aux_launches", C.c_int)]


class KinoCounters(C.Structure):
    _fields_ = [(n, C.c_longlong) for n in ("n_pop", "n_occ_lookup", "n_cloud_pts_tested", "n_hash_probe",
                                            "n_insert", "n_update", "n_heuristic", "n_shot")]


class PlanOptions(C.Structure):
    """uavmp_plan_options: what the pipeline builds between the search and the QP (time allocation, corridor rows)."""
    _fields_ = [("order", C.c_int), ("S", C.c_int), ("seg_time", C.c_double), ("time_alloc", C.c_int),
                ("corridor_samples", C.c_int), ("corridor_margin", C.c_double)]


class PlanInfo(C.Structure):
    """uavmp_plan_info: what uavmp_plan_wait reports about one batch."""
    _fields_ = [("error_flags", C.c_int), ("counters", KinoCounters), ("timings", Timings)]


# every symbol include/uavmp.h declares (tests/test_abi.py checks the .so exports all of them)
SYMBOLS = [
    "uavmp_ctx_create", "uavmp_ctx_destroy", "uavmp_last_error", "uavmp_ctx_stream", "uavmp_ctx_sync",
    "uavmp_version", "uavmp_kino_params_default", "uavmp_kino_params_launch", "uavmp_osqp_settings_default",
    "uavmp_kino_set_params", "uavmp_map_set", "uavmp_kino_search_batch", "uavmp_kino_get_paths",
    "uavmp_kino_set_trace", "uavmp_kino_get_trace", "uavmp_kino_get_counters", "uavmp_minctrl_solve_batch",
    "uavmp_plan_batch", "uavmp_plan_batch_dev", "uavmp_get_timings", "uavmp_fpmath_eval", "uavmp_kino_set_profile",
    "uavmp_kino_get_profile", "uavmp_map_set_from_cloud", "uavmp_map_get_occupancy", "uavmp_polytraj_eval_batch",
    "uavmp_plan_submit", "uavmp_plan_wait", "uavmp_plan_stream_wait", "uavmp_plan_max_in_flight",
    "uavmp_kino_set_path_cap", "uavmp_minctrl_solve_corridor_batch", "uavmp_plan_options_default", "uavmp_plan_submit_opt",
    "uavmp_astar_set_params", "uavmp_astar_search_batch", "uavmp_astar_get_paths",
    "uavmp_rrt_set_params", "uavmp_rrt_sample_seed", "uavmp_rrt_search_batch", "uavmp_rrt_get_paths",
    "uavmp_minctrl_solve_ragged_batch", "uavmp_rrt_plan_batch", "uavmp_rrt_plan_get_coef",
]

WORLDGEN_SYMBOLS = ["uavmp_mapgen_params_default", "uavmp_mapgen_cloud", "uavmp_grid_inflate_host"]

# test/launch/test_kino_astar_searching.launch:44-57 and kino_astar.cpp:8-19 — the same tables uavmp_kino_params_launch /
# uavmp_kino_params_default return (tests/test_abi.py keeps the two in step); here so that host-only code (the CPU reference
# arm of bench.py) never has to map the CUDA library
LAUNCH_PARAMS = dict(allocated_node_num=100000, collision_check_type=1, rou_time=50.0, lambda_heu=3.0, goal_tolerance=2.0,
                     time_step_size=0.075, max_velocity=7.0, max_accelration=10.0, acc_resolution=4.0, sample_tau=0.3,
                     robot_r=0.4, robot_h=0.1)
DEFAULT_PARAMS = dict(allocated_node_num=100000, collision_check_type=1, rou_time=1.0, lambda_heu=2.0, goal_tolerance=2.0,
                      time_step_size=0.1, max_velocity=5.0, max_accelration=7.0, acc_resolution=2.0, sample_tau=0.5,
                      robot_r=0.2, robot_h=0.1)


def launch_params(**overrides):
    p = KinoParams(**LAUNCH_PARAMS)
    for k, v in overrides.items():
        setattr(p, k, v)
    return p


_lib = None
_wg = None


def load_worldgen():
    """Load libuavmp_worldgen.so (host only, no CUDA): the synthetic-world generator of tests and bench.py."""
    global _wg
    if _wg is not None:
        return _wg
    if not os.path.exists(WORLDGEN_PATH):
        raise RuntimeError(f"{WORLDGEN_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(WORLDGEN_PATH)
    vp = C.c_void_p
    lib.uavmp_mapgen_params_default.argtypes = [C.POINTER(MapgenParams), C.c_double, C.c_double, C.c_uint32]
    lib.uavmp_mapgen_params_default.restype = None
    lib.uavmp_mapgen_cloud.argtypes = [C.POINTER(MapgenParams), vp, C.c_int]
    lib.uavmp_grid_inflate_host.argtypes = [vp, C.c_int, vp, vp, C.c_double, C.c_double, vp, C.c_int, C.c_int,
                                            C.c_int]
    _wg = lib
    return lib


def load():
    """Load libuavmp.so; raises (loudly) when it has not been built — there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(the CUDA extension is the only implementation; there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    vp, ip, dp = C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_double)
    lib.uavmp_ctx_create.argtypes = [C.POINTER(vp), C.c_int]
    lib.uavmp_ctx_destroy.argtypes = [vp]
    lib.uavmp_ctx_destroy.restype = None
    lib.uavmp_last_error.argtypes = [vp]
    lib.uavmp_last_error.restype = C.c_char_p
    lib.uavmp_ctx_stream.argtypes = [vp]
    lib.uavmp_ctx_stream.restype = vp
    lib.uavmp_ctx_sync.argtypes = [vp]
    lib.uavmp_version.restype = C.c_char_p
    lib.uavmp_kino_params_default.argtypes = [C.POINTER(KinoParams)]
    lib.uavmp_kino_params_launch.argtypes = [C.POINTER(KinoParams)]
    lib.uavmp_osqp_settings_default.argtypes = [C.POINTER(OsqpSettings)]
    lib.uavmp_kino_set_params.argtypes = [vp, C.POINTER(KinoParams)]
    lib.uavmp_map_set.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, C.c_double, vp, C.c_int]
    lib.uavmp_kino_search_batch.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.uavmp_kino_search_batch.restype = C.c_longlong
    lib.uavmp_kino_get_paths.argtypes = [vp, vp, C.c_longlong]
    lib.uavmp_kino_set_trace.argtypes = [vp, C.c_int]
    lib.uavmp_kino_get_trace.argtypes = [vp, C.c_int, vp, C.c_int]
    lib.uavmp_kino_get_counters.argtypes = [vp, C.POINTER(KinoCounters)]
    lib.uavmp_minctrl_solve_batch.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp,
                                              C.POINTER(OsqpSettings), vp, vp, vp, vp]
    lib.uavmp_plan_batch.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, C.c_double,
                                     C.POINTER(OsqpSettings), vp, vp, vp]
    lib.uavmp_plan_batch_dev.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, C.c_double,
                                         C.POINTER(OsqpSettings), vp, vp, vp]
    lib.uavmp_plan_submit.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, C.c_double,
                                      C.POINTER(OsqpSettings), C.c_uint, vp, vp, vp, C.POINTER(C.c_longlong)]
    lib.uavmp_plan_submit_opt.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.POINTER(PlanOptions), C.POINTER(OsqpSettings), C.c_uint,
                                          vp, vp, vp, C.POINTER(C.c_longlong)]
    lib.uavmp_plan_options_default.argtypes = [C.POINTER(PlanOptions)]
    lib.uavmp_plan_options_default.restype = None
    lib.uavmp_minctrl_solve_corridor_batch.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp,
                                                       C.POINTER(OsqpSettings), vp, vp, vp, vp]
    lib.uavmp_plan_wait.argtypes = [vp, C.c_longlong, C.POINTER(PlanInfo)]
    lib.uavmp_plan_stream_wait.argtypes = [vp, C.c_longlong, vp]
    lib.uavmp_kino_set_path_cap.argtypes = [vp, C.c_int]
    lib.uavmp_get_timings.argtypes = [vp, C.POINTER(Timings)]
    lib.uavmp_fpmath_eval.argtypes = [vp, C.c_int, C.c_int, vp, vp, C.c_longlong]
    lib.uavmp_map_set_from_cloud.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, C.c_double, C.c_double]
    lib.uavmp_map_get_occupancy.argtypes = [vp, vp, C.c_longlong]
    lib.uavmp_polytraj_eval_batch.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, vp, C.c_int, vp]
    lib.uavmp_astar_set_params.argtypes = [vp, C.c_double, C.c_int, C.c_int]
    lib.uavmp_astar_search_batch.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp]
    lib.uavmp_astar_search_batch.restype = C.c_longlong
    lib.uavmp_astar_get_paths.argtypes = [vp, vp, C.c_longlong]
    lib.uavmp_rrt_set_params.argtypes = [vp, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int]
    lib.uavmp_rrt_sample_seed.argtypes = [C.c_uint64, C.c_longlong]
    lib.uavmp_rrt_sample_seed.restype = C.c_uint32
    lib.uavmp_rrt_search_batch.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.uavmp_rrt_search_batch.restype = C.c_longlong
    lib.uavmp_rrt_get_paths.argtypes = [vp, vp, C.c_longlong]
    lib.uavmp_minctrl_solve_ragged_batch.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, C.POINTER(OsqpSettings), vp, vp, vp, vp]
    lib.uavmp_rrt_plan_batch.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_int, C.c_double, C.POINTER(OsqpSettings), vp, vp, vp, vp, vp, vp]
    lib.uavmp_rrt_plan_batch.restype = C.c_longlong
    lib.uavmp_rrt_plan_get_coef.argtypes = [vp, vp, C.c_longlong]
    lib.uavmp_kino_set_profile.argtypes = [vp, C.c_int]
    lib.uavmp_kino_get_profile.argtypes = [vp, vp, vp, C.c_int, ip]
    _lib = lib
    return lib


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def as_f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


class UavmpError(RuntimeError):
    pass


class Context:
    """Owns one uavmp_ctx (one CUDA device)."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.uavmp_ctx_create(C.byref(h), device)
        if rc != 0:
            raise UavmpError(f"uavmp_ctx_create failed ({rc}): no usable CUDA device — this library has no CPU path")
        self.h = h

    def check(self, rc):
        if rc < 0:
            raise UavmpError(f"uavmp error {rc}: {self.lib.uavmp_last_error(self.h).decode()}")
        return rc

    def close(self):
        if getattr(self, "h", None):
            self.lib.uavmp_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self):
        return self.lib.uavmp_ctx_stream(self.h)

    def sync(self):
        return self.check(self.lib.uavmp_ctx_sync(self.h))

    def timings(self):
        t = Timings()
        self.lib.uavmp_get_timings(self.h, C.byref(t))
        return {k: getattr(t, k) for k, _ in Timings._fields_}
