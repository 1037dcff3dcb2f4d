"""Host-side mirror of traj_optimization::MinimumControl (minimum_control.h:10-49) over the batched CUDA QP solver.

`solve` keeps the reference signature (one axis per call, returns bool, `getCoef1d` returns the 6S coefficients,
segment-major / ascending power / local time).  `solve_batch` is the B200 entry point: B independent 1-D problems.
order=5 is the reference's minimum jerk; order=7 (minimum snap) is the §9.3 generalisation (extension).
"""
import ctypes as C

import numpy as np

from . import _lib


def default_settings(**kw):
    s = _lib.OsqpSettings()
    _lib.load().uavmp_osqp_settings_default(C.byref(s))
    for k, v in kw.items():
        if not hasattr(s, k):
            raise KeyError(k)
        setattr(s, k, v)
    return s


class MinimumControl:
    def __init__(self, ctx=None, device=0, order=5):
        self.ctx = ctx if ctx is not None else _lib.Context(device)
        self.lib = self.ctx.lib
        self.order = order
        self.settings = default_settings()
        self._coef_1d = None
        self.last = {}

    def solve_batch(self, pos_1d, bound_vel, bound_acc, time_vec, bound_jerk=None, order=None, settings=None,
                    corridor_lo=None, corridor_hi=None, n_corridor=0):
        """n_corridor > 0 (extension, SURVEY.md §9.3): per segment, the position at n_corridor interior times must stay in
        [corridor_lo[b, s], corridor_hi[b, s]] — true inequality rows (uavmp_minctrl_solve_corridor_batch)."""
        order = self.order if order is None else order
        pos = _lib.as_f64(pos_1d)
        pos = pos.reshape(1, -1) if pos.ndim == 1 else pos
        B, S = pos.shape[0], pos.shape[1] - 1
        bv = _lib.as_f64(bound_vel).reshape(B, 2)
        ba = _lib.as_f64(bound_acc).reshape(B, 2)
        bj = None if order == 5 else _lib.as_f64(np.zeros((B, 2)) if bound_jerk is None else bound_jerk).reshape(B, 2)
        T = _lib.as_f64(time_vec).reshape(B, S)
        n = (order + 1) * S
        coef = np.zeros((B, n))
        solved, status, iters = np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32)
        st = settings or self.settings
        if n_corridor > 0:
            lo, hi = _lib.as_f64(corridor_lo).reshape(B, S), _lib.as_f64(corridor_hi).reshape(B, S)
            self.ctx.check(self.lib.uavmp_minctrl_solve_corridor_batch(
                self.ctx.h, order, S, n_corridor, B, _lib.ptr(pos), _lib.ptr(bv), _lib.ptr(ba), _lib.ptr(bj), _lib.ptr(T),
                _lib.ptr(lo), _lib.ptr(hi), C.byref(st), _lib.ptr(coef), _lib.ptr(solved), _lib.ptr(status), _lib.ptr(iters)))
        else:
            self.ctx.check(self.lib.uavmp_minctrl_solve_batch(
                self.ctx.h, order, S, B, _lib.ptr(pos), _lib.ptr(bv), _lib.ptr(ba), _lib.ptr(bj), _lib.ptr(T), C.byref(st),
                _lib.ptr(coef), _lib.ptr(solved), _lib.ptr(status), _lib.ptr(iters)))
        self.last = dict(coef=coef, solved=solved, status=status, iters=iters)
        return self.last

    def solve_batch_ragged(self, pos_1d, bound_vel, bound_acc, time_vec, S=None, bound_jerk=None, order=None, settings=None):
        """B problems with a different number of segments each, one call (uavmp_minctrl_solve_ragged_batch).  Either lists (pos_1d[b]:
        S_b + 1 waypoints, time_vec[b]: S_b times; S=None) or packed arrays plus S (B segment counts, problems in order).  bound_vel /
        bound_acc (/ bound_jerk): B x 2.  Returns packed coef with coef_offsets (B + 1, problem b's coefficients are
        coef[coef_offsets[b]:coef_offsets[b + 1]], segment-major as in solve_batch), solved, status, iters, S.  Every result is
        bit-identical to solve_batch on that problem alone."""
        order = self.order if order is None else order
        if S is None:
            S = np.array([len(t) for t in time_vec], np.int32)
            pos = _lib.as_f64(np.concatenate([np.asarray(p, np.float64).reshape(-1) for p in pos_1d]))
            T = _lib.as_f64(np.concatenate([np.asarray(t, np.float64).reshape(-1) for t in time_vec]))
        else:
            S = np.ascontiguousarray(S, np.int32).reshape(-1)
            pos, T = _lib.as_f64(pos_1d).reshape(-1), _lib.as_f64(time_vec).reshape(-1)
        B = len(S)
        if pos.size != int(S.sum()) + B or T.size != int(S.sum()):
            raise ValueError("pos_1d needs sum(S + 1) waypoints and time_vec sum(S) segment times")
        bv = _lib.as_f64(bound_vel).reshape(B, 2)
        ba = _lib.as_f64(bound_acc).reshape(B, 2)
        bj = None if order == 5 else _lib.as_f64(np.zeros((B, 2)) if bound_jerk is None else bound_jerk).reshape(B, 2)
        coef_offsets = np.zeros(B + 1, np.int64)
        coef_offsets[1:] = np.cumsum(S.astype(np.int64) * (order + 1))
        coef = np.zeros(int(coef_offsets[-1]))
        solved, status, iters = np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32)
        st = settings or self.settings
        self.ctx.check(self.lib.uavmp_minctrl_solve_ragged_batch(
            self.ctx.h, order, B, _lib.ptr(S), _lib.ptr(pos), _lib.ptr(bv), _lib.ptr(ba), _lib.ptr(bj), _lib.ptr(T), C.byref(st),
            _lib.ptr(coef), _lib.ptr(solved), _lib.ptr(status), _lib.ptr(iters)))
        self.last = dict(coef=coef, coef_offsets=coef_offsets, solved=solved, status=status, iters=iters, S=S)
        return self.last

    # bool solve(VectorXd& pos_1d, Vector2d& bound_vel, Vector2d& bound_acc, VectorXd& time_vec)
    def solve(self, pos_1d, bound_vel, bound_acc, time_vec):
        r = self.solve_batch(np.asarray(pos_1d)[None], np.asarray(bound_vel)[None], np.asarray(bound_acc)[None],
                             np.asarray(time_vec)[None])
        if not r["solved"][0]:
            print("solver solve failed!")  # minimum_control.cpp:182; coef_1d_ keeps its previous value
            return False
        self._coef_1d = r["coef"][0].copy()
        return True

    def getCoef1d(self):
        return self._coef_1d

    def reset(self):  # minimum_control.cpp:194-197
        if self._coef_1d is not None:
            self._coef_1d[:] = 0.0
