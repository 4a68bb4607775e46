"""Host-side mirror of the reference's `MSPlanner` back_end interface (batched).

planning_ddr_opt/back_end/include/back_end/optimizer.h:192-300: `minco_plan(flat_traj)` keeps its
name, argument and bool result; results are exposed like the reference's public members/getters
(`final_traj_` coefficients + durations, `get_current_Innerpoints`, `get_current_finalpieceTime`,
`get_current_finState`).  `minco_plan_batch` is the same call over a structure-of-arrays batch of
candidates — what the task-and-motion planner scores.  Everything forwards to the C ABI; there is no
CPU fallback.  The C++ twin is csrc/host/ms_planner.hpp.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi, front_end
from .sdf_map import SDFmap


class DeviceBatch:
    """A candidate batch resident in HBM (alore_batch_*): upload once, optimise many times."""

    def __init__(self, ctx: capi.Context, cands: capi.CandidateBatch):
        self.ctx, self.cands = ctx, cands
        self.h = C.c_void_p()
        cs = cands.as_struct()
        ctx.check(ctx.lib.alore_batch_upload(ctx.h, C.byref(cs), C.byref(self.h)))

    def run(self, prm: capi.Params, stream=None):
        self.ctx.check(self.ctx.lib.alore_batch_run(self.ctx.h, C.byref(prm), self.h, stream))

    def download(self) -> capi.ResultBatch:
        res = capi.ResultBatch(self.cands)
        rs = res.as_struct()
        self.ctx.check(self.ctx.lib.alore_batch_download(self.ctx.h, self.h, C.byref(rs)))
        return res

    def argmin(self):
        bc, bi = C.c_double(), C.c_int32()
        self.ctx.check(self.ctx.lib.alore_batch_argmin(self.ctx.h, self.h, C.byref(bc), C.byref(bi)))
        return float(bc.value), int(bi.value)

    def task_plan(self, n_objects, leg_from, leg_to, fixed_assignment=False, assign=None, with_matrix=False, width=None):
        """alore_batch_task_plan: the task plan (task_planner.TaskPlan) from the device results of the last run, one
        leg label per candidate of this batch.  width: None = the exact solver, an int = alore_batch_task_plan_beam."""
        from .task_planner import TaskCall
        call = TaskCall(n_objects, leg_from, leg_to, fixed_assignment, assign, with_matrix)
        if call.B != self.cands.B:
            raise ValueError(f"{call.B} leg labels for a batch of {self.cands.B} candidates")
        if width is None:
            self.ctx.check(self.ctx.lib.alore_batch_task_plan(self.ctx.h, self.h, C.byref(call.task), C.byref(call.out)))
            return call.result()
        exact = C.c_int32(-1)
        self.ctx.check(self.ctx.lib.alore_batch_task_plan_beam(self.ctx.h, self.h, C.byref(call.task), int(width),
                                                               C.byref(call.out), C.byref(exact)))
        return call.result(exact)

    def device_results(self):
        dc, dk = C.c_void_p(), C.c_void_p()
        self.ctx.check(self.ctx.lib.alore_batch_device_results(self.h, C.byref(dc), C.byref(dk)))
        return dc.value, dk.value

    def stats(self):
        """(algorithmic bytes, cost evaluations, L-BFGS iterations) summed over the batch of the last run."""
        ab, ev, it = C.c_double(), C.c_longlong(), C.c_longlong()
        self.ctx.check(self.ctx.lib.alore_batch_stats(self.ctx.h, self.h, C.byref(ab), C.byref(ev), C.byref(it)))
        return float(ab.value), int(ev.value), int(it.value)

    def kernel_ms(self) -> float:
        ms = C.c_float()
        self.ctx.check(self.ctx.lib.alore_batch_last_kernel_ms(self.h, C.byref(ms)))
        return float(ms.value)

    def close(self):
        if self.h:
            self.ctx.lib.alore_batch_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MSPlanner:
    def __init__(self, ctx: capi.Context, params: capi.Params, sdf_map: SDFmap):
        self.ctx, self.params, self.map_ = ctx, params, sdf_map
        self.last_result: capi.ResultBatch | None = None
        self._cands: capi.CandidateBatch | None = None

    # ---- the reference's entry point -------------------------------------------------------
    def minco_plan(self, flat_traj: front_end.FlatTrajData) -> bool:  # optimizer.cpp:169-220
        res = self.minco_plan_batch(front_end.pack_candidates([flat_traj]))
        return bool(res.ok[0])

    def minco_plan_batch(self, cands: capi.CandidateBatch, out: capi.ResultBatch | None = None) -> capi.ResultBatch:
        """Optimises every candidate of the batch.  `out`: a reusable (optionally page-locked) result store."""
        self.map_._check_owner()
        res = capi.ResultBatch(cands) if out is None else out.bind(cands.B, cands.total_pieces)
        cs, rs = cands.as_struct(), res.as_struct()
        self.ctx.check(self.ctx.lib.alore_opt_batch(self.ctx.h, C.byref(self.params), C.byref(cs), C.byref(rs)))
        self.last_result, self._cands = res, cands
        return res

    # ---- getters (optimizer.h:253-268) for candidate b of the last call -------------------------
    def _slice(self, b):
        p0, p1 = int(self._cands.piece_off[b]), int(self._cands.piece_off[b + 1])
        return p0, p1

    def get_current_Innerpoints(self, b=0):
        p0, p1 = self._slice(b)
        return self.last_result.inner_pts[p0 - b:p1 - b - 1].T.copy()       # 2 x (N-1)

    def get_current_finalpieceTime(self, b=0):
        p0, p1 = self._slice(b)
        return self.last_result.piece_T[p0:p1].copy()

    def get_current_finState(self, b=0):
        fs = self._cands.final_state[b].copy()
        fs[1, 0] = self.last_result.tail_s[b]
        return fs

    def final_traj(self, b=0):
        """(durations [N], coefficients [N, 6, 2] ascending powers) — Trajectory<5,2> final_traj_."""
        p0, p1 = self._slice(b)
        return self.last_result.piece_T[p0:p1].copy(), self.last_result.coeffs[p0:p1].copy()

    # ---- pieces of the path exposed for parity tests / benchmarks ---------------------------------
    def cost_batch(self, cands: capi.CandidateBatch, stage: int, x: np.ndarray, lam=None, rho=None, safe_dis=None,
                   g_init=None):
        """One costFunctionCallback (stage 1) / costFunctionCallbackPath (stage 0) per candidate."""
        self.map_._check_owner()
        B = cands.B
        x = np.ascontiguousarray(x, dtype=np.float64)
        assert x.size == cands.n_vars()
        g = np.zeros_like(x) if g_init is None else np.ascontiguousarray(g_init, dtype=np.float64).copy()
        cost, err = np.zeros(B), np.zeros((B, 2))
        cs = cands.as_struct()
        opt = lambda a, n: capi.dptr(np.ascontiguousarray(a, dtype=np.float64).reshape(n)) if a is not None else None
        keep = [opt(lam, 2 * B), opt(rho, 2 * B), opt(safe_dis, B)]
        self.ctx.check(self.ctx.lib.alore_cost_batch(self.ctx.h, C.byref(self.params), C.byref(cs), stage, capi.dptr(x),
                                                     keep[0], keep[1], keep[2], capi.dptr(cost), capi.dptr(g),
                                                     capi.dptr(err)))
        return cost, g, err

    def penalty_batch(self, piece_off, coeffs, piece_T, start_xy, final_xy):
        """attachPenaltyFunctional on given coefficients (BASELINE config 3)."""
        self.map_._check_owner()
        piece_off = np.ascontiguousarray(piece_off, dtype=np.int32)
        B, tot = piece_off.size - 1, int(piece_off[-1])
        cost, gC, gT, err = np.zeros(B), np.zeros((tot, 6, 2)), np.zeros(tot), np.zeros((B, 2))
        self.ctx.check(self.ctx.lib.alore_penalty_batch(
            self.ctx.h, C.byref(self.params), B, capi.iptr(piece_off), capi.dptr(np.ascontiguousarray(coeffs)),
            capi.dptr(np.ascontiguousarray(piece_T)), capi.dptr(np.ascontiguousarray(start_xy)),
            capi.dptr(np.ascontiguousarray(final_xy)), capi.dptr(cost), capi.dptr(gC), capi.dptr(gT), capi.dptr(err)))
        return cost, gC, gT, err

    def check_final_collision_batch(self, piece_off, coeffs, piece_T, start_xy):  # optimizer.cpp:474-571
        piece_off = np.ascontiguousarray(piece_off, dtype=np.int32)
        B = piece_off.size - 1
        col, md = np.zeros(B, np.int32), np.zeros(B)
        self.ctx.check(self.ctx.lib.alore_final_collision_batch(
            self.ctx.h, C.byref(self.params), B, capi.iptr(piece_off), capi.dptr(np.ascontiguousarray(coeffs)),
            capi.dptr(np.ascontiguousarray(piece_T)), capi.dptr(np.ascontiguousarray(start_xy)), capi.iptr(col),
            capi.dptr(md)))
        return col, md
