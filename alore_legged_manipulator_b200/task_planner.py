"""Task plan from the optimised candidates: which object to pick next and which target to put it on.

Task points: 0 is the robot, 1..n the objects, n+1..2n the targets.  Every candidate of a batch is labelled with the
leg it belongs to (`leg_from[b] -> leg_to[b]`, or `leg_from[b] = -1` for a candidate that is not a task leg).  The
library reduces the candidates to the leg cost matrix (cheapest counted candidate per leg, lowest index on ties) and
solves the visiting order (and, unless `fixed_assignment`, the object-to-target assignment) on the device: exactly up to
12 (free) / 20 (fixed) objects, or with `width=` by a bounded-width layered search up to 32 objects that reports whether
its result is proven optimal; see include/alore_b200.h for the contract.  `plan_tasks` takes host results (`alore_opt_batch`); `DeviceBatch.task_plan`
(ms_planner.py) reads the device results of a resident batch without downloading it.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import capi


@dataclass
class TaskPlan:
    cost: float                      # optimum of the left fold of the tour's leg costs; +inf when infeasible
    feasible: bool
    order: np.ndarray                # [n] object point picked k-th (-1 when infeasible)
    target: np.ndarray               # [n] target point it is placed on
    leg_cand: np.ndarray             # [2n] candidate index of every leg in tour order
    leg_cost: np.ndarray | None      # [P, P] leg matrix D (with_matrix)
    leg_best: np.ndarray | None      # [P, P] candidate index of every leg, -1 = none (with_matrix)
    exact: bool | None = None        # width search only: no layer was truncated, so the plan is the exact solver's

    def legs(self):
        """The tour's legs in order: [(from point, to point), ...]."""
        pts = [0]
        for o, t in zip(self.order.tolist(), self.target.tolist()):
            pts += [o, t]
        return list(zip(pts[:-1], pts[1:]))


class TaskCall:
    """The packed arguments and the output store of one task-plan call (keeps the arrays alive for the call)."""

    def __init__(self, n_objects, leg_from, leg_to, fixed_assignment=False, assign=None, with_matrix=False):
        n = int(n_objects)
        self.n, self.P = n, 2 * n + 1
        self.leg_from = np.ascontiguousarray(leg_from, dtype=np.int32).reshape(-1)
        self.leg_to = np.ascontiguousarray(leg_to, dtype=np.int32).reshape(-1)
        if self.leg_from.size != self.leg_to.size:
            raise ValueError("leg_from and leg_to differ in length")
        self.assign = None if assign is None else np.ascontiguousarray(assign, dtype=np.int32).reshape(-1)
        if self.assign is not None and self.assign.size != n:
            raise ValueError(f"assign has {self.assign.size} entries, expected {n}")
        nn = max(n, 1)
        self.order, self.target = np.full(nn, -1, np.int32), np.full(nn, -1, np.int32)
        self.leg_cand = np.full(2 * nn, -1, np.int32)
        self.leg_cost = np.zeros((self.P, self.P)) if with_matrix else None
        self.leg_best = np.zeros((self.P, self.P), np.int32) if with_matrix else None
        self.task = capi.Task(n, 1 if fixed_assignment else 0,
                              capi.iptr(self.assign) if self.assign is not None else None,
                              capi.iptr(self.leg_from), capi.iptr(self.leg_to))
        self.out = capi.TaskPlanOut(0.0, 0, 0, capi.iptr(self.order), capi.iptr(self.target), capi.iptr(self.leg_cand),
                                    capi.dptr(self.leg_cost) if with_matrix else None,
                                    capi.iptr(self.leg_best) if with_matrix else None)

    @property
    def B(self) -> int:
        return int(self.leg_from.size)

    def result(self, exact=None) -> TaskPlan:
        n = self.n
        return TaskPlan(float(self.out.cost), bool(self.out.feasible), self.order[:n].copy(), self.target[:n].copy(),
                        self.leg_cand[:2 * n].copy(),
                        None if self.leg_cost is None else self.leg_cost.copy(),
                        None if self.leg_best is None else self.leg_best.copy(),
                        None if exact is None else bool(exact.value))


def plan_tasks(ctx: capi.Context, n_objects, leg_from, leg_to, cost, ok, fixed_assignment=False, assign=None,
               with_matrix=False, width=None) -> TaskPlan:
    """alore_task_plan on host results: cost [B] (float64) and ok [B] (int32) of alore_opt_batch, one label per
    candidate.  fixed_assignment: object i goes to assign[i-1] (None: target n+i) and only the order is searched.
    width: None runs the exact solver; an int runs alore_task_plan_beam with that width, and the plan's `exact` tells
    whether no layer was truncated."""
    call = TaskCall(n_objects, leg_from, leg_to, fixed_assignment, assign, with_matrix)
    cost = np.ascontiguousarray(cost, dtype=np.float64).reshape(-1)
    ok = np.ascontiguousarray(ok, dtype=np.int32).reshape(-1)
    if cost.size != call.B or ok.size != call.B:
        raise ValueError(f"{call.B} labels but {cost.size} costs / {ok.size} ok flags")
    if width is None:
        ctx.check(ctx.lib.alore_task_plan(ctx.h, C.byref(call.task), call.B, capi.dptr(cost), capi.iptr(ok), C.byref(call.out)))
        return call.result()
    exact = C.c_int32(-1)
    ctx.check(ctx.lib.alore_task_plan_beam(ctx.h, C.byref(call.task), int(width), call.B, capi.dptr(cost), capi.iptr(ok),
                                           C.byref(call.out), C.byref(exact)))
    return call.result(exact)
