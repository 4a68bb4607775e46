"""GPU tests of the task plan (alore_task_plan, alore_batch_task_plan) against the sequential oracle, bit for bit:
optimum bits, feasibility, order, targets, leg candidates, the leg matrix and its candidate indices."""
import ctypes as C
import math

import numpy as np
import pytest

from alore_legged_manipulator_b200 import capi, plan_tasks, workloads
from alore_legged_manipulator_b200.ms_planner import DeviceBatch
from alore_legged_manipulator_b200.task_planner import TaskCall
from task_plan_util import assert_same_plan, assert_valid_plan, oracle_plan, random_assign, random_batch, task_leg_batch
from test_esdf_gpu import make_sdf

pytestmark = pytest.mark.gpu


def device_vs_oracle(ctx, n, batch, fixed=False, assign=None):
    lf, lt, cost, ok = batch
    got = plan_tasks(ctx, n, lf, lt, cost, ok, fixed, assign, with_matrix=True)
    ref = oracle_plan(n, lf, lt, cost, ok, fixed, assign)
    assert_same_plan(got, ref)
    if got.feasible:
        assert_valid_plan(got, n, fixed, assign)
    return got


@pytest.mark.parametrize("n", range(1, capi.ALORE_TASK_MAX_FREE + 1))
def test_free_mode_equals_oracle(ctx, n):
    rng = np.random.default_rng(n)
    kinds = ["mixed", "ties", "neg"] if n <= 9 else ["mixed"]
    feasible = 0
    for kind in kinds:
        for bad in ([0.16, 0.02] if n <= 9 else [0.02]):
            feasible += device_vs_oracle(ctx, n, random_batch(rng, n, kind, per_leg=(0, 3) if n <= 9 else (1, 2), bad=bad)).feasible
    assert feasible > 0


@pytest.mark.parametrize("n", range(1, capi.ALORE_TASK_MAX_FIXED + 1))
def test_fixed_mode_equals_oracle(ctx, n):
    rng = np.random.default_rng(100 + n)
    feasible = 0
    for rep, kind in enumerate(["ties", "mixed"] if n <= 16 else ["ties"]):
        assign = None if rep == 0 else random_assign(rng, n)
        feasible += device_vs_oracle(ctx, n, random_batch(rng, n, kind, per_leg=(1, 2), bad=0.01), True, assign).feasible
    if n <= 10:                                          # infeasible mixes too
        device_vs_oracle(ctx, n, random_batch(rng, n, "mixed", per_leg=(0, 2)), True, random_assign(rng, n))
    assert feasible > 0


def test_arena_reuse_growing_and_shrinking(ctx):
    sizes = [(4, False), (10, False), (2, False), (16, True), (3, True), (12, False), (20, True), (1, False), (7, True)]
    rng = np.random.default_rng(7)
    cases = [(n, fixed, random_assign(rng, n) if fixed else None, random_batch(rng, n, "mixed", per_leg=(1, 2), bad=0.02))
             for n, fixed in sizes]
    reused = [plan_tasks(ctx, n, *b, fixed, a, with_matrix=True) for n, fixed, a, b in cases]
    for (n, fixed, a, b), r in zip(cases, reused):
        fresh_ctx = capi.Context(0)
        try:
            assert_same_plan(r, plan_tasks(fresh_ctx, n, *b, fixed, a, with_matrix=True))
        finally:
            fresh_ctx.close()
        assert_same_plan(r, oracle_plan(n, *b, fixed, a))


def test_launch_count_and_matrix_optional(ctx):
    n = 5
    b = random_batch(np.random.default_rng(3), n, "ties", per_leg=(1, 2), bad=0.0)
    before = ctx.launches
    p = plan_tasks(ctx, n, *b)
    assert ctx.launches - before == 3 + 2 * n + 1          # leg key, leg index, leg matrix; 2n DP layers; backtrack
    assert p.leg_cost is None and p.leg_best is None
    assert_same_plan(p, oracle_plan(n, *b))


def test_minus_one_labels_never_influence_the_plan(ctx):
    rng = np.random.default_rng(11)
    for fixed, n in [(False, 6), (True, 9)]:
        lf, lt, cost, ok = random_batch(rng, n, "ties", per_leg=(1, 3), decoys=0.0, bad=0.05)
        assign = random_assign(rng, n) if fixed else None
        clean = plan_tasks(ctx, n, lf, lt, cost, ok, fixed, assign, with_matrix=True)
        # interleave decoys labelled -1 with every kind of cost, then map the indices back
        B = lf.size
        k = 3 * B
        where = np.sort(rng.choice(B + k, k, replace=False))
        keep = np.setdiff1d(np.arange(B + k), where)
        lf2, lt2 = np.full(B + k, -1, np.int32), rng.integers(-100, 100, B + k).astype(np.int32)
        cost2 = rng.choice([-1e300, -0.0, 0.0, -5.0, np.nan, -np.inf], B + k)
        ok2 = np.ones(B + k, np.int32)
        lf2[keep], lt2[keep], cost2[keep], ok2[keep] = lf, lt, cost, ok
        dirty = plan_tasks(ctx, n, lf2, lt2, cost2, ok2, fixed, assign, with_matrix=True)
        assert not np.isin(dirty.leg_best[dirty.leg_best >= 0], where).any()
        assert np.array_equal(keep[clean.leg_best[clean.leg_best >= 0]], dirty.leg_best[dirty.leg_best >= 0])
        assert clean.cost == dirty.cost and np.array_equal(clean.order, dirty.order)
        assert np.array_equal(clean.target, dirty.target)
        assert np.array_equal(np.where(clean.leg_cand >= 0, keep[np.maximum(clean.leg_cand, 0)], -1), dirty.leg_cand)
        assert_same_plan(dirty, oracle_plan(n, lf2, lt2, cost2, ok2, fixed, assign))


def test_invalid_inputs_return_einval_and_context_survives(ctx):
    lib = ctx.lib
    n = 3
    lf = np.array([0, 1, 4, -1], np.int32)
    lt = np.array([1, 4, 2, 99], np.int32)
    cost = np.array([1.0, 2.0, 3.0, 4.0])
    ok = np.ones(4, np.int32)

    def call(n_=n, lf_=lf, lt_=lt, fixed=False, assign=None, B=None):
        c = TaskCall(n_, lf_, lt_, fixed, assign)
        rc = lib.alore_task_plan(ctx.h, C.byref(c.task), c.B if B is None else B, capi.dptr(cost[:c.B].copy()),
                                 capi.iptr(ok[:c.B].copy()), C.byref(c.out))
        return rc, lib.alore_last_error(ctx.h).decode()

    bad = [
        dict(n_=0), dict(n_=capi.ALORE_TASK_MAX_FREE + 1), dict(n_=capi.ALORE_TASK_MAX_FIXED + 1, fixed=True),
        dict(lf_=np.array([0, 1, 4, -2], np.int32)),                  # label below -1
        dict(lf_=np.array([0, 1, 7, -1], np.int32)),                  # label >= P
        dict(lt_=np.array([1, 1, 2, 99], np.int32)),                  # from == to
        dict(lt_=np.array([1, 4, 7, 99], np.int32)),                  # leg_to >= P
        dict(lt_=np.array([-1, 4, 2, 99], np.int32)),                 # leg_to < 0 where leg_from >= 0
        dict(fixed=True, assign=np.array([4, 4, 6], np.int32)),        # not a bijection
        dict(fixed=True, assign=np.array([4, 5, 3], np.int32)),        # not a target
        dict(B=-1),
    ]
    for kw in bad:
        rc, msg = call(**kw)
        assert rc == -1 and msg.startswith("task plan:"), (kw, rc, msg)
    assert call()[0] == 0
    rng = np.random.default_rng(5)
    for fixed in (False, True):
        device_vs_oracle(ctx, 6, random_batch(rng, 6, "ties", per_leg=(1, 2), bad=0.0), fixed, random_assign(rng, 6) if fixed else None)


def test_batch_task_plan_on_a_real_optimised_batch(ctx):
    glx = gly = 240
    grid = workloads.random_map(glx, gly, 21, p_occ=0.0, p_unknown=0.0, wall=True, boxes=10, box_cells=(6, 16))
    m = make_sdf(ctx, glx, gly, 0.05, grid)
    m.updateESDF2d()
    n = 3
    pts = workloads.free_points(grid, m.geom(), m.distance_buffer_all_, 2 * n + 1, 3, min_clear=0.6)
    cands, lf, lt = task_leg_batch(pts, list(range(2 * n + 1)), [(0.0, 0.0), (0.0, math.pi / 2)])
    assert cands.B == 2 * (n + 2 * n * n)
    prm = capi.default_params()
    prm.alm_max_outer = 20
    db = DeviceBatch(ctx, cands)
    try:
        with pytest.raises(capi.AloreError):
            db.task_plan(n, lf, lt)                         # not run yet
        plans = []
        for safe in (0.6, 0.3):
            prm.safeDis = safe
            db.run(prm)
            for fixed, assign in [(False, None), (True, np.array([6, 4, 5], np.int32))]:
                dev = db.task_plan(n, lf, lt, fixed, assign, with_matrix=True)
                res = db.download()
                host = plan_tasks(ctx, n, lf, lt, res.cost, res.ok, fixed, assign, with_matrix=True)
                assert_same_plan(dev, host)
                assert_same_plan(dev, oracle_plan(n, lf, lt, res.cost, res.ok, fixed, assign))
                if dev.feasible:
                    assert_valid_plan(dev, n, fixed, assign)
                plans.append((dev, res.cost.copy()))
        assert plans[0][0].feasible
        # the second run's parameters change the optimised costs, and the plan reads the new results
        assert not np.array_equal(plans[0][1], plans[2][1])
        assert not np.array_equal(plans[0][0].leg_cost, plans[2][0].leg_cost)
    finally:
        db.close()
        m.close()
