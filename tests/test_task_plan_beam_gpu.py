"""GPU tests of the bounded-width task plan (alore_task_plan_beam, alore_batch_task_plan_beam) against the sequential
oracle orc_task_plan_beam and the exact solver, bit for bit: result bits, feasibility, order, targets, leg candidates,
the leg matrix and the `exact` flag."""
import ctypes as C
import math

import numpy as np
import pytest

from alore_legged_manipulator_b200 import capi, plan_tasks, workloads
from alore_legged_manipulator_b200.ms_planner import DeviceBatch
from alore_legged_manipulator_b200.task_planner import TaskCall
from task_plan_util import (assert_same_beam_plan, assert_same_plan, assert_valid_plan, oracle_plan_beam, random_assign,
                            random_batch, task_leg_batch)
from test_esdf_gpu import make_sdf

pytestmark = pytest.mark.gpu
MAXW = capi.ALORE_TASK_MAX_WIDTH


def device_vs_oracle(ctx, n, width, batch, fixed=False, assign=None):
    got = plan_tasks(ctx, n, *batch, fixed, assign, with_matrix=True, width=width)
    ref = oracle_plan_beam(n, width, *batch, fixed, assign)
    assert_same_beam_plan(got, ref)
    if got.feasible:
        assert_valid_plan(got, n, fixed, assign)
    return got


@pytest.mark.parametrize("fixed", [False, True])
@pytest.mark.parametrize("n", [1, 2, 5, 9, 13, 17, 24, 31, 32])
def test_device_equals_oracle(ctx, n, fixed):
    rng = np.random.default_rng(10 * n + fixed)
    widths = [1, 2, 7, 64, 1000, 4096] + ([MAXW] if n <= 5 else [])
    feasible = truncated = 0
    for w in widths:
        assign = random_assign(rng, n) if fixed and w % 2 == 0 else None
        # ties-heavy: truncation cuts through runs of equal values, and the merge sees equal minima
        p = device_vs_oracle(ctx, n, w, random_batch(rng, n, "ties", per_leg=(1, 2), bad=0.02), fixed, assign)
        feasible += p.feasible
        truncated += not p.exact
        if w in (1, 64, 4096):                           # infeasible mixes: missing legs, NaN / inf / ok = 0 candidates
            device_vs_oracle(ctx, n, w, random_batch(rng, n, "mixed", per_leg=(0, 2)), fixed, assign)
    assert feasible > 0
    assert truncated > 0 or n <= 2


@pytest.mark.parametrize("fixed", [False, True])
def test_wide_beam_equals_exact_solver(ctx, fixed):
    rng = np.random.default_rng(77 + fixed)
    for n in range(1, (15 if fixed else 8) + 1):
        for kind in ["ties", "mixed"]:
            assign = random_assign(rng, n) if fixed and kind == "mixed" else None
            b = random_batch(rng, n, kind, per_leg=(1, 2), bad=0.02)
            beam = plan_tasks(ctx, n, *b, fixed, assign, with_matrix=True, width=MAXW)
            assert beam.exact is True
            assert_same_plan(beam, plan_tasks(ctx, n, *b, fixed, assign, with_matrix=True))


def test_alternating_with_the_exact_solver_on_one_context(ctx):
    calls = [(4, False, None), (30, False, 4096), (2, True, 7), (20, True, None), (12, False, None), (32, True, MAXW),
             (3, False, 1), (16, True, 64), (9, False, MAXW), (1, True, None), (32, False, 1000), (6, True, 2)]
    rng = np.random.default_rng(19)
    cases = [(n, fixed, w, random_assign(rng, n) if fixed else None, random_batch(rng, n, "ties", per_leg=(1, 2), bad=0.02))
             for n, fixed, w in calls]
    reused = [plan_tasks(ctx, n, *b, fixed, a, with_matrix=True, width=w) for n, fixed, w, a, b in cases]
    for (n, fixed, w, a, b), r in zip(cases, reused):
        fresh_ctx = capi.Context(0)
        try:
            assert_same_beam_plan(r, plan_tasks(fresh_ctx, n, *b, fixed, a, with_matrix=True, width=w))
        finally:
            fresh_ctx.close()
        assert (r.exact is None) == (w is None)
        if w is not None and n >= 16:
            assert_same_beam_plan(r, oracle_plan_beam(n, w, *b, fixed, a))


def test_minus_one_labels_never_influence_the_plan(ctx):
    rng = np.random.default_rng(23)
    for fixed, n, w in [(False, 14, 64), (True, 25, 7)]:
        lf, lt, cost, ok = random_batch(rng, n, "ties", per_leg=(1, 2), decoys=0.0, bad=0.0)
        assign = random_assign(rng, n) if fixed else None
        clean = plan_tasks(ctx, n, lf, lt, cost, ok, fixed, assign, with_matrix=True, width=w)
        B = lf.size
        k = 2 * B
        where = np.sort(rng.choice(B + k, k, replace=False))
        keep = np.setdiff1d(np.arange(B + k), where)
        lf2, lt2 = np.full(B + k, -1, np.int32), rng.integers(-100, 100, B + k).astype(np.int32)
        cost2 = rng.choice([-1e300, -0.0, 0.0, -5.0, np.nan, -np.inf], B + k)
        ok2 = np.ones(B + k, np.int32)
        lf2[keep], lt2[keep], cost2[keep], ok2[keep] = lf, lt, cost, ok
        dirty = plan_tasks(ctx, n, lf2, lt2, cost2, ok2, fixed, assign, with_matrix=True, width=w)
        assert clean.feasible
        assert math.copysign(1, clean.cost) == math.copysign(1, dirty.cost) and clean.cost == dirty.cost
        assert np.array_equal(clean.order, dirty.order) and np.array_equal(clean.target, dirty.target)
        assert np.array_equal(keep[clean.leg_cand], dirty.leg_cand)
        assert clean.exact == dirty.exact
        assert_same_beam_plan(dirty, oracle_plan_beam(n, w, lf2, lt2, cost2, ok2, fixed, assign))


def test_invalid_inputs_return_einval_and_context_survives(ctx):
    lib = ctx.lib
    n = 3
    lf = np.array([0, 1, 4, -1], np.int32)
    lt = np.array([1, 4, 2, 99], np.int32)
    cost = np.array([1.0, 2.0, 3.0, 4.0])
    ok = np.ones(4, np.int32)

    def call(n_=n, lf_=lf, lt_=lt, fixed=False, assign=None, width=4):
        c = TaskCall(n_, lf_, lt_, fixed, assign)
        exact = C.c_int32(-7)
        rc = lib.alore_task_plan_beam(ctx.h, C.byref(c.task), width, c.B, capi.dptr(cost[:c.B].copy()),
                                      capi.iptr(ok[:c.B].copy()), C.byref(c.out), C.byref(exact))
        return rc, lib.alore_last_error(ctx.h).decode(), exact.value

    bad = [
        dict(width=0), dict(width=MAXW + 1), dict(width=-3),
        dict(n_=0), dict(n_=capi.ALORE_TASK_MAX_BEAM_N + 1), dict(n_=capi.ALORE_TASK_MAX_BEAM_N + 1, fixed=True),
        dict(lf_=np.array([0, 1, 4, -2], np.int32)),                  # label below -1
        dict(lf_=np.array([0, 1, 7, -1], np.int32)),                  # label >= P
        dict(lt_=np.array([1, 1, 2, 99], np.int32)),                  # from == to
        dict(lt_=np.array([-1, 4, 2, 99], np.int32)),                 # leg_to < 0 where leg_from >= 0
        dict(fixed=True, assign=np.array([4, 4, 6], np.int32)),        # not a bijection
        dict(fixed=True, assign=np.array([4, 5, 3], np.int32)),        # not a target
    ]
    before = ctx.launches
    for kw in bad:
        rc, msg, exact = call(**kw)
        assert rc == -1 and msg.startswith("task plan:"), (kw, rc, msg)
        assert exact == -7
    assert ctx.launches == before                                      # refused before any launch
    rc, _, exact = call()
    assert rc == 0 and exact == 1
    rng = np.random.default_rng(5)
    for fixed in (False, True):
        device_vs_oracle(ctx, 32, 16, random_batch(rng, 32, "ties", per_leg=(1, 1), bad=0.0), fixed,
                         random_assign(rng, 32) if fixed else None)


@pytest.mark.parametrize("fixed", [False, True])
def test_launch_count_formula(ctx, fixed):
    n = 7
    b = random_batch(np.random.default_rng(3), n, "ties", per_leg=(1, 2), bad=0.0)
    digits = 17                                          # cost key 8, O 4, T 4, last 1 in both modes
    for w in (1, 100):
        before = ctx.launches
        p = plan_tasks(ctx, n, *b, fixed, None, width=w)
        # leg key, leg index, leg matrix; per layer 2 expand + merge + radix-select digits + keep; backtrack
        assert ctx.launches - before == 3 + 2 * n * (4 + digits) + 1
        assert p.leg_cost is None and p.leg_best is None
        assert_same_beam_plan(p, oracle_plan_beam(n, w, *b, fixed, None, with_matrix=False))


def test_batch_task_plan_beam_on_a_real_optimised_batch(ctx):
    glx = gly = 240
    grid = workloads.random_map(glx, gly, 21, p_occ=0.0, p_unknown=0.0, wall=True, boxes=10, box_cells=(6, 16))
    m = make_sdf(ctx, glx, gly, 0.05, grid)
    m.updateESDF2d()
    n = 4
    pts = workloads.free_points(grid, m.geom(), m.distance_buffer_all_, 2 * n + 1, 3, min_clear=0.6)
    cands, lf, lt = task_leg_batch(pts, list(range(2 * n + 1)), [(0.0, 0.0), (0.0, math.pi / 2)])
    prm = capi.default_params()
    prm.alm_max_outer = 20
    db = DeviceBatch(ctx, cands)
    try:
        with pytest.raises(capi.AloreError):
            db.task_plan(n, lf, lt, width=4)              # not run yet
        db.run(prm)
        res = db.download()
        feasible = 0
        for fixed, assign in [(False, None), (True, np.array([7, 8, 5, 6], np.int32))]:
            for w in (1, 3, 40, MAXW):
                dev = db.task_plan(n, lf, lt, fixed, assign, with_matrix=True, width=w)
                host = plan_tasks(ctx, n, lf, lt, res.cost, res.ok, fixed, assign, with_matrix=True, width=w)
                assert_same_beam_plan(dev, host)
                assert_same_beam_plan(dev, oracle_plan_beam(n, w, lf, lt, res.cost, res.ok, fixed, assign))
                if dev.feasible:
                    assert_valid_plan(dev, n, fixed, assign)
                feasible += dev.feasible
                if w == MAXW:
                    assert dev.exact
                    assert_same_plan(dev, db.task_plan(n, lf, lt, fixed, assign, with_matrix=True))
        assert feasible > 0
    finally:
        db.close()
        m.close()
