"""The opt-in ESDF implementations must stay bit-identical to the default ones and to the oracle:
  ALORE_ESDF_DC=1     the divide-and-conquer ESDF column pass instead of the register-window / expanding search
  ALORE_ESDF_NO_BAND  the round-1 per-cell far search instead of the band lower-envelope kernel
  ALORE_ESDF_SB       rows per band of the lower-envelope kernel (32/64/128/256)
The library reads these knobs at call time, so a test can flip them around a call.  Also here: the device-pointer
penalty entry, the coefficient-space penalty kernel against the oracle, and the reusable pinned result store."""
import os
from contextlib import contextmanager

import numpy as np
import pytest

import oracle_lib
from alore_legged_manipulator_b200 import capi, workloads
from test_esdf_gpu import make_sdf
from test_optimizer_gpu import leg_batch, portable_trig, world  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu


@contextmanager
def env(**kw):
    old = {k: os.environ.get(k) for k in kw}
    os.environ.update({k: str(v) for k, v in kw.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.mark.parametrize("shape", [(257, 130), (64, 700), (1024, 1024)])
def test_esdf_divide_and_conquer_column_pass_bit_exact(shape):
    import alore_legged_manipulator_b200 as alore
    ctx = alore.Context(0)                # its own context: one context holds one device-resident map
    glx, gly = shape
    for seed, kw in ((1, dict(p_occ=0.02, p_unknown=0.01)), (2, dict(p_occ=0.0, p_unknown=0.0, boxes=6, box_cells=(4, 40))),
                     (3, dict(p_occ=0.7, p_unknown=0.05))):
        grid = workloads.random_map(glx, gly, seed, **kw)
        m = make_sdf(ctx, glx, gly, 0.05, grid)
        with env(ALORE_ESDF_DC=1):
            m.updateESDF2d()
        ref = np.full(glx * gly, np.finfo(np.float64).max)
        mn, mx = m.esdf_window()
        oracle_lib.esdf_update(m.geom(), grid, mn, mx, ref)
        assert np.array_equal(m.distance_buffer_all_.view(np.uint64), ref.view(np.uint64)), (shape, seed)
        m.close()
    ctx.close()


@pytest.mark.parametrize("knobs", [dict(ALORE_ESDF_NO_BAND=1), dict(ALORE_ESDF_SB=32), dict(ALORE_ESDF_SB=64),
                                   dict(ALORE_ESDF_SB=128), dict(ALORE_ESDF_SB=256)])
def test_esdf_far_field_paths_bit_exact(knobs):
    """Far cells (large empty / solid regions): the band lower-envelope kernel at every band height and the round-1
    per-cell search must all reproduce the oracle bit for bit, on maps that are nearly empty, nearly solid and mixed."""
    import alore_legged_manipulator_b200 as alore
    ctx = alore.Context(0)
    for (glx, gly), seed, kw in (((700, 300), 2, dict(p_occ=0.0, p_unknown=0.0, boxes=5, box_cells=(4, 40))),
                                 ((513, 257), 3, dict(p_occ=0.0, p_unknown=0.0, wall=False, boxes=1, box_cells=(2, 3))),
                                 ((300, 900), 4, dict(p_occ=0.0, p_unknown=0.0, boxes=30, box_cells=(40, 200))),
                                 ((1100, 260), 5, dict(p_occ=1.0, p_unknown=0.0))):
        grid = workloads.random_map(glx, gly, seed, **kw)
        if kw.get("p_occ") == 1.0:                           # a solid world with one free pocket and one free cell
            g2 = grid.reshape(glx, gly)
            g2[500:520, 100:130] = workloads.UNOCCUPIED
            g2[40, 200] = workloads.UNOCCUPIED
        m = make_sdf(ctx, glx, gly, 0.05, grid)
        with env(**knobs):
            m.updateESDF2d()
        ref = np.full(glx * gly, np.finfo(np.float64).max)
        mn, mx = m.esdf_window()
        oracle_lib.esdf_update(m.geom(), grid, mn, mx, ref)
        assert np.array_equal(m.distance_buffer_all_.view(np.uint64), ref.view(np.uint64)), ((glx, gly), seed, knobs)
        m.close()
    ctx.close()


def test_penalty_kernel_bit_identical_to_oracle(world, portable_trig):
    m, prm, pl, grid = world
    po, coeffs, T, s_xy, f_xy = workloads.random_spline_batch(24, 40, m.geom(), m.distance_buffer_all_, grid, seed=5)
    cost, gC, gT, _ = pl.penalty_batch(po, coeffs, T, s_xy, f_xy)
    cr, gCr, gTr, _ = oracle_lib.penalty_batch(prm, m.geom(), m.distance_buffer_all_, po, coeffs, T, s_xy, f_xy, 4)
    assert np.array_equal(cost, cr) and np.array_equal(gC, gCr) and np.array_equal(gT, gTr)


def test_device_penalty_entry_refuses_undeclared_piece_counts(world, ctx):
    """alore_penalty_batch_dev sizes its shared memory and scratch from max_pieces: a trajectory with more pieces than
    declared is not evaluated (cost NaN), nothing is written out of bounds (ADVICE r1: Nmax guess from total / B)."""
    import ctypes as C
    import torch
    m, prm, pl, grid = world
    po, coeffs, T, s_xy, f_xy = workloads.random_spline_batch(2, 6, m.geom(), m.distance_buffer_all_, grid, seed=7)
    po = np.array([0, 2, 8], np.int32)                  # pieces (2, 6): total divisible by B, NOT uniform
    dev = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()
    d = [dev(po, np.int32), dev(coeffs[:8], np.float64), dev(T[:8], np.float64), dev(s_xy, np.float64), dev(f_xy, np.float64)]
    o = [torch.zeros(n, dtype=torch.float64, device="cuda") for n in (2, 8 * 12, 8, 4)]
    pv = lambda t: C.c_void_p(t.data_ptr())
    for declared, want_nan in ((4, True), (6, False)):
        ctx.check(ctx.lib.alore_penalty_batch_dev(ctx.h, C.byref(prm), 2, declared, *[pv(t) for t in d], *[pv(t) for t in o], None))
        torch.cuda.synchronize()
        cost = o[0].cpu().numpy()
        assert np.isfinite(cost[0]) and bool(np.isnan(cost[1])) == want_nan


def test_reusable_pinned_result_store_gives_the_same_results(world, ctx):
    """`minco_plan_batch(cands, out=store)`: one page-locked result store reused by batches of different sizes."""
    m, prm, pl, grid = world
    big, small = leg_batch(world, max_legs=48), leg_batch(world, max_legs=20)
    store = capi.ResultBatch(capacity=(big.B, big.total_pieces)).pin(ctx)
    try:
        for cands in (big.pin(ctx), small, big):
            a = pl.minco_plan_batch(cands)
            b = pl.minco_plan_batch(cands, out=store)
            assert b is store and b.coeffs.shape == a.coeffs.shape
            for f in capi.ResultBatch._FIELDS:
                assert np.array_equal(getattr(a, f), getattr(b, f)), f
        with pytest.raises(ValueError):
            capi.ResultBatch(capacity=(4, 16)).bind(big.B, big.total_pieces)
    finally:
        big.unpin()
        store.unpin()
