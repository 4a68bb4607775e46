"""Entry points beside the main optimizer parity suite: the coefficient-space penalty kernel against the oracle, the
device-pointer penalty entry and the reusable pinned result store."""
import numpy as np
import pytest

import oracle_lib
from alore_legged_manipulator_b200 import capi, workloads
from test_optimizer_gpu import leg_batch, portable_trig, world  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu


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
