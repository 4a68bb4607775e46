"""GPU parity off the default parameters: every L-BFGS exit, history-ring wrap, ALM caps and tolerance sets, sampling
resolutions K / KF from 1 to 64, lateral check-points, the ICR and direct v/omega models, map edges and per-candidate
ALM state.  Every case is bit-identical to the CPU oracle (portable-trig contract, DESIGN.md section 3) AND asserts
that it reached the path it is named for; tests/test_param_space_oracle.py anchors the oracle on the same inputs."""
import math

import numpy as np
import pytest

import oracle_lib
from alore_legged_manipulator_b200 import capi, front_end, workloads
from alore_legged_manipulator_b200.ms_planner import DeviceBatch, MSPlanner
from test_esdf_gpu import make_sdf
from test_optimizer_gpu import check_results, leg_batch
from test_param_space_oracle import (CHECKPOINTS, set_checkpoints, stationary_known_answer, stationary_pose,
                                     stationary_spline)

pytestmark = pytest.mark.gpu

# lbfgs.hpp return codes
LBFGS_CONVERGENCE, LBFGS_STOP = 0, 1
LBFGSERR_INVALID_MEMSIZE = -1022
LBFGSERR_INVALID_FDECCOEFF = -1016
LBFGSERR_MINIMUMSTEP, LBFGSERR_MAXIMUMSTEP, LBFGSERR_MAXIMUMLINESEARCH = -1011, -1010, -1009
LBFGSERR_MAXIMUMITERATION, LBFGSERR_WIDTHTOOSMALL = -1008, -1007


@pytest.fixture(scope="module")
def portable_trig():
    lib = oracle_lib.load()
    lib.orc_set_trig_portable(1)
    yield
    lib.orc_set_trig_portable(0)


@pytest.fixture(scope="module")
def world(ctx):
    glx = gly = 400
    grid = workloads.random_map(glx, gly, 7, p_occ=0.0, p_unknown=0.0, wall=True, boxes=25, box_cells=(6, 24))
    m = make_sdf(ctx, glx, gly, 0.05, grid)
    m.updateESDF2d()
    prm = capi.default_params()
    prm.alm_max_outer = 20
    return m, prm, MSPlanner(ctx, prm, m), grid


def params(**kw) -> capi.Params:
    p = capi.default_params()
    p.alm_max_outer = 4
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def optimise(world, ctx, prm, cands):
    """Whole optimisations on the device and in the oracle: bit-identical; returns the oracle's results."""
    m = world[0]
    res = MSPlanner(ctx, prm, m).minco_plan_batch(cands)
    ref = oracle_lib.opt_batch(prm, m.geom(), m.distance_buffer_all_, cands, 8)
    assert check_results(res, ref, cands) == 0.0
    return ref


def costs(world, ctx, prm, cands, x, stages=(0, 1), lam=None, rho=None, safe_dis=None):
    """cost_batch on the device against the oracle's cost callback, bit for bit; returns the oracle's costs."""
    m = world[0]
    pl = MSPlanner(ctx, prm, m)
    out = []
    for stage in stages:
        cost, g, err = pl.cost_batch(cands, stage, x, lam=lam, rho=rho, safe_dis=safe_dis)
        for b in range(cands.B):
            o, n = cands.x_offset(b), 3 * int(cands.piece_off[b + 1] - cands.piece_off[b]) - 1
            kw = {} if lam is None else dict(lam=lam[b], rho=rho[b], safe_dis=safe_dis[b])
            cr, gr, er = oracle_lib.cost(prm, m.geom(), m.distance_buffer_all_, cands, b, stage, x[o:o + n], **kw)
            assert cost[b] == cr and np.array_equal(g[o:o + n], gr, equal_nan=True), (stage, b)
            if stage == 1:
                assert np.array_equal(err[b], er, equal_nan=True)
            out.append(cr)
    return np.array(out)


def penalties(world, ctx, prm, po, coeffs, T, s_xy, f_xy):
    m = world[0]
    got = MSPlanner(ctx, prm, m).penalty_batch(po, coeffs, T, s_xy, f_xy)
    ref = oracle_lib.penalty_batch(prm, m.geom(), m.distance_buffer_all_, po, np.ascontiguousarray(coeffs),
                                   np.ascontiguousarray(T), np.ascontiguousarray(s_xy), np.ascontiguousarray(f_xy), 8)
    for a, r in zip(got, ref):
        # equal_nan: at the map edges the bilinear gradient can mix DBL_MAX cells (inf - inf); NaN payloads may differ
        assert np.array_equal(a, r, equal_nan=True)
    return ref


def final_collisions(world, ctx, prm, po, coeffs, T, s_xy):
    m = world[0]
    col, md = MSPlanner(ctx, prm, m).check_final_collision_batch(po, coeffs, T, s_xy)
    for b in range(po.size - 1):
        sl = slice(int(po[b]), int(po[b + 1]))
        c, d = oracle_lib.final_collision(prm, m.geom(), m.distance_buffer_all_, sl.stop - sl.start,
                                          coeffs[sl], T[sl], s_xy[b])
        assert col[b] == c and md[b] == d, b
    return col, md


def ragged(po, coeffs, T, s_xy, f_xy):
    """Drops trailing pieces of every other trajectory."""
    keep, npo = [], [0]
    for b in range(po.size - 1):
        n = int(po[b + 1] - po[b])
        n = n if b % 2 == 0 else max(1, n - 1 - b % 5)
        keep.extend(range(int(po[b]), int(po[b]) + n))
        npo.append(npo[-1] + n)
    return np.array(npo, np.int32), np.ascontiguousarray(coeffs[keep]), np.ascontiguousarray(T[keep]), s_xy, f_xy


def perturbed_x(cands, scale, seed):
    rng = np.random.default_rng(seed)
    return np.concatenate([oracle_lib.initial_x(cands, b) for b in range(cands.B)]) + scale * rng.normal(size=cands.n_vars())


# ---- 1. L-BFGS exits and history ----------------------------------------------------------------------------------
@pytest.mark.parametrize("mem_a,mem_b", [(1, 3), (2, 5), (3, 1), (5, 2)])
def test_lbfgs_small_memory_and_history_wrap(world, portable_trig, ctx, mem_a, mem_b):
    prm = params()
    prm.path_lbfgs.mem_size, prm.lbfgs.mem_size = mem_a, mem_b
    cands = leg_batch(world, max_legs=12, seed=mem_a)
    optimise(world, ctx, prm, cands)
    # one candidate, one optimiser run per stage: its iteration count proves the ring (m = min(mem_size, mcap)) wrapped
    one = cands.subset([0])
    prm1 = params(alm_max_outer=1, safeReplanMaxTime=1)
    prm1.path_lbfgs.mem_size = prm1.lbfgs.mem_size = min(mem_a, mem_b)
    db = DeviceBatch(ctx, one)
    db.run(prm1)
    r = db.download()
    _, _, iters = db.stats()
    db.close()
    m = world[0]
    ref = oracle_lib.opt_batch(prm1, m.geom(), m.distance_buffer_all_, one, 1)
    check_results(r, ref, one)
    assert iters > 2 * 2 * min(mem_a, mem_b) + 4, iters


EXITS = {
    "max_iterations": (dict(max_iterations=3, past=0), {LBFGSERR_MAXIMUMITERATION}),
    "max_linesearch_1": (dict(max_linesearch=1), {LBFGSERR_MAXIMUMLINESEARCH}),
    "max_linesearch_2": (dict(max_linesearch=2), {LBFGSERR_MAXIMUMLINESEARCH}),
    "g_epsilon_first_check": (dict(g_epsilon=1e12, past=0), {LBFGS_CONVERGENCE}),
    "g_epsilon": (dict(g_epsilon=2e-2, past=0), {LBFGS_CONVERGENCE}),
    "min_step": (dict(min_step=0.3), {LBFGSERR_MINIMUMSTEP}),
    "max_step": (dict(max_step=1e-7), {LBFGSERR_MAXIMUMSTEP}),
    "machine_prec": (dict(machine_prec=0.9), {LBFGSERR_WIDTHTOOSMALL}),
    "past_64": (dict(past=64, delta=1e-2), {LBFGS_STOP}),
    "invalid_mem_size": (dict(mem_size=0), {LBFGSERR_INVALID_MEMSIZE}),
    "invalid_f_dec_coeff": (dict(f_dec_coeff=1.0), {LBFGSERR_INVALID_FDECCOEFF}),
}


@pytest.mark.parametrize("case", list(EXITS))
def test_lbfgs_exit_codes(world, portable_trig, ctx, case):
    """Stage-B settings (the status reported is the last stage-B optimiser's); each case must see its code."""
    kw, codes = EXITS[case]
    prm = params(alm_max_outer=2)
    for k, v in kw.items():
        setattr(prm.lbfgs, k, v)
    if case == "invalid_mem_size":
        prm.path_lbfgs.mem_size = 0
    if case == "past_64":           # both stage-A `past` branches in one batch: |initial tail s| against the horizon
        prm.path_lbfgs.past, prm.normal_past, prm.shot_path_past = 64, 64, 5
    cands = leg_batch(world, max_legs=16, seed=3)
    if case == "past_64":
        tail = np.abs(cands.final_state[:, 1, 0])
        prm.shot_path_horizon = float(np.median(tail))
        assert np.any(tail < prm.shot_path_horizon) and np.any(tail >= prm.shot_path_horizon)
    ref = optimise(world, ctx, prm, cands)
    seen = set(int(s) for s in ref.status)
    assert codes & seen, (case, seen)
    if case in ("max_iterations", "g_epsilon_first_check", "invalid_mem_size", "invalid_f_dec_coeff"):
        assert seen == codes, (case, seen)


def test_cautious_update_skip(world, portable_trig, ctx):
    """cautious_factor so large that every history update is skipped (steepest descent): the result differs from the
    default factor's, and both are bit-identical to the oracle."""
    cands = leg_batch(world, max_legs=8, seed=4)
    base = optimise(world, ctx, params(), cands)
    prm = params()
    prm.lbfgs.cautious_factor = prm.path_lbfgs.cautious_factor = 1e30
    skip = optimise(world, ctx, prm, cands)
    assert not np.array_equal(base.coeffs, skip.coeffs) and np.any(base.evals != skip.evals)


# ---- 2. ALM ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("capped", ["normal", "cut"])
def test_alm_hard_cap_and_tolerance_sets(world, portable_trig, ctx, capped):
    """alm_max_outer = 0 (hard cap only): the set with tolerance 0 runs to ALORE_ALM_HARD_CAP and saturates rho at its
    RhoMax; the other set stops after its first outer iteration.  safeReplanMaxTime = 1."""
    m, _, _, grid = world
    prm = params(alm_max_outer=0, safeReplanMaxTime=1)
    big = 1e9
    prm.EqualTolerance[0] = 0.0 if capped == "normal" else big
    prm.CutEqualTolerance[0] = 0.0 if capped == "cut" else big
    prm.EqualRhoMax[0] = prm.EqualRhoMax[1] = 3e4
    prm.CutEqualRhoMax[0] = prm.CutEqualRhoMax[1] = 2e3
    fe = front_end.FrontEndParams()
    fe.trajCutLength = 4.0
    pts = workloads.free_points(grid, m.geom(), m.distance_buffer_all_, 6, 11, min_clear=0.5)
    legs = workloads.leg_candidates(pts, headings=(0.0,), fe=fe, max_legs=30)
    cut, normal = np.flatnonzero(legs.if_cut == 1)[:3], np.flatnonzero(legs.if_cut == 0)[:3]
    assert len(cut) and len(normal)
    cands = legs.subset(list(cut) + list(normal))
    ref = optimise(world, ctx, prm, cands)
    is_capped = (cands.if_cut == 1) if capped == "cut" else (cands.if_cut == 0)
    assert np.all(ref.alm_iters[is_capped] == capi.ALORE_ALM_HARD_CAP)
    assert np.all(ref.alm_iters[~is_capped] == 1)
    assert np.all(ref.replans == 1)


# ---- 3. sampling resolutions -------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,KF", [(1, 2), (2, 17), (3, 1), (7, 64), (16, 2), (33, 17), (64, 1)])
def test_sampling_resolutions(world, portable_trig, ctx, K, KF):
    m, _, _, grid = world
    prm = params(sparseResolution=K, finalSafeDisCheckNum=KF, alm_max_outer=2)
    dflt = params(alm_max_outer=2)
    cands = leg_batch(world, max_legs=6, seed=K, dogleg=0.5)
    x = perturbed_x(cands, 0.03, K)
    c = costs(world, ctx, prm, cands, x)
    assert not np.array_equal(c, costs(world, ctx, dflt, cands, x))       # K is what was evaluated
    po, coeffs, T, s_xy, f_xy = workloads.random_spline_batch(8, 10, m.geom(), m.distance_buffer_all_, grid, seed=K)
    pc = penalties(world, ctx, prm, *ragged(po, coeffs, T, s_xy, f_xy))
    assert not np.array_equal(pc[0], penalties(world, ctx, dflt, *ragged(po, coeffs, T, s_xy, f_xy))[0])
    prm_f = params(sparseResolution=K, finalSafeDisCheckNum=KF, finalMinSafeDis=0.25)
    col, md = final_collisions(world, ctx, prm_f, po, coeffs, T, s_xy)
    col8, md8 = final_collisions(world, ctx, params(finalMinSafeDis=0.25), po, coeffs, T, s_xy)
    assert not np.array_equal(md, md8) or KF == 16                       # KF is what was sampled
    optimise(world, ctx, prm, leg_batch(world, max_legs=4, seed=K + 1))


def test_sixty_four_samples_log_more_than_512_terms(world, portable_trig, ctx):
    """K = 64, 8 check-points, low limits and a safety margin no cell reaches: every check-point of every even sample
    logs a collision term, 65 x 8 = 520 > 512 (the shared packing buffer) in one piece, plus the limit terms."""
    m, _, _, grid = world
    prm = params(sparseResolution=64, max_vel=0.05, max_acc=0.05, max_centripetal_acc=0.01, safeDis=50.0)
    set_checkpoints(prm, CHECKPOINTS[8])
    po, coeffs, T, s_xy, f_xy = workloads.random_spline_batch(6, 4, m.geom(), m.distance_buffer_all_, grid, seed=17)
    # starts near the centre: every sample and check-point of these <= 2.4 m splines stays well inside the map
    s_xy = np.array([[0.5 * (b - 3), 0.3 * b - 1.0] for b in range(6)])
    geom = m.geom()
    t = np.linspace(0.0, 1.0, 401)
    for b in range(6):
        reach = 0.5                      # check-point offsets + path length (|ds/dt| integrated densely)
        for i in range(int(po[b]), int(po[b + 1])):
            ds = sum(k * coeffs[i, k, 1] * (t * T[i]) ** (k - 1) for k in range(1, 6))
            reach += float(np.mean(np.abs(ds))) * T[i] * 1.01
        assert geom.x_lower + reach < s_xy[b, 0] < geom.x_upper - reach
        assert geom.y_lower + reach < s_xy[b, 1] < geom.y_upper - reach
    assert np.max(m.distance_buffer_all_[m.distance_buffer_all_ < 1e9]) < prm.safeDis
    cost, _, _, _ = penalties(world, ctx, prm, po, coeffs, T, s_xy, f_xy)
    prm0 = params(sparseResolution=64, max_vel=0.05, max_acc=0.05, max_centripetal_acc=0.01, safeDis=50.0)
    set_checkpoints(prm0, CHECKPOINTS[8])
    prm0.pw_collision = 0.0
    assert np.all(penalties(world, ctx, prm0, po, coeffs, T, s_xy, f_xy)[0] != cost)
    assert (2 * 64 // 2 + 1) * prm.n_checkpoints > 512


# ---- 4. check-point geometry and model variants --------------------------------------------------------------------
MODELS = {
    "no_checkpoints": dict(cps=[]),
    "three_lateral": dict(cps=CHECKPOINTS[3]),
    "eight_lateral": dict(cps=CHECKPOINTS[8]),
    "icr": dict(if_standard_diff=0, cps=CHECKPOINTS[3]),
    "direct_v_omega": dict(if_directly_constrain_v_omega=1, cps=CHECKPOINTS[3]),
}


def model_params(variant, **extra):
    kw = dict(MODELS[variant])
    cps = kw.pop("cps")
    prm = params(min_vel=0.0, **kw, **extra)
    set_checkpoints(prm, cps)
    return prm, cps


@pytest.mark.parametrize("variant", list(MODELS))
def test_checkpoints_and_models(world, portable_trig, ctx, variant):
    m, _, _, grid = world
    prm, cps = model_params(variant, safeDis=0.9)
    cands = leg_batch(world, max_legs=8, seed=6, dogleg=0.6)
    x = perturbed_x(cands, 0.05, 6)
    c = costs(world, ctx, prm, cands, x)
    po, coeffs, T, s_xy, f_xy = workloads.random_spline_batch(16, 8, m.geom(), m.distance_buffer_all_, grid, seed=23)
    pc = penalties(world, ctx, prm, po, coeffs, T, s_xy, f_xy)[0]
    pr = penalties(world, ctx, prm, *ragged(po, coeffs, T, s_xy, f_xy))[0]
    # the lateral check-points fire: moving only their lateral offsets inward changes the cost
    inward, _ = model_params(variant, safeDis=0.9)
    for k, (cx, cy) in enumerate(cps):
        inward.check_point[k][1] = 0.0
    pin = penalties(world, ctx, inward, po, coeffs, T, s_xy, f_xy)[0]
    if cps:
        assert np.any(pin != pc) and not np.array_equal(costs(world, ctx, inward, cands, x, stages=(1,)), c[cands.B:])
    else:
        nocol, _ = model_params(variant, safeDis=0.9, pw_collision=0.0)
        assert np.array_equal(penalties(world, ctx, nocol, po, coeffs, T, s_xy, f_xy)[0], pc)
    assert pr.shape == (16,)
    final_collisions(world, ctx, model_params(variant, finalMinSafeDis=0.25)[0], po, coeffs, T, s_xy)
    optimise(world, ctx, prm, leg_batch(world, max_legs=6, seed=8))


# ---- the stationary known answer, on the device --------------------------------------------------------------------
@pytest.mark.parametrize("ncp", [1, 3, 8])
@pytest.mark.parametrize("K", [1, 2, 3, 8, 64])
def test_stationary_collision_known_answer_on_device(world, portable_trig, ctx, K, ncp):
    m = world[0]
    geom, dist = m.geom(), m.distance_buffer_all_
    prm = params(sparseResolution=K, min_vel=0.0)
    prm.EqualLambda[0] = prm.EqualLambda[1] = 0.0
    set_checkpoints(prm, CHECKPOINTS[ncp])
    xy, theta, prm.safeDis = stationary_pose(geom, dist, CHECKPOINTS[ncp])
    T = [0.4, 0.7, 1.3]
    cost = penalties(world, ctx, prm, *stationary_spline(xy, theta, 2.5, T))[0]
    want = stationary_known_answer(prm, geom, dist, xy, theta, T)[0]
    assert want > 0.0 and math.isclose(cost[0], want, rel_tol=1e-13)


# ---- 5. map edges ------------------------------------------------------------------------------------------------------
def test_map_edges(world, portable_trig, ctx):
    m, _, _, grid = world
    g = m.geom()
    gi = g.grid_interval
    # standing-still splines (the samples sit exactly at their start point) and straight runs across the boundary
    poses = [(g.x_lower, 0.3, 0.0), (g.x_upper, -0.4, 1.0), (0.2, g.y_upper, 2.0), (g.x_upper, g.y_upper, 0.5),
             (g.x_upper - gi, 0.1, 0.0), (0.0, g.y_upper - 2 * gi, -1.2), (g.x_lower + 0.5 * gi, g.y_lower + 0.2 * gi, 3.0),
             (g.x_upper - 0.6 * gi, g.y_lower + 0.1, 0.0), (g.x_upper + 0.3, 0.0, 0.0)]
    N, Tp = 3, 0.4
    coeffs, T, s_xy = [], [], []
    for k, (x, y, th) in enumerate(poses):
        c = np.zeros((N, 6, 2))
        c[:, 0, 0] = th
        if k >= 6:                       # moving outward along x at 0.25 m/s
            c[:, 1, 1] = 0.25
            c[:, 0, 1] = 0.25 * Tp * np.arange(N)
        coeffs.append(c)
        T.append(np.full(N, Tp))
        s_xy.append((x, y))
    coeffs, T, s_xy = np.concatenate(coeffs), np.concatenate(T), np.array(s_xy, dtype=np.float64)
    B = len(poses)
    po = (np.arange(B + 1) * N).astype(np.int32)
    prm = params(safeDis=0.9)
    set_checkpoints(prm, [(0.3, 0.2), (-0.25, -0.15), (0.0, 0.35), (0.0, 0.0)])
    # sample positions (exact for the standing splines): some outside the map, some in its last row / column where the
    # bilinear lookup refuses to interpolate
    pts = []
    for k, (x, y, th) in enumerate(poses[:6]):
        for c in range(prm.n_checkpoints):
            cx, cy = prm.check_point[c][0], prm.check_point[c][1]
            pts.append((x + math.cos(th) * cx - math.sin(th) * cy, y + math.sin(th) * cx + math.cos(th) * cy))
    pts = np.array(pts)
    out = (pts[:, 0] < g.x_lower) | (pts[:, 0] > g.x_upper) | (pts[:, 1] < g.y_lower) | (pts[:, 1] > g.y_upper)
    ix = ((pts[:, 0] - g.x_lower) * g.inv_grid_interval - 0.5).astype(int)
    iy = ((pts[:, 1] - g.y_lower) * g.inv_grid_interval - 0.5).astype(int)
    last = ~out & ((ix >= g.glx - 1) | (iy >= g.gly - 1))
    assert out.any() and last.any() and (~out & ~last).any()
    assert np.any(pts[:, 0] == g.x_lower) and np.any(pts[:, 0] == g.x_upper)
    cost = penalties(world, ctx, prm, po, coeffs, T, s_xy, s_xy.copy())[0]
    prm0 = params(safeDis=0.9, pw_collision=0.0)
    set_checkpoints(prm0, [(0.3, 0.2), (-0.25, -0.15), (0.0, 0.35), (0.0, 0.0)])
    assert np.any(penalties(world, ctx, prm0, po, coeffs, T, s_xy, s_xy.copy())[0] != cost)
    col, md = final_collisions(world, ctx, params(finalMinSafeDis=0.05), po, coeffs, T, s_xy)
    assert np.any(md == 1e10) and col.any()
    # candidates that start one or two cells inside x_upper / y_upper and run out of the map
    fts = [front_end.make_flat_traj([(g.x_upper - gi, 0.0), (g.x_upper + 1.0, 0.5)], (g.x_upper - gi, 0.0, 0.0),
                                    (g.x_upper + 1.0, 0.5, 0.3)),
           front_end.make_flat_traj([(1.0, g.y_upper - 2 * gi), (0.5, g.y_upper + 1.5)], (1.0, g.y_upper - 2 * gi, 1.6),
                                    (0.5, g.y_upper + 1.5, 1.9))]
    cands = front_end.pack_candidates(fts)
    costs(world, ctx, prm, cands, perturbed_x(cands, 0.02, 9))


# ---- 6. per-candidate ALM state ------------------------------------------------------------------------------------
def test_cost_batch_per_candidate_alm_state(world, portable_trig, ctx):
    prm = params()
    cands = leg_batch(world, max_legs=10, seed=12, dogleg=0.4)
    x = perturbed_x(cands, 0.03, 12)
    rng = np.random.default_rng(12)
    lam = rng.normal(0.0, 50.0, size=(cands.B, 2))
    rho = rng.uniform(1e3, 1e5, size=(cands.B, 2))
    sd = rng.uniform(0.2, 1.0, size=cands.B)
    c = costs(world, ctx, prm, cands, x, stages=(1,), lam=lam, rho=rho, safe_dis=sd)
    assert np.all(c != costs(world, ctx, prm, cands, x, stages=(1,)))
