"""CPU anchors for the parameter combinations that tests/test_param_space_gpu.py runs on the device.

The GPU file proves that the kernels equal the oracle bit for bit off the default parameters; these tests prove that
the oracle is right there, independently of both:

* a closed-form known answer for the collision term of the coefficient-space functional (a robot standing still),
  for every sampling resolution and check-point set the GPU file uses;
* central finite differences of the cost callbacks for lateral check-points, three check-points, the ICR model,
  direct v/omega limits and coarse / fine sampling;
* central finite differences of the coefficient-space gradient (`penalty_batch`: gradC, gradT).
"""
import ctypes as C
import math

import numpy as np
import pytest

import oracle_lib
from alore_legged_manipulator_b200 import capi, workloads
from test_optimizer_oracle import _fd_check

# check-point sets with non-zero lateral components; the first is a single check-point off the centre line
CHECKPOINTS = {
    1: [(0.25, 0.2)],
    3: [(0.3, 0.2), (-0.25, -0.15), (0.0, 0.35)],
    8: [(0.3, 0.2), (-0.25, -0.15), (0.0, 0.35), (0.35, -0.1), (-0.3, 0.25), (0.1, -0.3), (-0.05, 0.0), (0.2, 0.3)],
}


def params(**kw) -> capi.Params:
    p = oracle_lib.default_params()
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def set_checkpoints(prm: capi.Params, cps):
    prm.n_checkpoints = len(cps)
    for c, (x, y) in enumerate(cps):
        prm.check_point[c][0], prm.check_point[c][1] = x, y


@pytest.fixture(scope="module")
def cfg1():
    geom, grid, cands = workloads.config1()
    dist = np.full(geom.glx * geom.gly, np.finfo(np.float64).max)
    oracle_lib.esdf_update(geom, grid, (0, 0), (geom.glx - 1, geom.gly - 1), dist)
    return geom, grid, cands, dist


@pytest.fixture(scope="module")
def exact_chain():
    lib = oracle_lib.load()
    lib.orc_set_exact_chain_weights(1)
    yield
    lib.orc_set_exact_chain_weights(0)


def smoothed_l1(eps, x):
    lib = oracle_lib.load()
    lib.orc_smoothed_l1.argtypes = [C.c_double, C.c_double, capi.c_double_p, capi.c_double_p]
    lib.orc_smoothed_l1.restype = None
    f, df = C.c_double(), C.c_double()
    lib.orc_smoothed_l1(eps, x, C.byref(f), C.byref(df))
    return f.value, df.value


def dist_grad3(geom, dist, pos, mindis):
    g = np.zeros(2)
    d = oracle_lib.load().orc_dist_grad3(C.byref(geom), capi.dptr(dist), capi.dptr(np.asarray(pos, dtype=np.float64)),
                                         capi.dptr(g), mindis)
    return d, g


def stationary_spline(xy, theta, s, T):
    """N pieces of a spline that stands still at `xy` with yaw `theta` and arc length `s`: every sample sees the same
    pose, the XY integral stays at the start point, and only the collision term can fire."""
    N = len(T)
    coeffs = np.zeros((N, 6, 2))
    coeffs[:, 0, 0], coeffs[:, 0, 1] = theta, s
    return (np.array([0, N], np.int32), coeffs, np.asarray(T, dtype=np.float64), np.array([xy], dtype=np.float64),
            np.array([xy], dtype=np.float64))


def stationary_known_answer(prm, geom, dist, xy, theta, T):
    """T_i * pw * sum_cp L1(safeDis - d(p + R(theta) c))  and  -T_i * pw * sum_cp L1'(v) (grad d . R'(theta) c):
    the cost and d cost / d (constant yaw coefficient) of piece i.  The sample weights omg * step sum to T_i."""
    cn, sn = math.cos(theta), math.sin(theta)
    vals, dvals, n_in = [], [], 0
    for c in range(prm.n_checkpoints):
        cx, cy = prm.check_point[c][0], prm.check_point[c][1]
        d, g = dist_grad3(geom, dist, (xy[0] + (cn * cx - sn * cy), xy[1] + (sn * cx + cn * cy)), prm.safeDis)
        v = prm.safeDis - d
        if v > 0.0:
            n_in += 1
            f, df = smoothed_l1(prm.smoothEps, v)
            vals.append(f)
            dvals.append(-df * (g[0] * (-sn * cx - cn * cy) + g[1] * (cn * cx - sn * cy)))
    l1 = math.fsum(vals)
    cost = math.fsum(Ti * prm.pw_collision * l1 for Ti in T)
    grad_yaw = [Ti * prm.pw_collision * math.fsum(dvals) for Ti in T]
    return cost, grad_yaw, prm.pw_collision * l1, n_in


def stationary_pose(geom, dist, cps):
    """A free pose next to an obstacle, and the safety margin half-way through its check-points' distances: some
    check-points are inside the margin and some are not."""
    d = dist.reshape(geom.glx, geom.gly)
    ix, iy = np.argwhere((d > 0.35) & (d < 0.45))[0]
    xy = (geom.x_lower + (ix + 0.37) * geom.grid_interval, geom.y_lower + (iy + 0.61) * geom.grid_interval)
    theta = 0.7
    cn, sn = math.cos(theta), math.sin(theta)
    ds = sorted(dist_grad3(geom, dist, (xy[0] + cn * x - sn * y, xy[1] + sn * x + cn * y), 1e9)[0] for x, y in cps)
    safe = 0.5 * (ds[len(ds) // 2 - 1] + ds[len(ds) // 2]) if len(ds) > 1 else ds[0] + 0.1
    return xy, theta, safe


@pytest.mark.parametrize("ncp", [1, 3, 8])
@pytest.mark.parametrize("K", [1, 2, 3, 8, 64])
def test_stationary_collision_known_answer(cfg1, K, ncp):
    geom, grid, cands, dist = cfg1
    prm = params(sparseResolution=K, min_vel=0.0)
    prm.EqualLambda[0] = prm.EqualLambda[1] = 0.0
    set_checkpoints(prm, CHECKPOINTS[ncp])
    xy, theta, prm.safeDis = stationary_pose(geom, dist, CHECKPOINTS[ncp])
    T = [0.4, 0.7, 1.3]
    po, coeffs, Tv, s_xy, f_xy = stationary_spline(xy, theta, 2.5, T)
    cost, gC, gT, err = oracle_lib.penalty_batch(prm, geom, dist, po, coeffs, Tv, s_xy, f_xy)
    want, grad_yaw, want_gT, n_in = stationary_known_answer(prm, geom, dist, xy, theta, T)
    # the pose is what the test says: some check-points inside the margin, some outside
    assert 0 < n_in < ncp or (ncp == 1 and n_in == 1)
    assert want > 0.0 and np.all(err == 0.0)
    assert math.isclose(cost[0], want, rel_tol=1e-13), (cost[0], want)
    for i in range(len(T)):
        assert math.isclose(gC[i, 0, 0], grad_yaw[i], rel_tol=1e-12, abs_tol=1e-12 * abs(want)), (i, gC[i, 0, 0], grad_yaw[i])
        assert math.isclose(gT[i], want_gT, rel_tol=1e-13), (i, gT[i], want_gT)
        assert gC[i, 0, 1] == 0.0              # the arc length enters the functional only through its derivatives


# ---- finite differences of the cost callbacks ---------------------------------------------------------------------
VARIANTS = {
    "lateral_checkpoints": dict(cps=[(0.3, 0.2), (-0.3, -0.2)]),
    "three_checkpoints": dict(cps=CHECKPOINTS[3]),
    "icr": dict(if_standard_diff=0),
    "direct_v_omega": dict(if_directly_constrain_v_omega=1),
    "K1": dict(sparseResolution=1),
    "K3": dict(sparseResolution=3),
    "K64": dict(sparseResolution=64),
}


ICR_SIGN = ("the ICR model's d(y-integrand)/d(yaw) carries -ds0*icr*sin(yaw) where the derivative of "
            "-ds0*icr*cos(yaw) is +ds0*icr*sin(yaw) (oracle and kernel alike, bit-identical)")


@pytest.mark.parametrize("variant", [pytest.param(v, marks=pytest.mark.xfail(strict=True, reason=ICR_SIGN)) if v == "icr"
                                     else v for v in VARIANTS])
def test_cost_gradient_finite_differences_variants(cfg1, exact_chain, variant):
    geom, grid, cands, dist = cfg1
    kw = dict(VARIANTS[variant])
    cps = kw.pop("cps", None)
    prm = params(**kw)
    if cps:
        set_checkpoints(prm, cps)
    N = cands.total_pieces
    rng = np.random.default_rng(7)
    x0 = oracle_lib.initial_x(cands, 0) + 0.05 * rng.normal(size=3 * N - 1)
    # the collision term fires at x0 (the check-points are what the lateral variants change)
    f, _, _ = oracle_lib.cost(prm, geom, dist, cands, 0, 1, x0)
    prm0 = params(**kw)
    prm0.pw_collision = 0.0
    assert oracle_lib.cost(prm0, geom, dist, cands, 0, 1, x0)[0] != f
    Psl, tail, tau = slice(0, 2 * (N - 1)), slice(2 * (N - 1), 2 * (N - 1) + 1), slice(2 * (N - 1) + 1, 3 * N - 1)
    for sl in (Psl, tail, tau):
        _fd_check(prm, geom, dist, cands, 1, x0, sl, rng, 1e-6)
    for sl in (Psl, tail):                     # stage 0: tau carries the reference's weight mix-up (see the FD test)
        _fd_check(prm, geom, dist, cands, 0, x0, sl, rng, 1e-6)


# ---- finite differences of the coefficient-space functional ------------------------------------------------------
@pytest.mark.parametrize("variant", ["default", "lateral_checkpoints", "K3",
                                     pytest.param("icr", marks=pytest.mark.xfail(strict=True, reason=ICR_SIGN))])
def test_penalty_batch_gradient_finite_differences(cfg1, exact_chain, variant):
    geom, grid, cands, dist = cfg1
    kw = dict(VARIANTS.get(variant, {}))
    cps = kw.pop("cps", None)
    prm = params(**kw)
    if cps:
        set_checkpoints(prm, cps)
    po, coeffs, T, s_xy, f_xy = workloads.random_spline_batch(4, 6, geom, dist, grid, seed=21)
    cost, gC, gT, _ = oracle_lib.penalty_batch(prm, geom, dist, po, coeffs, T, s_xy, f_xy)
    prm0 = params(**kw)
    prm0.pw_collision = 0.0
    assert np.any(oracle_lib.penalty_batch(prm0, geom, dist, po, coeffs, T, s_xy, f_xy)[0] != cost)
    rng = np.random.default_rng(5)
    h = 1e-6
    for b in range(po.size - 1):
        sl = slice(int(po[b]), int(po[b + 1]))
        one = np.array([0, sl.stop - sl.start], np.int32)

        def f(c, t):
            return oracle_lib.penalty_batch(prm, geom, dist, one, np.ascontiguousarray(c), np.ascontiguousarray(t),
                                            s_xy[b:b + 1].copy(), f_xy[b:b + 1].copy())[0][0]
        vc = rng.normal(size=coeffs[sl].shape)
        vc /= np.linalg.norm(vc)
        fd = (f(coeffs[sl] + h * vc, T[sl]) - f(coeffs[sl] - h * vc, T[sl])) / (2 * h)
        an = float(np.sum(gC[sl] * vc))
        assert math.isclose(fd, an, rel_tol=1e-6, abs_tol=1e-7 * max(1.0, abs(cost[b]))), (b, fd, an)
        vt = rng.normal(size=T[sl].shape)
        vt /= np.linalg.norm(vt)
        fd = (f(coeffs[sl], T[sl] + h * vt) - f(coeffs[sl], T[sl] - h * vt)) / (2 * h)
        an = float(gT[sl] @ vt)
        assert math.isclose(fd, an, rel_tol=1e-6, abs_tol=1e-7 * max(1.0, abs(cost[b]))), (b, fd, an)
