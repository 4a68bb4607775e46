"""GPU parity tests for the ESDF path: CUDA (through the C ABI) vs the CPU oracle, bit for bit."""
import numpy as np
import pytest

import oracle_lib
from alore_legged_manipulator_b200 import SDFmap, capi, workloads

pytestmark = pytest.mark.gpu
DBL_MAX = float(np.finfo(np.float64).max)


def make_sdf(ctx, glx, gly, gi, grid, odom=(0.0, 0.0), rng_m=1e6, ref_compat=True):
    # SDFmap derives GLX = ceil((upper-lower)/gi) like the reference (sdf_map.h:150-151); put the upper
    # bound half a cell inside the last cell so the ceil is robust to FP rounding of the product
    xl, yl = -0.5 * glx * gi, -0.5 * gly * gi
    m = SDFmap(ctx, gridmap_interval=gi, detection_range=rng_m, global_x_lower=xl, global_x_upper=xl + (glx - 0.5) * gi,
               global_y_lower=yl, global_y_upper=yl + (gly - 0.5) * gi, ref_compat=ref_compat)
    assert (m.GLX_SIZE_, m.GLY_SIZE_) == (glx, gly)
    m.gridmap_[:] = grid
    m.odom_pos_[:2] = odom
    m.has_map_ = True
    return m


def check_against_oracle(ctx, glx, gly, gi, grid, odom=(0.0, 0.0), rng_m=1e6, check_sq=True):
    m = make_sdf(ctx, glx, gly, gi, grid, odom, rng_m)
    m.distance_buffer_all_[:] = -3.0          # sentinel: cells the reference never writes must keep it
    m.updateESDF2d()
    mn, mx = m.esdf_window()
    ref = np.full(glx * gly, -3.0)
    sp, sn = oracle_lib.esdf_update(m.geom(), m.gridmap_, mn, mx, ref, want_sq=check_sq)
    assert np.array_equal(m.distance_buffer_all_, ref), "ESDF distances differ from the reference restatement"
    if check_sq:
        pos, neg = m.last_squared()
        NX, NY = mx[0] - mn[0] + 1, mx[1] - mn[1] + 1
        S = NY - 1
        if S > 0:
            # the reference's own buffer index is x*S + y (aliasing stride); compare y < S
            rp = sp[: NX * S].reshape(NX, S)
            rn = sn[: NX * S].reshape(NX, S)
            gp = np.where(pos[:, :S] == capi.ALORE_SQ_INF, DBL_MAX, pos[:, :S].astype(np.float64))
            gn = np.where(neg[:, :S] == capi.ALORE_SQ_INF, DBL_MAX, neg[:, :S].astype(np.float64))
            assert np.array_equal(gp, rp), "squared distances (+) differ"
            assert np.array_equal(gn, rn), "squared distances (-) differ"
    return m


@pytest.mark.parametrize("shape", [(48, 40), (33, 57), (64, 64), (20, 90), (70, 25), (2, 2), (3, 5), (5, 3), (1, 7),
                                   (200, 200), (130, 257), (257, 130), (24, 8193), (24, 16384)])
@pytest.mark.parametrize("dens", [0.0, 1 / 400, 1 / 23, 1 / 3, 1.0])
def test_small_maps_bit_exact(ctx, shape, dens):
    glx, gly = shape
    grid = workloads.random_map(glx, gly, seed=glx * 7 + gly + int(dens * 1000), p_occ=dens, p_unknown=0.05, wall=False)
    check_against_oracle(ctx, glx, gly, 0.05, grid)


def test_sub_window_and_stale_cells(ctx):
    glx, gly, gi = 300, 260, 0.1
    grid = workloads.random_map(glx, gly, seed=11, p_occ=0.03)
    m = check_against_oracle(ctx, glx, gly, gi, grid, odom=(1.3, -2.1), rng_m=6.37)
    mn, mx = m.esdf_window()
    assert mn[0] > 0 and mx[1] < gly - 1
    # second update with a moved window on the same context: cells outside keep the previous values
    prev = m.distance_buffer_all_.copy()
    m.odom_pos_[:2] = (-3.0, 2.0)
    m.gridmap_[:] = workloads.random_map(glx, gly, seed=12, p_occ=0.05)
    m.updateESDF2d()
    mn, mx = m.esdf_window()
    ref = prev.copy()
    oracle_lib.esdf_update(m.geom(), m.gridmap_, mn, mx, ref)
    assert np.array_equal(m.distance_buffer_all_, ref)


def test_clean_mode_matches_bruteforce(ctx):
    from test_esdf_oracle import brute_force_expected
    glx, gly, gi = 48, 40, 0.05
    grid = workloads.random_map(glx, gly, seed=3, p_occ=0.05, wall=False)
    m = make_sdf(ctx, glx, gly, gi, grid, ref_compat=False)
    m.updateESDF2d()
    exp, _, _, _ = brute_force_expected(grid.reshape(glx, gly), gi, ref_compat=False)
    assert np.array_equal(m.distance_buffer_all_.reshape(glx, gly), exp)


@pytest.mark.parametrize("name", ["bernoulli_0.02", "sparse_1e-4", "dense_0.5", "empty", "single_seed", "corridor",
                                  "all_occupied"])
def test_2048_variants_bit_exact(ctx, name):
    n = 2048
    if name == "bernoulli_0.02":
        grid = workloads.random_map(n, n, 2, p_occ=0.02)
    elif name == "sparse_1e-4":
        grid = workloads.random_map(n, n, 3, p_occ=1e-4, p_unknown=0.0, wall=False)
    elif name == "dense_0.5":
        grid = workloads.random_map(n, n, 4, p_occ=0.5)
    elif name == "empty":
        grid = np.full(n * n, capi.UNOCCUPIED, np.uint8)
    elif name == "single_seed":
        grid = np.full(n * n, capi.UNOCCUPIED, np.uint8)
        grid[777 * n + 1300] = capi.OCCUPIED
    elif name == "corridor":
        grid = workloads.corridor_map(n, n, 5, width_cells=64)
    else:
        grid = np.full(n * n, capi.OCCUPIED, np.uint8)
    check_against_oracle(ctx, n, n, 0.05, grid)


def test_config2_4096_bit_exact(ctx):
    n = 4096
    grid = workloads.random_map(n, n, 2, p_occ=0.02, p_unknown=0.01)
    m = check_against_oracle(ctx, n, n, 0.05, grid, check_sq=False)
    # size-independent properties on the full map
    d = m.distance_buffer_all_.reshape(n, n)[: n - 1, : n - 1]
    occ = grid.reshape(n, n)[: n - 1, : n - 1] == capi.OCCUPIED
    assert np.all(d[occ] <= 0.0) and np.all(d[~occ] > 0.0)
    # 1-Lipschitz in grid units between 4-neighbours (exact EDT property, tolerance one ulp-ish)
    gi = 0.05
    assert np.max(np.abs(np.diff(d[1:, 1:], axis=0))) <= gi * 2 + 1e-12   # sign change adds the +gi offset; quirk column excluded
    assert m.last_kernel_ms() > 0.0


def test_config5_shape_8192x2048_bit_exact(ctx):
    glx, gly = 8192, 2048
    grid = workloads.corridor_map(glx, gly, 5, width_cells=400, clutter=0.02)
    check_against_oracle(ctx, glx, gly, 0.005, grid, check_sq=False)


@pytest.mark.parametrize("shape", [(257, 130), (64, 700), (1024, 1024)])
def test_sparse_box_and_dense_maps_bit_exact(shape):
    """Sparse clutter, a box world and a dense map of each shape, on a context of their own."""
    import alore_legged_manipulator_b200 as alore
    ctx = alore.Context(0)                # its own context: one context holds one device-resident map
    glx, gly = shape
    for seed, kw in ((1, dict(p_occ=0.02, p_unknown=0.01)), (2, dict(p_occ=0.0, p_unknown=0.0, boxes=6, box_cells=(4, 40))),
                     (3, dict(p_occ=0.7, p_unknown=0.05))):
        grid = workloads.random_map(glx, gly, seed, **kw)
        m = make_sdf(ctx, glx, gly, 0.05, grid)
        m.updateESDF2d()
        ref = np.full(glx * gly, DBL_MAX)
        mn, mx = m.esdf_window()
        oracle_lib.esdf_update(m.geom(), grid, mn, mx, ref)
        assert np.array_equal(m.distance_buffer_all_.view(np.uint64), ref.view(np.uint64)), (shape, seed)
        m.close()
    ctx.close()


def far_field_maps():
    """(glx, gly, grid): nearly empty, nearly solid and mixed maps, where most cells are left to the band kernel."""
    out = []
    for (glx, gly), seed, kw in (((700, 300), 2, dict(p_occ=0.0, p_unknown=0.0, boxes=5, box_cells=(4, 40))),
                                 ((513, 257), 3, dict(p_occ=0.0, p_unknown=0.0, wall=False, boxes=1, box_cells=(2, 3))),
                                 ((300, 900), 4, dict(p_occ=0.0, p_unknown=0.0, boxes=30, box_cells=(40, 200))),
                                 ((1100, 260), 5, dict(p_occ=1.0, p_unknown=0.0))):
        grid = workloads.random_map(glx, gly, seed, **kw)
        if kw.get("p_occ") == 1.0:                           # a solid world with one free pocket and one free cell
            g2 = grid.reshape(glx, gly)
            g2[500:520, 100:130] = capi.UNOCCUPIED
            g2[40, 200] = capi.UNOCCUPIED
        out.append((glx, gly, grid))
    return out


def test_far_field_maps_bit_exact():
    """Far cells (large empty / solid regions) must reproduce the oracle bit for bit."""
    import alore_legged_manipulator_b200 as alore
    ctx = alore.Context(0)
    for glx, gly, grid in far_field_maps():
        m = make_sdf(ctx, glx, gly, 0.05, grid)
        m.updateESDF2d()
        ref = np.full(glx * gly, DBL_MAX)
        mn, mx = m.esdf_window()
        oracle_lib.esdf_update(m.geom(), grid, mn, mx, ref)
        assert np.array_equal(m.distance_buffer_all_.view(np.uint64), ref.view(np.uint64)), (glx, gly)
        m.close()
    ctx.close()


def patchwork_map(glx, gly, rng):
    """Rectangles of very different character side by side: solid, empty, cluttered, sparse seeds, unknown."""
    g = np.full((glx, gly), capi.UNOCCUPIED, dtype=np.uint8)
    for _ in range(int(rng.integers(3, 9))):
        w, h = int(rng.integers(8, max(9, glx // 2))), int(rng.integers(8, max(9, gly // 2)))
        x0, y0 = int(rng.integers(0, max(1, glx - w))), int(rng.integers(0, max(1, gly - h)))
        kind = int(rng.integers(0, 5))
        blk = g[x0:x0 + w, y0:y0 + h]
        if kind == 0:
            blk[:] = capi.OCCUPIED
        elif kind == 1:
            blk[:] = capi.UNOCCUPIED
        elif kind == 2:
            blk[rng.random(blk.shape) < 0.05] = capi.OCCUPIED
        elif kind == 3:
            blk[rng.random(blk.shape) < 0.6] = capi.OCCUPIED
        else:
            blk[:] = capi.UNKNOWN
    if rng.random() < 0.3:
        g[int(rng.integers(0, glx)), int(rng.integers(0, gly))] = capi.OCCUPIED
    return np.ascontiguousarray(g.reshape(-1))


@pytest.mark.parametrize("seed", range(24))
def test_patchwork_maps_and_windows_bit_exact(ctx, seed):
    """Near-field, far-field and dense regions in ONE map (every hand-over between K2, the deferred list and the band
    kernel inside a single tile), odd sizes, windows that start and end anywhere; distances and both squared planes."""
    rng = np.random.default_rng(1234 + seed)
    glx, gly = int(rng.integers(40, 700)), int(rng.integers(40, 700))
    grid = patchwork_map(glx, gly, rng)
    gi = 0.1
    if seed % 3 == 0:                                  # full map
        check_against_oracle(ctx, glx, gly, gi, grid)
    else:                                              # a window around a random odometry position
        odom = (float(rng.uniform(-0.4, 0.4) * glx * gi), float(rng.uniform(-0.4, 0.4) * gly * gi))
        check_against_oracle(ctx, glx, gly, gi, grid, odom=odom, rng_m=float(rng.uniform(2.0, 0.45 * min(glx, gly) * gi)))


def test_stale_handover_words_of_another_window_shape_are_never_read_as_flags():
    """K2 hands far cells to K2e through masks and per-tile flags kept in a per-context buffer; a flag is "set" when it
    holds the update's epoch.  Regression: with the flags BEHIND the (shape-dependent) mask planes, a mask word of an
    earlier, larger window could sit where a later window looks for a flag — and equal its epoch.  Window A (35 rows:
    the last band has 3 rows, every cell far from the only seed) leaves mask words of value 0b11; window B (two 64x128
    tiles, cluttered: nothing far) is then updated at every epoch from 2 to 12 — epoch 3 met the stale word."""
    import alore_legged_manipulator_b200 as alore
    ctx = alore.Context(0)
    ga = np.full((35, 1024), capi.UNOCCUPIED, np.uint8)
    ga[0, 0] = capi.OCCUPIED
    ga = np.ascontiguousarray(ga.reshape(-1))
    gb = workloads.random_map(100, 120, 5, p_occ=0.08, p_unknown=0.0, wall=False)
    for it in range(12):                                  # A once (epoch 1), then B at the epochs 2 .. 12
        glx, gly, grid = (35, 1024, ga) if it == 0 else (100, 120, gb)
        m = make_sdf(ctx, glx, gly, 0.1, grid)
        m.updateESDF2d()
        ref = np.full(glx * gly, DBL_MAX)
        mn, mx = m.esdf_window()
        oracle_lib.esdf_update(m.geom(), grid, mn, mx, ref)
        assert np.array_equal(m.distance_buffer_all_.view(np.uint64), ref.view(np.uint64)), (it, glx, gly)
        m.close()
    ctx.close()


def test_alternating_window_shapes_on_one_context():
    """Three window shapes alternate on ONE context for many updates (the hand-over buffer of K2e survives across
    updates and is re-used under every shape): every update must reproduce the oracle."""
    import alore_legged_manipulator_b200 as alore
    ctx = alore.Context(0)
    rng = np.random.default_rng(99)
    shapes = [(130, 520), (260, 260), (70, 900)]
    for it in range(120):
        glx, gly = shapes[it % len(shapes)]
        grid = patchwork_map(glx, gly, rng)
        m = make_sdf(ctx, glx, gly, 0.1, grid)            # takes the context's map over (one context = one map)
        m.updateESDF2d()
        ref = np.full(glx * gly, DBL_MAX)
        mn, mx = m.esdf_window()
        oracle_lib.esdf_update(m.geom(), grid, mn, mx, ref)
        assert np.array_equal(m.distance_buffer_all_.view(np.uint64), ref.view(np.uint64)), (it, glx, gly)
        m.close()
    ctx.close()
