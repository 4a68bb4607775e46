"""What the DEVICE sees of the ESDF: the device-resident entry points (alore_esdf_update_dev in its three modes,
alore_esdf_set) on a caller stream, the whole device distance buffer read back bit for bit, clean mode
(ref_compat = 0) against an exact EDT that does not go through the oracle, every row-pass kernel variant and the
16384-cell window limit.

`exact_esdf` is the reference for clean mode and, with the column-0 patch and the unwritten last row / column, for
ref_compat mode too.  It is pinned against the exhaustive brute force of test_esdf_oracle.py on small maps and pins
the C++ oracle on strips of 16384 cells (CPU tests in this file, no GPU needed)."""
import ctypes as C

import numpy as np
import pytest
from scipy import ndimage

import oracle_lib
from alore_legged_manipulator_b200 import capi, workloads
from test_esdf_gpu import far_field_maps as far_field_grids, patchwork_map
from test_esdf_oracle import SHAPES, brute_force_expected
from test_optimizer_gpu import check_results, portable_trig  # noqa: F401  (fixture)

gpu = pytest.mark.gpu
DBL_MAX = float(np.finfo(np.float64).max)
INF = np.int64(1) << 40          # "no seed of this kind" in the integer planes (as brute_force_expected)
# sentinel of cells nobody may write: no ESDF value can equal it (|value| <= gi*sqrt(DBL_MAX) + gi), whereas a small
# one like -3.0 is a real distance on some maps (gi - gi*sqrt(601^2) at gi = 0.005)
SENT = -1.0e300
OCC, FREE, UNK = capi.OCCUPIED, capi.UNOCCUPIED, capi.UNKNOWN
EINVAL, ENOMAP = -1, -3          # ALORE_EINVAL, ALORE_ENOMAP


# ---- exact reference ---------------------------------------------------------------------------------------------
def _sq_edt(seed):
    """Exact integer squared distance of every cell to the nearest True cell of `seed` (INF when there is none)."""
    if not seed.any():
        return np.full(seed.shape, INF, np.int64)
    ix, iy = ndimage.distance_transform_edt(~seed, return_distances=False, return_indices=True)
    X = np.arange(seed.shape[0], dtype=np.int64)[:, None]
    Y = np.arange(seed.shape[1], dtype=np.int64)[None, :]
    return (ix - X) ** 2 + (iy - Y) ** 2


def _envelope_1d(f):
    """min_q (x-q)^2 + f[q] for every x: Felzenszwalb's lower envelope in exact integer arithmetic (entries >= INF
    are absent), O(n)."""
    fl = [int(v) for v in f]
    qs = [q for q, v in enumerate(fl) if v < INF]
    out = np.full(len(fl), INF, np.int64)
    if not qs:
        return out
    v, z = [qs[0]], []                      # z[k] = (num, den): where parabola v[k+1] takes over from v[k]
    for q in qs[1:]:
        while True:
            p = v[-1]
            num, den = (fl[q] + q * q) - (fl[p] + p * p), 2 * (q - p)
            if z and num * z[-1][1] <= z[-1][0] * den:
                v.pop()
                z.pop()
                continue
            break
        v.append(q)
        z.append((num, den))
    k = 0
    for x in range(len(fl)):
        while k < len(z) and z[k][0] < x * z[k][1]:
            k += 1
        out[x] = (x - v[k]) ** 2 + fl[v[k]]
    return out


def exact_esdf(occ2d, gi, ref_compat):
    """(dist, written, pos_sq, neg_sq) of a full window = the whole (NX, NY) grid, as brute_force_expected states them.

    Squared distances are exact int64 from scipy's feature transform; dist = gi*sqrt(.) (gi*sqrt(DBL_MAX) without a
    seed), combined as the reference does.  ref_compat: window-local column 0, rows 1..NX-2, is the 1-D transform of
    the aliased column W(j) = row-pass value of (j, 0), W(NX) = row-pass value of (NX-1, NY-1); the last row and column
    are not written."""
    NX, NY = occ2d.shape
    occm = occ2d == OCC
    hp, hn = _sq_edt(occm), _sq_edt(~occm)
    if ref_compat and NX >= 2 and NY >= 2:
        for seed, h in ((occm, hp), (~occm, hn)):
            first = seed.argmax(axis=1).astype(np.int64)               # in-row distance of column 0
            g0 = np.where(seed.any(axis=1), first * first, INF)
            last = NY - 1 - int(seed[NX - 1, ::-1].argmax())
            gl = (NY - 1 - last) ** 2 if seed[NX - 1].any() else INF   # in-row distance of (NX-1, NY-1)
            t = _envelope_1d(np.concatenate([g0[1:], [gl]]))
            h[1:, 0] = t[: NX - 1]

    def to_d(h):
        return np.where(h >= INF, gi * np.sqrt(DBL_MAX), gi * np.sqrt(np.minimum(h, INF - 1).astype(np.float64)))

    pos, neg = to_d(hp), to_d(hn)
    allv = pos.copy()
    m = neg > 0.0
    allv[m] = pos[m] + (-neg[m] + gi)
    written = np.ones((NX, NY), bool)
    if ref_compat:
        written[NX - 1, :] = False
        written[:, NY - 1] = False
    return allv, written, hp, hn


def expected_clean(occ, glx, gly, gi, mn, mx, base):
    """`base` (flat glx*gly) with the window replaced by the clean-mode ESDF of the window's occupancy; planes too."""
    g = occ.reshape(glx, gly)[mn[0]:mx[0] + 1, mn[1]:mx[1] + 1]
    d, _, hp, hn = exact_esdf(g, gi, False)
    out = base.copy().reshape(glx, gly)
    out[mn[0]:mx[0] + 1, mn[1]:mx[1] + 1] = d
    return out.reshape(-1), hp, hn


def test_k1_dispatch_rule_restated():
    """The helper below restates esdf.cu's row-pass choice; the case table of the GPU test must reach every variant."""
    kernels = {k1_kernel(c[1], c[2], c[3], c[4]) for c in K1_CASES}
    assert kernels >= {"row_pass16<1>", "row_pass16<2>", "row_pass16<4>", "byte", "byte_unaligned", "byte_smem_optin"}
    assert "row_pass16<8>" not in kernels                       # unreachable under the 16384-cell limit
    fast_ragged = {c[3] % 16 for c in K1_CASES if k1_kernel(c[1], c[2], c[3], c[4]).startswith("row_pass16")}
    assert fast_ragged >= {0, 1, 7, 15}
    heights = {c[3] for c in K1_CASES}
    assert heights >= {4096, 4097, 4112, 8192, 8193, 8208, 16368, 16383, 16384}
    assert {c[4] for c in K1_CASES} >= {1, 7, 15}
    assert all(k1_kernel(c[1], c[2], c[3], c[4]) == c[5] for c in K1_CASES)


@pytest.mark.parametrize("shape", SHAPES + [(1, 7)])
@pytest.mark.parametrize("dens", [0.0, 1 / 400, 1 / 23, 1 / 3, 1.0])
@pytest.mark.parametrize("ref_compat", [False, True])
def test_exact_reference_matches_bruteforce(shape, dens, ref_compat):
    NX, NY = shape
    rng = np.random.default_rng(NX * 1000 + NY + int(dens * 1e4))
    u = rng.random((NX, NY))
    occ = np.full((NX, NY), FREE, np.uint8)
    occ[u < dens] = OCC
    occ[(u >= dens) & (u < dens + 0.05)] = UNK
    got = exact_esdf(occ, 0.05, ref_compat)
    exp = brute_force_expected(occ, 0.05, ref_compat=ref_compat)
    assert np.array_equal(got[0].view(np.uint64), exp[0].view(np.uint64))
    for a, b in zip(got[1:], exp[1:]):
        assert np.array_equal(a, b)


def strip_map(NX, NY, seed):
    """A strip with sparse clutter, a solid block, an empty band of rows and one seed in the corner."""
    rng = np.random.default_rng(seed)
    g = np.where(rng.random((NX, NY)) < 2e-4, OCC, FREE).astype(np.uint8)
    g[rng.random((NX, NY)) < 0.01] = UNK
    g[NX // 3: NX // 3 + max(1, NX // 50), NY // 4: NY // 2] = OCC
    g[NX // 2: NX // 2 + max(1, NX // 20), :] = FREE
    g[0, 0] = OCC
    return np.ascontiguousarray(g.reshape(-1))


@pytest.mark.parametrize("shape", [(16384, 48), (48, 16384), (8192, 64)])
def test_oracle_matches_exact_reference_on_long_strips(shape):
    """Pins the C++ oracle far beyond the brute force: 16384-cell sides, distances and both squared planes."""
    NX, NY = shape
    grid = strip_map(NX, NY, NX + NY)
    geom = workloads.make_geom(NX, NY, 0.05)
    dist = np.full(NX * NY, SENT)
    sp, sn = oracle_lib.esdf_update(geom, grid, (0, 0), (NX - 1, NY - 1), dist, want_sq=True)
    exp, written, hp, hn = exact_esdf(grid.reshape(NX, NY), 0.05, True)
    got = dist.reshape(NX, NY)
    assert np.array_equal(got[written].view(np.uint64), exp[written].view(np.uint64))
    assert np.all(got[~written] == SENT)
    S = NY - 1
    for plane, h in ((sp, hp), (sn, hn)):
        assert np.array_equal(plane[: NX * S].reshape(NX, S), np.where(h[:, :S] >= INF, DBL_MAX, h[:, :S].astype(np.float64)))


# ---- device helpers ----------------------------------------------------------------------------------------------
def new_ctx():
    import alore_legged_manipulator_b200 as alore
    return alore.Context(0)                  # one context per test: it holds one device-resident map


def stream_ptr(stream):
    return C.c_void_p(stream.cuda_stream)


def update_dev(ctx, geom, d_occ, mn, mx, d_dist, ref_compat, stream):
    """alore_esdf_update_dev; d_occ / d_dist are device addresses (int) or None.  Returns the status code."""
    return ctx.lib.alore_esdf_update_dev(ctx.h, C.byref(geom), C.c_void_p(d_occ) if d_occ else None, mn[0], mn[1], mx[0],
                                         mx[1], C.c_void_p(d_dist) if d_dist else None, int(ref_compat), stream_ptr(stream))


def host_update(ctx, geom, occ, mn, mx, dist, ref_compat):
    return ctx.lib.alore_esdf_update(ctx.h, C.byref(geom), capi.u8ptr(occ), mn[0], mn[1], mx[0], mx[1], capi.dptr(dist),
                                     int(ref_compat))


def device_readback(ctx, geom, occ, mn, mx, ref_compat, occ_offset=0):
    """Caller-buffer update on a non-default stream into a sentinel-filled device buffer; the WHOLE buffer back."""
    import torch
    n = geom.glx * geom.gly
    d_occ = torch.zeros(n + occ_offset, dtype=torch.uint8, device="cuda")
    d_occ[occ_offset:].copy_(torch.from_numpy(occ))
    d_dist = torch.full((n,), SENT, dtype=torch.float64, device="cuda")
    stream = torch.cuda.Stream()
    torch.cuda.synchronize()                          # the fills above ran on torch's current stream
    ctx.check(update_dev(ctx, geom, d_occ.data_ptr() + occ_offset, mn, mx, d_dist.data_ptr(), ref_compat, stream))
    stream.synchronize()
    return d_dist.cpu().numpy()


def last_sq(ctx, mn, mx):
    nx, ny = mx[0] - mn[0] + 1, mx[1] - mn[1] + 1
    pos, neg = np.zeros(nx * ny, np.int32), np.zeros(nx * ny, np.int32)
    ctx.check(ctx.lib.alore_esdf_last_sq(ctx.h, capi.iptr(pos), capi.iptr(neg)))
    return pos.reshape(nx, ny), neg.reshape(nx, ny)


def oracle_update(geom, occ, mn, mx, base, want_sq=False):
    out = np.array(base, dtype=np.float64, copy=True)
    s = oracle_lib.esdf_update(geom, occ, mn, mx, out, want_sq=want_sq)
    return (out, *s) if want_sq else out


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint64), np.asarray(b).view(np.uint64))


def check_sq_ref_compat(ctx, mn, mx, sp_, sn_):
    """last_sq against the oracle's planes (its own buffer index is x*S + y, S = NY-1: compare y < S)."""
    pos, neg = last_sq(ctx, mn, mx)
    NX, NY = pos.shape
    S = NY - 1
    if S <= 0:
        return
    for got, ref in ((pos, sp_), (neg, sn_)):
        g = np.where(got[:, :S] == capi.ALORE_SQ_INF, DBL_MAX, got[:, :S].astype(np.float64))
        assert np.array_equal(g, ref[: NX * S].reshape(NX, S))


def check_sq_clean(ctx, mn, mx, hp, hn):
    pos, neg = last_sq(ctx, mn, mx)
    for got, h in ((pos, hp), (neg, hn)):
        assert np.array_equal(got, np.where(h >= INF, capi.ALORE_SQ_INF, h).astype(np.int32))


def check_ref_compat(ctx, geom, occ, mn, mx, sq=False, occ_offset=0):
    got = device_readback(ctx, geom, occ, mn, mx, True, occ_offset)
    r = oracle_update(geom, occ, mn, mx, np.full(geom.glx * geom.gly, SENT), want_sq=sq)
    ref = r[0] if sq else r
    assert same_bits(got, ref), ("device write set / values differ from the oracle", geom.glx, geom.gly, mn, mx)
    if sq:
        check_sq_ref_compat(ctx, mn, mx, r[1], r[2])


def check_clean(ctx, geom, occ, mn, mx, sq=True, host=True, occ_offset=0):
    n = geom.glx * geom.gly
    got = device_readback(ctx, geom, occ, mn, mx, False, occ_offset)
    exp, hp, hn = expected_clean(occ, geom.glx, geom.gly, geom.grid_interval, mn, mx, np.full(n, SENT))
    win = got.reshape(geom.glx, geom.gly)[mn[0]:mx[0] + 1, mn[1]:mx[1] + 1]
    assert not np.any(win == SENT), "clean mode must write the whole window, last row and column included"
    assert same_bits(got, exp), ("clean mode differs from the exact EDT", geom.glx, geom.gly, mn, mx)
    if sq:
        check_sq_clean(ctx, mn, mx, hp, hn)
    if host:
        h = np.full(n, SENT)
        ctx.check(host_update(ctx, geom, occ, mn, mx, h, False))
        assert same_bits(h, got), "host path (alore_esdf_update, ref_compat=0) differs from the device path"


# ---- maps --------------------------------------------------------------------------------------------------------
def far_field_maps():
    """The four maps of test_esdf_gpu.test_far_field_maps_bit_exact (nearly empty, nearly solid, mixed), whole windows."""
    return [(glx, gly, grid, (0, 0), (glx - 1, gly - 1)) for glx, gly, grid in far_field_grids()]


def patchwork_windows(n, seed0=500):
    out = []
    for s in range(n):
        rng = np.random.default_rng(seed0 + s)
        glx, gly = int(rng.integers(40, 600)), int(rng.integers(40, 600))
        grid = patchwork_map(glx, gly, rng)
        x0, y0 = int(rng.integers(0, glx // 2)), int(rng.integers(0, gly // 2))
        x1, y1 = int(rng.integers(x0 + 1, glx)), int(rng.integers(y0 + 1, gly))
        out.append((glx, gly, grid, (x0, y0), (x1, y1)))
    return out


def uniform_maps():
    out = []
    for state in (OCC, FREE):
        glx, gly = 300, 200
        out.append((glx, gly, np.full(glx * gly, state, np.uint8), (0, 0), (glx - 1, gly - 1)))
        out.append((glx, gly, np.full(glx * gly, state, np.uint8), (17, 33), (250, 180)))
    return out


def degenerate_windows():
    glx, gly = 100, 90
    grid = workloads.random_map(glx, gly, 21, p_occ=0.05, p_unknown=0.02, wall=False)
    wins = [((10, 5), (10, 80)), ((3, 40), (95, 40)), ((50, 50), (51, 51)), ((0, 0), (1, 89)), ((0, 7), (99, 8)),
            ((99, 89), (99, 89)), ((98, 0), (99, 89))]     # 1xN, Nx1, 2x2, 2xN, Nx2, 1x1, the last two rows
    return [(glx, gly, grid, mn, mx) for mn, mx in wins]


@gpu
def test_device_write_set_equals_reference_write_set():
    """ref_compat: the device buffer holds exactly the reference's writes (window minus its last row and column);
    every other cell keeps its sentinel.  The largest map also checks both squared planes of the caller-buffer update."""
    ctx = new_ctx()
    cases = patchwork_windows(6) + far_field_maps() + uniform_maps() + degenerate_windows()
    largest = max(range(len(cases)), key=lambda i: (cases[i][4][0] - cases[i][3][0] + 1) * (cases[i][4][1] - cases[i][3][1] + 1))
    for i, (glx, gly, grid, mn, mx) in enumerate(cases):
        check_ref_compat(ctx, workloads.make_geom(glx, gly, 0.05), grid, mn, mx, sq=(i == largest))
    ctx.close()


def map_2048(name):
    n = 2048
    if name == "bernoulli_0.02":
        return workloads.random_map(n, n, 2, p_occ=0.02)
    if name == "sparse_1e-4":
        return workloads.random_map(n, n, 3, p_occ=1e-4, p_unknown=0.0, wall=False)
    if name == "dense_0.5":
        return workloads.random_map(n, n, 4, p_occ=0.5)
    if name == "corridor":
        return workloads.corridor_map(n, n, 5, width_cells=64)
    grid = np.full(n * n, OCC if name == "all_occupied" else FREE, np.uint8)
    if name == "single_seed":
        grid[777 * n + 1300] = OCC
    return grid


@gpu
@pytest.mark.parametrize("name", ["bernoulli_0.02", "sparse_1e-4", "dense_0.5", "empty", "single_seed", "corridor",
                                  "all_occupied"])
def test_clean_mode_2048_variants_exact(name):
    ctx = new_ctx()
    check_clean(ctx, workloads.make_geom(2048, 2048, 0.05), map_2048(name), (0, 0), (2047, 2047))
    ctx.close()


@gpu
def test_clean_mode_corridor_8192x2048_exact():
    ctx = new_ctx()
    glx, gly = 8192, 2048
    grid = workloads.corridor_map(glx, gly, 5, width_cells=400, clutter=0.02)
    check_clean(ctx, workloads.make_geom(glx, gly, 0.005), grid, (0, 0), (glx - 1, gly - 1), sq=False)
    ctx.close()


@gpu
def test_clean_mode_far_field_patchwork_and_uniform_exact():
    """Far cells in clean mode (the band kernel), windows anywhere, all-free and all-Occupied windows
    (gi*sqrt(DBL_MAX) for the missing kind), degenerate windows."""
    ctx = new_ctx()
    for glx, gly, grid, mn, mx in far_field_maps() + patchwork_windows(8, 900) + uniform_maps() + degenerate_windows():
        check_clean(ctx, workloads.make_geom(glx, gly, 0.05), grid, mn, mx)
    ctx.close()


# ---- every row-pass (K1) variant ---------------------------------------------------------------------------------
def k1_kernel(gly, min_y, NY, occ_offset):
    """esdf.cu's choice of row-pass kernel (alore_esdf_run), for a caller buffer `occ_offset` bytes past a 256-byte
    aligned allocation."""
    G16 = (NY + 15) // 16
    GP = (G16 + 255) // 256
    if occ_offset % 16 == 0 and gly % 16 == 0 and min_y % 16 == 0 and GP <= 8:
        return "row_pass16<%d>" % (1 if GP <= 1 else 2 if GP <= 2 else 4 if GP <= 4 else 8)
    smem = (((NY + 31 + 15) >> 4) << 4) + 2 * NY + 16
    if smem > 48 * 1024:
        return "byte_smem_optin"
    return "byte_unaligned" if occ_offset % 16 else "byte"


# (NX, gly, min_y, NY, occ byte offset, kernel); every window spans rows 0..NX-1, so it ends on the caller buffer's
# last row: with an offset base the byte path reads up to the end of the caller's allocation
K1_CASES = [
    (24, 4096, 0, 4096, 0, "row_pass16<1>"),
    (29, 1072, 16, 1031, 0, "row_pass16<1>"),           # ragged last group: 1031 % 16 = 7, window inside the row
    (33, 4112, 0, 4097, 0, "row_pass16<2>"),            # 4097 % 16 = 1
    (24, 4112, 0, 4112, 0, "row_pass16<2>"),
    (40, 8192, 0, 8192, 0, "row_pass16<2>"),
    (31, 8224, 16, 8193, 0, "row_pass16<4>"),           # 8193 % 16 = 1
    (24, 8208, 0, 8208, 0, "row_pass16<4>"),
    (25, 16384, 0, 16368, 0, "row_pass16<4>"),
    (26, 16384, 0, 16383, 0, "row_pass16<4>"),          # 16383 % 16 = 15
    (24, 16384, 0, 16384, 0, "row_pass16<4>"),
    (28, 4101, 3, 4097, 0, "byte"),
    (30, 16375, 2, 16368, 0, "byte"),                   # dynamic shared memory exactly 48 KB: no opt-in
    (27, 16380, 5, 16369, 0, "byte_smem_optin"),
    (24, 16390, 5, 16383, 0, "byte_smem_optin"),
    (25, 16385, 1, 16384, 0, "byte_smem_optin"),
    (24, 2048, 0, 2048, 1, "byte_unaligned"),
    (29, 2064, 16, 2041, 7, "byte_unaligned"),
    (33, 4112, 0, 4112, 15, "byte_unaligned"),
]


def k1_map(NX, gly, seed):
    """Sparse clutter and Unknown cells, a row without any Occupied cell, a solid row, a long solid run."""
    rng = np.random.default_rng(seed)
    g = np.where(rng.random((NX, gly)) < 1e-3, OCC, FREE).astype(np.uint8)
    g[rng.random((NX, gly)) < 0.01] = UNK
    g[1, :] = FREE
    g[2, :] = OCC
    g[NX // 2, gly // 5: gly // 5 + min(gly // 2, 9000)] = OCC
    g[NX - 1, gly - 1] = OCC
    return np.ascontiguousarray(g.reshape(-1))


@gpu
@pytest.mark.parametrize("case", K1_CASES, ids=["%s_ny%d_off%d" % (c[5], c[3], c[4]) for c in K1_CASES])
def test_every_row_pass_variant(case):
    """Each case lands on a known K1 kernel (k1_kernel restates the dispatch); distances and squared planes against
    the oracle (ref_compat) and against the exact EDT (clean)."""
    NX, gly, min_y, NY, off, _ = case
    ctx = new_ctx()
    geom = workloads.make_geom(NX, gly, 0.05)
    grid = k1_map(NX, gly, NX * gly + off)
    mn, mx = (0, min_y), (NX - 1, min_y + NY - 1)
    check_ref_compat(ctx, geom, grid, mn, mx, sq=True, occ_offset=off)
    check_clean(ctx, geom, grid, mn, mx, host=False, occ_offset=off)
    ctx.close()


# ---- the 16384-cell window limit ---------------------------------------------------------------------------------
def corner_strip(NX, NY, inverted):
    """One seed in a corner: row distances up to 16383 and column distances up to 16383 (16383^2 + 47^2 in the
    squared plane of a 16384 x 48 strip); inverted: all Occupied but one free corner cell (the other plane)."""
    g = np.full((NX, NY), OCC if inverted else FREE, np.uint8)
    g[0, 0] = FREE if inverted else OCC
    return np.ascontiguousarray(g.reshape(-1))


@gpu
@pytest.mark.parametrize("shape", [(16384, 48), (48, 16384)])
def test_window_limit_corner_seed_strips(shape):
    """16384-cell sides: far cells everywhere (band kernel, 512 blocks of minima per column on 16384 rows) and the
    aliased column over 16384 rows."""
    NX, NY = shape
    ctx = new_ctx()
    geom = workloads.make_geom(NX, NY, 0.05)
    for inverted in (False, True):
        grid = corner_strip(NX, NY, inverted)
        check_ref_compat(ctx, geom, grid, (0, 0), (NX - 1, NY - 1), sq=True)
        check_clean(ctx, geom, grid, (0, 0), (NX - 1, NY - 1), host=False)
        pos, neg = last_sq(ctx, (0, 0), (NX - 1, NY - 1))
        plane = neg if inverted else pos
        assert plane.max() == (NX - 1) ** 2 + (NY - 1) ** 2        # the far corner, exactly
    ctx.close()


@gpu
def test_window_limit_two_sub_band_kernel():
    """16384 x 512 = 8 Mcells: the default band kernel switches to two sub-bands per thread."""
    NX, NY = 16384, 512
    ctx = new_ctx()
    geom = workloads.make_geom(NX, NY, 0.05)
    grid = strip_map(NX, NY, 77)
    check_ref_compat(ctx, geom, grid, (0, 0), (NX - 1, NY - 1), sq=True)
    check_clean(ctx, geom, grid, (0, 0), (NX - 1, NY - 1), sq=False, host=False)
    ctx.close()


@gpu
def test_window_over_the_limit_is_refused_and_context_stays_exact():
    ctx = new_ctx()
    for (glx, gly), mn, mx in (((16385, 8), (1, 0), (16384, 7)), ((8, 16385), (0, 1), (7, 16384))):
        geom = workloads.make_geom(glx, gly, 0.05)
        grid = corner_strip(glx, gly, False)
        host = np.full(glx * gly, SENT)
        rc = host_update(ctx, geom, grid, (0, 0), (glx - 1, gly - 1), host, True)
        assert rc == EINVAL and np.all(host == SENT)
        # the next update, an in-limit window of the same map, on the same context is exact
        ctx.check(host_update(ctx, geom, grid, mn, mx, host, True))
        assert same_bits(host, oracle_update(geom, grid, mn, mx, np.full(glx * gly, SENT)))
    # a map larger than the limit, window of 16384 rows inside it, through the caller-buffer path
    glx, gly = 16500, 40
    grid = strip_map(glx, gly, 5)
    check_ref_compat(ctx, workloads.make_geom(glx, gly, 0.05), grid, (100, 3), (16483, 38), sq=True)
    ctx.close()


# ---- padding columns of the row buffer ----------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("ref_compat", [True, False])
@pytest.mark.parametrize("order", ["forward", "reverse"])
def test_row_buffer_padding_columns_never_reach_an_output(order, ref_compat):
    """Three windows of the same row pitch (256) on one context: A (250 cells per row, dense clutter: negative row
    distances in columns 200..249), B (200, nearly empty: far cells, the band kernel reads whole tiles), C (fast row
    pass with a ragged last group: 201 cells, stores up to column 207)."""
    NX = 300
    a = (NX, 250, workloads.random_map(NX, 250, 1, p_occ=0.45, p_unknown=0.02, wall=False), (0, 0), (NX - 1, 249))
    gb = np.full(NX * 200, FREE, np.uint8)
    gb[37 * 200 + 11] = OCC
    b = (NX, 200, gb, (0, 0), (NX - 1, 199))
    c = (NX, 208, workloads.random_map(NX, 208, 3, p_occ=0.002, p_unknown=0.0, wall=False), (0, 0), (NX - 1, 200))
    seq = [a, b, c, b, a, c] if order == "forward" else [c, b, a, c, b, a]
    ctx = new_ctx()
    for glx, gly, grid, mn, mx in seq:
        geom = workloads.make_geom(glx, gly, 0.1)
        host = np.full(glx * gly, SENT)
        ctx.check(host_update(ctx, geom, grid, mn, mx, host, ref_compat))
        if ref_compat:
            assert same_bits(host, oracle_update(geom, grid, mn, mx, np.full(glx * gly, SENT)))
        else:
            assert same_bits(host, expected_clean(grid, glx, gly, 0.1, mn, mx, np.full(glx * gly, SENT))[0])
    ctx.close()


# ---- the three update_dev modes and alore_esdf_set on a caller stream ---------------------------------------------
GLX = GLY = 400


def box_world(seed=7):
    return workloads.random_map(GLX, GLY, seed, p_occ=0.0, p_unknown=0.0, wall=True, boxes=25, box_cells=(6, 24))


def opt_params():
    prm = capi.default_params()
    prm.alm_max_outer = 20
    return prm


def dev_opt(ctx, prm, cands):
    res = capi.ResultBatch(cands)
    cs, rs = cands.as_struct(), res.as_struct()
    ctx.check(ctx.lib.alore_opt_batch(ctx.h, C.byref(prm), C.byref(cs), C.byref(rs)))
    return res


def dev_penalty(ctx, prm, po, coeffs, T, s_xy, f_xy):
    po, coeffs, T, s_xy, f_xy = (np.ascontiguousarray(a) for a in (po, coeffs, T, s_xy, f_xy))
    B, tot = po.size - 1, int(po[-1])
    cost, gC, gT, err = np.zeros(B), np.zeros((tot, 6, 2)), np.zeros(tot), np.zeros((B, 2))
    ctx.check(ctx.lib.alore_penalty_batch(ctx.h, C.byref(prm), B, capi.iptr(po), capi.dptr(coeffs), capi.dptr(T),
                                          capi.dptr(s_xy), capi.dptr(f_xy), capi.dptr(cost), capi.dptr(gC), capi.dptr(gT),
                                          capi.dptr(err)))
    return cost, gC, gT


def check_penalty(ctx, prm, geom, dist, splines):
    got = dev_penalty(ctx, prm, *splines)
    ref = oracle_lib.penalty_batch(prm, geom, dist, *splines, 4)
    for a, b in zip(got, ref[:3]):
        assert same_bits(a, b)
    return got


def legs(grid, geom, dist, n=40, seed=5):
    pts = workloads.free_points(grid, geom, dist, 9, seed, min_clear=0.8)
    return workloads.leg_candidates(pts, headings=(0.0, 1.57), max_legs=n)


@gpu
def test_resident_rebuild_and_device_grid_update_on_a_caller_stream(portable_trig):
    """(NULL, NULL): rebuild from the resident grid; (d_occ, NULL): the window's rows of a device grid replace the
    resident ones, then rebuild.  Both on a caller stream; checked through last_sq, penalty_batch and opt_batch."""
    import torch
    ctx = new_ctx()
    prm = opt_params()
    geom = workloads.make_geom(GLX, GLY, 0.05)
    full = ((0, 0), (GLX - 1, GLY - 1))
    g0 = box_world()
    # a host update of rows 50..349 on a fresh map (device ESDF at DBL_MAX): the resident grid's other rows stay Unknown
    host = np.full(GLX * GLY, DBL_MAX)
    hw = ((50, 0), (349, GLY - 1))
    ctx.check(host_update(ctx, geom, g0, *hw, host, True))
    expect = oracle_update(geom, g0, *hw, np.full(GLX * GLY, DBL_MAX))
    assert same_bits(host, expect)
    stream = torch.cuda.Stream()
    # 1. (NULL, NULL) over the full window
    ctx.check(update_dev(ctx, geom, None, *full, None, True, stream))
    stream.synchronize()
    resident = g0.copy().reshape(GLX, GLY)
    resident[:50] = UNK
    resident[350:] = UNK
    resident = np.ascontiguousarray(resident.reshape(-1))
    expect, sp_, sn_ = oracle_update(geom, resident, *full, expect, want_sq=True)
    check_sq_ref_compat(ctx, *full, sp_, sn_)
    cands = legs(g0, geom, expect)
    from alore_legged_manipulator_b200.ms_planner import DeviceBatch
    db = DeviceBatch(ctx, cands)
    db.run(prm, stream_ptr(stream))
    assert check_results(db.download(), oracle_lib.opt_batch(prm, geom, expect, cands, 8), cands) == 0.0
    db.close()
    # 2. (d_occ, NULL) with a sub-window: rows 100..299 of a new grid, columns 80..319 rebuilt
    g1 = box_world(8)
    d_g1 = torch.from_numpy(g1).cuda()
    torch.cuda.synchronize()
    sub = ((100, 80), (299, 319))
    ctx.check(update_dev(ctx, geom, d_g1.data_ptr(), *sub, None, True, stream))
    stream.synchronize()
    merged = resident.copy().reshape(GLX, GLY)
    merged[100:300] = g1.reshape(GLX, GLY)[100:300]
    merged = np.ascontiguousarray(merged.reshape(-1))
    expect, sp_, sn_ = oracle_update(geom, merged, *sub, expect, want_sq=True)
    check_sq_ref_compat(ctx, *sub, sp_, sn_)
    splines = workloads.random_spline_batch(24, 24, geom, expect, merged, seed=3)   # they cross the window's border
    check_penalty(ctx, prm, geom, expect, splines)
    cands = legs(g1, geom, expect, seed=6)
    assert check_results(dev_opt(ctx, prm, cands), oracle_lib.opt_batch(prm, geom, expect, cands, 8), cands) == 0.0
    # the resident grid really is the merge: a full rebuild from it
    ctx.check(update_dev(ctx, geom, None, *full, None, True, stream))
    stream.synchronize()
    expect = oracle_update(geom, merged, *full, expect)
    check_penalty(ctx, prm, geom, expect, splines)
    # 3. (d_occ, NULL) over the full window
    g2 = box_world(9)
    d_g2 = torch.from_numpy(g2).cuda()
    torch.cuda.synchronize()
    ctx.check(update_dev(ctx, geom, d_g2.data_ptr(), *full, None, True, stream))
    stream.synchronize()
    expect, sp_, sn_ = oracle_update(geom, g2, *full, expect, want_sq=True)
    check_sq_ref_compat(ctx, *full, sp_, sn_)
    before = check_penalty(ctx, prm, geom, expect, splines)
    # 4. caller buffers of another geometry: exact, and the resident map is untouched
    geom_c = workloads.make_geom(300, 520, 0.05)
    gc = workloads.random_map(300, 520, 12, p_occ=0.03)
    check_ref_compat(ctx, geom_c, gc, (7, 9), (290, 511), sq=True)
    after = dev_penalty(ctx, prm, *splines)
    for a, b in zip(before, after):
        assert same_bits(a, b)
    ctx.close()


@gpu
def test_update_dev_error_paths_leave_the_context_usable(portable_trig):
    import torch
    ctx = new_ctx()
    stream = torch.cuda.Stream()
    geom = workloads.make_geom(GLX, GLY, 0.05)
    full = ((0, 0), (GLX - 1, GLY - 1))
    g0 = box_world()
    d_g0 = torch.from_numpy(g0).cuda()
    d_dist = torch.zeros(GLX * GLY, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    assert update_dev(ctx, geom, None, *full, None, True, stream) == ENOMAP            # no resident map yet
    assert update_dev(ctx, geom, d_g0.data_ptr(), *full, None, True, stream) == ENOMAP
    host = np.full(GLX * GLY, DBL_MAX)
    ctx.check(host_update(ctx, geom, g0, *full, host, True))
    other = workloads.make_geom(200, 800, 0.05)                                            # same cell count
    assert update_dev(ctx, other, None, (0, 0), (199, 799), None, True, stream) == EINVAL
    assert update_dev(ctx, other, d_g0.data_ptr(), (0, 0), (199, 799), None, True, stream) == ENOMAP
    assert update_dev(ctx, geom, None, *full, d_dist.data_ptr(), True, stream) == EINVAL   # dist without occ
    assert update_dev(ctx, geom, None, (0, 0), (GLX, GLY - 1), None, True, stream) == EINVAL
    assert update_dev(ctx, geom, d_g0.data_ptr(), (0, 0), (GLX - 1, GLY), None, True, stream) == EINVAL
    assert update_dev(ctx, geom, d_g0.data_ptr(), (0, -1), (GLX - 1, 5), d_dist.data_ptr(), True, stream) == EINVAL
    # a refused device-grid update leaves the resident grid as it was
    g1 = np.ascontiguousarray(np.full(GLX * GLY, OCC, np.uint8))
    d_g1 = torch.from_numpy(g1).cuda()
    torch.cuda.synchronize()
    assert update_dev(ctx, geom, d_g1.data_ptr(), (0, 0), (GLX - 1, GLY + 3), None, True, stream) == EINVAL
    ctx.check(update_dev(ctx, geom, None, *full, None, True, stream))
    stream.synchronize()
    prm = opt_params()
    splines = workloads.random_spline_batch(16, 16, geom, host, g0, seed=4)
    check_penalty(ctx, prm, geom, oracle_update(geom, g0, *full, np.full(GLX * GLY, DBL_MAX)), splines)
    ctx.close()


@gpu
def test_esdf_set_gives_the_optimizer_the_same_map(portable_trig):
    """alore_esdf_set with the oracle's ESDF = alore_esdf_update of the same grid, bit for bit in opt_batch; a set of
    another geometry re-shapes the map."""
    prm = opt_params()
    geom = workloads.make_geom(GLX, GLY, 0.05)
    g0 = box_world()
    ref = oracle_update(geom, g0, (0, 0), (GLX - 1, GLY - 1), np.full(GLX * GLY, DBL_MAX))
    cands = legs(g0, geom, ref)
    a_ctx, b_ctx = new_ctx(), new_ctx()
    host = np.full(GLX * GLY, DBL_MAX)
    a_ctx.check(host_update(a_ctx, geom, g0, (0, 0), (GLX - 1, GLY - 1), host, True))
    a = dev_opt(a_ctx, prm, cands)
    b_ctx.check(b_ctx.lib.alore_esdf_set(b_ctx.h, C.byref(geom), capi.dptr(ref)))
    b = dev_opt(b_ctx, prm, cands)
    for f in capi.ResultBatch._FIELDS:
        assert np.array_equal(getattr(a, f).view(np.uint8), getattr(b, f).view(np.uint8)), f
    assert check_results(b, oracle_lib.opt_batch(prm, geom, ref, cands, 8), cands) == 0.0
    geom2 = workloads.make_geom(260, 610, 0.05)
    g2 = workloads.random_map(260, 610, 31, p_occ=0.0, p_unknown=0.0, boxes=20, box_cells=(6, 24))
    ref2 = oracle_update(geom2, g2, (0, 0), (259, 609), np.full(260 * 610, DBL_MAX))
    b_ctx.check(b_ctx.lib.alore_esdf_set(b_ctx.h, C.byref(geom2), capi.dptr(ref2)))
    check_penalty(b_ctx, prm, geom2, ref2, workloads.random_spline_batch(20, 20, geom2, ref2, g2, seed=9))
    a_ctx.close()
    b_ctx.close()


# ---- the benchmark's resident tick in miniature -------------------------------------------------------------------
def perturbed_tick(t, geom, grid0, pts0):
    """Tick t of a replanning loop: the robot's way-point moved by <= 0.3 m, one 10 x 10-cell box painted at a
    tick-dependent spot more than 2 m from every way-point."""
    rng = np.random.default_rng(1000 + t)
    pts = pts0.copy()
    pts[0] = pts0[0] + rng.uniform(-0.3, 0.3, 2)
    grid = grid0.copy()
    g = grid.reshape(geom.glx, geom.gly)
    while True:
        cx, cy = rng.integers(40, geom.glx - 50, 2)
        wx, wy = geom.x_lower + (cx + 5) * geom.grid_interval, geom.y_lower + (cy + 5) * geom.grid_interval
        if np.min(np.hypot(pts[:, 0] - wx, pts[:, 1] - wy)) > 2.0:
            break
    g[cx:cx + 10, cy:cy + 10] = OCC
    return grid, pts


@gpu
def test_resident_tick_device_grid_then_batch_run_on_a_caller_stream(portable_trig):
    """Per tick: alore_esdf_update_dev(d_occ) + alore_batch_run on the same caller stream + on-device argmin; every
    tick's results bit-identical to the oracle on that tick's grid."""
    import torch
    from alore_legged_manipulator_b200.ms_planner import DeviceBatch
    ctx = new_ctx()
    prm = opt_params()
    geom = workloads.make_geom(GLX, GLY, 0.05)
    full = ((0, 0), (GLX - 1, GLY - 1))
    g0 = box_world()
    host = np.full(GLX * GLY, DBL_MAX)
    ctx.check(host_update(ctx, geom, g0, *full, host, True))        # the map the ticks perturb, resident
    pts0 = workloads.free_points(g0, geom, host, 9, 5, min_clear=0.8)
    stream = torch.cuda.Stream()
    for t in (1, 2, 3):
        grid, pts = perturbed_tick(t, geom, g0, pts0)
        cands = workloads.leg_candidates(pts, headings=(0.0, 1.57), max_legs=48)
        db = DeviceBatch(ctx, cands)
        d_grid = torch.from_numpy(grid).cuda()
        torch.cuda.synchronize()
        ctx.check(update_dev(ctx, geom, d_grid.data_ptr(), *full, None, True, stream))
        db.run(prm, stream_ptr(stream))
        bc, bi = db.argmin()
        res = db.download()
        ref_dist = oracle_update(geom, grid, *full, np.full(GLX * GLY, DBL_MAX))
        ref = oracle_lib.opt_batch(prm, geom, ref_dist, cands, 8)
        assert check_results(res, ref, cands) == 0.0
        ok = np.flatnonzero(ref.ok == 1)
        if ok.size:
            best = ok[np.argmin(ref.cost[ok])]
            assert bi == best and bc == ref.cost[best]
        else:
            assert bi == -1
        db.close()
    ctx.close()
