"""Small, fixed workloads for ncu captures (one process, one GPU):  esdf | penalty | opt"""
import sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import numpy as np
import alore_legged_manipulator_b200 as alore
from alore_legged_manipulator_b200 import workloads, capi
from alore_legged_manipulator_b200.ms_planner import MSPlanner, DeviceBatch
from test_esdf_gpu import make_sdf

which = sys.argv[1]
ctx = alore.Context(0)
prm = alore.default_params()
if which == "esdf":
    n = 4096
    grid = workloads.random_map(n, n, 2, p_occ=0.02, p_unknown=0.01)
    m = make_sdf(ctx, n, n, 0.05, grid)
    for _ in range(3):
        m.updateESDF2d()
    print("esdf kernels ms", m.last_kernel_ms())
else:
    n = 2048
    grid = workloads.random_map(n, n, 4 if which == "bench" else 3, p_occ=0.0, p_unknown=0.0, wall=True, boxes=400, box_cells=(6, 30))
    m = make_sdf(ctx, n, n, 0.05, grid)
    m.updateESDF2d()
    pl = MSPlanner(ctx, prm, m)
    if which == "penalty":
        B = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
        po, coeffs, T, s_xy, f_xy = workloads.random_spline_batch(B, 64, m.geom(), m.distance_buffer_all_, grid, seed=3)
        for _ in range(2):
            c, gC, gT, err = pl.penalty_batch(po, coeffs, T, s_xy, f_xy)
        print("penalty done", float(c.mean()))
    elif which == "cost":
        # B copies of one ~64-piece leg: one full cost+gradient evaluation per warp (stage 1 then stage 0)
        import oracle_lib
        from alore_legged_manipulator_b200 import front_end
        B = int(sys.argv[2]) if len(sys.argv) > 2 else 1184
        pts = workloads.free_points(grid, m.geom(), m.distance_buffer_all_, 40, 4, min_clear=0.9)
        best = None
        for i in range(40):
            for j in range(40):
                if i != j:
                    ft = front_end.make_flat_traj([tuple(pts[i]), tuple(pts[j])], (pts[i][0], pts[i][1], 0.0), (pts[j][0], pts[j][1], 1.0))
                    if best is None or abs(ft.TrajNum - 64) < abs(best.TrajNum - 64):
                        best = ft
        print("pieces", best.TrajNum)
        cands = front_end.pack_candidates([best] * B)
        x = np.tile(oracle_lib.initial_x(cands, 0), B)
        for stage in (1, 0, 1):
            c, g, e = pl.cost_batch(cands, stage, x)
        print("cost done", c[0])
    elif which == "bench":
        # the exact per-GPU candidate block of bench.py (rank 0), one optimisation launch
        import bench
        B = int(sys.argv[2]) if len(sys.argv) > 2 else bench.PER_GPU
        cands = bench.build_candidates(m.geom(), grid, m.distance_buffer_all_, 0, B)
        db = DeviceBatch(ctx, cands)
        reps = int(sys.argv[3]) if len(sys.argv) > 3 else 1
        for rep in range(reps):
            db.run(prm)
            r = db.download()
            if reps > 1:
                print("  run", rep, "kernel ms", db.kernel_ms())
        print("bench block done: kernel ms", db.kernel_ms(), "ok", int(r.ok.sum()), "evals", int(r.evals.sum()), "alg bytes", db.stats()[0])
    else:
        B = int(sys.argv[2]) if len(sys.argv) > 2 else 256
        pts = workloads.free_points(grid, m.geom(), m.distance_buffer_all_, 40, 4, min_clear=0.9)
        legs = workloads.leg_candidates(pts, headings=(0.0,), max_legs=B)
        db = DeviceBatch(ctx, legs)
        db.run(prm)
        r = db.download()
        print("opt done: kernel ms", db.kernel_ms(), "ok", int(r.ok.sum()), "evals", int(r.evals.sum()))

import ctypes as C
ph = (C.c_ulonglong * 32)()
if ctx.lib.alore_debug_phase_cycles(ctx.h, ph, 1) == 0:
    names = {0: "T-powers", 1: "LU+fwd", 2: "back", 3: "energy", 4: "penalty cost", 7: "penalty grad", 5: "adjoint", 6: "grad-out", 8: "  passA", 9: "  cells/prefix",
             10: "  passB", 11: "  cost-sum", 12: "  fold", 13: "  passC", 17: "lbfgs s/y+dots", 18: "lbfgs two-loop", 20: "history steps (count, M)", 21: "skipped grads (count, M)"}
    tot = sum(ph[i] for i in (0, 1, 2, 3, 4, 5, 6, 7, 17, 18))
    for i, nme in names.items():
        print(f"phase {nme:16s} {ph[i]/1e6:12.1f} Mcycles  {100.0*ph[i]/max(tot,1):5.1f}%")
