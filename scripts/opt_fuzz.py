"""Sequential fuzz of minco_plan_batch on ONE context: random worlds (boxes), random leg batches (ragged piece counts,
doglegs, cut trajectories), every result against the CPU oracle bit for bit (portable-trig contract).  usage: python scripts/opt_fuzz.py [rounds] [seed]"""
import sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import numpy as np
import alore_legged_manipulator_b200 as alore
from alore_legged_manipulator_b200 import capi, front_end, workloads
from alore_legged_manipulator_b200.ms_planner import MSPlanner
import oracle_lib
from test_esdf_gpu import make_sdf
from test_optimizer_gpu import check_results
rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 12
seed = int(sys.argv[2]) if len(sys.argv) > 2 else 3
rng = np.random.default_rng(seed)
ctx = alore.Context(0)
olib = oracle_lib.load()
olib.orc_set_trig_portable(1)
total = 0
for it in range(rounds):
    glx, gly = int(rng.integers(300, 520)), int(rng.integers(300, 520))
    grid = workloads.random_map(glx, gly, int(rng.integers(1, 10**6)), p_occ=0.0, p_unknown=0.0, wall=True,
                                boxes=int(rng.integers(8, 40)), box_cells=(5, 26))
    m = make_sdf(ctx, glx, gly, 0.05, grid)
    m.updateESDF2d()
    prm = capi.default_params()
    prm.alm_max_outer = int(rng.integers(4, 20))
    if rng.random() < 0.3:
        prm.finalMinSafeDis = 0.45
        prm.safeReplanMaxTime = 2
    pl = MSPlanner(ctx, prm, m)
    fe = front_end.FrontEndParams()
    if rng.random() < 0.3:
        fe.trajCutLength = 4.0
    pts = workloads.free_points(grid, m.geom(), m.distance_buffer_all_, int(rng.integers(5, 10)), int(rng.integers(1, 10**6)), min_clear=0.6)
    cands = workloads.leg_candidates(pts, headings=(0.0, float(rng.uniform(0.5, 3.0))), fe=fe, max_legs=int(rng.integers(20, 70)),
                                     dogleg=float(rng.uniform(0.0, 0.7)))
    res = pl.minco_plan_batch(cands)
    ref = oracle_lib.opt_batch(prm, m.geom(), m.distance_buffer_all_, cands, 8)
    worst = check_results(res, ref, cands)
    assert worst == 0.0, (it, worst)
    total += cands.B
    print(f"round {it}: {glx}x{gly}, {cands.B} candidates, pieces {int(np.diff(cands.piece_off).min())}..{int(np.diff(cands.piece_off).max())}, "
          f"ok {int(res.ok.sum())}, replans max {int(res.replans.max())}: identical")
    m.close()
olib.orc_set_trig_portable(0)
print(f"opt fuzz: {rounds} rounds, {total} candidates ok (seed {seed})")
