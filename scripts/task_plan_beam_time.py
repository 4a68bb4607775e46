"""Bounded-width task plan on the whole bench world: python scripts/task_plan_beam_time.py [--calls 10] [--out FILE]

Builds the bench world (bench.build_world / bench.way_points) and optimises every task leg of all 32 chairs once with
DeviceBatch: robot -> chair, chair -> target, target -> chair (task point p = bench point p: 0 the robot, 1..32 the
chairs, 33..64 the targets) in the bench's 16 heading variants.  On those results it
- times alore_batch_task_plan_beam (n = 32) in both modes at widths 1, 256, 4096 and 65536: host clock around the
  blocking call, which ends in a stream synchronise; median of --calls calls after 2 warm-up calls;
- times the sequential oracle orc_task_plan_beam once per width on one host thread, asserts that its plan equals the
  device's bit for bit, and skips (and says so) a width whose oracle call would take more than about --oracle-limit s
  judging by the previous width;
- reports every width's cost relative to width 1;
- lists the chairs whose leg to their own target (chair i -> target 32+i) has no counted candidate, which makes the
  fixed-mode plan infeasible at every width;
- on the n = 12 free and n = 20 fixed sub-problems (chairs 1..n, targets 33..32+n) reports the gap of every width's
  cost to the exact optimum of alore_batch_task_plan.
Prints one JSON line with the GPU's name and power limit read in the same run.
"""
import argparse
import json
import math
import subprocess
import sys
import time
from pathlib import Path

sys.dont_write_bytecode = True
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import numpy as np  # noqa: E402

import bench  # noqa: E402
import alore_legged_manipulator_b200 as alore  # noqa: E402
from alore_legged_manipulator_b200.ms_planner import DeviceBatch  # noqa: E402
from task_plan_util import assert_same_beam_plan, oracle_plan_beam, task_leg_batch  # noqa: E402

N = 32
WIDTHS = [1, 256, 4096, 65536]
SUBPROBLEMS = [("free", 12), ("fixed", 20)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def median_time(fn, calls, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(calls):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)) * 1e3


def sub_labels(n, lf, lt):
    """Labels of the sub-problem with chairs 1..n and targets 33..32+n; every other candidate is not a task leg."""
    tp = {0: 0, **{i: i for i in range(1, n + 1)}, **{32 + i: n + i for i in range(1, n + 1)}}
    f = np.array([tp.get(int(a), -1) if int(b) in tp else -1 for a, b in zip(lf, lt)], np.int32)
    t = np.array([tp.get(int(b), -1) if x >= 0 else -1 for b, x in zip(lt, f)], np.int32)
    return f, t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--oracle-limit", type=float, default=60.0)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    info = gpu_info()
    ctx = alore.Context(0)
    geom, grid = bench.build_world()
    m = alore.SDFmap(ctx, gridmap_interval=0.05, detection_range=1e6, global_x_lower=geom.x_lower,
                     global_x_upper=geom.x_lower + (geom.glx - 0.5) * 0.05, global_y_lower=geom.y_lower,
                     global_y_upper=geom.y_lower + (geom.gly - 0.5) * 0.05)
    m.gridmap_[:] = grid
    m.has_map_ = True
    m.forceUpdateESDF()
    pts = bench.way_points(m.geom(), grid, m.distance_buffer_all_.copy())
    variants = [((v // 8) * math.pi / 2, (v % 8) * math.pi / 4) for v in range(16)]
    cands, lf, lt = task_leg_batch(pts, list(range(2 * N + 1)), variants)
    prm = alore.default_params()
    db = DeviceBatch(ctx, cands)
    t0 = time.perf_counter()
    db.run(prm)
    res = db.download()
    opt_s = time.perf_counter() - t0

    rows = []
    missing = None
    for mode in ("free", "fixed"):
        fixed = mode == "fixed"
        base = None
        oracle_s = None
        for i, w in enumerate(WIDTHS):
            gpu = db.task_plan(N, lf, lt, fixed, None, with_matrix=True, width=w)
            gpu_ms = median_time(lambda: db.task_plan(N, lf, lt, fixed, None, width=w), args.calls, 2)
            base = gpu.cost if base is None else base
            if missing is None:                      # fixed mode needs chair i -> target 32+i to have a counted candidate
                missing = [i for i in range(1, N + 1) if not np.isfinite(gpu.leg_cost[i, N + i])]
            row = {"mode": mode, "n": N, "width": w, "gpu_ms": round(gpu_ms, 3), "feasible": gpu.feasible,
                   "exact": gpu.exact, "cost": gpu.cost, "cost_vs_width_1": gpu.cost / base if gpu.feasible else None}
            guess = None if oracle_s is None else oracle_s * w / WIDTHS[i - 1]
            if guess is not None and guess > args.oracle_limit:
                row["oracle"] = f"skipped: about {guess:.0f} s expected from the previous width"
            else:
                t1 = time.perf_counter()
                ref = oracle_plan_beam(N, w, lf, lt, res.cost, res.ok, fixed, None)
                oracle_s = time.perf_counter() - t1
                assert_same_beam_plan(gpu, ref)
                row.update(oracle_ms=round(oracle_s * 1e3, 1), plan_equals_oracle=True)
            rows.append(row)

    gaps = []
    for mode, n in SUBPROBLEMS:
        fixed = mode == "fixed"
        f, t = sub_labels(n, lf, lt)
        ex = db.task_plan(n, f, t, fixed, None)
        for w in WIDTHS:
            p = db.task_plan(n, f, t, fixed, None, width=w)
            gaps.append({"mode": mode, "n": n, "width": w, "exact_flag": p.exact, "cost": p.cost, "optimum": ex.cost,
                         "gap_to_optimum": p.cost / ex.cost - 1.0 if ex.feasible and p.feasible else None})

    line = {"script": "task_plan_beam_time", **info,
            "batch": {"candidates": cands.B, "task_legs": int(cands.B // len(variants)), "ok": int(res.ok.sum()),
                      "optimise_s": round(opt_s, 3)},
            "timing": f"alore_batch_task_plan_beam: host clock around the blocking call, median of {args.calls} after "
                      "2 warm-up; oracle: orc_task_plan_beam on one host thread, one call",
            "fixed_mode_chairs_without_own_target_leg": missing, "n32": rows, "subproblem_gaps": gaps}
    print(json.dumps(line))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(line) + "\n")
    db.close()
    m.close()
    ctx.close()


if __name__ == "__main__":
    main()
