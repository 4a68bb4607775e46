"""Task-plan time on sub-problems of the bench world: python scripts/task_plan_time.py [--calls 20] [--out FILE]

Builds the bench world (bench.build_world / bench.way_points), takes the robot, chairs 1..20 and targets 33..52, and
optimises every task leg among them (robot -> chair, chair -> target, target -> chair) in the bench's 16 heading
variants once with DeviceBatch.  Each sub-problem of n objects (points 1..n as objects, 33..32+n as targets) labels
the candidates of its own legs and marks every other candidate -1.  It then times alore_batch_task_plan (host clock
around the blocking call, which ends in a stream synchronise; median of --calls calls after 3 warm-up calls) and the
sequential oracle orc_task_plan on one host thread (median of 3 calls) on the same results, asserts that both plans
are equal bit for bit, and prints one JSON line with the GPU's name and power limit read in the same run.
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
from task_plan_util import assert_same_plan, oracle_plan, task_leg_batch  # noqa: E402

CASES = [("free", 8), ("free", 10), ("free", 12), ("fixed", 12), ("fixed", 16), ("fixed", 20)]
NMAX = 20


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
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
    ids = [0] + list(range(1, NMAX + 1)) + list(range(33, 33 + NMAX))        # task point -> bench point
    variants = [((v // 8) * math.pi / 2, (v % 8) * math.pi / 4) for v in range(16)]
    cands, lf_max, lt_max = task_leg_batch(pts, ids, variants)
    prm = alore.default_params()
    db = DeviceBatch(ctx, cands)
    t0 = time.perf_counter()
    db.run(prm)
    res = db.download()
    opt_s = time.perf_counter() - t0
    bench_from, bench_to = np.array(ids)[lf_max], np.array(ids)[lt_max]
    rows = []
    for mode, n in CASES:
        # task point of every bench point of this sub-problem; candidates of any other leg are not task legs
        tp = {0: 0, **{i: i for i in range(1, n + 1)}, **{32 + i: n + i for i in range(1, n + 1)}}
        lf = np.array([tp.get(int(a), -1) if int(b) in tp else -1 for a, b in zip(bench_from, bench_to)], np.int32)
        lt = np.array([tp.get(int(b), -1) if l >= 0 else -1 for b, l in zip(bench_to, lf)], np.int32)
        fixed = mode == "fixed"
        gpu = db.task_plan(n, lf, lt, fixed, None, with_matrix=True)
        gpu_ms = median_time(lambda: db.task_plan(n, lf, lt, fixed, None), args.calls, 3)
        ref = oracle_plan(n, lf, lt, res.cost, res.ok, fixed, None)
        cpu_ms = median_time(lambda: oracle_plan(n, lf, lt, res.cost, res.ok, fixed, None, with_matrix=False), 3, 0)
        assert_same_plan(gpu, ref)
        states = sum(math.comb(n, k) * (1 if fixed else math.comb(n, k - 1)) * k + math.comb(n, k) * (1 if fixed else math.comb(n, k)) * k
                     for k in range(1, n + 1))
        rows.append({"mode": mode, "n": n, "task_legs_labelled": int((lf >= 0).sum()), "dp_states": states,
                     "gpu_ms": round(gpu_ms, 4), "oracle_ms": round(cpu_ms, 2), "speedup": round(cpu_ms / gpu_ms, 1),
                     "gpu_mstates_per_s": round(states / gpu_ms / 1e3, 1), "feasible": gpu.feasible,
                     "cost": gpu.cost, "plan_equals_oracle": True})
    line = {"script": "task_plan_time", **info,
            "batch": {"candidates": cands.B, "ok": int(res.ok.sum()), "optimise_s": round(opt_s, 3)},
            "timing": f"alore_batch_task_plan: host clock around the blocking call, median of {args.calls} after 3 warm-up; "
                      "oracle: orc_task_plan on one host thread, median of 3",
            "cases": rows}
    print(json.dumps(line))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(line) + "\n")
    db.close()
    m.close()
    ctx.close()


if __name__ == "__main__":
    main()
