#!/usr/bin/env python
"""bench.py — the measurement contract of the planning_ddr_opt hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W

One STEP = one replan tick of one rank: rebuild the ESDF of the 2048x2048 map from its occupancy grid, then run
MSPlanner::minco_plan (stage A L-BFGS + stage B augmented-Lagrangian L-BFGS loop + final collision check with replans)
on the rank's block of candidate trajectories, find the best candidate on the device and (N>1) all-gather
(best cost, index) over NCCL.

Workload (BASELINE.json configs[3] family, weak scaling): 65 way-points (32 chairs + 32 targets + the robot) on a
2048^2 @0.05 m map -> 4160 ordered legs x 16 heading variants = 66 560 candidates (the batch of configs[4]); rank r
optimises candidates [8320 r, 8320 (r+1)): 8320 per GPU is configs[3] at its 2-GPU point.
EVERY TICK IS PERTURBED (tick t differs from tick t-1): the robot way-point moves by up to 0.3 m (its 2 x 64 legs x 16
variants are re-timed by the front end) and one 0.5 m box is repainted somewhere else on the map, so the ESDF changes
and the schedule prediction (evaluation counts of the previous tick) is never exact.  `config.cold_kernel_ms` is the
same tick without any prediction.

Prints ONE JSON line (rank 0).  `value` = candidates optimised per second, inputs resident in HBM, device time
(CUDA events), max over ranks.  `e2e` = the same through the host-buffer C ABI (alore_esdf_update + alore_opt_batch)
with every copy inside the timed region.  The reference arm runs the CPU restatement on a bounded random sample of
the SAME block with the ESDF cost amortised over the sample fraction, so both arms measure the same workload.

`--dump-outputs DIR` (rank 0) writes what the last timed tick returned as DIR/<name>.npy (float64), see dump_outputs.
The inputs depend on the arguments only, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

sys.dont_write_bytecode = True     # the benchmark may run from a read-only tree and writes nothing into it
ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

PER_GPU = 8320
METRIC = "candidate trajs optimized/sec (ESDF Mcells/s under 'esdf')"
UNIT = "trajs/s"
SAMPLE = 2080                      # candidates of the rank-0 block the CPU arm optimises per step
DUMP_LIMIT = 64 << 20              # bytes --dump-outputs writes at most, .npy headers included
DUMP_ESDF_CELLS = 1 << 19          # ESDF cells --dump-outputs writes (a seeded sample of the 2048^2 map)


def workload_config(per_gpu):
    """The `config` both arms print: same workload, same block, same perturbation rule."""
    return {"workload": f"configs[3] family: per step and per GPU, ESDF 2048^2 rebuild + minco_plan of {per_gpu} candidates "
                        f"(block r of 4160 legs x 16 heading variants = 66 560; 2 GPUs = the ~16k batch of configs[3], "
                        f"8 GPUs = the 65k-candidate tick of configs[4]); every tick perturbed (robot way-point moved <= 0.3 m, "
                        f"one 0.5 m box repainted)",
            "candidates_per_gpu": per_gpu, "sparseResolution": 8, "lbfgs_mem_size": 256}


def build_world(seed=4):
    """configs[3]: 2048^2 map with 400 boxes (deterministic)."""
    from alore_legged_manipulator_b200 import workloads
    n = 2048
    grid = workloads.random_map(n, n, seed, p_occ=0.0, p_unknown=0.0, wall=True, boxes=400, box_cells=(6, 30))
    geom = workloads.make_geom(n, n, 0.05)
    return geom, grid


def way_points(geom, grid, dist, seed=4):
    from alore_legged_manipulator_b200 import workloads
    # inside the central 50 m x 50 m of the 102 m map: leg lengths give TrajNum = 3 .. ~80 (SURVEY.md section 8d, config 4)
    return workloads.free_points(grid, geom, dist, 65, seed, min_clear=0.9, margin_m=26.0)


def candidates_from_points(pts, lo, hi):
    """Candidates [lo, hi) of the deterministic enumeration (variant-major so that every block spans all leg lengths):
    variant v = 0..15 -> goal heading (v % 8) * pi/4, start heading (v // 8) * pi/2; then i -> j over the 65 points."""
    from alore_legged_manipulator_b200 import front_end
    fts = []
    idx = 0
    for v in range(16):
        gh, sh = (v % 8) * math.pi / 4, (v // 8) * math.pi / 2
        for i in range(65):
            for j in range(65):
                if i == j:
                    continue
                if lo <= idx < hi:
                    a, b = pts[i], pts[j]
                    fts.append(front_end.make_flat_traj([tuple(a), tuple(b)], (a[0], a[1], sh), (b[0], b[1], gh)))
                idx += 1
    return front_end.pack_candidates(fts)


def build_candidates(geom, grid, dist, lo, hi, seed=4):
    return candidates_from_points(way_points(geom, grid, dist, seed), lo, hi)


def tick_variant(t, geom, grid0, pts0):
    """Tick t of the replanning loop: (grid_t, pts_t).  t = 0 is the unperturbed world."""
    if t == 0:
        return grid0, pts0
    rng = np.random.default_rng(1000 + t)
    pts = pts0.copy()
    pts[0] = pts0[0] + rng.uniform(-0.3, 0.3, 2)                 # the robot has moved
    grid = grid0.copy()
    g = grid.reshape(geom.glx, geom.gly)
    while True:                                                  # one 10 x 10-cell box repainted at a tick-dependent free spot
        cx, cy = rng.integers(300, geom.glx - 300, 2)
        wx, wy = geom.x_lower + (cx + 5) * geom.grid_interval, geom.y_lower + (cy + 5) * geom.grid_interval
        if np.min(np.hypot(pts[:, 0] - wx, pts[:, 1] - wy)) > 2.0:
            break
    g[cx:cx + 10, cy:cy + 10] = 2
    return grid, pts


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nme in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


FP64_PEAK_TFLOPS = 37.2     # 148 SMs x 64 FP64 FMA lanes x 2 flop x 1.965 GHz (measured issue rate: 2 DFMA warp-instr/clk/SM, profiles/)


def sample_indices(n, k, seed=11):
    """Unbiased bounded sample of a block: k of n candidates, seeded, in index order."""
    return np.sort(np.random.default_rng(seed).choice(n, size=min(k, n), replace=False))


def dump_outputs(out_dir, res, cands, best, dist, limit=DUMP_LIMIT):
    """--dump-outputs: the results of one tick as float64 .npy files under `out_dir`, `limit` bytes at most.

    best_cost / best_index: the winner the step returns.  esdf_distance: the tick's ESDF at the cells listed in
    esdf_cells (a seeded sample).  For the candidates listed in `candidates` (the whole block while it fits the limit,
    else a seeded sample), in that order: ok, status, replans, alm_iters, evals, cost, tail_s (one value each) and their
    pieces, piece_T [P], coeffs [P, 6, 2], inner_pts [P - len(candidates), 2]."""
    rng = np.random.default_rng(0)
    cells = np.sort(rng.choice(dist.size, size=min(DUMP_ESDF_CELLS, dist.size), replace=False))
    room = limit - (1 << 20) - 8 * (2 + 2 * cells.size)          # 1 MB spare for the .npy headers
    n = np.diff(cands.piece_off).astype(np.int64)
    per_cand = 8 * (15 * n + 6)      # index + 7 scalars; 12 coefficients and one duration per piece; N - 1 inner points
    keep = np.arange(cands.B)
    if per_cand.sum() > room:
        order = rng.permutation(cands.B)
        keep = np.sort(order[:np.searchsorted(np.cumsum(per_cand[order]), room, side="right")])
    po = cands.piece_off
    pieces = np.concatenate([np.arange(0)] + [np.arange(po[b], po[b + 1]) for b in keep]).astype(np.int64)
    inner = np.concatenate([np.arange(0)] + [np.arange(po[b] - b, po[b + 1] - b - 1) for b in keep]).astype(np.int64)
    arrays = {"best_cost": [best[0]], "best_index": [best[1]], "esdf_cells": cells, "esdf_distance": dist[cells],
              "candidates": keep, "piece_T": res.piece_T[pieces], "coeffs": res.coeffs[pieces], "inner_pts": res.inner_pts[inner]}
    for f in ("ok", "status", "replans", "alm_iters", "evals", "cost", "tail_s"):
        arrays[f] = getattr(res, f)[keep]
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", np.asarray(a, dtype=np.float64))


def cpu_arm(steps, warmup, per_gpu):
    """The reference's CPU algorithm (oracle port; the real one needs ROS+Eigen+PCL and cannot be built here, see
    DESIGN.md) on all host threads: per step, one single-thread 2048^2 ESDF rebuild (the reference's ESDF is serial)
    and minco_plan of a bounded random sample of the rank-0 block.  value = sample / (t_opt + t_esdf * sample/block):
    the ESDF is amortised over the sample fraction, i.e. what the full block would read.  Loads nothing of the product."""
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle_lib
    lib = oracle_lib.load()
    cores = int(lib.orc_hardware_threads()) or os.cpu_count() or 1
    geom, grid = build_world()
    dist = np.full(geom.glx * geom.gly, np.finfo(np.float64).max)
    oracle_lib.esdf_update(geom, grid, (0, 0), (geom.glx - 1, geom.gly - 1), dist)
    full = build_candidates(geom, grid, dist, 0, per_gpu)
    idx = sample_indices(full.B, SAMPLE)
    cands = full.subset(idx)
    prm = oracle_lib.default_params()
    t_esdf, t_opt, res = [], [], None
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        oracle_lib.esdf_update(geom, grid, (0, 0), (geom.glx - 1, geom.gly - 1), dist)
        t1 = time.perf_counter()
        res = oracle_lib.opt_batch(prm, geom, dist, cands, cores)
        t2 = time.perf_counter()
        if it >= warmup:
            t_esdf.append(t1 - t0)
            t_opt.append(t2 - t1)
    frac = cands.B / full.B
    per_step = float(np.mean(t_opt)) + float(np.mean(t_esdf)) * frac
    val = cands.B / per_step
    info = {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{cands.B} random candidates (seed 11) of the {full.B}-candidate rank-0 block per step on {cores} threads "
                      f"({np.mean(t_opt):.2f} s) + the single-thread 2048^2 ESDF ({np.mean(t_esdf):.2f} s) amortised over the sample "
                      f"fraction {frac:.3f}",
            "esdf_mcells_per_s_1thread": geom.glx * geom.gly / float(np.mean(t_esdf)) / 1e6,
            "pieces_mean": float(np.diff(cands.piece_off).mean()), "pieces_mean_block": float(np.diff(full.piece_off).mean())}
    return info, per_step, res, idx, cands, full, (geom, grid, dist)


def run_reference(args, rank, world):
    """--impl reference.  Rank 0 only."""
    if rank != 0:
        return
    info, per_step, res, idx, cands, full, _ = cpu_arm(args.steps, args.warmup, args.per_gpu)
    # configs[0]: one minco_plan (B = 1) on the 200x200 map, single thread — the literal drop-in call
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle_lib
    from alore_legged_manipulator_b200 import workloads
    g1, grid1, c1 = workloads.config1()
    d1 = np.full(g1.glx * g1.gly, np.finfo(np.float64).max)
    oracle_lib.esdf_update(g1, grid1, (0, 0), (g1.glx - 1, g1.gly - 1), d1)
    prm = oracle_lib.default_params()
    t0 = time.perf_counter()
    for _ in range(5):
        oracle_lib.opt_batch(prm, g1, d1, c1, 1)
    b1_ms = (time.perf_counter() - t0) / 5 * 1e3
    line = {
        "impl": "reference", "metric": METRIC, "value": info["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.per_gpu),
        "cpu_baseline": info,
        "e2e": {"value": info["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "config0_b1_latency_ms": b1_ms,
        "ok_fraction": float(res.ok.mean()),
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--per-gpu", type=int, default=PER_GPU)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed tick as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import alore_legged_manipulator_b200 as alore
    from alore_legged_manipulator_b200 import capi, sharding, workloads
    from alore_legged_manipulator_b200.ms_planner import DeviceBatch, MSPlanner

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.Stream()          # a real (non-NULL) stream so that CUDA events bracket our kernels
    torch.cuda.set_stream(stream)
    sptr = C.c_void_p(stream.cuda_stream)

    ctx = alore.Context(local)
    prm = alore.default_params()
    peak, peak_src = measured_peak()
    pv = lambda t: C.c_void_p(t.data_ptr())

    def esdf_line(ctx, workload, nx, ny, gi, grid, reps=8):
        """Kernel-only ESDF rebuild of a resident map, L2 flushed between iterations; 13 algorithmic bytes per cell."""
        g = workloads.make_geom(nx, ny, gi)
        mm = alore.SDFmap(ctx, gridmap_interval=gi, detection_range=1e6, global_x_lower=g.x_lower,
                          global_x_upper=g.x_lower + (nx - 0.5) * gi, global_y_lower=g.y_lower, global_y_upper=g.y_lower + (ny - 0.5) * gi)
        mm.gridmap_[:] = grid
        mm.has_map_ = True
        e2e_t = []
        for _ in range(4):
            t0 = time.perf_counter()
            mm.updateESDF2d()
            e2e_t.append(time.perf_counter() - t0)
        gg = mm.geom()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        for a, b in evs:
            flush.fill_(1)                                    # L2 flush between timed iterations
            a.record(stream)
            ctx.check(ctx.lib.alore_esdf_update_dev(ctx.h, C.byref(gg), None, 0, 0, nx - 1, ny - 1, None, 1, sptr))
            b.record(stream)
        torch.cuda.synchronize()
        k_ms = float(np.median(sorted(a.elapsed_time(b) for a, b in evs)))
        cells = nx * ny
        mm.close()
        del flush
        return {"workload": workload, "kernel_ms": k_ms, "mcells_per_s": cells / k_ms / 1e3,
                "roofline": {"bound": "hbm", "achieved": 13 * cells / k_ms / 1e6, "peak": peak, "unit": "GB/s",
                             "frac": 13 * cells / k_ms / 1e6 / peak, "bytes_per_cell": 13},
                "e2e_ms": 1e3 * min(e2e_t[1:]), "e2e_mcells_per_s": cells / min(e2e_t[1:]) / 1e6, "l2_flush_between_iterations": True}

    geom, grid0 = build_world()

    # ---- ESDF on three maps: configs[1] (cluttered), configs[4] (corridor, mostly solid), the bench world (mostly empty) ----
    esdf_info = {}
    if rank == 0:
        esdf_info = esdf_line(ctx, "configs[1]: 4096x4096, Bernoulli(0.02) occupied + 1% unknown + wall, full-map window", 4096, 4096, 0.05,
                              workloads.random_map(4096, 4096, 2, p_occ=0.02, p_unknown=0.01))
        esdf_info["long_route"] = esdf_line(ctx, "configs[4] map: 8192x2048 corridor (2 m wide free lane, 2 % clutter, walls elsewhere), "
                                            "full-window rebuild", 8192, 2048, 0.005,
                                            workloads.corridor_map(8192, 2048, 5, width_cells=400, clutter=0.02), reps=6)
        esdf_info["box_world"] = esdf_line(ctx, "the candidate benchmark's own map: 2048x2048, 400 boxes, mostly free space", 2048, 2048, 0.05,
                                           grid0, reps=6)

    # ---- candidate workload: the base world and its perturbed ticks -----------------------------------------------------
    m = alore.SDFmap(ctx, gridmap_interval=0.05, detection_range=1e6, global_x_lower=geom.x_lower,
                     global_x_upper=geom.x_lower + (geom.glx - 0.5) * 0.05, global_y_lower=geom.y_lower,
                     global_y_upper=geom.y_lower + (geom.gly - 0.5) * 0.05)
    m.gridmap_[:] = grid0
    m.has_map_ = True
    m.forceUpdateESDF()                                        # also leaves the occupancy grid resident
    gm = m.geom()
    dist0 = m.distance_buffer_all_.copy()
    pts0 = way_points(gm, grid0, dist0)
    lo, hi = sharding.shard_range(rank, world, per_rank=args.per_gpu)
    n_ticks = 1 + args.warmup + args.steps
    ticks = []
    for t in range(n_ticks):
        grid_t, pts_t = tick_variant(t, gm, grid0, pts0)
        ticks.append((grid_t, candidates_from_points(pts_t, lo, hi)))
    cands0 = ticks[0][1]
    pl = MSPlanner(ctx, prm, m)
    d_grids = [torch.from_numpy(g).cuda() for g, _ in ticks]
    batches = [DeviceBatch(ctx, c) for _, c in ticks]

    # ---- BASELINE configs[2]: batched penalty + gradient of 4096 trajectories x 64 pieces on this 2048^2 ESDF ------
    penalty_info = {}
    if rank == 0:
        Bp, Np = 4096, 64
        po, coeffs, Tp, s_xy, f_xy = workloads.random_spline_batch(Bp, Np, gm, dist0, grid0, seed=3)
        dev = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()
        d_po, d_c, d_T, d_s, d_f = dev(po, np.int32), dev(coeffs, np.float64), dev(Tp, np.float64), dev(s_xy, np.float64), dev(f_xy, np.float64)
        d_cost = torch.zeros(Bp, dtype=torch.float64, device="cuda")
        d_gC = torch.zeros(Bp * Np * 12, dtype=torch.float64, device="cuda")
        d_gT = torch.zeros(Bp * Np, dtype=torch.float64, device="cuda")
        d_err = torch.zeros(Bp * 2, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(8)]
        for a, b in evs:
            a.record(stream)
            ctx.check(ctx.lib.alore_penalty_batch_dev(ctx.h, C.byref(prm), Bp, Np, pv(d_po), pv(d_c), pv(d_T), pv(d_s), pv(d_f),
                                                      pv(d_cost), pv(d_gC), pv(d_gT), pv(d_err), sptr))
            b.record(stream)
        torch.cuda.synchronize()
        p_ms = float(np.median(sorted(a.elapsed_time(b) for a, b in evs)[1:]))
        pbytes = Bp * (8 * (26 * Np + 1) + 32 * int(prm.n_checkpoints) * Np * (int(prm.sparseResolution) + 1))
        pflop = Bp * Np * 17 * 620.0          # FP64 operations per sample counted from the SASS of the three passes (DESIGN.md)
        penalty_info = {"workload": "configs[2]: 4096 trajectories x 64 pieces, 16 half-steps/piece, 2048^2 ESDF, coefficient space",
                        "kernel_ms": p_ms, "evals_per_s": Bp / p_ms * 1e3,
                        "roofline": {"bound": "hbm", "achieved": pbytes / p_ms / 1e6, "peak": peak, "unit": "GB/s",
                                     "frac": pbytes / p_ms / 1e6 / peak, "bytes_per_trajectory": pbytes // Bp},
                        "fp64_roofline": {"achieved_tflops": pflop / p_ms / 1e9, "peak_tflops": FP64_PEAK_TFLOPS / 2,
                                          "frac": pflop / p_ms / 1e9 / (FP64_PEAK_TFLOPS / 2),
                                          "note": "no FMA contraction is allowed on this path (parity with the reference's x86 build), so the "
                                                  "ceiling is one FP64 operation per lane per issue slot = half the FMA peak; this, not HBM, bounds the kernel"}}
        if not args.skip_cpu_baseline:            # the full-size batch against the oracle, once, outside the timed region
            sys.path.insert(0, str(ROOT / "tests"))
            import oracle_lib
            olib = oracle_lib.load()
            olib.orc_set_trig_portable(1)
            try:
                cr, gCr, gTr, _ = oracle_lib.penalty_batch(prm, gm, dist0, po, coeffs, Tp, s_xy, f_xy, int(olib.orc_hardware_threads()) or 1)
            finally:
                olib.orc_set_trig_portable(0)
            same = (np.array_equal(d_cost.cpu().numpy(), cr) and np.array_equal(d_gC.cpu().numpy().reshape(gCr.shape), gCr)
                    and np.array_equal(d_gT.cpu().numpy(), gTr))
            penalty_info["full_size_bit_identical_to_oracle"] = bool(same)
        del d_po, d_c, d_T, d_s, d_f, d_cost, d_gC, d_gT, d_err

    def step_resident(t):
        # resident update: the tick's occupancy grid (device) replaces the context's, the ESDF is rebuilt, the block optimised
        ctx.check(ctx.lib.alore_esdf_update_dev(ctx.h, C.byref(gm), pv(d_grids[t]), 0, 0, geom.glx - 1, geom.gly - 1, None, 1, sptr))
        batches[t].run(prm, sptr)
        bc, bi = batches[t].argmin()                           # on-device argmin of this rank's block
        # the only exchange: all-gather of (best cost, global index) per rank over NCCL
        return sharding.gather_best(bc, lo + bi if bi >= 0 else -1, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # cold tick: no prediction at all (piece counts only)
    os.environ["ALORE_NO_SCHED_PREDICTION"] = "1"
    step_resident(0)
    cold_ms = batches[0].kernel_ms()
    del os.environ["ALORE_NO_SCHED_PREDICTION"]
    for t in range(1, 1 + args.warmup):
        step_resident(t)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern_ms = []
    e0.record(stream)
    for t in range(1 + args.warmup, n_ticks):
        best = step_resident(t)
        kern_ms.append(batches[t].kernel_ms())
    e1.record(stream)
    barrier()
    launches = ctx.launches - l0
    clocks = sampler.stop()
    dev_ms = e0.elapsed_time(e1)
    alg_bytes, evals, iters = batches[-1].stats()
    res_last = batches[-1].download()
    res0 = batches[0].download()

    # ---- end to end through the host-buffer C ABI (same perturbed ticks) -------------------------------------------
    # host side as a planner keeps it: candidates in page-locked staging arrays, ONE page-locked result store reused
    # by every tick (a fresh 70 MB numpy result per call costs more in page faults than its PCIe transfer)
    store = capi.ResultBatch(capacity=(max(tk[1].B for tk in ticks), max(tk[1].total_pieces for tk in ticks))).pin(ctx)
    for tk in ticks:
        tk[1].pin(ctx)

    def step_e2e(t):
        m.gridmap_[:] = ticks[t][0]
        m.updateESDF2d()
        r = pl.minco_plan_batch(ticks[t][1], out=store)
        sharding.gather_best(*sharding.local_best(r.cost, r.ok, lo), device="cuda")
        return r

    step_e2e(args.warmup)                 # the tick before the first timed one (as in the resident loop: its evaluation
    barrier()                             # counts are what the first timed tick's schedule is predicted from)
    t0 = time.perf_counter()
    for t in range(1 + args.warmup, n_ticks):
        step_e2e(t)
    barrier()
    e2e_s = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:
        # the resident loop's last tick; the e2e loop ended on the same tick and left its ESDF in the map's host buffer
        dump_outputs(args.dump_outputs, res_last, ticks[-1][1], best, m.distance_buffer_all_)

    # ---- the heaviest candidate alone (what bounds a rank's step), ALM statistics ----------------------------------
    heavy = int(np.argmax(res_last.evals * np.diff(ticks[-1][1].piece_off)))
    hb = DeviceBatch(ctx, ticks[-1][1].subset([heavy]))
    hb.run(prm, sptr)
    hb.download()
    heavy_ms = hb.kernel_ms()
    hb.close()

    times = torch.tensor([dev_ms, e2e_s * 1e3, float(np.mean(kern_ms)), cold_ms, heavy_ms], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(cands0.B), float(cands0.total_pieces), alg_bytes, float(evals), float(iters), float(launches),
                        float(res_last.alm_iters.max()), float((res_last.alm_iters >= 64).sum())], dtype=torch.float64, device="cuda")
    per_rank = [times.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, times)
        tmax = times.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot[:6], op=dist.ReduceOp.SUM)
        dist.all_reduce(tot[6:7], op=dist.ReduceOp.MAX)
        dist.all_reduce(tot[7:8], op=dist.ReduceOp.SUM)
    else:
        tmax = times
    dev_ms, e2e_ms = float(tmax[0]), float(tmax[1])
    total_B = int(tot[0])

    if rank == 0:
        value = total_B * args.steps / (dev_ms / 1e3)
        e2e_val = total_B * args.steps / (e2e_ms / 1e3)
        k_avg = float(np.mean(kern_ms))
        k_all = [float(p[2]) for p in per_rank]
        cells = geom.glx * geom.gly
        c_last = ticks[-1][1]
        h2d = cells + sum(a.nbytes for a in (c_last.piece_off, c_last.inner_pts, c_last.init_T, c_last.inner_init_pos,
                                              c_last.start_state, c_last.final_state, c_last.start_xytheta,
                                              c_last.final_xytheta, c_last.if_cut))
        d2h = 8 * (geom.glx - 1) * (geom.gly - 1) + sum(a.nbytes for a in (res_last.ok, res_last.status, res_last.replans, res_last.alm_iters,
                                                                           res_last.evals, res_last.cost, res_last.inner_pts, res_last.tail_s,
                                                                           res_last.piece_T, res_last.coeffs))
        traffic = None
        tp = ROOT / "profiles" / "traffic.json"
        if tp.exists():
            try:
                traffic = json.loads(tp.read_text()).get("opt_kernel_dram_bytes_per_launch")
            except Exception:
                traffic = None
        cfg = workload_config(args.per_gpu)
        cfg.update({"candidates_total": total_B, "pieces_mean": float(tot[1]) / total_B,
                    "parallelism": f"candidate-sharded x{world}, ESDF replicated",
                    "l2": "working set (per-warp L-BFGS history + scratch, > 1 GB) is larger than L2; no flush needed",
                    "schedule": "work queue handed out longest-predicted-first; prediction = pieces x cost evaluations of the PREVIOUS (different, "
                                "perturbed) tick at the same candidate index; cold_kernel_ms = the same block with piece counts only",
                    "cold_kernel_ms": float(tmax[3]),
                    "kernel_ms_per_rank": {"min": min(k_all), "max": max(k_all), "all": k_all},
                    "longest_candidate_solo_ms": float(tmax[4]),
                    "alm_iters_max": int(tot[6]), "candidates_at_alm_hard_cap": int(tot[7])})
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "roofline": {"bound": "hbm", "kernel": "opt_kernel", "achieved": float(tot[2]) / world / (k_avg / 1e3) / 1e9,
                         "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                         "frac": float(tot[2]) / world / (k_avg / 1e3) / 1e9 / peak, "traffic": traffic,
                         "algorithmic_bytes_per_launch": float(tot[2]) / world, "kernel_ms_per_launch": k_avg,
                         "note": "not HBM bound: the step is bounded below by its heaviest candidate (longest_candidate_solo_ms), one warp walking "
                                 "dependent FP64 chains (banded LU, triangular sweeps, two-loop recursion); DESIGN.md section 6"},
            "esdf": esdf_info,
            "penalty": penalty_info,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(tot[5]),
            "clocks": clocks,
            "work": {"cost_evals_per_step": float(tot[3]), "lbfgs_iterations_per_step": float(tot[4]),
                     "ok_fraction": float(res_last.ok.mean())},
        }
        if world == 1 and not args.skip_cpu_baseline:
            info, per_step, ref, idx, _, _, _ = cpu_arm(1, 0, args.per_gpu)
            line["cpu_baseline"] = info
            # ---- parity of the sample: the CUDA results of tick 0 against the oracle with the reference's own (glibc) sin/cos.
            # Single evaluations agree to 1e-12 (tests); whole optimisations amplify 1-ulp differences through the
            # line-search / stopping decisions (DESIGN.md section 3), so what is asserted and reported is the distribution.
            g_ok, g_cost = res0.ok[idx], res0.cost[idx]
            both = (g_ok == 1) & (ref.ok == 1)
            rel = np.abs(g_cost - ref.cost) / np.maximum(1e-300, np.abs(ref.cost))
            wg = idx[np.argmin(np.where(g_ok == 1, g_cost, np.inf))]
            wr = idx[np.argmin(np.where(ref.ok == 1, ref.cost, np.inf))]
            sys.path.insert(0, str(ROOT / "tests"))
            import oracle_lib
            olib = oracle_lib.load()
            sub = cands0.subset(idx[:64])
            olib.orc_set_trig_portable(1)
            try:
                pr = oracle_lib.opt_batch(prm, gm, dist0, sub, info["cores"])
            finally:
                olib.orc_set_trig_portable(0)
            line["parity_sample"] = {
                "against": "oracle with glibc sin/cos (what the reference calls), same 2080-candidate sample, tick 0",
                "ok_flag_agreement": float((g_ok == ref.ok).mean()), "collision_free_fraction": [float(g_ok.mean()), float(ref.ok.mean())],
                "final_cost_rel_diff": {"median": float(np.median(rel[both])), "p99": float(np.percentile(rel[both], 99)), "max": float(rel[both].max())},
                "same_winner": bool(wg == wr),
                "bit_identical_to_portable_trig_oracle_first64": bool(np.array_equal(res0.coeffs[:0], pr.coeffs[:0]) and all(
                    np.array_equal(res0.coeffs[int(cands0.piece_off[b]):int(cands0.piece_off[b + 1])],
                                   pr.coeffs[int(sub.piece_off[k]):int(sub.piece_off[k + 1])]) for k, b in enumerate(idx[:64]))),
            }
            # configs[0]: the literal drop-in, one minco_plan (B = 1) on the 200x200 map: latency of both arms
            g1, grid1, c1 = workloads.config1()
            ctx1 = alore.Context(local)
            m1 = alore.SDFmap(ctx1, gridmap_interval=g1.grid_interval, detection_range=1e6, global_x_lower=g1.x_lower,
                              global_x_upper=g1.x_lower + (g1.glx - 0.5) * g1.grid_interval, global_y_lower=g1.y_lower,
                              global_y_upper=g1.y_lower + (g1.gly - 0.5) * g1.grid_interval)
            m1.gridmap_[:] = grid1
            m1.has_map_ = True
            m1.forceUpdateESDF()
            p1 = MSPlanner(ctx1, prm, m1)
            p1.minco_plan_batch(c1)
            t0 = time.perf_counter()
            for _ in range(5):
                p1.minco_plan_batch(c1)
            gpu_b1 = (time.perf_counter() - t0) / 5 * 1e3
            t0 = time.perf_counter()
            for _ in range(5):
                oracle_lib.opt_batch(prm, m1.geom(), m1.distance_buffer_all_, c1, 1)
            cpu_b1 = (time.perf_counter() - t0) / 5 * 1e3
            line["config0_b1_latency_ms"] = {"b200_e2e": gpu_b1, "cpu_1thread": cpu_b1,
                                             "note": "one candidate cannot fill a GPU: the batch is the product, B = 1 is the drop-in's worst case"}
            m1.close()
            ctx1.close()
        print(json.dumps(line), flush=True)
    for b in batches:
        b.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
