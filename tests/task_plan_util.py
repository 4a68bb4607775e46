"""Helpers of the task-plan tests: both oracles, brute force over every tour, random matrices and labelled batches."""
from __future__ import annotations

import ctypes as C
import hashlib
import itertools
import os
import struct
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from alore_legged_manipulator_b200 import capi
from alore_legged_manipulator_b200.task_planner import TaskCall, TaskPlan

INF = float("inf")
ROOT = Path(__file__).resolve().parent.parent
ORACLE_SRC = ROOT / "tests" / "cpp" / "task_plan_oracle.cpp"
_oracle = None


def load_oracle() -> C.CDLL:
    """The sequential task-plan oracles orc_task_plan and orc_task_plan_beam (tests/cpp/task_plan_oracle.cpp), compiled
    once into the temporary directory (the tree is left untouched) with the flags of the other CPU oracle: no FMA
    contraction, no fast-math."""
    global _oracle
    if _oracle is None:
        src = ORACLE_SRC.read_bytes() + (ROOT / "include" / "alore_b200.h").read_bytes()
        tag = hashlib.sha256(src).hexdigest()[:16]
        lib = Path(tempfile.gettempdir()) / f"alore_task_oracle_{os.getuid()}_{tag}.so"
        if not lib.exists():
            tmp = lib.with_suffix(f".{os.getpid()}.tmp")
            subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-O3", "-fPIC", "-ffp-contract=off", "-Wall",
                            "-shared", "-o", str(tmp), str(ORACLE_SRC)], check=True, capture_output=True)
            os.replace(tmp, lib)
        _oracle = C.CDLL(str(lib))
        _oracle.orc_task_plan.argtypes = [C.POINTER(capi.Task), C.c_int, capi.c_double_p, capi.c_int32_p,
                                          C.POINTER(capi.TaskPlanOut)]
        _oracle.orc_task_plan_beam.argtypes = [C.POINTER(capi.Task), C.c_int, C.c_int, capi.c_double_p, capi.c_int32_p,
                                               C.POINTER(capi.TaskPlanOut), C.POINTER(C.c_int32)]
    return _oracle


def bits(x: float) -> int:
    return struct.unpack("<Q", struct.pack("<d", x))[0]


def oracle_plan(n, leg_from, leg_to, cost, ok, fixed=False, assign=None, with_matrix=True) -> TaskPlan:
    call = TaskCall(n, leg_from, leg_to, fixed, assign, with_matrix)
    cost = np.ascontiguousarray(cost, dtype=np.float64)
    ok = np.ascontiguousarray(ok, dtype=np.int32)
    rc = load_oracle().orc_task_plan(C.byref(call.task), call.B, capi.dptr(cost), capi.iptr(ok), C.byref(call.out))
    assert rc == 0
    return call.result()


def oracle_plan_beam(n, width, leg_from, leg_to, cost, ok, fixed=False, assign=None, with_matrix=True) -> TaskPlan:
    call = TaskCall(n, leg_from, leg_to, fixed, assign, with_matrix)
    cost = np.ascontiguousarray(cost, dtype=np.float64)
    ok = np.ascontiguousarray(ok, dtype=np.int32)
    exact = C.c_int32(-1)
    rc = load_oracle().orc_task_plan_beam(C.byref(call.task), int(width), call.B, capi.dptr(cost), capi.iptr(ok),
                                          C.byref(call.out), C.byref(exact))
    assert rc == 0
    return call.result(exact)


def targets_of(n, fixed, assign):
    """Fixed mode: target point of object point i (1..n)."""
    if not fixed:
        return None
    return {i: (int(assign[i - 1]) if assign is not None else n + i) for i in range(1, n + 1)}


def fold(D, order, target) -> float:
    """The tour's cost: left fold of its leg costs in tour order (Python floats are IEEE doubles)."""
    c, prev = None, 0
    for o, t in zip(order, target):
        c = D[prev, o] if c is None else c + D[prev, o]
        c = c + D[o, t]
        prev = t
    return float(c)


def brute_force(D, n, fixed=False, assign=None):
    """Every tour's fold: [(fold, order, target)]."""
    tmap = targets_of(n, fixed, assign)
    objs, tgts = list(range(1, n + 1)), list(range(n + 1, 2 * n + 1))
    out = []
    for order in itertools.permutations(objs):
        for target in ([tuple(tmap[o] for o in order)] if fixed else itertools.permutations(tgts)):
            out.append((fold(D, order, target), order, target))
    return out


def random_tour(rng, n, fixed=False, assign=None):
    order = [int(x) for x in rng.permutation(n) + 1]
    tmap = targets_of(n, fixed, assign)
    target = [tmap[o] for o in order] if fixed else [int(x) for x in rng.permutation(n) + n + 1]
    return order, target


def tour_legs(order, target):
    pts = [0]
    for o, t in zip(order, target):
        pts += [o, t]
    return list(zip(pts[:-1], pts[1:]))


def random_matrix(rng, n, kind, fixed=False, assign=None) -> np.ndarray:
    """P x P leg matrix (diagonal +inf).  kind: ties (costs from {1, 2, 3}), inf (some +inf legs), neg (negative costs),
    zero (+0 / -0 / small), all_inf, one_tour (exactly one feasible tour)."""
    P = 2 * n + 1
    if kind == "ties":
        D = rng.integers(1, 4, (P, P)).astype(np.float64)
    elif kind == "inf":
        D = rng.integers(1, 4, (P, P)).astype(np.float64) + rng.uniform(0, 1, (P, P)).round(1)
        D[rng.uniform(size=(P, P)) < 0.35] = INF
    elif kind == "neg":
        D = rng.uniform(-5, 5, (P, P)).round(2)
        D[rng.uniform(size=(P, P)) < 0.1] = INF
    elif kind == "zero":
        D = rng.choice(np.array([0.0, -0.0, 1.0, -1.0, 0.5]), (P, P))
    elif kind == "all_inf":
        D = np.full((P, P), INF)
    elif kind == "one_tour":
        D = np.full((P, P), INF)
        order, target = random_tour(rng, n, fixed, assign)
        for i, j in tour_legs(order, target):
            D[i, j] = float(rng.integers(1, 4))
    else:
        raise ValueError(kind)
    np.fill_diagonal(D, INF)
    return D


def batch_of_matrix(D):
    """One candidate per finite off-diagonal entry; +inf entries become a candidate with ok = 0 or cost +inf."""
    P = D.shape[0]
    lf, lt, cost, ok = [], [], [], []
    for i in range(P):
        for j in range(P):
            if i == j:
                continue
            lf.append(i), lt.append(j)
            cost.append(D[i, j] if np.isfinite(D[i, j]) else (1.0 if (i + j) % 2 else INF))
            ok.append(1 if np.isfinite(D[i, j]) else ((i + j + 1) % 2))
    return (np.array(lf, np.int32), np.array(lt, np.int32), np.array(cost), np.array(ok, np.int32))


def random_batch(rng, n, kind="mixed", per_leg=(0, 4), decoys=0.1, bad=0.16):
    """A labelled batch over every leg of P points: 0..per_leg candidates per leg whose costs tie often, with ok = 0,
    NaN, +/-inf and -0 candidates mixed in, and candidates labelled -1 (cheaper than anything) sprinkled between."""
    P = 2 * n + 1
    lf, lt, cost, ok = [], [], [], []
    slots = [(i, j) for i in range(P) for j in range(P) if i != j
             for _ in range(int(rng.integers(per_leg[0], per_leg[1] + 1)))]
    rng.shuffle(slots)
    for i, j in slots:
        if rng.uniform() < decoys:                       # not a task leg: any leg_to, a cost below everything
            lf.append(-1), lt.append(int(rng.integers(-5, P + 5))), cost.append(-1e9), ok.append(1)
        if kind == "ties":
            c = float(rng.integers(1, 4))
        elif kind == "neg":
            c = round(float(rng.uniform(-3, 3)), 1)
        else:
            c = float(rng.choice([1.0, 2.0, 2.5, 3.0, 0.0, -0.0, -1.5]))
        k, r = 1, rng.uniform() * 0.16 / bad if bad > 0 else 1.0
        if r < 0.08:
            k = int(rng.choice([0, 2, -1]))              # only ok == 1 counts
        elif r < 0.12:
            c = float("nan")
        elif r < 0.16:
            c = INF if rng.uniform() < 0.5 else -INF
        lf.append(i), lt.append(j), cost.append(c), ok.append(k)
    return (np.array(lf, np.int32), np.array(lt, np.int32), np.array(cost, np.float64), np.array(ok, np.int32))


def numpy_matrix(P, leg_from, leg_to, cost, ok):
    """The leg matrix by numpy: D = cost of the lowest-index counted candidate equal to its leg's minimum."""
    D = np.full((P, P), INF)
    best = np.full((P, P), -1, np.int32)
    counted = (leg_from >= 0) & (ok == 1) & np.isfinite(cost)
    for i in range(P):
        for j in range(P):
            idx = np.nonzero(counted & (leg_from == i) & (leg_to == j))[0]
            if idx.size:
                m = cost[idx].min()
                b = int(idx[np.nonzero(cost[idx] == m)[0][0]])
                D[i, j], best[i, j] = cost[b], b
    return D, best


def random_assign(rng, n):
    return (rng.permutation(n) + n + 1).astype(np.int32)


def assert_valid_plan(p: TaskPlan, n, fixed=False, assign=None):
    """order / target form a tour (and respect the fixed assignment); leg_cand are the matrix's candidates."""
    assert sorted(p.order.tolist()) == list(range(1, n + 1))
    assert sorted(p.target.tolist()) == list(range(n + 1, 2 * n + 1))
    tmap = targets_of(n, fixed, assign)
    if fixed:
        assert [tmap[o] for o in p.order.tolist()] == p.target.tolist()
    if p.leg_best is not None:
        assert p.leg_cand.tolist() == [int(p.leg_best[i, j]) for i, j in p.legs()]


def assert_same_plan(a: TaskPlan, b: TaskPlan):
    """Bit for bit: optimum, feasibility, plan, and the matrix when both carry it."""
    assert bits(a.cost) == bits(b.cost), (a.cost, b.cost)
    assert a.feasible == b.feasible
    assert np.array_equal(a.order, b.order) and np.array_equal(a.target, b.target), (a, b)
    assert np.array_equal(a.leg_cand, b.leg_cand)
    if a.leg_cost is not None and b.leg_cost is not None:
        assert np.array_equal(a.leg_cost.view(np.uint64), b.leg_cost.view(np.uint64))
        assert np.array_equal(a.leg_best, b.leg_best)


def assert_same_beam_plan(a: TaskPlan, b: TaskPlan):
    """assert_same_plan, and the same `exact` flag."""
    assert_same_plan(a, b)
    assert a.exact == b.exact, (a.exact, b.exact)


def task_legs(n):
    """The legs a tour can use: robot -> object, object -> target, target -> object."""
    objs, tgts = range(1, n + 1), range(n + 1, 2 * n + 1)
    return ([(0, o) for o in objs] + [(o, t) for o in objs for t in tgts] + [(t, o) for t in tgts for o in objs])


def task_leg_batch(points, point_ids, variants):
    """One candidate per task leg x heading variant (start heading, goal heading), straight paths through the front
    end's time allocation.  points: xy of every task point; point_ids: which row of `points` is task point p.
    Returns (candidates, leg_from, leg_to)."""
    from alore_legged_manipulator_b200 import front_end
    n = (len(point_ids) - 1) // 2
    fts, lf, lt = [], [], []
    for sh, gh in variants:
        for i, j in task_legs(n):
            a, b = points[point_ids[i]], points[point_ids[j]]
            fts.append(front_end.make_flat_traj([tuple(a), tuple(b)], (a[0], a[1], sh), (b[0], b[1], gh)))
            lf.append(i), lt.append(j)
    return front_end.pack_candidates(fts), np.array(lf, np.int32), np.array(lt, np.int32)
