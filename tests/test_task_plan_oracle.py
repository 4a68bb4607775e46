"""CPU tests of the task plan's sequential oracle (orc_task_plan): the DP against brute force over every tour, the leg
matrix assembly against numpy, and the ctypes mirrors of the two C structs.  No GPU."""
import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

from alore_legged_manipulator_b200 import capi
from task_plan_util import (INF, assert_valid_plan, batch_of_matrix, bits, brute_force, fold, numpy_matrix, oracle_plan,
                            random_assign, random_batch, random_matrix)

ROOT = Path(__file__).resolve().parent.parent
KINDS = ["ties", "inf", "neg", "zero", "all_inf", "one_tour"]


def check_against_brute_force(D, n, fixed, assign):
    lf, lt, cost, ok = batch_of_matrix(D)
    p = oracle_plan(n, lf, lt, cost, ok, fixed, assign)
    assert np.array_equal(p.leg_cost.view(np.uint64), D.view(np.uint64))   # one candidate per finite leg: D itself
    tours = brute_force(D, n, fixed, assign)
    m = min(f for f, _, _ in tours)
    if not m < INF:
        assert p.cost == INF and not p.feasible
        assert (p.order == -1).all() and (p.target == -1).all() and (p.leg_cand == -1).all()
        return
    assert p.feasible
    assert p.cost == m
    # bit-equal to the minimum; with +0 / -0 both minimal, to one of the minimal tours' folds
    assert bits(p.cost) in {bits(f) for f, _, _ in tours if f == m}
    assert_valid_plan(p, n, fixed, assign)
    assert bits(fold(D, p.order.tolist(), p.target.tolist())) == bits(p.cost)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5])
def test_free_dp_equals_brute_force(n, kind):
    rng = np.random.default_rng(100 * n + KINDS.index(kind))
    for _ in range(6 if n <= 4 else 2):
        check_against_brute_force(random_matrix(rng, n, kind), n, False, None)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 6, 7])
def test_fixed_dp_equals_brute_force(n, kind):
    rng = np.random.default_rng(1000 + 100 * n + KINDS.index(kind))
    for rep in range(4):
        assign = None if rep == 0 else random_assign(rng, n)
        check_against_brute_force(random_matrix(rng, n, kind, True, assign), n, True, assign)


def test_plan_order_breaks_ties_by_lowest_point_index():
    # every leg costs 1: all tours tie, the DP's scans in ascending point index give one defined plan
    n = 3
    D = np.ones((7, 7))
    np.fill_diagonal(D, INF)
    p = oracle_plan(n, *batch_of_matrix(D))
    assert p.cost == 6.0 and p.feasible
    assert_valid_plan(p, n)
    assert p.order.tolist() == oracle_plan(n, *batch_of_matrix(D)).order.tolist()   # deterministic


@pytest.mark.parametrize("seed", range(6))
def test_leg_matrix_equals_numpy(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 5))
    P = 2 * n + 1
    lf, lt, cost, ok = random_batch(rng, n, kind=["mixed", "ties", "neg"][seed % 3], per_leg=(0, 5))
    assert (lf == -1).any() and (ok != 1).any() and np.isnan(cost).any()
    D, best = numpy_matrix(P, lf, lt, cost, ok)
    p = oracle_plan(n, lf, lt, cost, ok, with_matrix=True)
    assert np.array_equal(p.leg_cost.view(np.uint64), D.view(np.uint64))
    assert np.array_equal(p.leg_best, best)
    assert not np.isin(p.leg_best[p.leg_best >= 0], np.nonzero(lf < 0)[0]).any()


def test_leg_matrix_cases():
    # leg 0 -> 1 (n = 1, P = 3): ok = 0, NaN, inf, -1 label, then ties of -0 / +0 / 0.0 broken to the lowest index
    lf = np.array([0, 0, 0, -1, 0, 0, 0, 1, 1], np.int32)
    lt = np.array([1, 1, 1, 1, 1, 1, 1, 2, 2], np.int32)
    cost = np.array([-5.0, np.nan, -INF, -9.0, 0.0, -0.0, 0.0, 3.0, 3.0])
    ok = np.array([0, 1, 1, 1, 1, 1, 1, 1, 1], np.int32)
    p = oracle_plan(1, lf, lt, cost, ok, with_matrix=True)
    assert p.leg_best[0, 1] == 4 and bits(p.leg_cost[0, 1]) == bits(0.0)
    assert p.leg_best[1, 2] == 7 and p.leg_cost[1, 2] == 3.0
    assert p.leg_best[2, 0] == -1 and p.leg_cost[2, 0] == INF
    assert p.feasible and p.cost == 3.0 and p.leg_cand.tolist() == [4, 7]
    cost[4] = 1.0                                           # now -0.0 (index 5) is the first minimum
    p = oracle_plan(1, lf, lt, cost, ok, with_matrix=True)
    assert p.leg_best[0, 1] == 5 and bits(p.leg_cost[0, 1]) == bits(-0.0)


def test_struct_sizes_match_ctypes():
    src = r'''
    #include "alore_b200.h"
    #include <stdio.h>
    int main(void) { printf("%zu %zu\n", sizeof(alore_task_t), sizeof(alore_task_plan_t)); return 0; }
    '''
    with tempfile.TemporaryDirectory() as d:
        (Path(d) / "t.c").write_text(src)
        subprocess.run(["gcc", "-I", str(ROOT / "include"), "-o", f"{d}/t", f"{d}/t.c"], check=True)
        out = subprocess.run([f"{d}/t"], check=True, capture_output=True, text=True).stdout.split()
    assert [int(x) for x in out] == [C.sizeof(capi.Task), C.sizeof(capi.TaskPlanOut)]
