"""CPU tests of the bounded-width task plan's sequential oracle (orc_task_plan_beam): a pure-Python statement of the
same rules, the exact solver where every layer fits, a greedy walk at width 1, and brute force over every tour.  No GPU."""
import numpy as np
import pytest

from alore_legged_manipulator_b200 import capi
from task_plan_beam_util import oracle_plan_beam
from task_plan_util import (INF, assert_same_plan, assert_valid_plan, batch_of_matrix, bits, brute_force, fold,
                            oracle_plan, random_assign, random_batch, random_matrix)

KINDS = ["ties", "inf", "neg", "zero", "all_inf", "one_tour"]
WIDTHS = [1, 2, 3, 7, 64, capi.ALORE_TASK_MAX_WIDTH]


def python_beam(D, n, width, fixed=False, assign=None):
    """The contract in plain Python: dict merge per layer, `sorted` truncation.  -> (cost, order, target, exact)."""
    tgt = [(int(assign[i]) if fixed and assign is not None else n + 1 + i) - n - 1 for i in range(n)]
    layers = [[(0, 0, -1, 0.0, -1, -1)]]                 # (O, T, last, value, predecessor's last, parent index)
    truncated = False
    for l in range(1, 2 * n + 1):
        merged = {}
        for s, (O, T, last, v, _, _) in enumerate(layers[-1]):
            for q in range(n):
                if l % 2:
                    if O >> q & 1:
                        continue
                    c = (O | 1 << q, T, q, D[0, 1 + q] if l == 1 else v + D[n + 1 + last, 1 + q], last, s)
                else:
                    if T >> q & 1 or (fixed and tgt[last] != q):
                        continue
                    c = (O, T | 1 << q, q, v + D[1 + last, n + 1 + q], last, s)
                if not c[3] < INF:
                    continue
                old = merged.get(c[:3])
                if old is None or c[3] < old[3] or (c[3] == old[3] and c[4] < old[4]):
                    merged[c[:3]] = c
        cur = list(merged.values())
        if len(cur) > width:
            truncated = True
            cur = sorted(cur, key=lambda st: (st[3] + 0.0, st[0], st[1], st[2]))[:width]   # + 0.0: -0 sorts as +0
        layers.append(cur)
    best, at = INF, -1
    for s in range(n):
        u = tgt[s] if fixed else s
        for i, st in enumerate(layers[-1]):
            if st[2] == u and st[3] < best:
                best, at = st[3], i
    if at < 0:
        return INF, None, None, not truncated
    order, target = [0] * n, [0] * n
    for l in range(2 * n, 0, -1):
        st = layers[l][at]
        if l % 2:
            order[l // 2] = 1 + st[2]
        else:
            target[l // 2 - 1] = n + 1 + st[2]
        at = st[5]
    return best, order, target, not truncated


def greedy(D, n, fixed=False, assign=None):
    """Width 1 from its definition: step to the next point minimising fl(value + D[last][next]), ties (==) to the
    lowest point index.  -> (cost, order, target) or (inf, None, None)."""
    tmap = {i: (int(assign[i - 1]) if assign is not None else n + i) for i in range(1, n + 1)}
    objs, tgts = set(range(1, n + 1)), set(range(n + 1, 2 * n + 1))
    c, at, order, target = None, 0, [], []

    def step(points):
        best, bv = None, INF
        for p in sorted(points):                         # ascending point index, replace on strict <
            v = D[at, p] if c is None else c + D[at, p]
            if v < bv:
                best, bv = p, v
        return best, bv

    for _ in range(n):
        o, c1 = step(objs)
        if o is None:
            return INF, None, None
        objs.discard(o), order.append(o)
        c, at = c1, o
        t, c1 = step({tmap[o]} if fixed else tgts)
        if t is None:
            return INF, None, None
        tgts.discard(t), target.append(t)
        c, at = c1, t
    return c, order, target


def cases(n_max, seed):
    rng = np.random.default_rng(seed)
    for n in range(1, n_max + 1):
        for kind in KINDS:
            for fixed in (False, True):
                assign = random_assign(rng, n) if fixed and rng.uniform() < 0.7 else None
                yield n, kind, fixed, assign, random_matrix(rng, n, kind, fixed, assign)


@pytest.mark.parametrize("width", WIDTHS)
def test_python_rules_equal_oracle(width):
    checked = truncated = 0
    for n, kind, fixed, assign, D in cases(8, width):
        if width > 64 and not fixed and n > 6:
            continue                                     # the Python layers get slow; the C++ oracle is checked below
        cost, order, target, exact = python_beam(D, n, width, fixed, assign)
        p = oracle_plan_beam(n, width, *batch_of_matrix(D), fixed, assign)
        assert bits(p.cost) == bits(cost), (n, kind, fixed, p.cost, cost)
        assert p.exact == exact
        assert p.feasible == (order is not None)
        if order is not None:
            assert p.order.tolist() == order and p.target.tolist() == target
        checked += 1
        truncated += not exact
    assert checked > 50
    assert truncated > 0 or width == capi.ALORE_TASK_MAX_WIDTH


@pytest.mark.parametrize("fixed", [False, True])
def test_wide_enough_equals_exact_solver(fixed):
    rng = np.random.default_rng(41 + fixed)
    for n in range(1, (12 if fixed else 7) + 1):
        for kind in ["mixed", "ties", "neg"]:
            assign = random_assign(rng, n) if fixed else None
            b = random_batch(rng, n, kind, per_leg=(0, 3), bad=0.05)
            p = oracle_plan_beam(n, capi.ALORE_TASK_MAX_WIDTH, *b, fixed, assign)
            assert p.exact
            assert_same_plan(p, oracle_plan(n, *b, fixed, assign))


def test_width_one_is_the_greedy_walk():
    for n, kind, fixed, assign, D in cases(8, 7):
        p = oracle_plan_beam(n, 1, *batch_of_matrix(D), fixed, assign)
        cost, order, target = greedy(D, n, fixed, assign)
        assert bits(p.cost) == bits(cost), (n, kind, fixed)
        if order is not None:
            assert p.order.tolist() == order and p.target.tolist() == target


@pytest.mark.parametrize("width", WIDTHS)
def test_plans_are_tours_and_bounded_by_brute_force(width):
    for n, kind, fixed, assign, D in cases(6, 100 + width):
        p = oracle_plan_beam(n, width, *batch_of_matrix(D), fixed, assign)
        if p.feasible:
            assert_valid_plan(p, n, fixed, assign)
            assert bits(fold(D, p.order.tolist(), p.target.tolist())) == bits(p.cost)
        else:
            assert (p.order == -1).all() and (p.target == -1).all() and (p.leg_cand == -1).all()
        if n <= (6 if fixed else 5):
            m = min(f for f, _, _ in brute_force(D, n, fixed, assign))
            assert p.cost >= m
            if p.exact:
                assert p.cost == m
