"""Helpers of the bounded-width task-plan tests: the sequential oracle orc_task_plan_beam and a plan comparison that
includes the `exact` flag.  The shared task-plan helpers (batches, matrices, brute force) live in task_plan_util."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from alore_legged_manipulator_b200 import capi
from alore_legged_manipulator_b200.task_planner import TaskCall, TaskPlan
from task_plan_util import assert_same_plan

ROOT = Path(__file__).resolve().parent.parent
BEAM_ORACLE_SRC = ROOT / "tests" / "cpp" / "task_plan_beam_oracle.cpp"
_beam_oracle = None


def load_beam_oracle() -> C.CDLL:
    """tests/cpp/task_plan_beam_oracle.cpp, compiled once into the temporary directory (the tree is left untouched)
    with the flags of the exact oracle: no FMA contraction, no fast-math."""
    global _beam_oracle
    if _beam_oracle is None:
        src = BEAM_ORACLE_SRC.read_bytes() + (ROOT / "include" / "alore_b200.h").read_bytes()
        tag = hashlib.sha256(src).hexdigest()[:16]
        lib = Path(tempfile.gettempdir()) / f"alore_task_beam_oracle_{os.getuid()}_{tag}.so"
        if not lib.exists():
            tmp = lib.with_suffix(f".{os.getpid()}.tmp")
            subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-O3", "-fPIC", "-ffp-contract=off", "-Wall",
                            "-shared", "-o", str(tmp), str(BEAM_ORACLE_SRC)], check=True, capture_output=True)
            os.replace(tmp, lib)
        _beam_oracle = C.CDLL(str(lib))
        _beam_oracle.orc_task_plan_beam.argtypes = [C.POINTER(capi.Task), C.c_int, C.c_int, capi.c_double_p,
                                                    capi.c_int32_p, C.POINTER(capi.TaskPlanOut), C.POINTER(C.c_int32)]
    return _beam_oracle


def oracle_plan_beam(n, width, leg_from, leg_to, cost, ok, fixed=False, assign=None, with_matrix=True) -> TaskPlan:
    call = TaskCall(n, leg_from, leg_to, fixed, assign, with_matrix)
    cost = np.ascontiguousarray(cost, dtype=np.float64)
    ok = np.ascontiguousarray(ok, dtype=np.int32)
    exact = C.c_int32(-1)
    rc = load_beam_oracle().orc_task_plan_beam(C.byref(call.task), int(width), call.B, capi.dptr(cost), capi.iptr(ok),
                                               C.byref(call.out), C.byref(exact))
    assert rc == 0
    return call.result(exact)


def assert_same_beam_plan(a: TaskPlan, b: TaskPlan):
    """assert_same_plan, and the same `exact` flag."""
    assert_same_plan(a, b)
    assert a.exact == b.exact, (a.exact, b.exact)
