"""alore_legged_manipulator_b200 — B200-native (sm_100a) hot path of ALORE's planning_ddr_opt stack.

Only what the path needs: `csrc/` (CUDA kernels + the C ABI of include/alore_b200.h, built into
`libalore_b200.so`) and the host-side mirrors of the reference interfaces (`SDFmap`, `MSPlanner`).
There is no CPU fallback: every op fails loudly when the CUDA library is missing.
"""
from .capi import (AloreError, CandidateBatch, Context, MapGeom, Params, ResultBatch, Task, TaskPlanOut,  # noqa: F401
                   default_params, load_library)
from .sdf_map import SDFmap  # noqa: F401
from .task_planner import TaskPlan, plan_tasks  # noqa: F401

__all__ = ["AloreError", "CandidateBatch", "Context", "MapGeom", "Params", "ResultBatch", "SDFmap", "Task", "TaskPlan",
           "TaskPlanOut", "default_params", "load_library", "plan_tasks"]
