"""ctypes view of include/alore_b200.h (the drop-in C ABI).

The structures below mirror the header field for field; `load_library()` loads the in-tree
`libalore_b200.so` and FAILS LOUDLY when it is missing — there is no CPU fallback in the product.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
# ALORE_B200_LIB: developer override used by the tuning scripts to A/B differently compiled builds of the same sources
LIB_PATH = Path(os.environ.get("ALORE_B200_LIB") or (PKG_DIR / "libalore_b200.so"))

ALORE_MAX_CHECKPOINTS = 8
ALORE_SQ_INF = 0x7FFFFFFF
ALORE_ALM_HARD_CAP = 64
UNKNOWN, UNOCCUPIED, OCCUPIED = 0, 1, 2

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_uint8_p = C.POINTER(C.c_uint8)


class LbfgsParams(C.Structure):
    """lbfgs::lbfgs_parameter_t (gcopter/lbfgs.hpp:15-129)."""

    _fields_ = [
        ("mem_size", C.c_int32), ("past", C.c_int32), ("max_iterations", C.c_int32), ("max_linesearch", C.c_int32),
        ("g_epsilon", C.c_double), ("delta", C.c_double), ("min_step", C.c_double), ("max_step", C.c_double),
        ("f_dec_coeff", C.c_double), ("s_curv_coeff", C.c_double), ("cautious_factor", C.c_double),
        ("machine_prec", C.c_double),
    ]


class MapGeom(C.Structure):
    _fields_ = [
        ("glx", C.c_int32), ("gly", C.c_int32),
        ("x_lower", C.c_double), ("y_lower", C.c_double), ("x_upper", C.c_double), ("y_upper", C.c_double),
        ("grid_interval", C.c_double), ("inv_grid_interval", C.c_double),
    ]


class Params(C.Structure):
    """Every MSPlanner / Config parameter (back_end/src/optimizer.cpp:17-166, optimizer.h:31-82)."""

    _fields_ = [
        ("max_vel", C.c_double), ("min_vel", C.c_double), ("max_acc", C.c_double), ("max_omega", C.c_double),
        ("max_domega", C.c_double), ("max_centripetal_acc", C.c_double),
        ("if_directly_constrain_v_omega", C.c_int32), ("if_standard_diff", C.c_int32),
        ("ICR", C.c_double * 3),
        ("mean_time_lowBound", C.c_double), ("mean_time_uppBound", C.c_double),
        ("smoothEps", C.c_double), ("safeDis", C.c_double), ("finalMinSafeDis", C.c_double),
        ("finalSafeDisCheckNum", C.c_int32), ("safeReplanMaxTime", C.c_int32),
        ("pw_time", C.c_double), ("pw_acc", C.c_double), ("pw_domega", C.c_double), ("pw_collision", C.c_double),
        ("pw_moment", C.c_double), ("pw_mean_time", C.c_double), ("pw_cen_acc", C.c_double),
        ("ppw_time", C.c_double), ("ppw_bigpath_sdf", C.c_double), ("ppw_mean_time", C.c_double),
        ("ppw_moment", C.c_double), ("ppw_acc", C.c_double), ("ppw_domega", C.c_double),
        ("energyWeights", C.c_double * 2),
        ("EqualLambda", C.c_double * 2), ("EqualRho", C.c_double * 2), ("EqualRhoMax", C.c_double * 2),
        ("EqualGamma", C.c_double * 2), ("EqualTolerance", C.c_double * 2),
        ("CutEqualLambda", C.c_double * 2), ("CutEqualRho", C.c_double * 2), ("CutEqualRhoMax", C.c_double * 2),
        ("CutEqualGamma", C.c_double * 2), ("CutEqualTolerance", C.c_double * 2),
        ("path_lbfgs", LbfgsParams),
        ("normal_past", C.c_int32), ("shot_path_past", C.c_int32), ("shot_path_horizon", C.c_double),
        ("lbfgs", LbfgsParams),
        ("sparseResolution", C.c_int32), ("n_checkpoints", C.c_int32),
        ("check_point", (C.c_double * 2) * ALORE_MAX_CHECKPOINTS),
        ("alm_max_outer", C.c_int32), ("reserved0", C.c_int32),
    ]


class Candidates(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("piece_off", c_int32_p), ("inner_pts", c_double_p), ("init_T", c_double_p),
        ("inner_init_pos", c_double_p), ("start_state", c_double_p), ("final_state", c_double_p),
        ("start_xytheta", c_double_p), ("final_xytheta", c_double_p), ("if_cut", c_uint8_p),
    ]


class Results(C.Structure):
    _fields_ = [
        ("ok", c_int32_p), ("status", c_int32_p), ("replans", c_int32_p), ("alm_iters", c_int32_p),
        ("evals", c_int32_p), ("cost", c_double_p), ("inner_pts", c_double_p), ("tail_s", c_double_p),
        ("piece_T", c_double_p), ("coeffs", c_double_p),
    ]


def dptr(a: np.ndarray):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_double_p)


def iptr(a: np.ndarray):
    assert a.dtype == np.int32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_int32_p)


def u8ptr(a: np.ndarray):
    assert a.dtype == np.uint8 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_uint8_p)


class CandidateBatch:
    """Host-side structure-of-arrays batch of FlatTrajData (front_end/traj_representation.h:46-76)."""

    def __init__(self, piece_off, inner_pts, init_T, inner_init_pos, start_state, final_state, start_xytheta,
                 final_xytheta, if_cut):
        self.piece_off = np.ascontiguousarray(piece_off, dtype=np.int32)
        self.B = int(self.piece_off.size - 1)
        tot = int(self.piece_off[-1])
        self.inner_pts = np.ascontiguousarray(inner_pts, dtype=np.float64).reshape(max(tot - self.B, 0), 2)
        self.init_T = np.ascontiguousarray(init_T, dtype=np.float64).reshape(self.B)
        self.inner_init_pos = np.ascontiguousarray(inner_init_pos, dtype=np.float64).reshape(tot, 3)
        self.start_state = np.ascontiguousarray(start_state, dtype=np.float64).reshape(self.B, 2, 3)
        self.final_state = np.ascontiguousarray(final_state, dtype=np.float64).reshape(self.B, 2, 3)
        self.start_xytheta = np.ascontiguousarray(start_xytheta, dtype=np.float64).reshape(self.B, 3)
        self.final_xytheta = np.ascontiguousarray(final_xytheta, dtype=np.float64).reshape(self.B, 3)
        self.if_cut = np.ascontiguousarray(if_cut, dtype=np.uint8).reshape(self.B)
        if self.inner_pts.size == 0:  # keep a valid pointer for B x (N=1)
            self.inner_pts = np.zeros((1, 2))

    @property
    def total_pieces(self) -> int:
        return int(self.piece_off[-1])

    def _arrays(self):
        return (self.piece_off, self.inner_pts, self.init_T, self.inner_init_pos, self.start_state, self.final_state,
                self.start_xytheta, self.final_xytheta, self.if_cut)

    def pin(self, ctx: "Context") -> "CandidateBatch":
        """Page-locks the batch's arrays (a front end that fills the same staging buffers every tick does this once)."""
        self._pins = getattr(self, "_pins", [])
        for a in self._arrays():
            if a.nbytes and ctx.lib.alore_host_register(ctx.h, a.ctypes.data, a.nbytes) == 0:
                self._pins.append((ctx, a))
        return self

    def unpin(self):
        for ctx, a in getattr(self, "_pins", []):
            if ctx.h:
                ctx.lib.alore_host_unregister(ctx.h, a.ctypes.data)
        self._pins = []

    def n_vars(self) -> int:
        return 3 * self.total_pieces - self.B

    def x_offset(self, b: int) -> int:
        return 3 * int(self.piece_off[b]) - b

    def as_struct(self) -> Candidates:
        return Candidates(self.B, iptr(self.piece_off), dptr(self.inner_pts), dptr(self.init_T),
                          dptr(self.inner_init_pos), dptr(self.start_state), dptr(self.final_state),
                          dptr(self.start_xytheta), dptr(self.final_xytheta), u8ptr(self.if_cut))

    def subset(self, idx) -> "CandidateBatch":
        idx = list(idx)
        po = [0]
        ip, pos = [], []
        for b in idx:
            p0, p1 = int(self.piece_off[b]), int(self.piece_off[b + 1])
            po.append(po[-1] + p1 - p0)
            ip.append(self.inner_pts[p0 - b:p1 - b - 1])
            pos.append(self.inner_init_pos[p0:p1])
        ipc = np.concatenate(ip) if ip and sum(len(a) for a in ip) else np.zeros((0, 2))
        return CandidateBatch(po, ipc, self.init_T[idx], np.concatenate(pos), self.start_state[idx],
                              self.final_state[idx], self.start_xytheta[idx], self.final_xytheta[idx], self.if_cut[idx])

    @staticmethod
    def concat(batches) -> "CandidateBatch":
        po = [0]
        for b in batches:
            for i in range(b.B):
                po.append(po[-1] + int(b.piece_off[i + 1] - b.piece_off[i]))
        tot_inner = [b.inner_pts[: b.total_pieces - b.B] for b in batches]
        return CandidateBatch(po, np.concatenate(tot_inner), np.concatenate([b.init_T for b in batches]),
                              np.concatenate([b.inner_init_pos for b in batches]),
                              np.concatenate([b.start_state for b in batches]),
                              np.concatenate([b.final_state for b in batches]),
                              np.concatenate([b.start_xytheta for b in batches]),
                              np.concatenate([b.final_xytheta for b in batches]),
                              np.concatenate([b.if_cut for b in batches]))


class ResultBatch:
    """Host-side results of one batch.  `capacity=(B, total_pieces)` allocates a REUSABLE result store: a planner that
    replans every tick keeps one (page-locked with `pin`) and passes it as `out=` to `minco_plan_batch`, which binds the
    public arrays to the leading part the tick's candidates need."""

    _FIELDS = ("ok", "status", "replans", "alm_iters", "evals", "cost", "inner_pts", "tail_s", "piece_T", "coeffs")

    def __init__(self, cands: CandidateBatch | None = None, *, capacity: tuple[int, int] | None = None):
        B, tot = capacity if capacity is not None else (cands.B, cands.total_pieces)
        self.capacity = (int(B), int(tot))
        self._base = {
            "ok": np.zeros(B, np.int32), "status": np.zeros(B, np.int32), "replans": np.zeros(B, np.int32),
            "alm_iters": np.zeros(B, np.int32), "evals": np.zeros(B, np.int32), "cost": np.zeros(B),
            "inner_pts": np.zeros((max(tot - 1, 1), 2)), "tail_s": np.zeros(B), "piece_T": np.zeros(tot),
            "coeffs": np.zeros((tot, 6, 2)),
        }
        self._pins: list = []
        self.bind(B, tot)

    def bind(self, B: int, tot: int) -> "ResultBatch":
        """Points the public arrays at the leading (B, tot) part of the store."""
        cb, ct = self.capacity
        if B > cb or tot > ct:
            raise ValueError(f"result store holds {cb} candidates / {ct} pieces, batch needs {B} / {tot}")
        n = {"inner_pts": max(tot - B, 1), "piece_T": tot, "coeffs": tot}
        for f in self._FIELDS:
            setattr(self, f, self._base[f][: n.get(f, B)])
        return self

    def pin(self, ctx: "Context") -> "ResultBatch":
        """Page-locks the store (cudaHostRegister through the C ABI); released by unpin() or when `ctx` is closed."""
        for a in self._base.values():
            if ctx.lib.alore_host_register(ctx.h, a.ctypes.data, a.nbytes) == 0:
                self._pins.append((ctx, a))
        return self

    def unpin(self):
        for ctx, a in self._pins:
            if ctx.h:
                ctx.lib.alore_host_unregister(ctx.h, a.ctypes.data)
        self._pins = []

    def as_struct(self) -> Results:
        return Results(iptr(self.ok), iptr(self.status), iptr(self.replans), iptr(self.alm_iters), iptr(self.evals),
                       dptr(self.cost), dptr(self.inner_pts), dptr(self.tail_s), dptr(self.piece_T), dptr(self.coeffs))


_lib = None


def load_library(path: os.PathLike | None = None) -> C.CDLL:
    """Loads libalore_b200.so.  Raises RuntimeError if it has not been built (no fallback)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path else LIB_PATH
    if not p.exists():
        raise RuntimeError(
            f"{p} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc -gencode arch=compute_100a,code=sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(str(p))
    vp = C.c_void_p
    lib.alore_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.alore_create.restype = C.c_int
    lib.alore_destroy.argtypes = [vp]
    lib.alore_destroy.restype = None
    lib.alore_last_error.argtypes = [vp]
    lib.alore_last_error.restype = C.c_char_p
    lib.alore_device_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.alore_host_register.argtypes = [vp, vp, C.c_size_t]
    lib.alore_host_unregister.argtypes = [vp, vp]
    lib.alore_params_default.argtypes = [C.POINTER(Params)]
    lib.alore_params_default.restype = None
    lib.alore_esdf_update.argtypes = [vp, C.POINTER(MapGeom), c_uint8_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      c_double_p, C.c_int]
    lib.alore_esdf_update_dev.argtypes = [vp, C.POINTER(MapGeom), vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp]
    lib.alore_esdf_set.argtypes = [vp, C.POINTER(MapGeom), c_double_p]
    lib.alore_esdf_reset.argtypes = [vp, C.POINTER(MapGeom)]
    lib.alore_esdf_last_sq.argtypes = [vp, c_int32_p, c_int32_p]
    lib.alore_esdf_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.alore_launch_count.argtypes = [vp]
    lib.alore_create_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    lib.alore_destroy_multi.argtypes = [vp]
    lib.alore_destroy_multi.restype = None
    lib.alore_multi_size.argtypes = [vp]
    lib.alore_multi_ctx.argtypes = [vp, C.c_int]
    lib.alore_multi_ctx.restype = vp
    lib.alore_multi_last_error.argtypes = [vp]
    lib.alore_multi_last_error.restype = C.c_char_p
    lib.alore_multi_esdf_update.argtypes = [vp, C.POINTER(MapGeom), c_uint8_p, C.c_int, C.c_int, C.c_int, C.c_int, c_double_p, C.c_int]
    lib.alore_multi_opt_batch.argtypes = [vp, C.POINTER(Params), C.POINTER(Candidates), C.POINTER(Results), C.POINTER(C.c_double),
                                          C.POINTER(C.c_int32), c_int32_p]
    lib.alore_launch_count.restype = C.c_longlong
    if hasattr(lib, "alore_penalty_batch"):
        lib.alore_penalty_batch.argtypes = [vp, C.POINTER(Params), C.c_int, c_int32_p, c_double_p, c_double_p,
                                            c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p]
        lib.alore_penalty_batch_dev.argtypes = [vp, C.POINTER(Params), C.c_int, C.c_int] + [vp] * 10
        lib.alore_cost_batch.argtypes = [vp, C.POINTER(Params), C.POINTER(Candidates), C.c_int, c_double_p, c_double_p,
                                         c_double_p, c_double_p, c_double_p, c_double_p, c_double_p]
        lib.alore_opt_batch.argtypes = [vp, C.POINTER(Params), C.POINTER(Candidates), C.POINTER(Results)]
        lib.alore_batch_upload.argtypes = [vp, C.POINTER(Candidates), C.POINTER(vp)]
        lib.alore_batch_run.argtypes = [vp, C.POINTER(Params), vp, vp]
        lib.alore_batch_download.argtypes = [vp, vp, C.POINTER(Results)]
        lib.alore_batch_device_results.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
        lib.alore_batch_argmin.argtypes = [vp, vp, C.POINTER(C.c_double), C.POINTER(C.c_int32)]
        lib.alore_batch_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
        lib.alore_batch_stats.argtypes = [vp, vp, C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
        lib.alore_batch_free.argtypes = [vp]
        lib.alore_batch_free.restype = None
        lib.alore_final_collision_batch.argtypes = [vp, C.POINTER(Params), C.c_int, c_int32_p, c_double_p, c_double_p,
                                                    c_double_p, c_int32_p, c_double_p]
        lib.alore_debug_force_exact_division.argtypes = [vp, C.c_int]
        lib.alore_debug_set_norm_guard.argtypes = [vp, C.c_double]
        lib.alore_debug_phase_cycles.argtypes = [vp, C.POINTER(C.c_ulonglong), C.c_int]
        lib.alore_selftest_division.argtypes = [vp, C.c_longlong, C.c_ulonglong, C.POINTER(C.c_longlong)]
    if path is None:
        _lib = lib
    return lib


# Symbols include/alore_b200.h declares (checked by the CPU test-suite without touching a GPU).
EXPORTED_SYMBOLS = [
    "alore_create", "alore_destroy", "alore_last_error", "alore_device_info", "alore_params_default",
    "alore_host_register", "alore_host_unregister",
    "alore_esdf_update", "alore_esdf_update_dev", "alore_esdf_set", "alore_esdf_reset", "alore_esdf_last_sq",
    "alore_esdf_last_kernel_ms", "alore_penalty_batch", "alore_penalty_batch_dev", "alore_cost_batch",
    "alore_opt_batch", "alore_batch_upload", "alore_batch_run", "alore_batch_download",
    "alore_batch_device_results", "alore_batch_argmin", "alore_batch_last_kernel_ms", "alore_batch_stats", "alore_batch_free",
    "alore_final_collision_batch", "alore_selftest_division", "alore_debug_force_exact_division", "alore_debug_set_norm_guard", "alore_debug_phase_cycles", "alore_launch_count",
    "alore_create_multi", "alore_destroy_multi", "alore_multi_size", "alore_multi_ctx", "alore_multi_last_error",
    "alore_multi_esdf_update", "alore_multi_opt_batch",
]


def default_params() -> Params:
    p = Params()
    load_library().alore_params_default(C.byref(p))
    return p


class AloreError(RuntimeError):
    pass


class Context:
    """RAII wrapper of alore_ctx (one CUDA device)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        self.h = C.c_void_p()
        rc = self.lib.alore_create(device, C.byref(self.h))
        if rc != 0:
            raise AloreError(f"alore_create({device}) failed rc={rc}: {self.lib.alore_last_error(None).decode()}")

    def check(self, rc: int):
        if rc != 0:
            raise AloreError(f"rc={rc}: {self.lib.alore_last_error(self.h).decode()}")

    def close(self):
        if self.h:
            self.lib.alore_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self) -> int:
        return int(self.lib.alore_launch_count(self.h))
