/*
 * alore_b200.h — C ABI of the B200-native planning_ddr_opt hot path.
 *
 * Drop-in boundary for the reference's (Zhihaibi/ALORE_Legged_Manipulator) grid-map and
 * back_end C++ interfaces.  Paths below are relative to the reference tree,
 * PDO = planning_ddr_opt.
 *
 *   SDFmap::updateESDF2d / forceUpdateESDF    PDO/utils/plan_env/include/plan_env/sdf_map.h:239,260
 *                                             PDO/utils/plan_env/src/sdf_map.cpp:618-715
 *   SDFmap::getDistWithGradBilinear (3 ovl.)  sdf_map.cpp:760-863   (device side, inside the kernels)
 *   MSPlanner::minco_plan / optimizer         PDO/back_end/include/back_end/optimizer.h:207-213
 *                                             PDO/back_end/src/optimizer.cpp:169-472
 *   MSPlanner::costFunctionCallback[Path]     optimizer.cpp:631-692, 1272-1317
 *   MSPlanner::attachPenaltyFunctional[Path]  optimizer.cpp:694-1067, 1319-1591
 *   MSPlanner::check_final_collision          optimizer.cpp:474-571
 *   lbfgs::lbfgs_optimize                     PDO/back_end/include/gcopter/lbfgs.hpp:440-751
 *   minco::MINCO_S3NU / BandedSystem          PDO/back_end/include/gcopter/minco.hpp:43-198, 751-1209
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success and a
 * negative ALORE_E* code on failure (never throws across the ABI); alore_last_error() gives
 * the message.  All functions are blocking unless they take a cuda_stream.  A context is bound to ONE CUDA device and
 * is not re-entrant (the reference runs everything on one ros::spin() thread): at most ONE operation per context may be
 * in flight — the *_dev / alore_batch_run entry points that are asynchronous on a caller stream share the context's
 * scratch (optimizer state, history, work counters), so the caller must order a second call after the first (same
 * stream, or an event).  Use one context per concurrent stream, or alore_create_multi for several GPUs.
 *
 * Grid layout is the reference's: cell (x, y) lives at index x*GLY + y (y contiguous),
 * sdf_map.cpp:525-527.  Cell states: 0 Unknown, 1 Unoccupied, 2 Occupied (sdf_map.h:98).
 */
#ifndef ALORE_B200_H
#define ALORE_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ALORE_OK 0
#define ALORE_EINVAL (-1)   /* bad argument */
#define ALORE_ECUDA (-2)    /* CUDA runtime error (message in alore_last_error) */
#define ALORE_ENOMAP (-3)   /* optimizer called before any ESDF is resident on the device */
#define ALORE_ENOMEM (-4)

#define ALORE_MAX_CHECKPOINTS 8

/* Cell states, sdf_map.h:98  enum {Unknown, Unoccupied, Occupied}. */
enum { ALORE_UNKNOWN = 0, ALORE_UNOCCUPIED = 1, ALORE_OCCUPIED = 2 };

/* lbfgs::lbfgs_parameter_t, lbfgs.hpp:15-129 (same fields, same defaults). */
typedef struct alore_lbfgs_params {
  int32_t mem_size;        /* 8 */
  int32_t past;            /* 3 */
  int32_t max_iterations;  /* 0 */
  int32_t max_linesearch;  /* 64 */
  double g_epsilon;        /* 1e-5 */
  double delta;            /* 1e-6 */
  double min_step;         /* 1e-20 */
  double max_step;         /* 1e+20 */
  double f_dec_coeff;      /* 1e-4 */
  double s_curv_coeff;     /* 0.9 */
  double cautious_factor;  /* 1e-6 */
  double machine_prec;     /* 1e-16 */
} alore_lbfgs_params_t;

/* Grid geometry: the members SDFmap derives in its constructor, sdf_map.h:120-160. */
typedef struct alore_map_geom {
  int32_t glx, gly;                 /* GLX_SIZE_, GLY_SIZE_ */
  double x_lower, y_lower;          /* global_x_lower_, global_y_lower_ */
  double x_upper, y_upper;          /* global_x_upper_, global_y_upper_ */
  double grid_interval;             /* grid_interval_ */
  double inv_grid_interval;         /* inv_grid_interval_ = 1/grid_interval_ (sdf_map.h:121) */
} alore_map_geom_t;

/*
 * Every parameter MSPlanner reads from the ROS parameter server in its constructor
 * (optimizer.cpp:17-166) plus Config (optimizer.h:31-52).  Field names follow the
 * reference's members; yaml defaults are PDO/back_end/config/global_planning3ms.yaml and
 * PDO/plan_tester/config/car3ms.yaml (see alore_params_default()).
 */
typedef struct alore_params {
  /* Config, optimizer.h:31-52 */
  double max_vel, min_vel, max_acc, max_omega, max_domega, max_centripetal_acc;
  int32_t if_directly_constrain_v_omega;
  int32_t if_standard_diff;              /* optimizer.cpp:166 */
  double ICR[3];                         /* ICR_.x (yl), .y (yr), .z (xv): optimizer.cpp:162-164 */

  double mean_time_lowBound, mean_time_uppBound;   /* dead code in the reference, kept for layout parity */
  double smoothEps;                      /* smoothingFactor */
  double safeDis;                        /* safeDis_ */
  double finalMinSafeDis;
  int32_t finalSafeDisCheckNum;
  int32_t safeReplanMaxTime;

  /* PenaltyWeights, optimizer.h:54-63 */
  double pw_time, pw_acc, pw_domega, pw_collision, pw_moment, pw_mean_time, pw_cen_acc;
  /* PathpenaltyWeights, optimizer.h:66-73 */
  double ppw_time, ppw_bigpath_sdf, ppw_mean_time, ppw_moment, ppw_acc, ppw_domega;

  double energyWeights[2];

  /* Augmented Lagrangian, optimizer.cpp:52-110 (normal and cut variants) */
  double EqualLambda[2], EqualRho[2], EqualRhoMax[2], EqualGamma[2], EqualTolerance[2];
  double CutEqualLambda[2], CutEqualRho[2], CutEqualRhoMax[2], CutEqualGamma[2], CutEqualTolerance[2];

  /* PathLbfgsParams, optimizer.h:76-81 */
  alore_lbfgs_params_t path_lbfgs;
  int32_t normal_past, shot_path_past;
  double shot_path_horizon;
  /* lbfgs_params_ */
  alore_lbfgs_params_t lbfgs;

  int32_t sparseResolution;
  int32_t n_checkpoints;
  double check_point[ALORE_MAX_CHECKPOINTS][2];

  /* The reference's ALM loop is `while(ros::ok())` (optimizer.cpp:376) with no cap.
   * 0 = reference behaviour, except that the device loop is still bounded by
   * ALORE_ALM_HARD_CAP so a pathological candidate cannot hang the GPU. */
  int32_t alm_max_outer;
  int32_t reserved0;
} alore_params_t;

#define ALORE_ALM_HARD_CAP 64

/*
 * A batch of candidate trajectories (one candidate = one FlatTrajData,
 * PDO/front_end/include/front_end/traj_representation.h:46-76), structure-of-arrays with
 * CSR offsets because TrajNum differs per candidate.  N_b = piece_off[b+1]-piece_off[b]
 * is MSPlanner::TrajNum (= UnOccupied_traj_pts.size()+1, optimizer.cpp:227), N_b >= 1.
 */
typedef struct alore_candidates {
  int32_t B;
  const int32_t* piece_off;      /* [B+1], piece_off[0] = 0 */
  const double* inner_pts;       /* [(sum N_b) - B][2]: (yaw, s) of UnOccupied_traj_pts; candidate b starts at row piece_off[b]-b */
  const double* init_T;          /* [B]  UnOccupied_initT */
  const double* inner_init_pos;  /* [sum N_b][3]: UnOccupied_positions followed by final_state_XYTheta (optimizer.cpp:234-235); candidate b starts at row piece_off[b] */
  const double* start_state;     /* [B][2][3] row 0 = yaw (P,V,A), row 1 = s (P,V,A) */
  const double* final_state;     /* [B][2][3] */
  const double* start_xytheta;   /* [B][3] */
  const double* final_xytheta;   /* [B][3] */
  const uint8_t* if_cut;         /* [B] */
} alore_candidates_t;

/* Result of MSPlanner::minco_plan for each candidate (same CSR offsets as the input). */
typedef struct alore_results {
  int32_t* ok;            /* [B] 1 = minco_plan returned true */
  int32_t* status;        /* [B] lbfgs return code of the last stage-B lbfgs_optimize (lbfgs.hpp:135-184) */
  int32_t* replans;       /* [B] number of optimizer() runs (replan_num_for_coll+1, capped at safeReplanMaxTime) */
  int32_t* alm_iters;     /* [B] stage-B lbfgs_optimize calls in the last optimizer() run */
  int32_t* evals;         /* [B] total cost-function evaluations (stage A + B, all replans) */
  double* cost;           /* [B] final stage-B cost */
  double* inner_pts;      /* [(sum N_b) - B][2] finalInnerpoints */
  double* tail_s;         /* [B] finState(1,0) after optimisation */
  double* piece_T;        /* [sum N_b] finalpieceTime */
  double* coeffs;         /* [sum N_b][6][2] MINCO coefficients b(6i+k, dim), ascending powers (minco.hpp:762) */
} alore_results_t;

typedef struct alore_ctx alore_ctx;

/* ---- lifetime ---------------------------------------------------------------------- */
int alore_create(int device, alore_ctx** out);
void alore_destroy(alore_ctx* ctx);
const char* alore_last_error(const alore_ctx* ctx);     /* ctx may be NULL: last creation error */
int alore_device_info(const alore_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor);

/* Optional: page-lock a caller-owned host buffer (SDFmap::gridmap_, distance_buffer_all_) for the
 * lifetime the CALLER guarantees, so the ESDF copies run at full PCIe speed.  The owner must call
 * alore_host_unregister before freeing the buffer (SDFmap's destructor, sdf_map.h:186-189).
 * Unregistered buffers work too (pageable copies, slower). */
int alore_host_register(alore_ctx* ctx, const void* ptr, size_t bytes);
int alore_host_unregister(alore_ctx* ctx, const void* ptr);

/* Fills *p with the reference's yaml defaults (global_planning3ms.yaml + plan_tester car3ms.yaml). */
void alore_params_default(alore_params_t* p);

/* ---- ESDF: replaces the body of SDFmap::updateESDF2d (sdf_map.cpp:618-680) ------------ */
/*
 * occ        host, geom.glx*geom.gly bytes (SDFmap::gridmap_)
 * min/max    inclusive window corners min_esdf/max_esdf as computed by the caller with the
 *            reference's own FP expression (sdf_map.cpp:619-621), so truncation is identical
 * dist_inout host, glx*gly doubles (SDFmap::distance_buffer_all_).  Only the cells the
 *            reference writes are written (window minus its last row and last column when
 *            ref_compat != 0); everything else keeps its previous value.
 * ref_compat 1: reproduce the reference's buffer-aliasing quirks bit for bit (SURVEY §8a-E1);
 *            0: clean EDT over the whole window (last row/col included, no column-0 alias).
 * On return the host mirror is valid AND a device-resident copy of the full distance buffer
 * plus geometry is retained in ctx for the optimizer entry points.  The device copy starts at
 * DBL_MAX (alore_esdf_reset) and then sees exactly the writes the host buffer sees.
 */
int alore_esdf_update(alore_ctx* ctx, const alore_map_geom_t* geom, const uint8_t* occ,
                      int min_x, int min_y, int max_x, int max_y,
                      double* dist_inout, int ref_compat);

/* Same, with occ and dist already in device memory (HBM-resident path used for kernel timing),
 * asynchronous on cuda_stream.  d_occ == NULL and d_dist_inout == NULL: rebuild the context's own
 * resident ESDF from the occupancy grid the last alore_esdf_update left on the device (rows never uploaded read as
 * Unknown, the constructor value of SDFmap::gridmap_); geom must then equal the resident map's geometry (ALORE_EINVAL
 * otherwise).  d_occ != NULL and d_dist_inout == NULL: the window's rows of the DEVICE grid d_occ are first copied into
 * the context's resident grid (what alore_esdf_update does from the host), then the resident ESDF is rebuilt.  With both
 * caller buffers, geom describes those buffers only and the context's resident map is untouched. */
int alore_esdf_update_dev(alore_ctx* ctx, const alore_map_geom_t* geom, const uint8_t* d_occ,
                          int min_x, int min_y, int max_x, int max_y,
                          double* d_dist_inout, int ref_compat, void* cuda_stream);

/* A new SDFmap on this context: (re)allocates the device grid for geom and fills the device
 * distance buffer with DBL_MAX, the value SDFmap's constructor gives distance_buffer_all_
 * (sdf_map.h:160), so that device and host agree in cells no update has written yet. */
int alore_esdf_reset(alore_ctx* ctx, const alore_map_geom_t* geom);

/* Make an existing HOST distance buffer the optimizer's ESDF (uploads it). */
int alore_esdf_set(alore_ctx* ctx, const alore_map_geom_t* geom, const double* dist);

/* Integer squared distances of the last alore_esdf_update[_dev] window (parity tests):
 * pos_sq/neg_sq host arrays of (max_x-min_x+1)*(max_y-min_y+1) int32, window-local index
 * x*NY + y; value ALORE_SQ_INF where the reference holds DBL_MAX.  Also after a caller-buffer
 * alore_esdf_update_dev (then those buffers' planes, whatever the resident map is).  Waits for
 * the device to be idle first, so a *_dev update still running on a caller stream is included. */
#define ALORE_SQ_INF 0x7fffffff
int alore_esdf_last_sq(alore_ctx* ctx, int32_t* pos_sq, int32_t* neg_sq);

/* Device time (ms, CUDA events on the launch stream) of the kernels of the last ESDF update. */
int alore_esdf_last_kernel_ms(const alore_ctx* ctx, float* ms);

/* ---- penalty + gradient, batched (replaces costFunctionCallback & friends) ----------- */
/*
 * Coefficient space (BASELINE config 3): attachPenaltyFunctional on given MINCO
 * coefficients, optimizer.cpp:694-1067.  Starts from cost=0, gradC=0, gradT=0 (no energy
 * term), with EqualLambda/EqualRho taken from params (normal set) and safeDis = params.safeDis.
 *   piece_off [B+1]; coeffs [sum N][6][2]; piece_T [sum N]; start_xy [B][2]; final_xy [B][2]
 *   out: cost [B]; gradC [sum N][6][2]; gradT [sum N]; xy_err [B][2] (FinalIntegralXYError)
 * All pointers are HOST pointers.
 */
int alore_penalty_batch(alore_ctx* ctx, const alore_params_t* prm, int B, const int32_t* piece_off,
                        const double* coeffs, const double* piece_T,
                        const double* start_xy, const double* final_xy,
                        double* cost, double* gradC, double* gradT, double* xy_err);

/* Same with DEVICE pointers, asynchronous on cuda_stream (kernel timing / HBM-resident path).
 * max_pieces = an upper bound on N_b = piece_off[b+1]-piece_off[b] over the batch (the offsets live on the device, so
 * the caller states it; shared memory and scratch are sized from it).  A trajectory with more pieces than declared is
 * NOT evaluated: its cost comes back NaN and nothing is written out of bounds. */
int alore_penalty_batch_dev(alore_ctx* ctx, const alore_params_t* prm, int B, int max_pieces,
                            const int32_t* d_piece_off, const double* d_coeffs, const double* d_piece_T,
                            const double* d_start_xy, const double* d_final_xy,
                            double* d_cost, double* d_gradC, double* d_gradT, double* d_xy_err,
                            void* cuda_stream);

/*
 * Decision-variable space: one call of MSPlanner::costFunctionCallback (stage 1,
 * optimizer.cpp:631-692) or costFunctionCallbackPath (stage 0, optimizer.cpp:1272-1317)
 * per candidate.  x/g layout is the reference's (optimizer.cpp:277-286):
 * [yaw_1,s_1,...,yaw_{N-1},s_{N-1} | tail_s | tau_1..tau_N], 3N-1 entries, candidate b
 * at offset 3*piece_off[b]-b.  lambda/rho [B][2] are EqualLambda/EqualRho (NULL = params'),
 * safe_dis [B] (NULL = params.safeDis).  HOST pointers.
 */
int alore_cost_batch(alore_ctx* ctx, const alore_params_t* prm, const alore_candidates_t* cands,
                     int stage, const double* x, const double* lambda, const double* rho,
                     const double* safe_dis, double* cost, double* g, double* xy_err);

/* ---- full optimisation, batched: B x MSPlanner::minco_plan (optimizer.cpp:169-220) ---- */
/* HOST pointers in cands/out.  B = 1 reproduces one minco_plan call.  Blocking.  The device copies of the batch are
 * carved from an arena the context keeps (no cudaMalloc/cudaFree per call), and the hand-out order of the candidates
 * to the resident warps uses the evaluation counts of the previous optimisation on this context with a similar batch
 * (same B, same piece count at the same index for >= 3/4 of the candidates; a replanning planner re-optimises mostly
 * the same legs every tick): longest predicted work first, piece counts alone otherwise (env ALORE_NO_SCHED_PREDICTION=1
 * forces the latter).  Neither affects a result: every candidate is optimised independently and deterministically. */
int alore_opt_batch(alore_ctx* ctx, const alore_params_t* prm, const alore_candidates_t* cands,
                    alore_results_t* out);

/* Upload once / optimise many: device-resident candidate batch (HBM-resident timing path).  alore_batch_run is
 * asynchronous on cuda_stream (NULL = the context's stream) except that a handle which is run AGAIN first reads
 * back its previous evaluation counts (one small blocking copy on that stream) to re-order its work queue. */
typedef struct alore_batch alore_batch;
int alore_batch_upload(alore_ctx* ctx, const alore_candidates_t* cands, alore_batch** out);
int alore_batch_run(alore_ctx* ctx, const alore_params_t* prm, alore_batch* batch, void* cuda_stream);
int alore_batch_download(alore_ctx* ctx, alore_batch* batch, alore_results_t* out);
/* Device pointers to the per-candidate final cost [B] (double) and ok flag [B] (int32) of the
 * last alore_batch_run, for an on-device argmin / NCCL gather by the caller. */
int alore_batch_device_results(alore_batch* batch, const double** d_cost, const int32_t** d_ok);
/* Best (lowest final cost among ok candidates) of the last run: computed on the device. */
int alore_batch_argmin(alore_ctx* ctx, alore_batch* batch, double* best_cost, int32_t* best_idx);
/* Totals over the batch of the last run: algorithmic bytes (SURVEY.md section 8d: per evaluation
 * 8*(2n+1) + 32*C*N*(K+1) [stage 1], per L-BFGS update 8*n*(4*bound+4)), cost evaluations, L-BFGS iterations. */
int alore_batch_stats(alore_ctx* ctx, alore_batch* batch, double* alg_bytes, long long* evals, long long* iters);
/* Device time (ms) of the optimisation kernel(s) of the last alore_batch_run / alore_opt_batch. */
int alore_batch_last_kernel_ms(const alore_batch* batch, float* ms);
void alore_batch_free(alore_batch* batch);

/* MSPlanner::check_final_collision (optimizer.cpp:474-571) on given coefficients; HOST pointers.
 *   collided [B] (1 = returns true), min_dist [B] (min SDF seen before the early return). */
int alore_final_collision_batch(alore_ctx* ctx, const alore_params_t* prm, int B,
                                const int32_t* piece_off, const double* coeffs,
                                const double* piece_T, const double* start_xy,
                                int32_t* collided, double* min_dist);

/* ---- several GPUs of one box behind one object (SURVEY.md section 8b ownership row, 8e) -------------------------------
 * The reference's caller is one C++ process (PlanManager, plan_manager.hpp:120-123, :662-670); alore_multi gives it the
 * multi-GPU path without a launcher: one host thread per device inside the library, the ESDF replicated (every device
 * rebuilds it from the 1 B/cell occupancy grid), the candidate array cut into contiguous blocks of (nearly) equal
 * piece counts, and ONE exchange: an all-gather over NCCL of (best cost, global index), 16 bytes per device.  Results
 * are written into the caller's arrays exactly where alore_opt_batch would write them (a candidate's result does not
 * depend on which device or block it ran in).  best_idx = -1 when no candidate succeeded.  block_offsets [n+1] (may be
 * NULL) receives the block boundaries.  NCCL is loaded at run time (dlopen) and only when n > 1. */
typedef struct alore_multi alore_multi;
int alore_create_multi(const int* devices, int n, alore_multi** out);
void alore_destroy_multi(alore_multi* m);
int alore_multi_size(const alore_multi* m);
alore_ctx* alore_multi_ctx(alore_multi* m, int i);           /* the per-device context (owned by m) */
const char* alore_multi_last_error(const alore_multi* m);
int alore_multi_esdf_update(alore_multi* m, const alore_map_geom_t* geom, const uint8_t* occ,
                            int min_x, int min_y, int max_x, int max_y, double* dist_inout, int ref_compat);
int alore_multi_opt_batch(alore_multi* m, const alore_params_t* prm, const alore_candidates_t* cands,
                          alore_results_t* out, double* best_cost, int32_t* best_idx, int32_t* block_offsets);

/* Self-test of the kernels' split IEEE division (csrc/traj_opt.cuh: rcp_refine + div_rcp, used on the dependent
 * chains of the banded LU / triangular sweeps that replace minco.hpp:99-197) against the compiler's a / b on
 * n_pairs generated operand pairs (all exponents, specials, solver-range magnitudes).  *mismatches = differing bits. */
int alore_selftest_division(alore_ctx* ctx, long long n_pairs, unsigned long long seed, long long* mismatches);
/* Test hook: on != 0 makes every banded-solver pass use the compiler's division (the path taken when a quotient
 * leaves the split division's range); results must not change.  Process-wide for the context's device. */
int alore_debug_force_exact_division(alore_ctx* ctx, int on);
/* Test hook: the optimizer's cost evaluations return 0 without touching the gradient when ||x|| > threshold (the
 * reference's `return inf;` with `#define inf 1 >> 30`, threshold 1e4 = the default).  A lower threshold makes that
 * path reachable on ordinary candidates; threshold must lie in (0, 1e4].  Process-wide for the context's device. */
int alore_debug_set_norm_guard(alore_ctx* ctx, double threshold);
/* Developer hook: per-phase cycle totals of the optimizer kernels (only in builds with -DALORE_PHASE_TIMING;
 * the product build returns ALORE_EINVAL).  out32[0..6] = cost_eval phases ([4] penalty cost half, [7] penalty gradient half), [8..13] = penalty passes,
 * [17..18] = L-BFGS update, [20] = history steps (a count), [21] = line-search trials whose gradient was skipped (a count). */
int alore_debug_phase_cycles(alore_ctx* ctx, unsigned long long* out32, int reset);

/* Number of kernels this library has launched since alore_create (bench `gpu_launches`). */
long long alore_launch_count(const alore_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* ALORE_B200_H */
