// common.cuh — shared host-side plumbing of libalore_b200 (context, error handling).
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/alore_b200.h"

struct alore_ctx {
  int device = 0;
  int sm_count = 0, cc_major = 0, cc_minor = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;                  // side stream: the ref_compat column runs beside K1b/K2
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  std::string err;
  long long launches = 0;

  // ---- ESDF state (device-resident grid map) ----
  alore_map_geom_t geom{};
  bool have_map = false;
  uint8_t* d_occ = nullptr;      // glx*gly
  double* d_dist = nullptr;      // glx*gly  (SDFmap::distance_buffer_all_ mirror)
  size_t map_cells = 0;
  int16_t* d_row = nullptr;      // window-local signed row distances, pitch row_pitch
  uint32_t* d_blk = nullptr;     // per (32-row block, column): lo16 = min g+ , hi16 = min g-
  size_t row_cap = 0, blk_cap = 0;
  void* d_band = nullptr;        // far-cell masks of the ESDF superband envelope kernel (K2e)
  size_t band_cap = 0;
  int band_epoch = 0;            // flags of K2e are 'set' when they hold the current run's epoch
  int row_pitch = 0;
  int win[4] = {0, 0, -1, -1};   // min_x, min_y, max_x, max_y of the last update
  alore_map_geom_t win_geom{};   // geometry of the grid the last update read (a caller buffer's, or the resident map's)
  int last_ref_compat = 1;
  float esdf_kernel_ms = 0.f;
  // host buffers page-locked through alore_host_register (lifetime guaranteed by the caller)
  struct Reg { const void* p; size_t bytes; };
  std::vector<Reg> regs;

  // ---- optimizer scratch (see traj_opt.cu) ----
  void* opt_scratch = nullptr;
  size_t opt_scratch_bytes = 0;
  void* opt_hist = nullptr;      // L-BFGS history ring of every resident warp
  size_t opt_hist_bytes = 0;
  // Scheduling memory across replan ticks: cost evaluations each candidate needed the last time a batch with the same
  // structure (B, piece_off) was optimised.  The persistent kernel hands out the predicted-longest work first
  // (results do not depend on the order; tests/test_optimizer_gpu.py::test_result_independent_of_batch_composition).
  // Device arena of the one-shot batch path (alore_opt_batch & co.): grown on demand, reused across calls, so that a
  // replan tick does not pay ~50 cudaMalloc/cudaFree round trips.  One pooled batch at a time; others use cudaMalloc.
  void* batch_pool = nullptr;
  size_t batch_pool_bytes = 0;
  bool batch_pool_busy = false;
  std::vector<int32_t> sched_piece_off;
  std::vector<int32_t> sched_evals;
  void* last_batch = nullptr;                      // alore_batch of the last persistent-kernel run (its evals feed the next schedule)
  int l2_max_persist = -1, l2_max_window = -1;     // per device (set_l2_window)
};

inline int alore_fail(alore_ctx* ctx, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  return code;
}

#define ALORE_CUDA(ctx, call)                                                                          \
  do {                                                                                                 \
    cudaError_t e__ = (call);                                                                          \
    if (e__ != cudaSuccess)                                                                            \
      return alore_fail((ctx), ALORE_ECUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
  } while (0)

// esdf.cu
int alore_esdf_run(alore_ctx* ctx, const alore_map_geom_t* geom, const uint8_t* d_occ, double* d_dist, int min_x, int min_y, int max_x, int max_y,
                   int ref_compat, cudaStream_t st, int32_t* d_pos_sq, int32_t* d_neg_sq);
// capi.cu: alore_esdf_update with an optional host mirror (dist_inout == NULL: keep the result in HBM only)
int alore_esdf_update_impl(alore_ctx* ctx, const alore_map_geom_t* geom, const uint8_t* occ, int min_x, int min_y, int max_x,
                           int max_y, double* dist_inout, int ref_compat);
