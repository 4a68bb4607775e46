// capi.cu — extern "C" entry points: context lifetime, parameter defaults, ESDF update.
// (Optimizer entry points live in traj_opt.cu.)  See include/alore_b200.h for the contract.
#include <mutex>

#include "common.cuh"

static std::string g_create_err;

extern "C" {

int alore_create(int device, alore_ctx** out) {
  if (!out) return ALORE_EINVAL;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    g_create_err = std::string("no CUDA device: ") + cudaGetErrorString(e);
    (void)cudaGetLastError();
    return ALORE_ECUDA;
  }
  if (device < 0 || device >= n) { g_create_err = "device index out of range"; return ALORE_EINVAL; }
  e = cudaSetDevice(device);
  if (e != cudaSuccess) { g_create_err = cudaGetErrorString(e); return ALORE_ECUDA; }
  alore_ctx* c = new alore_ctx();
  c->device = device;
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  c->sm_count = prop.multiProcessorCount;
  c->cc_major = prop.major;
  c->cc_minor = prop.minor;
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess) {
    g_create_err = "stream/event creation failed";
    delete c;
    return ALORE_ECUDA;
  }
  *out = c;
  return ALORE_OK;
}

void alore_destroy(alore_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (auto& r : ctx->regs) cudaHostUnregister(const_cast<void*>(r.p));
  if (ctx->d_occ) cudaFree(ctx->d_occ);
  if (ctx->d_dist) cudaFree(ctx->d_dist);
  if (ctx->d_row) cudaFree(ctx->d_row);
  if (ctx->d_blk) cudaFree(ctx->d_blk);
  if (ctx->d_band) cudaFree(ctx->d_band);
  if (ctx->opt_scratch) cudaFree(ctx->opt_scratch);
  if (ctx->opt_hist) cudaFree(ctx->opt_hist);
  if (ctx->batch_pool) cudaFree(ctx->batch_pool);
  cudaEventDestroy(ctx->ev0);
  cudaEventDestroy(ctx->ev1);
  cudaEventDestroy(ctx->ev_fork);
  cudaEventDestroy(ctx->ev_join);
  cudaStreamDestroy(ctx->stream2);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

int alore_host_register(alore_ctx* ctx, const void* p, size_t bytes) {
  if (!ctx || !p || !bytes) return ALORE_EINVAL;
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  for (auto& r : ctx->regs)
    if (r.p == p) return r.bytes == bytes ? ALORE_OK : alore_fail(ctx, ALORE_EINVAL, "buffer already registered with another size");
  ALORE_CUDA(ctx, cudaHostRegister(const_cast<void*>(p), bytes, cudaHostRegisterDefault));
  ctx->regs.push_back({p, bytes});
  return ALORE_OK;
}

int alore_host_unregister(alore_ctx* ctx, const void* p) {
  if (!ctx || !p) return ALORE_EINVAL;
  for (size_t i = 0; i < ctx->regs.size(); i++)
    if (ctx->regs[i].p == p) {
      cudaSetDevice(ctx->device);
      cudaStreamSynchronize(ctx->stream);
      cudaHostUnregister(const_cast<void*>(p));
      ctx->regs.erase(ctx->regs.begin() + i);
      return ALORE_OK;
    }
  return alore_fail(ctx, ALORE_EINVAL, "buffer was not registered");
}

const char* alore_last_error(const alore_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int alore_device_info(const alore_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor) {
  if (!ctx) return ALORE_EINVAL;
  if (sm_count) *sm_count = ctx->sm_count;
  if (cc_major) *cc_major = ctx->cc_major;
  if (cc_minor) *cc_minor = ctx->cc_minor;
  return ALORE_OK;
}

long long alore_launch_count(const alore_ctx* ctx) { return ctx ? ctx->launches : 0; }

static void lbfgs_defaults(alore_lbfgs_params_t* l) {  // lbfgs.hpp:15-129
  l->mem_size = 8; l->past = 3; l->max_iterations = 0; l->max_linesearch = 64;
  l->g_epsilon = 1.0e-5; l->delta = 1.0e-6; l->min_step = 1.0e-20; l->max_step = 1.0e+20;
  l->f_dec_coeff = 1.0e-4; l->s_curv_coeff = 0.9; l->cautious_factor = 1.0e-6; l->machine_prec = 1.0e-16;
}

// planning_ddr_opt/back_end/config/global_planning3ms.yaml + plan_tester/config/car3ms.yaml
// + plan_tester/launch/planner_sim.launch:41-46 (ICR, if_standard_diff).
void alore_params_default(alore_params_t* p) {
  std::memset(p, 0, sizeof(*p));
  p->max_vel = 3.0; p->min_vel = -3.0; p->max_acc = 2.0; p->max_omega = 3.0; p->max_domega = 4.0;
  p->max_centripetal_acc = 50.0; p->if_directly_constrain_v_omega = 0;
  p->if_standard_diff = 1;
  p->ICR[0] = 0.3; p->ICR[1] = -0.3; p->ICR[2] = 0.2;
  p->mean_time_lowBound = 0.5; p->mean_time_uppBound = 2.0;
  p->smoothEps = 0.01; p->safeDis = 0.6; p->finalMinSafeDis = 0.10;
  p->finalSafeDisCheckNum = 16; p->safeReplanMaxTime = 3;
  p->pw_time = 50; p->pw_acc = 300; p->pw_domega = 300; p->pw_collision = 500000; p->pw_moment = 300;
  p->pw_mean_time = 300; p->pw_cen_acc = 300;
  p->ppw_time = 20; p->ppw_bigpath_sdf = 200000; p->ppw_mean_time = 100; p->ppw_moment = 1000;
  p->ppw_acc = 100; p->ppw_domega = 100;
  p->energyWeights[0] = 0.33; p->energyWeights[1] = 1.0;
  for (int i = 0; i < 2; i++) {
    p->EqualLambda[i] = 0; p->EqualRho[i] = 10000.0; p->EqualRhoMax[i] = 1.0e10; p->EqualGamma[i] = 9.0;
    p->CutEqualLambda[i] = 0; p->CutEqualRho[i] = 1000.0; p->CutEqualRhoMax[i] = 1.0e10; p->CutEqualGamma[i] = 5.0;
  }
  p->EqualTolerance[0] = 0.01; p->EqualTolerance[1] = 0.0;
  p->CutEqualTolerance[0] = 0.5; p->CutEqualTolerance[1] = 0.0;
  lbfgs_defaults(&p->path_lbfgs);
  p->path_lbfgs.mem_size = 256; p->path_lbfgs.past = 2; p->path_lbfgs.g_epsilon = 0.0; p->path_lbfgs.min_step = 0.0;
  p->path_lbfgs.delta = 5.0e-2; p->path_lbfgs.max_iterations = 8000;
  p->normal_past = 2; p->shot_path_past = 8; p->shot_path_horizon = 0.5;
  lbfgs_defaults(&p->lbfgs);
  p->lbfgs.mem_size = 256; p->lbfgs.past = 3; p->lbfgs.g_epsilon = 0.0; p->lbfgs.min_step = 1.0e-32;
  p->lbfgs.delta = 5.0e-4; p->lbfgs.max_iterations = 8000;
  p->sparseResolution = 8;
  p->n_checkpoints = 1; p->check_point[0][0] = 0.0; p->check_point[0][1] = 0.0;
  p->alm_max_outer = 0;
}

__global__ void fill_f64(double* p, size_t n, double v) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

// (Re)allocates the device grid for `geom`.  A fresh or re-shaped device distance buffer starts at
// DBL_MAX like SDFmap's constructor (sdf_map.h:160), so device and host agree in never-updated cells.
static int ensure_map(alore_ctx* ctx, const alore_map_geom_t* geom, bool force_fill = false) {
  if (!geom || geom->glx <= 0 || geom->gly <= 0) return alore_fail(ctx, ALORE_EINVAL, "bad map geometry");
  const size_t cells = (size_t)geom->glx * geom->gly;
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  if (cells != ctx->map_cells) {
    if (ctx->d_occ) cudaFree(ctx->d_occ);
    if (ctx->d_dist) cudaFree(ctx->d_dist);
    ctx->d_occ = nullptr; ctx->d_dist = nullptr; ctx->map_cells = 0;
    ctx->have_map = false;
    ALORE_CUDA(ctx, cudaMalloc(&ctx->d_occ, cells));
    ALORE_CUDA(ctx, cudaMalloc(&ctx->d_dist, cells * sizeof(double)));
    // rows no alore_esdf_update has uploaded yet read as Unknown, the state SDFmap's constructor gives gridmap_
    ALORE_CUDA(ctx, cudaMemsetAsync(ctx->d_occ, ALORE_UNKNOWN, cells, ctx->stream));
    ctx->map_cells = cells;
    force_fill = true;
  }
  if (std::memcmp(&ctx->geom, geom, sizeof(*geom)) != 0) { ctx->geom = *geom; force_fill = true; }
  if (force_fill) {
    fill_f64<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(ctx->d_dist, cells, 1.7976931348623157e308);
    ctx->launches++;
    ALORE_CUDA(ctx, cudaGetLastError());
    ctx->have_map = false;
  }
  return ALORE_OK;
}

}  // extern "C"

// dist_inout == NULL: no host mirror is written (replica devices of alore_multi keep the ESDF in HBM only)
int alore_esdf_update_impl(alore_ctx* ctx, const alore_map_geom_t* geom, const uint8_t* occ, int min_x, int min_y, int max_x,
                           int max_y, double* dist_inout, int ref_compat) {
  if (!ctx) return ALORE_EINVAL;
  if (!occ) return alore_fail(ctx, ALORE_EINVAL, "null buffer");
  int rc = ensure_map(ctx, geom);
  if (rc) return rc;
  const int NX = max_x - min_x + 1, NY = max_y - min_y + 1;
  if (NX <= 0 || NY <= 0 || min_x < 0 || min_y < 0 || max_x >= geom->glx || max_y >= geom->gly)
    return alore_fail(ctx, ALORE_EINVAL, "esdf window outside the grid");
  const size_t gly = geom->gly;
  cudaStream_t st = ctx->stream;
  // H2D: the window's rows of the occupancy grid (contiguous chunk).
  ALORE_CUDA(ctx, cudaMemcpyAsync(ctx->d_occ + (size_t)min_x * gly, occ + (size_t)min_x * gly, (size_t)NX * gly,
                                  cudaMemcpyHostToDevice, st));
  ALORE_CUDA(ctx, cudaEventRecord(ctx->ev0, st));
  rc = alore_esdf_run(ctx, &ctx->geom, ctx->d_occ, ctx->d_dist, min_x, min_y, max_x, max_y, ref_compat, st, nullptr, nullptr);
  if (rc) return rc;
  ALORE_CUDA(ctx, cudaEventRecord(ctx->ev1, st));
  // D2H: exactly the rectangle the reference writes.
  const int wx = ref_compat ? NX - 1 : NX, wy = ref_compat ? NY - 1 : NY;
  if (dist_inout && wx > 0 && wy > 0) {
    const size_t o = (size_t)min_x * gly + min_y;
    ALORE_CUDA(ctx, cudaMemcpy2DAsync(dist_inout + o, gly * sizeof(double), ctx->d_dist + o, gly * sizeof(double),
                                      (size_t)wy * sizeof(double), wx, cudaMemcpyDeviceToHost, st));
  }
  ALORE_CUDA(ctx, cudaStreamSynchronize(st));
  ALORE_CUDA(ctx, cudaEventElapsedTime(&ctx->esdf_kernel_ms, ctx->ev0, ctx->ev1));
  ctx->have_map = true;
  return ALORE_OK;
}

extern "C" {

int alore_esdf_update(alore_ctx* ctx, const alore_map_geom_t* geom, const uint8_t* occ, int min_x, int min_y, int max_x,
                      int max_y, double* dist_inout, int ref_compat) {
  if (!ctx) return ALORE_EINVAL;
  if (!dist_inout) return alore_fail(ctx, ALORE_EINVAL, "null buffer");
  return alore_esdf_update_impl(ctx, geom, occ, min_x, min_y, max_x, max_y, dist_inout, ref_compat);
}

int alore_esdf_update_dev(alore_ctx* ctx, const alore_map_geom_t* geom, const uint8_t* d_occ, int min_x, int min_y,
                          int max_x, int max_y, double* d_dist_inout, int ref_compat, void* cuda_stream) {
  if (!ctx) return ALORE_EINVAL;
  if (!geom || geom->glx <= 0 || geom->gly <= 0) return alore_fail(ctx, ALORE_EINVAL, "bad map geometry");
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  const bool resident = (d_occ == nullptr && d_dist_inout == nullptr);
  if (resident) {
    // HBM-resident path: rebuild the context's own ESDF from the occupancy grid a previous alore_esdf_update left on the
    // device.  The geometry must be the one that map was created with: a different shape with the same cell count
    // (4096x4096 vs 8192x2048) would silently re-stride the buffers.
    if (!ctx->d_occ || !ctx->d_dist || (size_t)geom->glx * geom->gly != ctx->map_cells)
      return alore_fail(ctx, ALORE_ENOMAP, "no resident occupancy grid of this geometry: call alore_esdf_update first");
    if (std::memcmp(&ctx->geom, geom, sizeof(*geom)) != 0)
      return alore_fail(ctx, ALORE_EINVAL, "geometry differs from the resident map's (%dx%d): call alore_esdf_update / alore_esdf_reset first",
                        ctx->geom.glx, ctx->geom.gly);
    d_occ = ctx->d_occ;
    d_dist_inout = ctx->d_dist;
  } else if (d_occ && !d_dist_inout) {
    // resident update from a DEVICE occupancy grid: the window's rows are copied into the context's grid (device to
    // device, what alore_esdf_update does from the host) and the resident ESDF is rebuilt
    if (!ctx->d_occ || !ctx->d_dist || (size_t)geom->glx * geom->gly != ctx->map_cells || std::memcmp(&ctx->geom, geom, sizeof(*geom)) != 0)
      return alore_fail(ctx, ALORE_ENOMAP, "no resident map of this geometry: call alore_esdf_update / alore_esdf_reset first");
    // the whole window is checked before the copy: a refused call leaves the resident grid as it was
    if (min_x < 0 || max_x >= geom->glx || max_x < min_x || min_y < 0 || max_y >= geom->gly || max_y < min_y)
      return alore_fail(ctx, ALORE_EINVAL, "esdf window outside the grid");
    cudaStream_t st2 = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    const size_t gly = geom->gly;
    ALORE_CUDA(ctx, cudaMemcpyAsync(ctx->d_occ + (size_t)min_x * gly, d_occ + (size_t)min_x * gly, (size_t)(max_x - min_x + 1) * gly,
                                    cudaMemcpyDeviceToDevice, st2));
    int rc2 = alore_esdf_run(ctx, geom, ctx->d_occ, ctx->d_dist, min_x, min_y, max_x, max_y, ref_compat, st2, nullptr, nullptr);
    if (rc2 == ALORE_OK) ctx->have_map = true;
    return rc2;
  } else if (!d_occ || !d_dist_inout) {
    return alore_fail(ctx, ALORE_EINVAL, "pass both device buffers, the occupancy alone, or neither");
  }
  // caller-buffer mode: the caller's geometry describes the caller's buffers only; the context's resident map (and the
  // geometry the optimizer entry points read) is left untouched
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
  int rc = alore_esdf_run(ctx, geom, d_occ, d_dist_inout, min_x, min_y, max_x, max_y, ref_compat, st, nullptr, nullptr);
  if (rc == ALORE_OK && resident) ctx->have_map = true;
  return rc;
}

int alore_esdf_set(alore_ctx* ctx, const alore_map_geom_t* geom, const double* dist) {
  if (!ctx) return ALORE_EINVAL;
  if (!dist) return alore_fail(ctx, ALORE_EINVAL, "null buffer");
  int rc = ensure_map(ctx, geom);
  if (rc) return rc;
  ALORE_CUDA(ctx, cudaMemcpyAsync(ctx->d_dist, dist, ctx->map_cells * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  ALORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->have_map = true;
  return ALORE_OK;
}

int alore_esdf_reset(alore_ctx* ctx, const alore_map_geom_t* geom) {
  if (!ctx) return ALORE_EINVAL;
  int rc = ensure_map(ctx, geom, true);
  if (rc) return rc;
  ALORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return ALORE_OK;
}

int alore_esdf_last_sq(alore_ctx* ctx, int32_t* pos_sq, int32_t* neg_sq) {
  if (!ctx) return ALORE_EINVAL;
  if (!pos_sq || !neg_sq) return alore_fail(ctx, ALORE_EINVAL, "null buffer");
  if (ctx->win[2] < ctx->win[0]) return alore_fail(ctx, ALORE_EINVAL, "no ESDF update has run on this context");
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  // the last update may still run on a caller stream (alore_esdf_update_dev): its row pass is what is re-read here
  ALORE_CUDA(ctx, cudaDeviceSynchronize());
  const int NX = ctx->win[2] - ctx->win[0] + 1, NY = ctx->win[3] - ctx->win[1] + 1;
  const size_t n = (size_t)NX * NY;
  int32_t *dp = nullptr, *dn = nullptr;
  ALORE_CUDA(ctx, cudaMalloc(&dp, n * sizeof(int32_t)));
  if (cudaMalloc(&dn, n * sizeof(int32_t)) != cudaSuccess) { cudaFree(dp); return alore_fail(ctx, ALORE_ENOMEM, "cudaMalloc"); }
  // the window is checked against the grid the last update read: after a caller-buffer update that is the caller's
  // geometry, not the resident map's (which may be absent or of another shape); the squared planes need no grid data
  int rc = alore_esdf_run(ctx, &ctx->win_geom, ctx->d_occ, ctx->d_dist, ctx->win[0], ctx->win[1], ctx->win[2], ctx->win[3],
                          ctx->last_ref_compat, ctx->stream, dp, dn);
  if (rc == ALORE_OK) {
    cudaMemcpyAsync(pos_sq, dp, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(neg_sq, dn, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) rc = alore_fail(ctx, ALORE_ECUDA, "%s", cudaGetErrorString(e));
  }
  cudaFree(dp);
  cudaFree(dn);
  return rc;
}

int alore_esdf_last_kernel_ms(const alore_ctx* ctx, float* ms) {
  if (!ctx || !ms) return ALORE_EINVAL;
  *ms = ctx->esdf_kernel_ms;
  return ALORE_OK;
}

}  // extern "C"
