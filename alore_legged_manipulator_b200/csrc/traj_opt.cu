// traj_opt.cu — kernels and C-ABI entry points of the batched trajectory optimizer.
// Device code: traj_opt.cuh.  One warp (= one 32-thread CTA) per candidate trajectory, persistent
// over the whole minco_plan (stage A L-BFGS, stage B augmented-Lagrangian loop of L-BFGS runs,
// final collision check, collision replans) — no host round trip per iteration.
#include <algorithm>
#include <cstdlib>
#include <numeric>

#include "traj_opt.cuh"

using namespace topt;

namespace {

struct KParams {
  alore_params_t P;
  MapDev map;
  Layout L;
  int mcap;
};

__device__ void carve(Warp& w, const Layout& L, double* smem, double* slab, double* hist, int N, int K) {
  w.lane = threadIdx.x & 31;
  w.N = N; w.n = 3 * N - 1; w.npad = (3 * N) & ~1; w.n6 = 6 * N; w.K = K; w.S1 = 2 * K + 1;
  const int Nm = L.Nmax;
  double* s = smem;
  w.T1 = s; s += Nm; w.T2 = s; s += Nm; w.T3 = s; s += Nm; w.T4 = s; s += Nm; w.T5 = s; s += Nm;
  w.gT = s; s += Nm;
  w.pXY = s; s += 2 * (Nm + 1);
  w.sumT = s; s += Nm + 1 + 3;
  s = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(s) + 15) & ~uintptr_t(15));   // stg/stgb are accessed as double2
  w.ring = s; s += 256;
  w.mbar = s; s += 6;                 // 4 mbarriers + phase word (TMA history variant), keeps 16-byte alignment
  w.d = s; s += L.npadmax;
  w.stg = s;
  w.hbuf = s;
  w.Nm = Nm;
  w.cf = slab + L.cf; w.gC = slab + L.gC;
  w.x = slab + L.x; w.g = slab + L.g; w.xp = slab + L.xp; w.gp = slab + L.gp;
  w.lm_s = hist + L.lm_s; w.lm_y = hist + L.lm_y;
  w.pf = slab + L.pf; w.Uf = slab + L.Ab; w.Lf = slab + L.Ab + (size_t)8 * 6 * Nm; w.zb = slab + L.zb; w.cs = slab + L.cs; w.ax = slab + L.ax; w.ay = slab + L.ay;
  w.cellP = slab + L.cellP; w.g2p = slab + L.g2p;
  w.terms = slab + L.terms; w.cg = slab + L.cg; w.fold = slab + L.fold;
  w.nterm = reinterpret_cast<int*>(slab + L.nterm); w.rank = reinterpret_cast<int*>(slab + L.rank);
  w.TS = L.TS; w.tsum = 0.0;
  w.evals = 0;
  w.iters = 0;
  w.alg_bytes = 0.0;
  w.err[0] = w.err[1] = 0.0;
}

// get_state (optimizer.cpp:222-249): candidate -> planner state.
__device__ void load_candidate(Warp& w, const BatchDev& bt, int b, int p0) {
  for (int d = 0; d < 2; d++)
    for (int k = 0; k < 3; k++) {
      w.head[d][k] = bt.start_state[6 * (size_t)b + 3 * d + k];
      w.tail[d][k] = bt.final_state[6 * (size_t)b + 3 * d + k];
    }
  w.sx = bt.start_xytheta[3 * (size_t)b]; w.sy = bt.start_xytheta[3 * (size_t)b + 1];
  w.fx = bt.final_xytheta[3 * (size_t)b]; w.fy = bt.final_xytheta[3 * (size_t)b + 1];
  w.init_pos = bt.inner_init_pos + 3 * (size_t)p0;
}

// x0 = [Innerpoints | finState(1,0) | RealT2VirtualT(pieceTime)]            optimizer.cpp:277-286
__device__ void initial_x(Warp& w, const BatchDev& bt, int b, int p0) {
  const int N = w.N, lane = w.lane;
  const double* ip = bt.inner_pts + 2 * (size_t)(p0 - b);
  for (int i = lane; i < 2 * (N - 1); i += 32) w.x[i] = ip[i];
  if (lane == 0) w.x[2 * (N - 1)] = w.tail[1][0];
  const double T = bt.init_T[b];
  const double vt = T > 1.0 ? (sqrt(2.0 * T - 1.0) - 1.0) : (1.0 - sqrt(2.0 / T - 1.0));
  for (int i = lane; i < N; i += 32) w.x[2 * (N - 1) + 1 + i] = vt;
  __syncwarp();
}

// Minco.setTConditions(finState); Minco.setParameters(P, T) from x            optimizer.cpp:452-464
__device__ void coefficients_from_x(Warp& w) {
  const int N = w.N, lane = w.lane;
  const double* tau = w.x + 2 * (N - 1) + 1;
  w.tail[1][0] = w.x[2 * (N - 1)];
  for (int i = lane; i < N; i += 32) {
    const double t = tau[i];
    const double T = t > 0.0 ? ((0.5 * t + 1.0) * t + 1.0) : 1.0 / ((0.5 * t - 1.0) * t + 1.0);
    w.T1[i] = T;
    const double t2 = T * T;
    w.T2[i] = t2; w.T3[i] = t2 * T; w.T4[i] = t2 * t2; w.T5[i] = (t2 * t2) * T;
  }
  __syncwarp();
  minco_lu_forward(w, w.x);
  minco_back(w);
}

// MSPlanner::minco_plan for candidate b                                       optimizer.cpp:169-220
__device__ void minco_plan(Warp& w, const KParams& kp, const BatchDev& bt, int b, const ResultDev& out) {
  const alore_params_t& P = kp.P;
  const int p0 = bt.piece_off[b];
  const int lane = w.lane, N = w.N;
  load_candidate(w, bt, b, p0);
  const double start_safe_dis = dist_real(kp.map, w.sx, w.sy) * 0.85;
  w.safeDis = fmin(start_safe_dis, P.safeDis);
  w.time_weight = P.pw_time;
  w.evals = 0;
  const bool cut = bt.if_cut[b] != 0;
  int replan = 0, status = 0, alm_iters = 0;
  double cost = 0.0;
  for (; replan < P.safeReplanMaxTime; replan++) {
    load_candidate(w, bt, b, p0);  // get_state: iniState / finState restored from the FlatTrajData
    for (int d = 0; d < 2; d++) {
      w.lam[d] = cut ? P.CutEqualLambda[d] : P.EqualLambda[d];
      w.rho[d] = cut ? P.CutEqualRho[d] : P.EqualRho[d];
    }
    initial_x(w, bt, b, p0);
    // stage A: path pre-processing                                             optimizer.cpp:296-309
    alore_lbfgs_params_t pa = P.path_lbfgs;
    pa.past = (fabs(w.tail[1][0]) < P.shot_path_horizon) ? P.shot_path_past : P.normal_past;
    status = lbfgs_optimize(w, P, kp.map, 0, pa, cost, kp.mcap);
    // (the reference's extra printing evaluation at optimizer.cpp:341 only re-derives state from x)
    // stage B: augmented-Lagrangian loop                                       optimizer.cpp:376-418
    alm_iters = 0;
    const int cap = P.alm_max_outer > 0 ? min(P.alm_max_outer, ALORE_ALM_HARD_CAP) : ALORE_ALM_HARD_CAP;
    while (true) {
      status = lbfgs_optimize(w, P, kp.map, 1, P.lbfgs, cost, kp.mcap);
      alm_iters++;
      const double nrm = sqrt(w.err[0] * w.err[0] + w.err[1] * w.err[1]);
      if (nrm < (cut ? P.CutEqualTolerance[0] : P.EqualTolerance[0])) break;
      w.lam[0] += w.rho[0] * w.err[0];
      w.lam[1] += w.rho[1] * w.err[1];
      for (int d = 0; d < 2; d++) {
        const double gm = cut ? P.CutEqualGamma[d] : P.EqualGamma[d];
        const double rm = cut ? P.CutEqualRhoMax[d] : P.EqualRhoMax[d];
        w.rho[d] = fmin((1 + gm) * w.rho[d], rm);
      }
      if (alm_iters >= cap) break;
    }
    coefficients_from_x(w);
    const int coll = final_collision(w, P, kp.map, nullptr);
    if (coll) w.time_weight *= 0.75;
    else break;
  }
  const bool ok = replan != P.safeReplanMaxTime;
  if (lane == 0) {
    out.ok[b] = ok ? 1 : 0;
    out.status[b] = status;
    out.replans[b] = min(replan + 1, P.safeReplanMaxTime);
    out.alm_iters[b] = alm_iters;
    out.evals[b] = w.evals;
    out.cost[b] = cost;
    out.tail_s[b] = w.x[2 * (N - 1)];
    out.alg_bytes[b] = w.alg_bytes;
    out.iters[b] = w.iters;
  }
  double* oi = out.inner_pts + 2 * (size_t)(p0 - b);
  for (int i = lane; i < 2 * (N - 1); i += 32) oi[i] = w.x[i];
  for (int i = lane; i < N; i += 32) out.piece_T[p0 + i] = w.T1[i];
  for (int i = lane; i < 12 * N; i += 32) out.coeffs[12 * (size_t)p0 + i] = w.cf[i];
  __syncwarp();
}

__device__ __forceinline__ int next_job(int* counter, int lane) {
  int j = 0;
  if (lane == 0) j = atomicAdd(counter, 1);
  return __shfl_sync(FULL, j, 0);
}

#ifndef ALORE_OPT_MINBLOCKS
#define ALORE_OPT_MINBLOCKS 8
#endif
#ifdef ALORE_CAND_TIMING   // developer build: wall time of every candidate inside the persistent kernel (scripts/cand_timing.py)
__device__ unsigned long long g_cand_ns[3 * 16384];
__device__ __forceinline__ unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#endif
__global__ void __launch_bounds__(32, ALORE_OPT_MINBLOCKS)
opt_kernel(const __grid_constant__ KParams kp, BatchDev bt, ResultDev out, double* slabs, double* hists, int* counter) {
  extern __shared__ __align__(16) double smem[];
  double* slab = slabs + (size_t)blockIdx.x * kp.L.total;
  double* hist = hists + (size_t)blockIdx.x * kp.L.hist_total;
  const int lane = threadIdx.x & 31;
#ifdef ALORE_TMA_HISTORY
  {
    Warp w0;
    carve(w0, kp.L, smem, slab, hist, 1, kp.P.sparseResolution);
    lbfgs_tma_init(w0.mbar);
  }
#endif
  for (;;) {
    const int job = next_job(counter, lane);
    if (job >= bt.B) break;
    const int b = bt.order ? bt.order[job] : job;
    const int N = bt.piece_off[b + 1] - bt.piece_off[b];
    Warp w;
    carve(w, kp.L, smem, slab, hist, N, kp.P.sparseResolution);
#ifdef ALORE_CAND_TIMING
    const unsigned long long t0 = gtimer();
#endif
    minco_plan(w, kp, bt, b, out);
#ifdef ALORE_CAND_TIMING
    if (lane == 0 && b < 16384) {
      unsigned smid;
      asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
      g_cand_ns[3 * b] = t0; g_cand_ns[3 * b + 1] = gtimer(); g_cand_ns[3 * b + 2] = smid;
    }
#endif
  }
}

// One cost evaluation per candidate at a caller-supplied x (parity tests / config-3-style timing in x space).
__global__ void __launch_bounds__(32)
cost_kernel(const __grid_constant__ KParams kp, BatchDev bt, int stage, const double* xs, const double* lam, const double* rho,
            const double* safe_dis, double* cost, double* gs, double* err, double* slabs, int* counter) {
  extern __shared__ __align__(16) double smem[];
  double* slab = slabs + (size_t)blockIdx.x * kp.L.total;
  const int lane = threadIdx.x & 31;
  for (;;) {
    const int b = next_job(counter, lane);
    if (b >= bt.B) break;
    const int p0 = bt.piece_off[b];
    const int N = bt.piece_off[b + 1] - p0;
    Warp w;
    carve(w, kp.L, smem, slab, slab, N, kp.P.sparseResolution);
    load_candidate(w, bt, b, p0);
    for (int d = 0; d < 2; d++) {
      w.lam[d] = lam ? lam[2 * b + d] : kp.P.EqualLambda[d];
      w.rho[d] = rho ? rho[2 * b + d] : kp.P.EqualRho[d];
    }
    w.safeDis = safe_dis ? safe_dis[b] : kp.P.safeDis;
    w.time_weight = kp.P.pw_time;
    const size_t xo = 3 * (size_t)p0 - b;
    for (int i = lane; i < w.n; i += 32) { w.x[i] = xs[xo + i]; w.g[i] = gs[xo + i]; }
    __syncwarp();
    const double f = cost_eval(w, kp.P, kp.map, stage, w.x, w.g);
    for (int i = lane; i < w.n; i += 32) gs[xo + i] = w.g[i];
    if (lane == 0) {
      cost[b] = f;
      if (err) { err[2 * b] = w.err[0]; err[2 * b + 1] = w.err[1]; }
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(32)
collision_kernel(const __grid_constant__ KParams kp, int B, const int* piece_off, const double* coeffs, const double* Ts,
                 const double* start_xy, int* collided, double* min_dist, double* slabs, int* counter) {
  extern __shared__ __align__(16) double smem[];
  double* slab = slabs + (size_t)blockIdx.x * kp.L.total;
  const int lane = threadIdx.x & 31;
  for (;;) {
    const int b = next_job(counter, lane);
    if (b >= B) break;
    const int p0 = piece_off[b];
    const int N = piece_off[b + 1] - p0;
    Warp w;
    carve(w, kp.L, smem, slab, slab, N, kp.P.sparseResolution);
    w.sx = start_xy[2 * b]; w.sy = start_xy[2 * b + 1];
    const double* c = coeffs + 12 * (size_t)p0;
    for (int i = lane; i < 12 * N; i += 32) w.cf[i] = c[i];
    for (int i = lane; i < N; i += 32) w.T1[i] = Ts[p0 + i];
    __syncwarp();
    double md;
    const int hit = final_collision(w, kp.P, kp.map, &md);
    if (lane == 0) { collided[b] = hit; if (min_dist) min_dist[b] = md; }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------
// coefficient-space penalty kernel (alore_penalty_batch[_dev]): one 64-thread CTA per trajectory
// ---------------------------------------------------------------------------------------------
// scratch of the penalty passes (per resident CTA, stays in L2)
struct PenLayout {
  size_t cs, ax, ay, cellP, g2p, terms, nterm, rank, cg, fold, total;
  int TS;
  __host__ __device__ void init(int Nmax, int K, int KF, int ncp) {
    const int Kbig = K > KF ? K : KF;
    const size_t Smax = (size_t)Nmax * (2 * Kbig + 1);
    size_t o = 0;
    auto take = [&](size_t cnt) { size_t r = o; o += (cnt + 3) & ~size_t(3); return r; };
    cs = take(2 * Smax); ax = take(Smax + 64); ay = take(Smax + 64);
    cellP = take(2 * (size_t)Nmax * Kbig); g2p = take(2 * (size_t)Nmax * (Kbig + 1));
    TS = (K + 1) * (7 + ncp) + 1;
    terms = take((size_t)Nmax * TS); nterm = take(Nmax); rank = take((size_t)Nmax * (K + 1) + 32);
    cg = take(2 * (size_t)Nmax * (K + 1)); fold = take(2 * (size_t)Nmax * (K + 1));
    total = o;
  }
};

struct PenParams {
  alore_params_t P;
  MapDev map;
  PenLayout L;
  int Nmax;
};

constexpr int PEN_NT = 64;   // threads per trajectory
inline size_t pen_smem_doubles(int Nmax) {
  // T1[N] gT[N] pXY[2(N+1)] bcast[4] | stg[1024] (cell-prefix chunks 2 x 256, cost-term packing 512)
  return (size_t)Nmax + Nmax + 2 * (Nmax + 1) + 4 + 2 + 1024;
}
__device__ __forceinline__ void pen_carve(Warp& w, const PenLayout& L, double* smem, double* slab, int Nmax, int N, int K) {
  w.lane = threadIdx.x;
  w.N = N; w.n = 3 * N - 1; w.npad = (3 * N) & ~1; w.n6 = 6 * N; w.K = K; w.S1 = 2 * K + 1;
  double* s = smem;
  w.T1 = s; s += Nmax; w.gT = s; s += Nmax; w.pXY = s; s += 2 * (Nmax + 1); w.sumT = s; s += 4;
  s = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(s) + 15) & ~uintptr_t(15));
  w.stg = s;
  w.Nm = Nmax;
  w.cs = slab + L.cs; w.ax = slab + L.ax; w.ay = slab + L.ay; w.cellP = slab + L.cellP; w.g2p = slab + L.g2p;
  w.terms = slab + L.terms; w.cg = slab + L.cg; w.fold = slab + L.fold;
  w.nterm = reinterpret_cast<int*>(slab + L.nterm); w.rank = reinterpret_cast<int*>(slab + L.rank);
  w.TS = L.TS;
  w.err[0] = w.err[1] = 0.0;
}

// attachPenaltyFunctional on given coefficients (BASELINE configs[2]), one CTA per trajectory, reading the caller's
// coefficient / duration arrays and accumulating straight into the caller's gradient arrays.
__global__ void __launch_bounds__(PEN_NT, 6)
penalty_cta_kernel(const __grid_constant__ PenParams kp, int B, const int* piece_off, const double* coeffs, const double* Ts,
                   const double* start_xy, const double* final_xy, double* cost, double* gradC, double* gradT, double* err, double* slabs) {
  extern __shared__ __align__(16) double smem[];
  double* slab = slabs + (size_t)blockIdx.x * kp.L.total;
  const int tid = threadIdx.x;
#pragma unroll 1
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int p0 = piece_off[b], N = piece_off[b + 1] - p0;
    if (N < 1 || N > kp.Nmax) {                               // more pieces than the caller declared: refuse, loudly (NaN), never overrun
      if (tid == 0) { cost[b] = __longlong_as_double(0x7ff8000000000000ll); err[2 * b] = err[2 * b + 1] = 0.0; }
      continue;
    }
    Warp w;
    pen_carve(w, kp.L, smem, slab, kp.Nmax, N, kp.P.sparseResolution);
    w.cf = const_cast<double*>(coeffs) + 12 * (size_t)p0;
    w.gC = gradC + 12 * (size_t)p0;
    w.sx = start_xy[2 * b]; w.sy = start_xy[2 * b + 1];
    w.fx = final_xy[2 * b]; w.fy = final_xy[2 * b + 1];
    for (int d = 0; d < 2; d++) { w.lam[d] = kp.P.EqualLambda[d]; w.rho[d] = kp.P.EqualRho[d]; }
    w.safeDis = kp.P.safeDis;
    w.init_pos = nullptr;
    tsync<PEN_NT>();
    for (int i = tid; i < 12 * N; i += PEN_NT) w.gC[i] = 0.0;
    for (int i = tid; i < N; i += PEN_NT) { w.T1[i] = Ts[p0 + i]; w.gT[i] = 0.0; }
    tsync<PEN_NT>();
    const double f = penalty_passes_t<PEN_NT>(w, kp.P, kp.map, 1, 0.0);
    for (int i = tid; i < N; i += PEN_NT) gradT[p0 + i] = w.gT[i];
    if (tid == 0) { cost[b] = f; err[2 * b] = w.err[0]; err[2 * b + 1] = w.err[1]; }
  }
}

// Lowest final cost among candidates with ok == 1 (ties -> lowest index).  One CTA.
__global__ void argmin_kernel(int B, const double* cost, const int* ok, double* best_cost, int* best_idx) {
  __shared__ double sc[256];
  __shared__ int si[256];
  double bc = DBL_MAX;
  int bi = -1;
  for (int i = threadIdx.x; i < B; i += blockDim.x)
    if (ok[i] && (cost[i] < bc || (cost[i] == bc && i < bi))) { bc = cost[i]; bi = i; }
  sc[threadIdx.x] = bc; si[threadIdx.x] = bi;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      const double c2 = sc[threadIdx.x + o];
      const int i2 = si[threadIdx.x + o];
      if (i2 >= 0 && (si[threadIdx.x] < 0 || c2 < sc[threadIdx.x] || (c2 == sc[threadIdx.x] && i2 < si[threadIdx.x]))) {
        sc[threadIdx.x] = c2; si[threadIdx.x] = i2;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { *best_cost = sc[0]; *best_idx = si[0]; }
}

// Self-test of the division split (traj_opt.cuh: rcp_refine / div_rcp) against the compiler's own a / b.
// Operand pairs come from a counter-based generator: mode 0 = raw 64-bit patterns (every exponent, NaN/Inf/subnormal
// included), mode 1 = magnitudes 2^-40 .. 2^40 (what the banded solves see), mode 2 = near-equal mantissas.
__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}
__global__ void division_selftest_kernel(long long n, unsigned long long seed, unsigned long long* mismatches) {
  unsigned long long bad = 0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const unsigned long long ra = mix64(seed + 2 * (unsigned long long)i), rb = mix64(seed + 2 * (unsigned long long)i + 1);
    double a, b;
    const int mode = (int)(i % 3);
    if (mode == 0) {
      a = __longlong_as_double((long long)ra);
      b = __longlong_as_double((long long)rb);
    } else {
      const unsigned long long ma = ra & 0x000fffffffffffffull, mb = mode == 2 ? (ma ^ (rb & 0xffull)) : (rb & 0x000fffffffffffffull);
      const unsigned long long ea = 1023 - 40 + ((ra >> 52) % 81), eb = 1023 - 40 + ((rb >> 52) % 81);
      a = __longlong_as_double((long long)(((ra >> 63) << 63) | (ea << 52) | ma));
      b = __longlong_as_double((long long)(((rb >> 63) << 63) | (eb << 52) | mb));
    }
    const double q_ref = a / b;
    const double q = div_rcp(a, b, rcp_refine(b));
    const bool same = __double_as_longlong(q) == __double_as_longlong(q_ref) || (q != q && q_ref != q_ref);
    if (!same) bad++;
  }
  if (bad) atomicAdd(mismatches, bad);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct Launch {
  KParams kp;
  int slots = 0;
  size_t smem = 0;
  double* slabs = nullptr;
  double* hists = nullptr;
  int* counter = nullptr;
};

int validate_opt_params(alore_ctx* ctx, const alore_params_t* prm) {
  if (prm->sparseResolution < 1 || prm->sparseResolution > 64) return alore_fail(ctx, ALORE_EINVAL, "sparseResolution out of range");
  if (prm->finalSafeDisCheckNum < 1 || prm->finalSafeDisCheckNum > 64) return alore_fail(ctx, ALORE_EINVAL, "finalSafeDisCheckNum out of range");
  if (prm->n_checkpoints < 0 || prm->n_checkpoints > ALORE_MAX_CHECKPOINTS) return alore_fail(ctx, ALORE_EINVAL, "n_checkpoints out of range");
  // the past-cost ring of lbfgs_optimize (lbfgs.hpp:511) is carved as 64 doubles per candidate
  for (int past : {prm->lbfgs.past, prm->path_lbfgs.past, prm->normal_past, prm->shot_path_past})
    if (past < 0 || past > 64) return alore_fail(ctx, ALORE_EINVAL, "lbfgs `past` must be in [0, 64]");
  if (prm->safeReplanMaxTime < 1) return alore_fail(ctx, ALORE_EINVAL, "safeReplanMaxTime must be >= 1");
  return ALORE_OK;
}

template <typename Kern>
int prepare_launch(alore_ctx* ctx, const alore_params_t* prm, int Nmax, int B, Kern kern, Launch& L, bool need_history) {
  if (!ctx->have_map || !ctx->d_dist) return alore_fail(ctx, ALORE_ENOMAP, "no ESDF resident on the device: call alore_esdf_update / alore_esdf_set first");
  {
    const int vrc = validate_opt_params(ctx, prm);
    if (vrc) return vrc;
  }
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  L.kp.P = *prm;
  const alore_map_geom_t& g = ctx->geom;
  L.kp.map = MapDev{ctx->d_dist, g.glx, g.gly, g.x_lower, g.y_lower, g.x_upper, g.y_upper, g.grid_interval, g.inv_grid_interval};
  const int mcap = need_history ? std::max(prm->path_lbfgs.mem_size, prm->lbfgs.mem_size) : 1;
  L.kp.mcap = std::max(1, mcap);
  L.kp.L.init(Nmax, L.kp.mcap, prm->sparseResolution, prm->finalSafeDisCheckNum, prm->n_checkpoints);
  L.smem = smem_doubles(Nmax) * sizeof(double);
  if (L.smem > 200 * 1024) return alore_fail(ctx, ALORE_EINVAL, "trajectory with %d pieces exceeds the shared-memory budget", Nmax);
  ALORE_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem));
  int per_sm = 0;
  ALORE_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32, L.smem));
  if (per_sm < 1) return alore_fail(ctx, ALORE_EINVAL, "kernel does not fit on an SM");
  if (const char* e = getenv("ALORE_OPT_WARPS_PER_SM")) {   // tuning knob: resident candidate warps per SM (default: occupancy limit)
    const int v = atoi(e);
    if (v >= 1) per_sm = std::min(per_sm, v);
  }
  L.slots = std::max(1, std::min(B, per_sm * ctx->sm_count));
  const size_t need = (size_t)L.slots * L.kp.L.total * sizeof(double) + 256;
  if (need > ctx->opt_scratch_bytes) {
    if (ctx->opt_scratch) cudaFree(ctx->opt_scratch);
    ctx->opt_scratch = nullptr; ctx->opt_scratch_bytes = 0;
    ALORE_CUDA(ctx, cudaMalloc(&ctx->opt_scratch, need));
    ctx->opt_scratch_bytes = need;
  }
  L.counter = reinterpret_cast<int*>(ctx->opt_scratch);
  L.slabs = reinterpret_cast<double*>(reinterpret_cast<char*>(ctx->opt_scratch) + 256);
  if (need_history) {
    const size_t hneed = (size_t)L.slots * L.kp.L.hist_total * sizeof(double);
    if (hneed > ctx->opt_hist_bytes) {
      if (ctx->opt_hist) cudaFree(ctx->opt_hist);
      ctx->opt_hist = nullptr; ctx->opt_hist_bytes = 0;
      ALORE_CUDA(ctx, cudaMalloc(&ctx->opt_hist, hneed));
      ctx->opt_hist_bytes = hneed;
    }
    L.hists = reinterpret_cast<double*>(ctx->opt_hist);
  }
  return ALORE_OK;
}

// Ask L2 to keep the per-warp evaluation scratch (factors, coefficients, sin/cos, ...) resident while the L-BFGS
// history — touched once per iteration, ~1 MB per warp — streams through (it would otherwise evict the scratch).
void set_l2_window(alore_ctx* ctx, cudaStream_t st, void* base, size_t bytes) {
  if (ctx->l2_max_persist < 0) {                 // limits of THIS context's device
    cudaDeviceGetAttribute(&ctx->l2_max_persist, cudaDevAttrMaxPersistingL2CacheSize, ctx->device);
    cudaDeviceGetAttribute(&ctx->l2_max_window, cudaDevAttrMaxAccessPolicyWindowSize, ctx->device);
    if (ctx->l2_max_persist > 0) cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)ctx->l2_max_persist);
  }
  if (ctx->l2_max_persist <= 0 || ctx->l2_max_window <= 0) return;
  if (getenv("ALORE_NO_L2_WINDOW")) return;   // tuning knob
  cudaStreamAttrValue v{};
  v.accessPolicyWindow.base_ptr = base;
  v.accessPolicyWindow.num_bytes = std::min(bytes, (size_t)ctx->l2_max_window);
  v.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)ctx->l2_max_persist / (double)std::max<size_t>(v.accessPolicyWindow.num_bytes, 1));
  v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
  v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  if (cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess) (void)cudaGetLastError();
}
// the caller's stream (e.g. torch's) must not keep our window after the launch that wanted it
void clear_l2_window(cudaStream_t st) {
  cudaStreamAttrValue v{};
  v.accessPolicyWindow.num_bytes = 0;
  if (cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess) (void)cudaGetLastError();
}

template <typename T>
int dev_copy(alore_ctx* ctx, T** dst, const T* src, size_t n, cudaStream_t st, char** arena_cur = nullptr, char* arena_end = nullptr) {
  *dst = nullptr;
  const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
  if (arena_cur && *arena_cur) {
    const size_t need = (bytes + 255) & ~size_t(255);
    if (*arena_cur + need > arena_end) return alore_fail(ctx, ALORE_ECUDA, "batch arena exhausted");
    *dst = reinterpret_cast<T*>(*arena_cur);
    *arena_cur += need;
  } else {
    ALORE_CUDA(ctx, cudaMalloc(dst, bytes));
  }
  if (n && src) ALORE_CUDA(ctx, cudaMemcpyAsync(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice, st));
  return ALORE_OK;
}

int max_pieces(const int32_t* po, int B) {
  int m = 0;
  for (int b = 0; b < B; b++) m = std::max(m, po[b + 1] - po[b]);
  return m;
}

}  // namespace

static void lpt_order(const std::vector<int32_t>& po, const int32_t* evals, std::vector<int>& order);
struct alore_batch {
  alore_ctx* ctx = nullptr;
  int B = 0, tot = 0, Nmax = 0;
  BatchDev bt{};
  ResultDev res{};
  std::vector<void*> allocs;
  float kernel_ms = 0.f;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  double* d_best = nullptr;
  int* d_best_idx = nullptr;
  std::vector<int32_t> piece_off;   // host copy (scheduling)
  int* d_order = nullptr;
  int runs = 0;
  bool predicted = false;           // d_order currently holds a predicted (not piece-count) order
  bool pooled = false;              // device arrays carved from ctx->batch_pool
  char* pool_cur = nullptr;
  char* pool_end = nullptr;
};

// Longest-processing-time-first order.  Work estimate of a candidate = pieces x cost evaluations of the previous
// optimisation of the same batch structure when known (replanning re-optimises nearly the same candidates every
// tick), else pieces alone.  Only the hand-out order of the work queue changes, never a result.
static void lpt_order(const std::vector<int32_t>& po, const int32_t* evals, std::vector<int>& order) {
  const int B = (int)po.size() - 1;
  order.resize(B);
  std::iota(order.begin(), order.end(), 0);
  std::vector<long long> key(B);
  for (int b = 0; b < B; b++) key[b] = (long long)(po[b + 1] - po[b]) * (evals ? std::max(1, evals[b]) : 1);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return key[a] > key[b]; });
}
// Evaluation counts to predict from, for a batch with piece offsets `po`: the previous tick's counts where the previous
// batch had the same number of candidates and (for at least 3 in 4 of them) the same piece count at the same index —
// a replanning planner re-optimises mostly the same legs; candidates whose piece count changed get the mean count.
// Returns false (piece counts only) when the previous batch does not look like this one.
static bool predicted_evals(const alore_ctx* ctx, const std::vector<int32_t>& po, std::vector<int32_t>& pred) {
  const int B = (int)po.size() - 1;
  if ((int)ctx->sched_evals.size() != B || (int)ctx->sched_piece_off.size() != B + 1) return false;
  long long same = 0, sum = 0;
  for (int b = 0; b < B; b++) {
    same += (po[b + 1] - po[b]) == (ctx->sched_piece_off[b + 1] - ctx->sched_piece_off[b]);
    sum += ctx->sched_evals[b];
  }
  if (4 * same < 3LL * B) return false;
  const int32_t mean = (int32_t)std::max<long long>(1, sum / B);
  pred.resize(B);
  for (int b = 0; b < B; b++)
    pred[b] = (po[b + 1] - po[b]) == (ctx->sched_piece_off[b + 1] - ctx->sched_piece_off[b]) ? ctx->sched_evals[b] : mean;
  return true;
}

static int validate_cands(alore_ctx* ctx, const alore_candidates_t* c) {
  if (!c || c->B <= 0 || !c->piece_off) return alore_fail(ctx, ALORE_EINVAL, "empty candidate batch");
  if (c->piece_off[0] != 0) return alore_fail(ctx, ALORE_EINVAL, "piece_off[0] must be 0");
  for (int b = 0; b < c->B; b++)
    if (c->piece_off[b + 1] - c->piece_off[b] < 1) return alore_fail(ctx, ALORE_EINVAL, "candidate %d has no piece", b);
  return ALORE_OK;
}

extern "C" {

int alore_debug_force_exact_division(alore_ctx* ctx, int on) {
  if (!ctx) return ALORE_EINVAL;
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  ALORE_CUDA(ctx, cudaDeviceSynchronize());
  const int v = on ? 1 : 0;
  ALORE_CUDA(ctx, cudaMemcpyToSymbol(g_force_exact_div, &v, sizeof(int)));
  return ALORE_OK;
}

int alore_debug_set_norm_guard(alore_ctx* ctx, double threshold) {
  if (!ctx) return ALORE_EINVAL;
  if (!(threshold > 0.0 && threshold <= 1e4)) return alore_fail(ctx, ALORE_EINVAL, "norm guard %g outside (0, 1e4]", threshold);
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  ALORE_CUDA(ctx, cudaDeviceSynchronize());
  ALORE_CUDA(ctx, cudaMemcpyToSymbol(g_norm_guard, &threshold, sizeof(double)));
  return ALORE_OK;
}

int alore_debug_phase_cycles(alore_ctx* ctx, unsigned long long* out32, int reset) {
  if (!ctx || !out32) return ALORE_EINVAL;
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  ALORE_CUDA(ctx, cudaDeviceSynchronize());
#ifdef ALORE_PHASE_TIMING
  ALORE_CUDA(ctx, cudaMemcpyFromSymbol(out32, g_phase_cycles, 32 * sizeof(unsigned long long)));
  if (reset) { unsigned long long z[32] = {0}; ALORE_CUDA(ctx, cudaMemcpyToSymbol(g_phase_cycles, z, sizeof(z))); }
  return ALORE_OK;
#else
  (void)reset;
  std::memset(out32, 0, 32 * sizeof(unsigned long long));
  return alore_fail(ctx, ALORE_EINVAL, "library built without -DALORE_PHASE_TIMING");
#endif
}

int alore_selftest_division(alore_ctx* ctx, long long n_pairs, unsigned long long seed, long long* mismatches) {
  if (!ctx || !mismatches || n_pairs <= 0) return ALORE_EINVAL;
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  unsigned long long* d = nullptr;
  ALORE_CUDA(ctx, cudaMalloc(&d, sizeof(unsigned long long)));
  cudaMemsetAsync(d, 0, sizeof(unsigned long long), ctx->stream);
  division_selftest_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(n_pairs, seed, d);
  ctx->launches++;
  unsigned long long h = 0;
  cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream);
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (e == cudaSuccess) e = cudaGetLastError();
  cudaFree(d);
  if (e != cudaSuccess) return alore_fail(ctx, ALORE_ECUDA, "division self-test: %s", cudaGetErrorString(e));
  *mismatches = (long long)h;
  return ALORE_OK;
}

static int batch_upload_impl(alore_ctx* ctx, const alore_candidates_t* c, alore_batch** out, bool use_arena) {
  if (!ctx || !out) return ALORE_EINVAL;
  *out = nullptr;
  int rc = validate_cands(ctx, c);
  if (rc) return rc;
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  alore_batch* bh = new alore_batch();
  bh->ctx = ctx;
  const int B = c->B, tot = c->piece_off[B];
  bh->B = B; bh->tot = tot; bh->Nmax = max_pieces(c->piece_off, B);
  cudaStream_t st = ctx->stream;
  bh->piece_off.assign(c->piece_off, c->piece_off + B + 1);
  std::vector<int> order;
  lpt_order(bh->piece_off, nullptr, order);            // piece-count order; alore_batch_run refines it from the previous tick
  int* d_po; int* d_order; double *d_ip, *d_T, *d_pos, *d_ss, *d_fs, *d_sx, *d_fx; unsigned char* d_cut;
  if (use_arena && !ctx->batch_pool_busy) {   // one-shot calls carve every device array from the context's arena
    const size_t need = 8 * (48 * (size_t)B + 40 * (size_t)tot) + 64 * 1024;
    if (need > ctx->batch_pool_bytes) {
      if (ctx->batch_pool) { cudaDeviceSynchronize(); cudaFree(ctx->batch_pool); }
      ctx->batch_pool = nullptr; ctx->batch_pool_bytes = 0;
      if (cudaMalloc(&ctx->batch_pool, need) == cudaSuccess) ctx->batch_pool_bytes = need;
      else (void)cudaGetLastError();
    }
    if (ctx->batch_pool) {
      ctx->batch_pool_busy = true;
      bh->pooled = true;
      bh->pool_cur = static_cast<char*>(ctx->batch_pool);
      bh->pool_end = bh->pool_cur + ctx->batch_pool_bytes;
    }
  }
#define UP(dst, src, n)                                  \
  rc = dev_copy(ctx, &dst, src, (size_t)(n), st, bh->pooled ? &bh->pool_cur : nullptr, bh->pool_end); \
  if (rc) { alore_batch_free(bh); return rc; }           \
  if (!bh->pooled) bh->allocs.push_back(dst);
  UP(d_po, c->piece_off, B + 1)
  UP(d_order, order.data(), B)
  UP(d_ip, c->inner_pts, 2 * (size_t)(tot - B))
  UP(d_T, c->init_T, B)
  UP(d_pos, c->inner_init_pos, 3 * (size_t)tot)
  UP(d_ss, c->start_state, 6 * (size_t)B)
  UP(d_fs, c->final_state, 6 * (size_t)B)
  UP(d_sx, c->start_xytheta, 3 * (size_t)B)
  UP(d_fx, c->final_xytheta, 3 * (size_t)B)
  UP(d_cut, c->if_cut, B)
  bh->bt = BatchDev{B, d_po, d_ip, d_T, d_pos, d_ss, d_fs, d_sx, d_fx, d_cut, d_order};
  bh->d_order = d_order;
  ResultDev& r = bh->res;
  const int* nul_i = nullptr; const double* nul_d = nullptr;
  UP(r.ok, nul_i, B) UP(r.status, nul_i, B) UP(r.replans, nul_i, B) UP(r.alm_iters, nul_i, B) UP(r.evals, nul_i, B)
  UP(r.cost, nul_d, B) UP(r.inner_pts, nul_d, 2 * (size_t)(tot - B)) UP(r.tail_s, nul_d, B) UP(r.piece_T, nul_d, tot)
  UP(r.coeffs, nul_d, 12 * (size_t)tot)
  UP(r.alg_bytes, nul_d, B) UP(r.iters, nul_i, B)
  UP(bh->d_best, nul_d, 1) UP(bh->d_best_idx, nul_i, 1)
#undef UP
  cudaEventCreate(&bh->e0);
  cudaEventCreate(&bh->e1);
  ALORE_CUDA(ctx, cudaStreamSynchronize(st));  // `order` is a host temporary
  *out = bh;
  return ALORE_OK;
}

int alore_batch_upload(alore_ctx* ctx, const alore_candidates_t* c, alore_batch** out) { return batch_upload_impl(ctx, c, out, false); }

int alore_batch_run(alore_ctx* ctx, const alore_params_t* prm, alore_batch* bh, void* cuda_stream) {
  if (!ctx || !prm || !bh) return ALORE_EINVAL;
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
  Launch L;
  int rc = prepare_launch(ctx, prm, bh->Nmax, bh->B, opt_kernel, L, true);
  if (rc) return rc;
  // Hand-out order of the work queue: longest predicted work first.  Prediction = pieces x cost evaluations the
  // candidate at the same index needed on the PREVIOUS tick (this handle's last run, or the last run of any handle
  // on this context with the same structure: a replanning planner re-optimises mostly the same legs), else pieces.
  if (ctx->last_batch) {                            // collect the previous tick's evaluation counts (it has finished: same-context ordering)
    alore_batch* pb = static_cast<alore_batch*>(ctx->last_batch);
    ALORE_CUDA(ctx, cudaEventSynchronize(pb->e1));   // that run may have been enqueued on another stream
    std::vector<int32_t> ev(pb->B);
    ALORE_CUDA(ctx, cudaMemcpyAsync(ev.data(), pb->res.evals, pb->B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    ALORE_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->sched_piece_off = pb->piece_off;
    ctx->sched_evals.swap(ev);
    ctx->last_batch = nullptr;
  }
  {
    std::vector<int32_t> pred;
    if (!getenv("ALORE_NO_SCHED_PREDICTION") && predicted_evals(ctx, bh->piece_off, pred)) {
      std::vector<int> order;
      lpt_order(bh->piece_off, pred.data(), order);
      ALORE_CUDA(ctx, cudaMemcpyAsync(bh->d_order, order.data(), bh->B * sizeof(int), cudaMemcpyHostToDevice, st));
      ALORE_CUDA(ctx, cudaStreamSynchronize(st));
      bh->predicted = true;
    } else if (bh->predicted) {                     // back to the piece-count order
      std::vector<int> order;
      lpt_order(bh->piece_off, nullptr, order);
      ALORE_CUDA(ctx, cudaMemcpyAsync(bh->d_order, order.data(), bh->B * sizeof(int), cudaMemcpyHostToDevice, st));
      ALORE_CUDA(ctx, cudaStreamSynchronize(st));
      bh->predicted = false;
    }
  }
  bh->runs++;
  ALORE_CUDA(ctx, cudaMemsetAsync(L.counter, 0, sizeof(int), st));
  ALORE_CUDA(ctx, cudaEventRecord(bh->e0, st));
  set_l2_window(ctx, st, L.slabs, (size_t)L.slots * L.kp.L.total * sizeof(double));
  opt_kernel<<<L.slots, 32, L.smem, st>>>(L.kp, bh->bt, bh->res, L.slabs, L.hists, L.counter);
  ctx->launches++;
  clear_l2_window(st);
  ALORE_CUDA(ctx, cudaGetLastError());
  ALORE_CUDA(ctx, cudaEventRecord(bh->e1, st));
  ctx->last_batch = bh;
#ifdef ALORE_CAND_TIMING
  if (const char* f = getenv("ALORE_CAND_TIMING_DUMP")) {
    cudaDeviceSynchronize();
    std::vector<unsigned long long> h(3 * 16384);
    cudaMemcpyFromSymbol(h.data(), g_cand_ns, h.size() * sizeof(unsigned long long));
    if (FILE* fp = fopen(f, "wb")) { fwrite(h.data(), sizeof(unsigned long long), h.size(), fp); fclose(fp); }
  }
#endif
  return ALORE_OK;
}

int alore_batch_download(alore_ctx* ctx, alore_batch* bh, alore_results_t* out) {
  if (!ctx || !bh || !out) return ALORE_EINVAL;
  cudaStream_t st = ctx->stream;
  ALORE_CUDA(ctx, cudaDeviceSynchronize());
  const int B = bh->B, tot = bh->tot;
  const ResultDev& r = bh->res;
#define DN(dst, src, n) \
  if (dst && (n)) ALORE_CUDA(ctx, cudaMemcpyAsync(dst, src, (size_t)(n) * sizeof(*dst), cudaMemcpyDeviceToHost, st));
  DN(out->ok, r.ok, B) DN(out->status, r.status, B) DN(out->replans, r.replans, B) DN(out->alm_iters, r.alm_iters, B)
  DN(out->evals, r.evals, B) DN(out->cost, r.cost, B) DN(out->inner_pts, r.inner_pts, 2 * (size_t)(tot - B))
  DN(out->tail_s, r.tail_s, B) DN(out->piece_T, r.piece_T, tot) DN(out->coeffs, r.coeffs, 12 * (size_t)tot)
#undef DN
  ALORE_CUDA(ctx, cudaStreamSynchronize(st));
  cudaEventElapsedTime(&bh->kernel_ms, bh->e0, bh->e1);
  (void)cudaGetLastError();
  return ALORE_OK;
}

int alore_batch_device_results(alore_batch* bh, const double** d_cost, const int32_t** d_ok) {
  if (!bh) return ALORE_EINVAL;
  if (d_cost) *d_cost = bh->res.cost;
  if (d_ok) *d_ok = bh->res.ok;
  return ALORE_OK;
}

int alore_batch_argmin(alore_ctx* ctx, alore_batch* bh, double* best_cost, int32_t* best_idx) {
  if (!ctx || !bh) return ALORE_EINVAL;
  cudaStream_t st = ctx->stream;
  ALORE_CUDA(ctx, cudaDeviceSynchronize());
  argmin_kernel<<<1, 256, 0, st>>>(bh->B, bh->res.cost, bh->res.ok, bh->d_best, bh->d_best_idx);
  ctx->launches++;
  double bc; int bi;
  ALORE_CUDA(ctx, cudaMemcpyAsync(&bc, bh->d_best, sizeof(double), cudaMemcpyDeviceToHost, st));
  ALORE_CUDA(ctx, cudaMemcpyAsync(&bi, bh->d_best_idx, sizeof(int), cudaMemcpyDeviceToHost, st));
  ALORE_CUDA(ctx, cudaStreamSynchronize(st));
  if (best_cost) *best_cost = bc;
  if (best_idx) *best_idx = bi;
  return ALORE_OK;
}

int alore_batch_stats(alore_ctx* ctx, alore_batch* bh, double* alg_bytes, long long* evals, long long* iters) {
  if (!ctx || !bh) return ALORE_EINVAL;
  ALORE_CUDA(ctx, cudaDeviceSynchronize());
  std::vector<double> hb(bh->B);
  std::vector<int> hi(bh->B), he(bh->B);
  ALORE_CUDA(ctx, cudaMemcpy(hb.data(), bh->res.alg_bytes, bh->B * sizeof(double), cudaMemcpyDeviceToHost));
  ALORE_CUDA(ctx, cudaMemcpy(hi.data(), bh->res.iters, bh->B * sizeof(int), cudaMemcpyDeviceToHost));
  ALORE_CUDA(ctx, cudaMemcpy(he.data(), bh->res.evals, bh->B * sizeof(int), cudaMemcpyDeviceToHost));
  double sb = 0.0;
  long long si = 0, se = 0;
  for (int b = 0; b < bh->B; b++) { sb += hb[b]; si += hi[b]; se += he[b]; }
  if (alg_bytes) *alg_bytes = sb;
  if (iters) *iters = si;
  if (evals) *evals = se;
  return ALORE_OK;
}

int alore_batch_last_kernel_ms(const alore_batch* bh, float* ms) {
  if (!bh || !ms) return ALORE_EINVAL;
  float t = 0.f;
  if (cudaEventElapsedTime(&t, bh->e0, bh->e1) != cudaSuccess) { (void)cudaGetLastError(); t = bh->kernel_ms; }
  *ms = t;
  return ALORE_OK;
}

void alore_batch_free(alore_batch* bh) {
  if (!bh) return;
  if (bh->ctx) cudaSetDevice(bh->ctx->device);
  cudaDeviceSynchronize();
  if (bh->ctx && bh->ctx->last_batch == bh) {        // keep this tick's evaluation counts for the next tick's schedule
    std::vector<int32_t> ev(bh->B);
    if (cudaMemcpy(ev.data(), bh->res.evals, bh->B * sizeof(int32_t), cudaMemcpyDeviceToHost) == cudaSuccess) {
      bh->ctx->sched_piece_off = bh->piece_off;
      bh->ctx->sched_evals.swap(ev);
    } else {
      (void)cudaGetLastError();
    }
    bh->ctx->last_batch = nullptr;
  }
  for (void* p : bh->allocs) cudaFree(p);
  if (bh->pooled && bh->ctx) bh->ctx->batch_pool_busy = false;
  if (bh->e0) cudaEventDestroy(bh->e0);
  if (bh->e1) cudaEventDestroy(bh->e1);
  delete bh;
}

int alore_opt_batch(alore_ctx* ctx, const alore_params_t* prm, const alore_candidates_t* cands, alore_results_t* out) {
  if (!ctx || !prm || !out) return ALORE_EINVAL;
  alore_batch* bh = nullptr;
  int rc = batch_upload_impl(ctx, cands, &bh, true);
  if (rc) return rc;
  rc = alore_batch_run(ctx, prm, bh, nullptr);
  if (rc == ALORE_OK) rc = alore_batch_download(ctx, bh, out);
  alore_batch_free(bh);
  return rc;
}

int alore_cost_batch(alore_ctx* ctx, const alore_params_t* prm, const alore_candidates_t* cands, int stage, const double* x,
                     const double* lambda, const double* rho, const double* safe_dis, double* cost, double* g, double* xy_err) {
  if (!ctx || !prm || !x || !cost || !g) return ALORE_EINVAL;
  if (stage != 0 && stage != 1) return alore_fail(ctx, ALORE_EINVAL, "stage must be 0 (path) or 1");
  alore_batch* bh = nullptr;
  int rc = batch_upload_impl(ctx, cands, &bh, true);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  const int B = bh->B;
  const size_t nv = 3 * (size_t)bh->tot - B;
  double *d_x = nullptr, *d_g = nullptr, *d_lam = nullptr, *d_rho = nullptr, *d_sd = nullptr, *d_cost = nullptr, *d_err = nullptr;
  Launch L;
  auto cleanup = [&]() {
    cudaStreamSynchronize(st);
    for (double* p : {d_x, d_g, d_lam, d_rho, d_sd, d_cost, d_err}) if (p) cudaFree(p);
    alore_batch_free(bh);
  };
#define TRY(e) rc = (e); if (rc) { cleanup(); return rc; }
  TRY(dev_copy(ctx, &d_x, x, nv, st))
  TRY(dev_copy(ctx, &d_g, g, nv, st))     // g is in/out: untouched when ||x|| > 1e4 (the reference's `inf` quirk)
  if (lambda) { TRY(dev_copy(ctx, &d_lam, lambda, 2 * (size_t)B, st)) }
  if (rho) { TRY(dev_copy(ctx, &d_rho, rho, 2 * (size_t)B, st)) }
  if (safe_dis) { TRY(dev_copy(ctx, &d_sd, safe_dis, (size_t)B, st)) }
  TRY(dev_copy(ctx, &d_cost, (const double*)nullptr, (size_t)B, st))
  TRY(dev_copy(ctx, &d_err, (const double*)nullptr, 2 * (size_t)B, st))
  TRY(prepare_launch(ctx, prm, bh->Nmax, B, cost_kernel, L, false))
  cudaMemsetAsync(L.counter, 0, sizeof(int), st);
  cudaMemsetAsync(d_err, 0, 2 * (size_t)B * sizeof(double), st);
  cost_kernel<<<L.slots, 32, L.smem, st>>>(L.kp, bh->bt, stage, d_x, d_lam, d_rho, d_sd, d_cost, d_g, d_err, L.slabs, L.counter);
  ctx->launches++;
  cudaMemcpyAsync(cost, d_cost, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st);
  cudaMemcpyAsync(g, d_g, nv * sizeof(double), cudaMemcpyDeviceToHost, st);
  if (xy_err) cudaMemcpyAsync(xy_err, d_err, 2 * (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st);
  cudaError_t e = cudaStreamSynchronize(st);
  if (e == cudaSuccess) e = cudaGetLastError();
  cleanup();
#undef TRY
  if (e != cudaSuccess) return alore_fail(ctx, ALORE_ECUDA, "cost kernel: %s", cudaGetErrorString(e));
  return ALORE_OK;
}

// shared launcher of the coefficient-space penalty kernel (device pointers)
static int penalty_launch(alore_ctx* ctx, const alore_params_t* prm, int B, int Nmax, const int32_t* d_piece_off, const double* d_coeffs,
                          const double* d_piece_T, const double* d_start_xy, const double* d_final_xy, double* d_cost, double* d_gradC,
                          double* d_gradT, double* d_xy_err, cudaStream_t st) {
  if (!ctx->have_map || !ctx->d_dist) return alore_fail(ctx, ALORE_ENOMAP, "no ESDF resident on the device: call alore_esdf_update / alore_esdf_set first");
  int rc = validate_opt_params(ctx, prm);
  if (rc) return rc;
  if (Nmax < 1) return alore_fail(ctx, ALORE_EINVAL, "max_pieces must be >= 1");
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  PenParams kp;
  kp.P = *prm;
  const alore_map_geom_t& g = ctx->geom;
  kp.map = MapDev{ctx->d_dist, g.glx, g.gly, g.x_lower, g.y_lower, g.x_upper, g.y_upper, g.grid_interval, g.inv_grid_interval};
  kp.L.init(Nmax, prm->sparseResolution, prm->finalSafeDisCheckNum, prm->n_checkpoints);
  kp.Nmax = Nmax;
  // 64 threads per trajectory, as many resident CTAs as fit (6 per SM), the per-sample intermediates in the per-CTA
  // L2-resident slab: chosen by measurement on configs[2] (B200, DESIGN.md section 6): 0.65 ms; 128 threads 0.84, one
  // warp 0.81, shared-memory intermediates 0.77 (8 warps per SM), more CTAs 0.69+, fewer CTAs (5 / 4 / 3 per SM)
  // 0.71 / 0.80 / 0.98, a persisting-L2 window on the slabs 0.70: the 888 slabs of 160 KB exceed L2, but the kernel
  // needs the parallelism more than the hit rate
  const size_t smem = pen_smem_doubles(Nmax) * sizeof(double);
  if (smem > 200 * 1024) return alore_fail(ctx, ALORE_EINVAL, "trajectory with %d pieces exceeds the shared-memory budget", Nmax);
  ALORE_CUDA(ctx, cudaFuncSetAttribute(penalty_cta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  ALORE_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, penalty_cta_kernel, PEN_NT, smem));
  if (occ < 1) return alore_fail(ctx, ALORE_EINVAL, "kernel does not fit on an SM");
  const int grid = std::max(1, std::min(B, occ * ctx->sm_count));
  const size_t need = (size_t)grid * kp.L.total * sizeof(double);
  if (need > ctx->opt_scratch_bytes) {
    if (ctx->opt_scratch) { cudaDeviceSynchronize(); cudaFree(ctx->opt_scratch); }
    ctx->opt_scratch = nullptr; ctx->opt_scratch_bytes = 0;
    ALORE_CUDA(ctx, cudaMalloc(&ctx->opt_scratch, need));
    ctx->opt_scratch_bytes = need;
  }
  penalty_cta_kernel<<<grid, PEN_NT, smem, st>>>(kp, B, d_piece_off, d_coeffs, d_piece_T, d_start_xy, d_final_xy, d_cost, d_gradC,
                                                 d_gradT, d_xy_err, reinterpret_cast<double*>(ctx->opt_scratch));
  ctx->launches++;
  ALORE_CUDA(ctx, cudaGetLastError());
  return ALORE_OK;
}

int alore_penalty_batch_dev(alore_ctx* ctx, const alore_params_t* prm, int B, int max_pieces, const int32_t* d_piece_off,
                            const double* d_coeffs, const double* d_piece_T, const double* d_start_xy, const double* d_final_xy,
                            double* d_cost, double* d_gradC, double* d_gradT, double* d_xy_err, void* cuda_stream) {
  if (!ctx || !prm || B <= 0) return ALORE_EINVAL;
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
  return penalty_launch(ctx, prm, B, max_pieces, d_piece_off, d_coeffs, d_piece_T, d_start_xy, d_final_xy, d_cost, d_gradC, d_gradT,
                        d_xy_err, st);
}

int alore_penalty_batch(alore_ctx* ctx, const alore_params_t* prm, int B, const int32_t* piece_off, const double* coeffs,
                        const double* piece_T, const double* start_xy, const double* final_xy, double* cost, double* gradC,
                        double* gradT, double* xy_err) {
  if (!ctx || !prm || B <= 0 || !piece_off || !coeffs || !piece_T || !start_xy || !final_xy || !cost || !gradC || !gradT || !xy_err)
    return ALORE_EINVAL;
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int tot = piece_off[B];
  const int Nmax = max_pieces(piece_off, B);
  int* d_po = nullptr;
  double *d_c = nullptr, *d_T = nullptr, *d_s = nullptr, *d_f = nullptr, *d_cost = nullptr, *d_gC = nullptr, *d_gT = nullptr, *d_e = nullptr;
  int rc = ALORE_OK;
  auto cleanup = [&]() {
    cudaStreamSynchronize(st);
    if (d_po) cudaFree(d_po);
    for (double* p : {d_c, d_T, d_s, d_f, d_cost, d_gC, d_gT, d_e}) if (p) cudaFree(p);
  };
#define TRY(e) rc = (e); if (rc) { cleanup(); return rc; }
  TRY(dev_copy(ctx, &d_po, piece_off, (size_t)B + 1, st))
  TRY(dev_copy(ctx, &d_c, coeffs, 12 * (size_t)tot, st))
  TRY(dev_copy(ctx, &d_T, piece_T, (size_t)tot, st))
  TRY(dev_copy(ctx, &d_s, start_xy, 2 * (size_t)B, st))
  TRY(dev_copy(ctx, &d_f, final_xy, 2 * (size_t)B, st))
  TRY(dev_copy(ctx, &d_cost, (const double*)nullptr, (size_t)B, st))
  TRY(dev_copy(ctx, &d_gC, (const double*)nullptr, 12 * (size_t)tot, st))
  TRY(dev_copy(ctx, &d_gT, (const double*)nullptr, (size_t)tot, st))
  TRY(dev_copy(ctx, &d_e, (const double*)nullptr, 2 * (size_t)B, st))
  TRY(penalty_launch(ctx, prm, B, Nmax, d_po, d_c, d_T, d_s, d_f, d_cost, d_gC, d_gT, d_e, st))
  cudaMemcpyAsync(cost, d_cost, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st);
  cudaMemcpyAsync(gradC, d_gC, 12 * (size_t)tot * sizeof(double), cudaMemcpyDeviceToHost, st);
  cudaMemcpyAsync(gradT, d_gT, (size_t)tot * sizeof(double), cudaMemcpyDeviceToHost, st);
  cudaMemcpyAsync(xy_err, d_e, 2 * (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st);
  cudaError_t e = cudaStreamSynchronize(st);
  if (e == cudaSuccess) e = cudaGetLastError();
  cleanup();
#undef TRY
  if (e != cudaSuccess) return alore_fail(ctx, ALORE_ECUDA, "penalty kernel: %s", cudaGetErrorString(e));
  return ALORE_OK;
}

int alore_final_collision_batch(alore_ctx* ctx, const alore_params_t* prm, int B, const int32_t* piece_off, const double* coeffs,
                                const double* piece_T, const double* start_xy, int32_t* collided, double* min_dist) {
  if (!ctx || !prm || B <= 0 || !piece_off || !coeffs || !piece_T || !start_xy || !collided) return ALORE_EINVAL;
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int tot = piece_off[B];
  const int Nmax = max_pieces(piece_off, B);
  int *d_po = nullptr, *d_col = nullptr;
  double *d_c = nullptr, *d_T = nullptr, *d_s = nullptr, *d_md = nullptr;
  int rc = ALORE_OK;
  auto cleanup = [&]() {
    cudaStreamSynchronize(st);
    if (d_po) cudaFree(d_po);
    if (d_col) cudaFree(d_col);
    for (double* p : {d_c, d_T, d_s, d_md}) if (p) cudaFree(p);
  };
#define TRY(e) rc = (e); if (rc) { cleanup(); return rc; }
  TRY(dev_copy(ctx, &d_po, piece_off, (size_t)B + 1, st))
  TRY(dev_copy(ctx, &d_col, (const int*)nullptr, (size_t)B, st))
  TRY(dev_copy(ctx, &d_c, coeffs, 12 * (size_t)tot, st))
  TRY(dev_copy(ctx, &d_T, piece_T, (size_t)tot, st))
  TRY(dev_copy(ctx, &d_s, start_xy, 2 * (size_t)B, st))
  TRY(dev_copy(ctx, &d_md, (const double*)nullptr, (size_t)B, st))
  {
    Launch L;
    TRY(prepare_launch(ctx, prm, Nmax, B, collision_kernel, L, false))
    cudaMemsetAsync(L.counter, 0, sizeof(int), st);
    collision_kernel<<<L.slots, 32, L.smem, st>>>(L.kp, B, d_po, d_c, d_T, d_s, d_col, d_md, L.slabs, L.counter);
    ctx->launches++;
  }
  cudaMemcpyAsync(collided, d_col, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st);
  if (min_dist) cudaMemcpyAsync(min_dist, d_md, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st);
  cudaError_t e = cudaStreamSynchronize(st);
  if (e == cudaSuccess) e = cudaGetLastError();
  cleanup();
#undef TRY
  if (e != cudaSuccess) return alore_fail(ctx, ALORE_ECUDA, "collision kernel: %s", cudaGetErrorString(e));
  return ALORE_OK;
}

}  // extern "C"
