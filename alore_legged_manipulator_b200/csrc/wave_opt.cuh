// wave_opt.cuh — the batched trajectory optimizer as a WAVEFRONT of small kernels.
//
// Reference (paths relative to planning_ddr_opt/): the same functions as traj_opt.cuh —
//   back_end/src/optimizer.cpp:169-472 (minco_plan / optimizer), :631-692, 1272-1317 (cost callbacks),
//   back_end/include/gcopter/minco.hpp:99-197, 817-898, 1139-1209 (banded LU, solves, adjoint),
//   back_end/include/gcopter/lbfgs.hpp:276-390, 440-751 (line search, L-BFGS).
//
// Why a wavefront.  One candidate is a long chain of dependent FP64 operations whose phases want very different
// shapes: the banded LU keeps 7 lanes busy, a triangular sweep 2, the penalty functional hundreds, the L-BFGS
// recursion 32.  A persistent warp per candidate (round 1) left 75-95 % of its lanes idle in the sequential phases and
// was limited to 8 warps per SM by its 255 registers.  Here every candidate's optimizer state lives in HBM and one
// ROUND advances every unfinished candidate by exactly one cost evaluation with four kernels, each shaped for its
// phase:
//   solve    8-lane groups, 4 candidates per warp : row generation + LU + forward substitution + back substitution
//   penalty  one CTA (128 threads) per candidate  : energy + attachPenaltyFunctional[Path]
//   adjoint  8-lane groups                         : U^T z = b, L^T x = z
//   step     one warp per candidate                : gradient assembly, then the optimizer's control flow as a resumable
//                                                    state machine (line search -> L-BFGS update + two-loop recursion ->
//                                                    ALM loop -> final collision check -> replans) up to the next
//                                                    evaluation request; survivors are appended to the next round's list
// The host only enqueues rounds (no per-iteration round trip: it polls the survivor count, asynchronously, every few
// rounds to know when to stop).  The floating-point operations and their order are those of traj_opt.cuh, so every
// result is bit-identical to the one-warp-per-candidate kernel and to the oracle.
#pragma once
#include "traj_opt.cuh"

namespace wave {
using namespace topt;

enum { PH_NEW = 0, PH_INIT = 1, PH_LS = 2, PH_FINAL = 3, PH_DONE = 4 };
#ifndef ALORE_TL_NB
#define ALORE_TL_NB 4
#endif
constexpr int TL_NB = ALORE_TL_NB;   // history pairs in flight (power of two): the recursion is bound by (memory latency) / TL_NB

// Developer counters (alore_debug_wave_counters): [0] LU warp-cycles, [1] back-substitution warp-cycles, [2] LU warps,
// [3] exact-division reruns of the LU, [4] of the back substitution, [5] of the adjoint, [6] adjoint-upper warp-cycles,
// [7] adjoint-lower warp-cycles, [8] two-loop warp-cycles, [9] two-loop history steps, [10] step-kernel warp-cycles, [11] step warps
__device__ unsigned long long g_wave_dbg[16];
#define WDBG_ADD(i, v) do { if ((threadIdx.x & 31) == 0) atomicAdd(&g_wave_dbg[i], (unsigned long long)(v)); } while (0)

// Optimizer state of one candidate between rounds (everything that was a register of the persistent warp).
struct CandState {
  double f;                 // energy + penalties of the pending evaluation (penalty kernel)
  double tsum;              // pieceTime.sum() of that evaluation
  double err[2];            // FinalIntegralXYError of the last stage-B evaluation
  double fx, step, mu, nu, finit, dgtest, dstest;
  double lam[2], rho[2];
  double safeDis, time_weight, alg_bytes, cost;
  int phase, stage, skip, k, end, bound, count, brackt, touched, past, alm_iters, replan, evals, iters, status, pad_;
};

struct WaveDev {
  int B, m;                       // candidates; L-BFGS history capacity
  const int* piece_off;
  const size_t* hist_off;         // [B] offset (doubles) of candidate b's history ring
  double *x, *g, *xp, *gp, *d;    // [3 tot] each, candidate b at 3*piece_off[b]
  double *T1, *gT;                // [tot]
  double *cf, *gC, *zb;           // [12 tot]
  double *Uf, *Lf;                // [48 tot]  (8 doubles per matrix row)
  double* pf;                     // [64 B]
  double* hist;
  CandState* st;
  int* list0; int* list1;         // survivor lists (double buffered)
  int* count;                     // count[0], count[1]
};

// scratch of the penalty / final-collision passes (per resident CTA, stays in L2)
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

struct WParams {
  alore_params_t P;
  MapDev map;
  PenLayout L;
  int Nmax, npadmax, mcap;
};

// =====================================================================================================
// 8-lane groups: banded LU and triangular sweeps (minco.hpp:99-197), 4 candidates per warp
//
// These kernels are chains of dependent issues (a lone warp issues one instruction every ~4.6 cycles), so their time
// is their instruction count: the pivot loop is unrolled by 7 with the entry of column j in register j % 7 (nothing
// ever shifts), the sweeps are unrolled by 2 with ping-pong operand sets (loads of the next row are issued before the
// quotient of the current one), and the per-lane generator constants live in a shared table.
// =====================================================================================================
constexpr int CH = 12;           // rows per sweep chunk
constexpr int SB = 180;          // doubles per staging buffer: 18 records of 8 + 18 rhs pairs
constexpr int GS = 368;          // doubles of shared memory per group: LU row ring (256) + T-power table (8) / sweep staging (2 x 180)
constexpr int GTAB = 6 * 16;     // generator table entries (row type q = 0..5, ring column 0..15), once per CTA

__device__ __forceinline__ double gshfl(double v, int src) { return __shfl_sync(FULL, v, src, 8); }

// Rows r of A for a candidate with n6 rows, generic form (head rows, tail rows, the all-zero rows past the matrix
// edge, and every row of very short trajectories).  Lane l8 writes columns l8 and l8 + 8 of the 16-double ring record.
__device__ __noinline__ void gen_row_generic(double* ring, int r, int n6, const double* T1g, const double* hs, const double* ts,
                                             double tail_s, const double* xg, int l8) {
#pragma unroll 1
  for (int h = 0; h < 2; h++) {
    const int col = l8 + 8 * h;
    double v = 0.0;
    if (r < n6 && col < 15) {
      int p;
      const int ty = row_type(r, n6, p);
      if (col < 13) {
        const int pw = g_row_pow[ty][col];
        if (pw >= 0) {
          double tp = 1.0;
          if (pw > 0) {
            const double T = T1g[p], t2 = T * T;
            tp = pw == 1 ? T : pw == 2 ? t2 : pw == 3 ? t2 * T : pw == 4 ? t2 * t2 : (t2 * t2) * T;
          }
          v = g_row_coef[ty][col] * tp;
        }
      } else {
        const int d = col - 13;
        if (ty >= 6 && ty <= 8) v = hs[3 * d + ty - 6];
        else if (ty >= 9) v = (d == 1 && ty == 9) ? tail_s : ts[3 * d + ty - 9];   // finState(1,0) is the relaxed tail arc length
        else if (ty == 2) v = xg[2 * p + d];
      }
    }
    ring[(r & (RING_ROWS - 1)) * 16 + col] = v;
  }
}

// The CTA-wide generator table: coefficient and T-power index of ring column `col` of knot row type q.
__device__ __forceinline__ void gen_table_init(double* gcoef, int* gidx) {
  for (int e = threadIdx.x; e < GTAB; e += blockDim.x) {
    const int q = e >> 4, col = e & 15;
    const int pw = col < 13 ? g_row_pow[q][col] : -1;
    gcoef[e] = pw >= 0 ? g_row_coef[q][col] : 0.0;             // structural zero: 0.0 * 1.0
    gidx[e] = pw > 0 ? pw : 0;                                 // index into tp[]: 0 -> 1.0
  }
}

struct GenState {          // row generator of one group (warp-uniform gen_next; Tn / rn fetched one block ahead)
  int gen_next;
  double Tn, rn;
};
// Rows gen_next .. gen_next + 5 -> ring.  Knot blocks from the table (12 values per lane), blocks past the matrix edge
// as zeros, the blocks holding head / tail rows through the generic generator.
__device__ __noinline__ void gen_block(double* ring, double* tp, const double* gcoef, const int* gidx, GenState& gsn, int n6,
                                       const double* xg, const double* T1g, const double* hs, const double* ts, double tail_s) {
  const int l8 = lane_id() & 7;
  const int gen_next = gsn.gen_next;
  const bool knot = gen_next < n6 - 3;
  const bool beyond = gen_next >= n6;                        // the whole block lies past the matrix edge: zero rows
  const bool rhs_lane = l8 == 5 || l8 == 6;                  // ring columns 13 / 14 of row type 2: rhs = inner point p
  if (knot) {
    const double Tn = gsn.Tn, t2 = Tn * Tn;
    const double pv = l8 == 1 ? Tn : l8 == 2 ? t2 : l8 == 3 ? t2 * Tn : l8 == 4 ? t2 * t2 : (t2 * t2) * Tn;
    if (l8 >= 1 && l8 < 6) tp[l8] = pv;
  }
  __syncwarp();
  if (knot || beyond) {
#pragma unroll
    for (int q = 0; q < 6; q++) {
      const int slot = (gen_next + q) & (RING_ROWS - 1);
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int e = q * 16 + l8 + 8 * h;
        double v = gcoef[e] * tp[gidx[e]];
        if (q == 2 && h == 1 && rhs_lane) v = gsn.rn;
        ring[slot * 16 + l8 + 8 * h] = beyond ? 0.0 : v;
      }
    }
  } else {
#pragma unroll 1
    for (int q = 0; q < 6; q++) gen_row_generic(ring, gen_next + q, n6, T1g, hs, ts, tail_s, xg, l8);
  }
  gsn.gen_next = gen_next + 6;
  if (gen_next + 6 < n6 - 3) {
    const int p = (gen_next + 3) / 6;
    gsn.Tn = T1g[p];
    if (rhs_lane) gsn.rn = xg[2 * p + l8 - 5];
  }
  __syncwarp();
}

// LU (factorizeLU, minco.hpp:99-131) fused with the forward substitution of solve() (:140-150), for the four
// candidates of a warp at once: lane 8c + (i % 7) holds row i of candidate c as a 7-wide register window, the entry of
// column j in register j % 7 (same operations per matrix element as topt::minco_lu_forward_t).  n6 = 0: the group has
// no work.  kmax = the largest n6 in the warp (loop bound, warp-uniform).  Returns true in every lane of a group whose
// quotients left the range of the split division.
template <bool EXACT>
__device__ __noinline__ bool group_lu_forward(double* gs, const double* gcoef, const int* gidx, int n6, int kmax, const double* xg,
                                              const double* T1g, const double* hs, const double* ts, double tail_s, double* Uf, double* Lf,
                                              double* yv) {
  const int lane = lane_id(), l8 = lane & 7;
  double* ring = gs;
  double* tp = gs + 256;
  if (l8 == 0) tp[0] = 1.0;
  gen_row_generic(ring, 0, n6, T1g, hs, ts, tail_s, xg, l8);
  gen_row_generic(ring, 1, n6, T1g, hs, ts, tail_s, xg, l8);
  gen_row_generic(ring, 2, n6, T1g, hs, ts, tail_s, xg, l8);
  GenState gsn;
  gsn.gen_next = 3; gsn.Tn = 0.0; gsn.rn = 0.0;
  if (3 < n6 - 3) { gsn.Tn = T1g[0]; if (l8 == 5 || l8 == 6) gsn.rn = xg[l8 - 5]; }
  __syncwarp();
  gen_block(ring, tp, gcoef, gidx, gsn, n6, xg, T1g, hs, ts, tail_s);          // rows 3..8
  const bool lu_lane = l8 < 7;
  const unsigned ring_s = smem_addr(ring);
  unsigned rowp = ring_s + (lu_lane ? l8 : 0) * 128;
  unsigned nxtp = rowp + (13 - l8) * 8;
  double wr[7], rb0, rb1;
#pragma unroll
  for (int c = 0; c < 7; c++) wr[c] = lu_lane ? lds64(rowp + (c - l8 + 6) * 8) : 0.0;
  rb0 = lds64(rowp + 13 * 8);
  rb1 = lds64(rowp + 14 * 8);
  bool bad = false;
  double* Up = Uf;
  double* yp = yv;
  double* Lp = Lf + l8;
#pragma unroll 1
  for (int k0 = 0; k0 < kmax; k0 += 7) {
#pragma unroll
    for (int kk = 0; kk < 7; kk++) {
      const int k = k0 + kk;
      if (gsn.gen_next <= k + 8) gen_block(ring, tp, gcoef, gidx, gsn, n6, xg, T1g, hs, ts, tail_s);   // warp-uniform
      const bool live = k < n6;
      double u[7];
#pragma unroll
      for (int c = 0; c < 7; c++) u[c] = gshfl(wr[(kk + c) % 7], kk);
      const double y0 = gshfl(rb0, kk), y1 = gshfl(rb1, kk);
      const double yk = rcp_refine(u[0]);
      if (l8 == kk) {
        if (live) {
          stg128(Up, u[0], yk);
          stg128(Up + 2, u[1], u[2]);
          stg128(Up + 4, u[3], u[4]);
          stg128(Up + 6, u[5], u[6]);
          stg128(yp, rb0, rb1);
        }
        // the owner takes row k+7: columns k+1 .. k+7 (band offsets 0..6) -> registers (kk+1+c) % 7
        rowp = ring_s + ((k + 7) & (RING_ROWS - 1)) * 128;
        const double2 v01 = lds128(rowp), v23 = lds128(rowp + 16), v45 = lds128(rowp + 32);
        wr[(kk + 1) % 7] = v01.x; wr[(kk + 2) % 7] = v01.y; wr[(kk + 3) % 7] = v23.x; wr[(kk + 4) % 7] = v23.y;
        wr[(kk + 5) % 7] = v45.x; wr[(kk + 6) % 7] = v45.y;
        wr[kk] = lds64(rowp + 48);
        rb0 = lds64(rowp + 13 * 8);
        rb1 = lds64(rowp + 14 * 8);
        nxtp = rowp + 7 * 8;
      } else if (lu_lane) {
        const double a = wr[kk];                             // A(myrow, k); rows past the matrix edge are all-zero
        double l = 0.0;
        if (a != 0.0) {
          l = quot_spec<EXACT>(a, u[0], yk, bad);
          // (the reference also tests A(k,j) != 0 per column; subtracting l*0 is the identity)
#pragma unroll
          for (int c = 1; c < 7; c++) wr[(kk + c) % 7] -= l * u[c];
          rb0 -= l * y0;
          rb1 -= l * y1;
        }
        if (live) stg64(Lp, l);
        wr[kk] = lds64(nxtp);                                // column k+7 enters: A(myrow, k+7)
        nxtp += 8;
      }
      Up += 8; yp += 2; Lp += 8;
    }
  }
  __syncwarp();
  const unsigned bal = __ballot_sync(FULL, bad);
  return ((bal >> (lane & ~7)) & 0xffu) != 0;
}

// 18 records [recA0, recA0+18) of A8 (8 doubles each) and 18 rhs pairs [recB0, ...) -> buf; rows outside [0, n6) read as zero
__device__ __forceinline__ void gstage(double* buf, const double* A8, const double* rhs, int recA0, int recB0, int n6, int l8) {
#pragma unroll
  for (int i = 0; i < 9; i++) {
    const int e = l8 + 8 * i;                                 // 72 16-byte chunks of records
    const int row = recA0 + (e >> 2);
    const bool ok = row >= 0 && row < n6;
    cp_async16(buf + 2 * e, A8 + (ok ? (size_t)row * 8 + (e & 3) * 2 : 0), ok);
  }
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const int e = l8 + 8 * i;
    if (e < 18) {
      const int row = recB0 + e;
      const bool ok = row >= 0 && row < n6;
      cp_async16(buf + 144 + 2 * e, rhs + (ok ? 2 * (size_t)row : 0), ok);
    }
  }
}

// Back substitution U x = y (minco.hpp:151-162): lanes 0/1 of the group = the two right-hand sides.
// Column-oriented like the reference: x_j = b_j / U(j,j), then b_i -= U(i,j) x_j for i = j-6..j-1.
struct BackOps { double2 d; double c1, c2, c3, c4, c5, c6, f; };
__device__ __forceinline__ void back_load(BackOps& o, unsigned ua, unsigned fa) {
  o.d = lds128(ua);
  o.c1 = lds64(ua - 48); o.c2 = lds64(ua - 104); o.c3 = lds64(ua - 160); o.c4 = lds64(ua - 216); o.c5 = lds64(ua - 272);
  o.c6 = lds64(ua - 328); o.f = lds64(fa);
}
template <bool EXACT>
__device__ __noinline__ bool group_back(double* gs, int n6, int kmax, const double* Uf, const double* __restrict__ y, double* __restrict__ x) {
  const int lane = lane_id(), l8 = lane & 7;
  const unsigned S_s = smem_addr(gs);
  const bool act = l8 < 2 && n6 > 0;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0, a4 = 0.0, a5 = 0.0;
  if (act) {
    a0 = y[2 * (n6 - 1) + l8]; a1 = y[2 * (n6 - 2) + l8]; a2 = y[2 * (n6 - 3) + l8];
    a3 = y[2 * (n6 - 4) + l8]; a4 = y[2 * (n6 - 5) + l8]; a5 = y[2 * (n6 - 6) + l8];
  }
  bool bad = false;
  int c0 = n6 > 0 ? ((n6 - 1) / CH) * CH : -CH, cur = 0;
  const int nch = (kmax - 1) / CH + 1;
  gstage(gs, Uf, y, c0 - 6, c0 - 6, n6, l8);
#pragma unroll 1
  for (int it = 0; it < nch; it++, c0 -= CH) {
    cp_async_wait_all();
    __syncwarp();
    gstage(gs + (cur ^ 1) * SB, Uf, y, c0 - CH - 6, c0 - CH - 6, c0 > 0 ? n6 : 0, l8);
    if (act && c0 >= 0) {
      const int rows = min(CH, n6 - c0);                     // even (n6 and CH are multiples of 6)
      unsigned ua = S_s + (cur * SB + (rows + 5) * 8) * 8;   // record of row j = c0 + i
      unsigned fa = S_s + (cur * SB + 144 + 2 * (rows - 1) + l8) * 8;
      double* xo = x + 2 * (c0 + rows - 1) + l8;
      BackOps A, B;
      back_load(A, ua, fa);
#define ALORE_BACK_STEP(CUR, NXT, more)                                        \
      {                                                                        \
        ua -= 64; fa -= 16;                                                    \
        if (more) back_load(NXT, ua, fa);                                      \
        const double xv = quot_spec<EXACT>(a0, CUR.d.x, CUR.d.y, bad);         \
        stg64(xo, xv);                                                         \
        xo -= 2;                                                               \
        a0 = a1 - CUR.c1 * xv;                                                 \
        a1 = a2 - CUR.c2 * xv;                                                 \
        a2 = a3 - CUR.c3 * xv;                                                 \
        a3 = a4 - CUR.c4 * xv;                                                 \
        a4 = a5 - CUR.c5 * xv;                                                 \
        a5 = CUR.f - CUR.c6 * xv;                                              \
      }
#pragma unroll 1
      for (int i = rows; i > 0; i -= 2) {
        ALORE_BACK_STEP(A, B, true)
        ALORE_BACK_STEP(B, A, i > 2)
      }
#undef ALORE_BACK_STEP
    }
    __syncwarp();
    cur ^= 1;
  }
  cp_async_wait_all();
  __syncwarp();
  const unsigned bal = __ballot_sync(FULL, bad);
  return ((bal >> (lane & ~7)) & 0xffu) != 0;
}

// U^T z = b ascending (minco.hpp:170-183): z_j = b_j / U(j,j), then b_i -= U(j,i) z_j, i = j+1..j+6.
struct UpOps { double2 r01, r23, r45, r67; double f; };
__device__ __forceinline__ void up_load(UpOps& o, unsigned ua, unsigned fa) {
  o.r01 = lds128(ua); o.r23 = lds128(ua + 16); o.r45 = lds128(ua + 32); o.r67 = lds128(ua + 48); o.f = lds64(fa);
}
template <bool EXACT>
__device__ __noinline__ bool group_adj_upper(double* gs, int n6, int kmax, const double* Uf, const double* __restrict__ b, double* __restrict__ z) {
  const int lane = lane_id(), l8 = lane & 7;
  const unsigned S_s = smem_addr(gs);
  const bool act = l8 < 2 && n6 > 0;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0, a4 = 0.0, a5 = 0.0;
  if (act) { a0 = b[l8]; a1 = b[2 + l8]; a2 = b[4 + l8]; a3 = b[6 + l8]; a4 = b[8 + l8]; a5 = b[10 + l8]; }
  bool bad = false;
  int cur = 0;
  gstage(gs, Uf, b, 0, 6, n6, l8);
#pragma unroll 1
  for (int c0 = 0; c0 < kmax; c0 += CH) {
    cp_async_wait_all();
    __syncwarp();
    gstage(gs + (cur ^ 1) * SB, Uf, b, c0 + CH, c0 + CH + 6, n6, l8);
    if (act && c0 < n6) {
      const int rows = min(CH, n6 - c0);                     // even
      unsigned ua = S_s + (cur * SB) * 8;
      unsigned fa = S_s + (cur * SB + 144 + l8) * 8;
      double* zo = z + 2 * c0 + l8;
      UpOps A, B;
      up_load(A, ua, fa);
#define ALORE_UP_STEP(CUR, NXT, more)                                          \
      {                                                                        \
        ua += 64; fa += 16;                                                    \
        if (more) up_load(NXT, ua, fa);                                        \
        const double zv = quot_spec<EXACT>(a0, CUR.r01.x, CUR.r01.y, bad);     \
        stg64(zo, zv);                                                         \
        zo += 2;                                                               \
        a0 = a1 - CUR.r23.x * zv;                                              \
        a1 = a2 - CUR.r23.y * zv;                                              \
        a2 = a3 - CUR.r45.x * zv;                                              \
        a3 = a4 - CUR.r45.y * zv;                                              \
        a4 = a5 - CUR.r67.x * zv;                                              \
        a5 = CUR.f - CUR.r67.y * zv;                                           \
      }
#pragma unroll 1
      for (int i = rows; i > 0; i -= 2) {
        ALORE_UP_STEP(A, B, true)
        ALORE_UP_STEP(B, A, i > 2)
      }
#undef ALORE_UP_STEP
    }
    __syncwarp();
    cur ^= 1;
  }
  cp_async_wait_all();
  __syncwarp();
  const unsigned bal = __ballot_sync(FULL, bad);
  return ((bal >> (lane & ~7)) & 0xffu) != 0;
}

// L^T x = z descending (minco.hpp:184-196): b_i -= L(j,i) b_j for i = j-6..j-1; L(j,i) = Lf[8i + j % 7]
struct LowOps { double c1, c2, c3, c4, c5, c6, f; };
__device__ __forceinline__ void low_load(LowOps& o, unsigned la, unsigned fa) {
  o.c1 = lds64(la - 64); o.c2 = lds64(la - 128); o.c3 = lds64(la - 192); o.c4 = lds64(la - 256); o.c5 = lds64(la - 320);
  o.c6 = lds64(la - 384); o.f = lds64(fa);
}
__device__ __noinline__ void group_adj_lower(double* gs, int n6, int kmax, const double* Lf, const double* __restrict__ z, double* __restrict__ x) {
  const int lane = lane_id(), l8 = lane & 7;
  const unsigned S_s = smem_addr(gs);
  const bool act = l8 < 2 && n6 > 0;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0, a4 = 0.0, a5 = 0.0;
  if (act) {
    a0 = z[2 * (n6 - 1) + l8]; a1 = z[2 * (n6 - 2) + l8]; a2 = z[2 * (n6 - 3) + l8];
    a3 = z[2 * (n6 - 4) + l8]; a4 = z[2 * (n6 - 5) + l8]; a5 = z[2 * (n6 - 6) + l8];
  }
  int c0 = n6 > 0 ? ((n6 - 1) / CH) * CH : -CH, cur = 0;
  const int nch = (kmax - 1) / CH + 1;
  gstage(gs, Lf, z, c0 - 6, c0 - 6, n6, l8);
#pragma unroll 1
  for (int it = 0; it < nch; it++, c0 -= CH) {
    cp_async_wait_all();
    __syncwarp();
    gstage(gs + (cur ^ 1) * SB, Lf, z, c0 - CH - 6, c0 - CH - 6, c0 > 0 ? n6 : 0, l8);
    if (act && c0 >= 0) {
      const int rows = min(CH, n6 - c0);                     // even
      int jm = (c0 + rows - 1) % 7;
      unsigned la = S_s + (cur * SB + (rows + 5) * 8 + jm) * 8;   // record of column j = c0 + i, slot j % 7
      unsigned fa = S_s + (cur * SB + 144 + 2 * (rows - 1) + l8) * 8;
      double* xo = x + 2 * (c0 + rows - 1) + l8;
      LowOps A, B;
      low_load(A, la, fa);
#define ALORE_LOW_STEP(CUR, NXT, more)                                         \
      {                                                                        \
        la -= (jm == 0) ? (64 - 48) : (64 + 8);                                \
        jm = jm == 0 ? 6 : jm - 1;                                             \
        fa -= 16;                                                              \
        if (more) low_load(NXT, la, fa);                                       \
        const double xv = a0;                                                  \
        stg64(xo, xv);                                                         \
        xo -= 2;                                                               \
        a0 = a1 - CUR.c1 * xv;                                                 \
        a1 = a2 - CUR.c2 * xv;                                                 \
        a2 = a3 - CUR.c3 * xv;                                                 \
        a3 = a4 - CUR.c4 * xv;                                                 \
        a4 = a5 - CUR.c5 * xv;                                                 \
        a5 = CUR.f - CUR.c6 * xv;                                              \
      }
#pragma unroll 1
      for (int i = rows; i > 0; i -= 2) {
        ALORE_LOW_STEP(A, B, true)
        ALORE_LOW_STEP(B, A, i > 2)
      }
#undef ALORE_LOW_STEP
    }
    __syncwarp();
    cur ^= 1;
  }
  cp_async_wait_all();
  __syncwarp();
}

__device__ __forceinline__ int warp_max_i(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(FULL, v, o));
  return v;
}

// ---- kernel 1 of a round: coefficients of every pending evaluation (Minco.setParameters) ----------------------------
constexpr int SOLVE_WARPS = 4;
__global__ void __launch_bounds__(32 * SOLVE_WARPS)
wave_solve_kernel(const __grid_constant__ WParams kp, BatchDev bt, WaveDev wd, int cur) {
  extern __shared__ __align__(16) double smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, grp = lane >> 3;
  double* gs = smem + (size_t)(wib * 4 + grp) * GS;
  double* gcoef = smem + (size_t)SOLVE_WARPS * 4 * GS;
  int* gidx = reinterpret_cast<int*>(gcoef + GTAB);
  gen_table_init(gcoef, gidx);
  __syncthreads();
  const int* list = cur ? wd.list1 : wd.list0;
  const int nact = wd.count[cur];
  if (blockIdx.x == 0 && threadIdx.x == 0) wd.count[cur ^ 1] = 0;    // the step kernel of this round appends there
  const int ngrp_total = gridDim.x * SOLVE_WARPS * 4;
#pragma unroll 1
  for (int base = (blockIdx.x * SOLVE_WARPS + wib) * 4; base < nact; base += ngrp_total) {
    const int slot = base + grp;
    int n6 = 0, b = 0, p0 = 0, N = 0;
    if (slot < nact) {
      b = list[slot];
      const CandState* s = wd.st + b;
      p0 = bt.piece_off[b];
      N = bt.piece_off[b + 1] - p0;
      if (s->phase != PH_DONE && !(s->phase != PH_FINAL && s->skip)) n6 = 6 * N;
    }
    const int kmax = warp_max_i(n6);
    if (kmax == 0) continue;                                          // warp-uniform
    const double* xg = wd.x + 3 * (size_t)p0;
    const double* T1g = wd.T1 + p0;
    const double* hs = bt.start_state + 6 * (size_t)b;
    const double* ts = bt.final_state + 6 * (size_t)b;
    double* Ug = wd.Uf + 48 * (size_t)p0;
    double* Lg = wd.Lf + 48 * (size_t)p0;
    double* yg = wd.gC + 12 * (size_t)p0;
    double* cg = wd.cf + 12 * (size_t)p0;
    const double tail_s = n6 ? xg[2 * (N - 1)] : 0.0;
    bool bad = g_force_exact_div != 0;
    const long long t0 = clock64();
    if (!bad) bad = group_lu_forward<false>(gs, gcoef, gidx, n6, kmax, xg, T1g, hs, ts, tail_s, Ug, Lg, yg);
    if (__any_sync(FULL, bad)) {                                      // rare: redo the affected groups with the compiler's division
      const int n6x = bad ? n6 : 0;
      group_lu_forward<true>(gs, gcoef, gidx, n6x, warp_max_i(n6x), xg, T1g, hs, ts, tail_s, Ug, Lg, yg);
      WDBG_ADD(3, 1);
    }
    const long long t1 = clock64();
    bad = g_force_exact_div != 0;
    if (!bad) bad = group_back<false>(gs, n6, kmax, Ug, yg, cg);
    if (__any_sync(FULL, bad)) {
      const int n6x = bad ? n6 : 0;
      group_back<true>(gs, n6x, warp_max_i(n6x), Ug, yg, cg);
      WDBG_ADD(4, 1);
    }
    const long long t2 = clock64();
    WDBG_ADD(0, t1 - t0); WDBG_ADD(1, t2 - t1); WDBG_ADD(2, 1); WDBG_ADD(12, kmax);
  }
}

// ---- kernel 3 of a round: solveAdj on gradC (propogateArcYawLenghGrad's band solve) ---------------------------------
__global__ void __launch_bounds__(32 * SOLVE_WARPS)
wave_adjoint_kernel(const __grid_constant__ WParams kp, BatchDev bt, WaveDev wd, int cur) {
  extern __shared__ __align__(16) double smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, grp = lane >> 3;
  double* gs = smem + (size_t)(wib * 4 + grp) * GS;
  const int* list = cur ? wd.list1 : wd.list0;
  const int nact = wd.count[cur];
  const int ngrp_total = gridDim.x * SOLVE_WARPS * 4;
#pragma unroll 1
  for (int base = (blockIdx.x * SOLVE_WARPS + wib) * 4; base < nact; base += ngrp_total) {
    const int slot = base + grp;
    int n6 = 0, p0 = 0;
    if (slot < nact) {
      const int b = list[slot];
      const CandState* s = wd.st + b;
      p0 = bt.piece_off[b];
      if ((s->phase == PH_INIT || s->phase == PH_LS) && !s->skip) n6 = 6 * (bt.piece_off[b + 1] - p0);
    }
    const int kmax = warp_max_i(n6);
    if (kmax == 0) continue;
    const double* Ug = wd.Uf + 48 * (size_t)p0;
    const double* Lg = wd.Lf + 48 * (size_t)p0;
    double* gCg = wd.gC + 12 * (size_t)p0;
    double* zg = wd.zb + 12 * (size_t)p0;
    bool bad = g_force_exact_div != 0;
    const long long t0 = clock64();
    if (!bad) bad = group_adj_upper<false>(gs, n6, kmax, Ug, gCg, zg);
    if (__any_sync(FULL, bad)) {
      const int n6x = bad ? n6 : 0;
      group_adj_upper<true>(gs, n6x, warp_max_i(n6x), Ug, gCg, zg);
      WDBG_ADD(5, 1);
    }
    const long long t1 = clock64();
    group_adj_lower(gs, n6, kmax, Lg, zg, gCg);
    WDBG_ADD(6, t1 - t0); WDBG_ADD(7, clock64() - t1);
  }
}

// =====================================================================================================
// kernel 2 of a round: energy + penalty functional, one CTA per candidate
// =====================================================================================================
constexpr int PEN_NT = 128;
__host__ __device__ inline size_t pen_smem_doubles(int Nmax) {
  // T1[N] gT[N] pXY[2(N+1)] bcast[4] | stg[1024] (cell-prefix chunks 2 x 256, cost-term packing 512)
  return (size_t)Nmax + Nmax + 2 * (Nmax + 1) + 4 + 2 + 1024;
}
// + the per-sample intermediates on chip: cs[2S] | ax[S+64] ay[S+64] (dead after the cell integrals; g2p[2N(K+1)] takes
// their place from pass B on) | cellP[2NK]
__host__ __device__ inline size_t pen_smem_doubles_onchip(int Nmax, int K) {
  const size_t S = (size_t)Nmax * (2 * K + 1);
  const size_t axy = 2 * (S + 64), g2 = 2 * (size_t)Nmax * (K + 1);
  return pen_smem_doubles(Nmax) + 2 * S + (axy > g2 ? axy : g2) + 2 * (size_t)Nmax * K + 8;
}
template <bool SH>
__device__ __forceinline__ void pen_carve(Warp& w, const PenLayout& L, double* smem, double* slab, int Nmax, int N, int K) {
  w.lane = threadIdx.x;
  w.N = N; w.n = 3 * N - 1; w.npad = (3 * N) & ~1; w.n6 = 6 * N; w.K = K; w.S1 = 2 * K + 1;
  double* s = smem;
  w.T1 = s; s += Nmax; w.gT = s; s += Nmax; w.pXY = s; s += 2 * (Nmax + 1); w.sumT = s; s += 4;
  s = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(s) + 15) & ~uintptr_t(15));
  w.stg = s; s += 1024;
  w.Nm = Nmax;
  if (SH) {
    const size_t S = (size_t)Nmax * (2 * K + 1);
    w.cs = s; s += 2 * S;
    w.ax = s; w.ay = s + S + 64; w.g2p = s;
    const size_t axy = 2 * (S + 64), g2 = 2 * (size_t)Nmax * (K + 1);
    s += (axy > g2 ? axy : g2);
    w.cellP = s;
  } else {
    w.cs = slab + L.cs; w.ax = slab + L.ax; w.ay = slab + L.ay; w.cellP = slab + L.cellP; w.g2p = slab + L.g2p;
  }
  w.terms = slab + L.terms; w.cg = slab + L.cg; w.fold = slab + L.fold;
  w.nterm = reinterpret_cast<int*>(slab + L.nterm); w.rank = reinterpret_cast<int*>(slab + L.rank);
  w.TS = L.TS;
  w.err[0] = w.err[1] = 0.0;
}

// energy and its partial gradients (minco.hpp:915-992) with NT threads; returns the energy, w.tsum = pieceTime.sum()
template <int NT>
__device__ __forceinline__ double energy_cta(Warp& w, const alore_params_t& P) {
  const int tid = w.lane, N = w.N;
  const double e0 = P.energyWeights[0], e1 = P.energyWeights[1];
  for (int i = tid; i < N; i += NT) {
    const double* c = w.cf + 12 * i;
    const double t1 = w.T1[i], t2 = t1 * t1, t3 = t2 * t1, t4 = t2 * t2, t5 = (t2 * t2) * t1;
    auto wd = [&](int a, int b) { return (c[2 * a] * e0) * c[2 * b] + (c[2 * a + 1] * e1) * c[2 * b + 1]; };
    w.ax[i] = 36.0 * wd(3, 3) * t1 + 144.0 * wd(4, 3) * t2 + 192.0 * wd(4, 4) * t3 + 240.0 * wd(5, 3) * t3 +
              720.0 * wd(5, 4) * t4 + 720.0 * wd(5, 5) * t5;
    w.gT[i] = 36.0 * wd(3, 3) + 288.0 * wd(4, 3) * t1 + 576.0 * wd(4, 4) * t2 + 720.0 * wd(5, 3) * t2 +
              2880.0 * wd(5, 4) * t3 + 3600.0 * wd(5, 5) * t4;
    double* gc = w.gC + 12 * i;
    for (int d = 0; d < 2; d++) {
      const double ew = d == 0 ? e0 : e1;
      gc[2 * 5 + d] = 240.0 * c[2 * 3 + d] * ew * t3 + 720.0 * c[2 * 4 + d] * ew * t4 + 1440.0 * c[2 * 5 + d] * ew * t5;
      gc[2 * 4 + d] = 144.0 * c[2 * 3 + d] * ew * t2 + 384.0 * c[2 * 4 + d] * ew * t3 + 720.0 * c[2 * 5 + d] * ew * t4;
      gc[2 * 3 + d] = 72.0 * c[2 * 3 + d] * ew * t1 + 144.0 * c[2 * 4 + d] * ew * t2 + 240.0 * c[2 * 5 + d] * ew * t3;
      gc[d] = 0.0; gc[2 + d] = 0.0; gc[4 + d] = 0.0;
    }
  }
  tsync<NT>();
  // `energy += ...` per piece and pieceTime.sum(): sequential, in piece order (threads 0 and 1 in parallel)
  double* bc = w.sumT + 2;
  if (tid < 2) {
    double acc = 0.0;
    if (tid == 0) for (int i = 0; i < N; i++) acc += w.ax[i];
    else for (int i = 0; i < N; i++) acc += w.T1[i];
    bc[tid] = acc;
  }
  tsync<NT>();
  w.tsum = bc[1];
  return bc[0];
}

__global__ void __launch_bounds__(PEN_NT, 3)
wave_penalty_kernel(const __grid_constant__ WParams kp, BatchDev bt, WaveDev wd, int cur, double* slabs) {
  extern __shared__ __align__(16) double smem[];
  double* slab = slabs + (size_t)blockIdx.x * kp.L.total;
  const int tid = threadIdx.x;
  const int* list = cur ? wd.list1 : wd.list0;
  const int nact = wd.count[cur];
#pragma unroll 1
  for (int slot = blockIdx.x; slot < nact; slot += gridDim.x) {
    const int b = list[slot];
    CandState* s = wd.st + b;
    if (!((s->phase == PH_INIT || s->phase == PH_LS) && !s->skip)) continue;     // CTA-uniform
    const int p0 = bt.piece_off[b], N = bt.piece_off[b + 1] - p0;
    const int stage = s->stage;
    Warp w;
    pen_carve<false>(w, kp.L, smem, slab, kp.Nmax, N, kp.P.sparseResolution);
    w.cf = wd.cf + 12 * (size_t)p0;
    w.gC = wd.gC + 12 * (size_t)p0;
    w.sx = bt.start_xytheta[3 * (size_t)b]; w.sy = bt.start_xytheta[3 * (size_t)b + 1];
    w.fx = bt.final_xytheta[3 * (size_t)b]; w.fy = bt.final_xytheta[3 * (size_t)b + 1];
    w.init_pos = bt.inner_init_pos + 3 * (size_t)p0;
    w.lam[0] = s->lam[0]; w.lam[1] = s->lam[1]; w.rho[0] = s->rho[0]; w.rho[1] = s->rho[1];
    w.safeDis = s->safeDis;
    __syncthreads();                                         // the previous candidate's shared arrays are free
    for (int i = tid; i < N; i += PEN_NT) w.T1[i] = wd.T1[p0 + i];
    __syncthreads();
    double cost = energy_cta<PEN_NT>(w, kp.P);
    cost = penalty_passes_t<PEN_NT>(w, kp.P, kp.map, stage, cost);
    for (int i = tid; i < N; i += PEN_NT) wd.gT[p0 + i] = w.gT[i];
    if (tid == 0) {
      s->f = cost;
      s->tsum = w.tsum;
      if (stage == 1) { s->err[0] = w.err[0]; s->err[1] = w.err[1]; }
    }
  }
}

// =====================================================================================================
// kernel 4 of a round: gradient assembly + the optimizer's control flow, one warp per candidate
// =====================================================================================================
__host__ __device__ inline size_t step_smem_doubles(int Nmax) {
  const size_t npad = (size_t)((3 * Nmax) & ~1);
  return (size_t)Nmax + (Nmax + 1) + 3 + 2 + (TL_NB + 2) + npad + (TL_NB > 4 ? TL_NB : 4) * (2 * npad + 4) + 8;
}

// tail of costFunctionCallback[Path] (optimizer.cpp:675-689 / 1299-1315): adjoint -> gradient w.r.t. points, tail s, tau
__device__ __forceinline__ double assemble_gradient(const Warp& w, const alore_params_t& P, int stage, const double* T1g, const double* gTg,
                                                    double f_partial, double tsum, double time_weight) {
  const int lane = w.lane, N = w.N, n6 = w.n6;
  const double* tau = w.x + 2 * (N - 1) + 1;
  double* g = w.g;
  for (int i = lane; i < N; i += 32) {
    const double* c = w.cf + 12 * i;
    const double* a = w.gC;
    const double t1 = T1g[i], t2 = t1 * t1, t3 = t2 * t1, t4 = t2 * t2;
    double gt = 0.0;
    if (i < N - 1) {
      double s = 0.0;
      for (int d = 0; d < 2; d++) {
        const double nv = -(c[2 * 1 + d] + 2.0 * t1 * c[2 * 2 + d] + 3.0 * t2 * c[2 * 3 + d] + 4.0 * t3 * c[2 * 4 + d] + 5.0 * t4 * c[2 * 5 + d]);
        const double na = -(2.0 * c[2 * 2 + d] + 6.0 * t1 * c[2 * 3 + d] + 12.0 * t2 * c[2 * 4 + d] + 20.0 * t3 * c[2 * 5 + d]);
        const double nj = -(6.0 * c[2 * 3 + d] + 24.0 * t1 * c[2 * 4 + d] + 60.0 * t2 * c[2 * 5 + d]);
        const double ns = -(24.0 * c[2 * 4 + d] + 120.0 * t1 * c[2 * 5 + d]);
        const double nc = -120.0 * c[2 * 5 + d];
        const double B1[6] = {ns, nc, nv, nv, na, nj};
        for (int r = 0; r < 6; r++) s += B1[r] * a[2 * (6 * i + 3 + r) + d];
      }
      gt = s;
      g[2 * i] = a[2 * (6 * i + 5)];
      g[2 * i + 1] = a[2 * (6 * i + 5) + 1];
    } else {
      double s = 0.0;
      for (int d = 0; d < 2; d++) {
        const double nv = -(c[2 * 1 + d] + 2.0 * t1 * c[2 * 2 + d] + 3.0 * t2 * c[2 * 3 + d] + 4.0 * t3 * c[2 * 4 + d] + 5.0 * t4 * c[2 * 5 + d]);
        const double na = -(2.0 * c[2 * 2 + d] + 6.0 * t1 * c[2 * 3 + d] + 12.0 * t2 * c[2 * 4 + d] + 20.0 * t3 * c[2 * 5 + d]);
        const double nj = -(6.0 * c[2 * 3 + d] + 24.0 * t1 * c[2 * 4 + d] + 60.0 * t2 * c[2 * 5 + d]);
        const double B2[3] = {nv, na, nj};
        for (int r = 0; r < 3; r++) s += B2[r] * a[2 * (n6 - 3 + r) + d];
      }
      gt = s;
      g[2 * (N - 1)] = a[2 * (n6 - 3) + 1];
    }
    gt += gTg[i];
    gt += time_weight * 1.0;
    const double t = tau[i];
    double gr;
    if (t > 0) gr = t + 1.0;
    else {
      const double den = (0.5 * t - 1.0) * t + 1.0;
      gr = (1.0 - t) / (den * den);
    }
    g[2 * (N - 1) + 1 + i] = gt * gr;
  }
  __syncwarp();
  return f_partial + (stage == 1 ? time_weight : P.ppw_time) * tsum;
}

// The same recursion with the history pairs moved by TMA: ONE lane issues two 1-D bulk copies per pair
// (cp.async.bulk, completion counted on an mbarrier) instead of every lane issuing cp.async chunks and computing their
// addresses — the staging drops from ~50 to ~12 warp-instructions per step; the consumers wait on the barrier's
// phase.  mb = 4 mbarriers + a phase word in shared memory (initialised once per kernel by two_loop_tma_init).
__device__ __forceinline__ void two_loop_tma_init(double* mbar) {
  if (lane_id() == 0) {
    const unsigned b0 = smem_addr(mbar);
    for (int i = 0; i < TL_NB; i++) mbar_init(b0 + 8 * i, 1);
    reinterpret_cast<int*>(mbar + TL_NB)[0] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
}
template <int EPL>
__device__ __noinline__ void two_loop_tma(Warp& w, int m, int end, int bound, double ys, double yy) {
  constexpr int NB = TL_NB, PF = 16;
  const int n = w.n, lane = w.lane, np = w.npad, hs = np + 4, bs = 2 * np + 4;
  double* dsh = as_shared(w.d);
  double* H = as_shared(w.hbuf);
  double* lm_s = as_global(w.lm_s);
  const double* lm_y = as_global(w.lm_y);
  const unsigned H_s = smem_addr(H), bar0 = smem_addr(w.mbar);
  int* phw = reinterpret_cast<int*>(as_shared(w.mbar) + TL_NB);
  unsigned ph = (unsigned)*phw;
  auto issue = [&](int stage, int jj) {
    if (lane == 0) {
      const unsigned bar = bar0 + 8 * stage, dst = H_s + (unsigned)(stage * bs) * 8;
      mbar_expect_tx(bar, (unsigned)(hs + np) * 8);
      tma_load_1d(dst, lm_s + (size_t)jj * hs, (unsigned)hs * 8, bar);
      tma_load_1d(dst + (unsigned)hs * 8, lm_y + (size_t)jj * np, (unsigned)np * 8, bar);
    }
  };
  auto wait = [&](int stage) {
    mbar_wait(bar0 + 8 * stage, (ph >> stage) & 1u);
    ph ^= 1u << stage;
  };
  auto prefetch = [&](int jj) {                      // one 128-byte line per lane: s-record then y-record (HBM -> L2)
    const int line = lane * 16;
    if (line < hs) prefetch_l2(lm_s + (size_t)jj * hs + line);
    if (line < np) prefetch_l2(lm_y + (size_t)jj * np + line);
  };
  double d[EPL];
#pragma unroll
  for (int q = 0; q < EPL; q++) d[q] = (lane + 32 * q < n) ? dsh[lane + 32 * q] : 0.0;
  const bool last_ok = lane + 32 * (EPL - 1) < n;    // only the last element of a lane can lie past n
  asm volatile("fence.proxy.async;" ::: "memory");   // the newest pair was written with ordinary stores
  __syncwarp();
  int j = end, jn = end, jp = end;
#pragma unroll 1
  for (int a = 0; a < PF; a++) { jp = jp == 0 ? m - 1 : jp - 1; if (a < bound) prefetch(jp); }
#pragma unroll 1
  for (int a = 0; a < NB - 1; a++) { jn = jn == 0 ? m - 1 : jn - 1; if (a < bound) issue(a, jn); }
#pragma unroll 1
  for (int it = 0; it < bound; ++it) {
    j = j == 0 ? m - 1 : j - 1;
    wait(it & (NB - 1));
    __syncwarp();                                    // every lane has left the buffer that is refilled next
    jn = jn == 0 ? m - 1 : jn - 1;
    if (it + NB - 1 < bound) issue((it + NB - 1) & (NB - 1), jn);
    jp = jp == 0 ? m - 1 : jp - 1;
    if (it + PF < bound) prefetch(jp);
    // explicit shared-space addresses: through the dynamic stage index the compiler would fall back to generic loads
    const unsigned sj = H_s + (unsigned)((it & (NB - 1)) * bs + lane) * 8;
    const unsigned yj = sj + (unsigned)hs * 8;
    double sv[EPL], yv[EPL];
#pragma unroll
    for (int q = 0; q < EPL; q++) { sv[q] = (q < EPL - 1 || last_ok) ? lds64(sj + 256 * q) : 0.0; yv[q] = (q < EPL - 1 || last_ok) ? lds64(yj + 256 * q) : 0.0; }
    const double2 yr = lds128(sj + (unsigned)(np - lane) * 8);
    double ps = 0.0;
#pragma unroll
    for (int q = 0; q < EPL; q++)
      if (q < EPL - 1 || last_ok) ps += sv[q] * d[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ps += shfl_xor_d(ps, o);
    const double alpha = div_rcp(ps, yr.x, yr.y);
    if (lane == 0) stg64(lm_s + (size_t)j * hs + np + 2, alpha);
    const double c = -alpha;
#pragma unroll
    for (int q = 0; q < EPL; q++)
      if (q < EPL - 1 || last_ok) d[q] += c * yv[q];
  }
  {
    const double c = ys / yy;
#pragma unroll
    for (int q = 0; q < EPL; q++) d[q] *= c;
  }
  asm volatile("fence.proxy.async;" ::: "memory");   // alpha_j (ordinary stores by lane 0) travels back with the s-records
  __syncwarp();
  jn = j == 0 ? m - 1 : j - 1;
  jp = jn;
#pragma unroll 1
  for (int a = 0; a < PF; a++) { jp = jp == m - 1 ? 0 : jp + 1; if (a < bound) prefetch(jp); }
#pragma unroll 1
  for (int a = 0; a < NB - 1; a++) { jn = jn == m - 1 ? 0 : jn + 1; if (a < bound) issue(a, jn); }
#pragma unroll 1
  for (int it = 0; it < bound; ++it) {
    wait(it & (NB - 1));
    __syncwarp();
    jn = jn == m - 1 ? 0 : jn + 1;
    if (it + NB - 1 < bound) issue((it + NB - 1) & (NB - 1), jn);
    jp = jp == m - 1 ? 0 : jp + 1;
    if (it + PF < bound) prefetch(jp);
    const unsigned sj = H_s + (unsigned)((it & (NB - 1)) * bs + lane) * 8;
    const unsigned yj = sj + (unsigned)hs * 8;
    double sv[EPL], yv[EPL];
#pragma unroll
    for (int q = 0; q < EPL; q++) { sv[q] = (q < EPL - 1 || last_ok) ? lds64(sj + 256 * q) : 0.0; yv[q] = (q < EPL - 1 || last_ok) ? lds64(yj + 256 * q) : 0.0; }
    const double2 yr = lds128(sj + (unsigned)(np - lane) * 8);
    const double aj = lds64(sj + (unsigned)(np + 2 - lane) * 8);
    double ps = 0.0;
#pragma unroll
    for (int q = 0; q < EPL; q++)
      if (q < EPL - 1 || last_ok) ps += yv[q] * d[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ps += shfl_xor_d(ps, o);
    const double beta = div_rcp(ps, yr.x, yr.y);
    const double c = aj - beta;
#pragma unroll
    for (int q = 0; q < EPL; q++)
      if (q < EPL - 1 || last_ok) d[q] += c * sv[q];
  }
#pragma unroll
  for (int q = 0; q < EPL; q++)
    if (lane + 32 * q < n) dsh[lane + 32 * q] = d[q];
  __syncwarp();
  if (lane == 0) *phw = (int)ph;
  __syncwarp();
}
__device__ __forceinline__ void two_loop_dispatch(Warp& w, int m, int end, int bound, double ys, double yy) {
  switch ((w.n + 31) >> 5) {
    case 1: two_loop_tma<1>(w, m, end, bound, ys, yy); break;
    case 2: two_loop_tma<2>(w, m, end, bound, ys, yy); break;
    case 3: two_loop_tma<3>(w, m, end, bound, ys, yy); break;
    case 4: two_loop_tma<4>(w, m, end, bound, ys, yy); break;
    case 5: two_loop_tma<5>(w, m, end, bound, ys, yy); break;
    case 6: two_loop_tma<6>(w, m, end, bound, ys, yy); break;
    case 7: two_loop_tma<7>(w, m, end, bound, ys, yy); break;
    case 8: two_loop_tma<8>(w, m, end, bound, ys, yy); break;
    default: lbfgs_two_loop(w, m, end, bound, ys, yy); break;    // very long trajectories: the rolled version
  }
}

__device__ __forceinline__ int lbfgs_param_check(const alore_lbfgs_params_t& prm, int n, int m) {   // lbfgs.hpp:456-500
  if (n <= 0) return LBFGSERR_INVALID_N;
  if (m <= 0) return LBFGSERR_INVALID_MEMSIZE;
  if (prm.g_epsilon < 0.0) return LBFGSERR_INVALID_GEPSILON;
  if (prm.past < 0) return LBFGSERR_INVALID_TESTPERIOD;
  if (prm.delta < 0.0) return LBFGSERR_INVALID_DELTA;
  if (prm.min_step < 0.0) return LBFGSERR_INVALID_MINSTEP;
  if (prm.max_step < prm.min_step) return LBFGSERR_INVALID_MAXSTEP;
  if (!(prm.f_dec_coeff > 0.0 && prm.f_dec_coeff < 1.0)) return LBFGSERR_INVALID_FDECCOEFF;
  if (!(prm.s_curv_coeff < 1.0 && prm.s_curv_coeff > prm.f_dec_coeff)) return LBFGSERR_INVALID_SCURVCOEFF;
  if (!(prm.machine_prec > 0.0)) return LBFGSERR_INVALID_MACHINEPREC;
  if (prm.max_linesearch <= 0) return LBFGSERR_INVALID_MAXLINESEARCH;
  return 0;
}

enum { A_START_OPT, A_START_LBFGS, A_INIT_DONE, A_ITER_BEGIN, A_LS_TRIAL, A_LS_DONE, A_LS_RET, A_LBFGS_RET, A_REQ_FINAL, A_FINAL, A_REQUEST, A_FINISH };

// Advances candidate b from the completion of its pending evaluation to its next evaluation request (or to the end
// of minco_plan).  Returns true while the candidate is unfinished.  Every branch is warp-uniform.
__device__ __noinline__ bool step_candidate(const WParams& kp, const BatchDev& bt, const ResultDev& out, const WaveDev& wd, int b,
                                            double* smem, double* slab) {
  const alore_params_t& P = kp.P;
  const int lane = lane_id();
  const int p0 = bt.piece_off[b], N = bt.piece_off[b + 1] - p0, n = 3 * N - 1;
  CandState* sp = wd.st + b;
  CandState s = *sp;
  Warp w;
  w.lane = lane; w.N = N; w.n = n; w.npad = (3 * N) & ~1; w.n6 = 6 * N; w.K = P.sparseResolution; w.S1 = 2 * w.K + 1;
  w.Nm = kp.Nmax;
  {
    double* q = smem;
    w.T1 = q; q += kp.Nmax; w.sumT = q; q += kp.Nmax + 1 + 3;
    q = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(q) + 15) & ~uintptr_t(15));
    w.mbar = q; q += TL_NB + 2;
    w.d = q; q += kp.npadmax;
    w.hbuf = q; w.stg = q;
  }
  w.x = wd.x + 3 * (size_t)p0; w.g = wd.g + 3 * (size_t)p0; w.xp = wd.xp + 3 * (size_t)p0; w.gp = wd.gp + 3 * (size_t)p0;
  w.cf = wd.cf + 12 * (size_t)p0; w.gC = wd.gC + 12 * (size_t)p0;
  w.pf = wd.pf + 64 * (size_t)b;
  w.lm_s = wd.hist + wd.hist_off[b];
  w.lm_y = w.lm_s + (size_t)wd.m * (w.npad + 4);
  w.ax = slab + kp.L.ax; w.ay = slab + kp.L.ay; w.cellP = slab + kp.L.cellP;
  w.sx = bt.start_xytheta[3 * (size_t)b]; w.sy = bt.start_xytheta[3 * (size_t)b + 1];
  double* dglob = wd.d + 3 * (size_t)p0;
  double* T1g = wd.T1 + p0;
  const bool cut = bt.if_cut[b] != 0;

  alore_lbfgs_params_t prm = s.stage == 0 ? P.path_lbfgs : P.lbfgs;
  if (s.stage == 0) prm.past = s.past;
  int m = min(prm.mem_size, kp.mcap);

  int act, ls = 0, ret = 0;
  double f = 0.0;
  bool d_dirty = false;
  if (s.phase == PH_NEW) {
    // MSPlanner::minco_plan prologue (optimizer.cpp:176-177)
    s.safeDis = fmin(dist_real(kp.map, w.sx, w.sy) * 0.85, P.safeDis);
    s.time_weight = P.pw_time;
    s.evals = 0; s.iters = 0; s.replan = 0; s.alg_bytes = 0.0; s.err[0] = s.err[1] = 0.0; s.cost = 0.0; s.status = 0; s.alm_iters = 0;
    act = A_START_OPT;
  } else if (s.phase == PH_FINAL) {
    act = A_FINAL;
  } else {
    for (int i = lane; i < n; i += 32) w.d[i] = dglob[i];
    __syncwarp();
    if (!s.skip) {
      f = assemble_gradient(w, P, s.stage, T1g, wd.gT + p0, s.f, s.tsum, s.time_weight);
      s.evals++;
      s.alg_bytes += 8.0 * (2 * n + 1) + (s.stage == 1 ? 32.0 * P.n_checkpoints * N * (w.K + 1) : 0.0);
    }
    act = s.phase == PH_INIT ? A_INIT_DONE : A_LS_DONE;
  }

#pragma unroll 1
  for (;;) {
    if (act == A_START_OPT) {
      // get_state (optimizer.cpp:222-249) + x0 (optimizer.cpp:277-286)
      for (int d = 0; d < 2; d++) {
        s.lam[d] = cut ? P.CutEqualLambda[d] : P.EqualLambda[d];
        s.rho[d] = cut ? P.CutEqualRho[d] : P.EqualRho[d];
      }
      const double tail_s0 = bt.final_state[6 * (size_t)b + 3];
      const double* ip = bt.inner_pts + 2 * (size_t)(p0 - b);
      for (int i = lane; i < 2 * (N - 1); i += 32) w.x[i] = ip[i];
      if (lane == 0) w.x[2 * (N - 1)] = tail_s0;
      const double T = bt.init_T[b];
      const double vt = T > 1.0 ? (sqrt(2.0 * T - 1.0) - 1.0) : (1.0 - sqrt(2.0 / T - 1.0));
      for (int i = lane; i < N; i += 32) w.x[2 * (N - 1) + 1 + i] = vt;
      __syncwarp();
      s.stage = 0;
      s.past = (fabs(tail_s0) < P.shot_path_horizon) ? P.shot_path_past : P.normal_past;   // optimizer.cpp:296-300
      prm = P.path_lbfgs; prm.past = s.past;
      m = min(prm.mem_size, kp.mcap);
      act = A_START_LBFGS;
    } else if (act == A_START_LBFGS) {
      const int bad = lbfgs_param_check(prm, n, m);
      if (bad) { ret = bad; s.fx = s.cost; act = A_LBFGS_RET; }   // lbfgs_optimize returns before touching f
      else { s.phase = PH_INIT; act = A_REQUEST; }
    } else if (act == A_INIT_DONE) {                         // lbfgs.hpp:524-551
      s.fx = f;
      if (lane == 0) w.pf[0] = s.fx;
      double ga = 0.0, xa = 0.0, dd = 0.0;
#pragma unroll 1
      for (int i = lane; i < n; i += 32) {
        const double gi = w.g[i];
        w.d[i] = -gi;
        ga = fmax(ga, fabs(gi));
        xa = fmax(xa, fabs(w.x[i]));
        dd += gi * gi;
      }
      ga = warp_max(ga); xa = warp_max(xa); dd = warp_sum(dd);
      __syncwarp();
      d_dirty = true;
      if (ga / fmax(1.0, xa) < prm.g_epsilon) { ret = LBFGS_CONVERGENCE; act = A_LBFGS_RET; }
      else { s.step = 1.0 / sqrt(dd); s.k = 1; s.end = 0; s.bound = 0; act = A_ITER_BEGIN; }
    } else if (act == A_ITER_BEGIN) {                        // lbfgs.hpp:553-600 + line search prologue :276-310
#pragma unroll 1
      for (int i = lane; i < n; i += 32) { w.xp[i] = w.x[i]; w.gp[i] = w.g[i]; }
      __syncwarp();
      s.count = 0; s.brackt = 0; s.touched = 0; s.mu = 0.0; s.nu = prm.max_step;
      if (!(s.step > 0.0)) { ls = LBFGSERR_INVALIDPARAMETERS; act = A_LS_RET; }
      else {
        const double dginit = wdot(w.gp, w.d, n, lane);
        if (0.0 < dginit) { ls = LBFGSERR_INCREASEGRADIENT; act = A_LS_RET; }
        else {
          s.finit = s.fx;
          s.dgtest = prm.f_dec_coeff * dginit;
          s.dstest = prm.s_curv_coeff * dginit;
          act = A_LS_TRIAL;
        }
      }
    } else if (act == A_LS_TRIAL) {
#pragma unroll 1
      for (int i = lane; i < n; i += 32) w.x[i] = w.xp[i] + s.step * w.d[i];
      __syncwarp();
      s.phase = PH_LS;
      act = A_REQUEST;
    } else if (act == A_LS_DONE) {                           // lbfgs.hpp:317-388
      s.fx = f;
      ++s.count;
      act = A_LS_RET;
      if (isinf(f) || isnan(f)) ls = LBFGSERR_INVALID_FUNCVAL;
      else if (prm.past > 0 && fabs(s.finit - f) / (fabs(s.finit) + 1.0) < prm.delta / prm.past) ls = s.count;   // lbfgs.hpp:326-329
      else {
        bool decided = false;
        if (f > s.finit + s.step * s.dgtest) { s.nu = s.step; s.brackt = 1; }
        else {
          if (wdot(w.g, w.d, n, lane) < s.dstest) s.mu = s.step;
          else { ls = s.count; decided = true; }
        }
        if (!decided) {
          if (prm.max_linesearch <= s.count) ls = LBFGSERR_MAXIMUMLINESEARCH;
          else if (s.brackt && (s.nu - s.mu) < prm.machine_prec * s.nu) ls = LBFGSERR_WIDTHTOOSMALL;
          else {
            if (s.brackt) s.step = 0.5 * (s.mu + s.nu);
            else s.step *= 2.0;
            if (s.step < prm.min_step) ls = LBFGSERR_MINIMUMSTEP;
            else {
              bool go = true;
              if (s.step > prm.max_step) {
                if (s.touched) { ls = LBFGSERR_MAXIMUMSTEP; go = false; }
                else { s.touched = 1; s.step = prm.max_step; }
              }
              if (go) act = A_LS_TRIAL;
            }
          }
        }
      }
    } else if (act == A_LS_RET) {                            // lbfgs.hpp:602-745
      if (ls < 0) {
#pragma unroll 1
        for (int i = lane; i < n; i += 32) { w.x[i] = w.xp[i]; w.g[i] = w.gp[i]; }
        __syncwarp();
        ret = ls;
        act = A_LBFGS_RET;
      } else {
        double ga = 0.0, xa = 0.0;
#pragma unroll 1
        for (int i = lane; i < n; i += 32) { ga = fmax(ga, fabs(w.g[i])); xa = fmax(xa, fabs(w.x[i])); }
        ga = warp_max(ga); xa = warp_max(xa);
        bool stop = false;
        if (ga / fmax(1.0, xa) < prm.g_epsilon) { ret = LBFGS_CONVERGENCE; stop = true; }
        if (!stop && 0 < prm.past) {
          if (prm.past <= s.k) {
            const double rate = fabs(w.pf[s.k % prm.past] - s.fx) / fmax(1.0, fabs(s.fx));
            if (rate < prm.delta) { ret = LBFGS_STOP; stop = true; }
          }
          if (!stop) {
            __syncwarp();
            if (lane == 0) w.pf[s.k % prm.past] = s.fx;
            __syncwarp();
          }
        }
        if (!stop && prm.max_iterations != 0 && prm.max_iterations <= s.k) { ret = LBFGSERR_MAXIMUMITERATION; stop = true; }
        if (stop) act = A_LBFGS_RET;
        else {
          ++s.k;
          double* sc = w.lm_s + (size_t)s.end * (w.npad + 4);
          double* yc = w.lm_y + (size_t)s.end * w.npad;
          double pys = 0.0, pyy = 0.0, pss = 0.0, pgg = 0.0;
#pragma unroll 1
          for (int i = lane; i < n; i += 32) {
            const double gpv = w.gp[i], gv = w.g[i];
            const double sv = w.x[i] - w.xp[i], yv = gv - gpv;
            sc[i] = sv; yc[i] = yv;
            pys += yv * sv; pyy += yv * yv; pss += sv * sv;
            pgg += gpv * gpv;
            w.d[i] = -gv;
          }
          const double ys = warp_sum(pys), yy = warp_sum(pyy);
          const double ss = warp_sum(pss), gg = warp_sum(pgg);
          if (lane == 0) { sc[w.npad] = ys; sc[w.npad + 1] = rcp_refine(ys); }
          __syncwarp();
          d_dirty = true;
          const double cau = ss * sqrt(gg) * prm.cautious_factor;
          s.iters++;
          if (ys > cau) {
            ++s.bound;
            s.bound = m < s.bound ? m : s.bound;
            s.alg_bytes += 8.0 * n * (4.0 * s.bound + 4.0);
            s.end = (s.end + 1) % m;
            const long long tl0 = clock64();
            two_loop_dispatch(w, m, s.end, s.bound, ys, yy);
            WDBG_ADD(8, clock64() - tl0); WDBG_ADD(9, s.bound);
          }
          s.step = 1.0;
          act = A_ITER_BEGIN;
        }
      }
    } else if (act == A_LBFGS_RET) {                         // back in MSPlanner::optimizer (optimizer.cpp:303-418)
      s.status = ret;
      s.cost = s.fx;
      if (s.stage == 0) {
        s.stage = 1;
        s.alm_iters = 0;
        prm = P.lbfgs;
        m = min(prm.mem_size, kp.mcap);
        act = A_START_LBFGS;
      } else {
        s.alm_iters++;
        const int cap = P.alm_max_outer > 0 ? min(P.alm_max_outer, ALORE_ALM_HARD_CAP) : ALORE_ALM_HARD_CAP;
        const double nrm = sqrt(s.err[0] * s.err[0] + s.err[1] * s.err[1]);
        if (nrm < (cut ? P.CutEqualTolerance[0] : P.EqualTolerance[0])) act = A_REQ_FINAL;
        else {
          s.lam[0] += s.rho[0] * s.err[0];
          s.lam[1] += s.rho[1] * s.err[1];
          for (int d = 0; d < 2; d++) {
            const double gm = cut ? P.CutEqualGamma[d] : P.EqualGamma[d];
            const double rm = cut ? P.CutEqualRhoMax[d] : P.EqualRhoMax[d];
            s.rho[d] = fmin((1 + gm) * s.rho[d], rm);
          }
          act = s.alm_iters >= cap ? A_REQ_FINAL : A_START_LBFGS;
        }
      }
    } else if (act == A_REQ_FINAL) {                         // Minco.setParameters(finalInnerpoints, finalpieceTime), optimizer.cpp:452-464
      s.phase = PH_FINAL;
      act = A_REQUEST;
    } else if (act == A_FINAL) {                             // check_final_collision + retry (optimizer.cpp:191-207)
      for (int i = lane; i < N; i += 32) w.T1[i] = T1g[i];
      __syncwarp();
      const int coll = final_collision(w, P, kp.map, nullptr);
      if (coll) {
        s.time_weight *= 0.75;
        s.replan++;
        act = s.replan < P.safeReplanMaxTime ? A_START_OPT : A_FINISH;
      } else {
        act = A_FINISH;
      }
    } else if (act == A_REQUEST) {
      // what the solve kernel needs: piece times from tau (VirtualT2RealT, optimizer.cpp:583-591) and the `inf` guard
      const double* tau = w.x + 2 * (N - 1) + 1;
      for (int i = lane; i < N; i += 32) {
        const double t = tau[i];
        T1g[i] = t > 0.0 ? ((0.5 * t + 1.0) * t + 1.0) : 1.0 / ((0.5 * t - 1.0) * t + 1.0);
      }
      s.skip = 0;
      if (s.phase != PH_FINAL) {
        const double ss = wdot(w.x, w.x, n, lane);
        if (sqrt(ss) > g_norm_guard) s.skip = 1;                      // costFunctionCallback returns `inf` (= 0) without touching g
        if (d_dirty) for (int i = lane; i < n; i += 32) dglob[i] = w.d[i];
      }
      break;
    } else {                                                 // A_FINISH
      const bool ok = s.replan != P.safeReplanMaxTime;
      if (lane == 0) {
        out.ok[b] = ok ? 1 : 0;
        out.status[b] = s.status;
        out.replans[b] = min(s.replan + 1, P.safeReplanMaxTime);
        out.alm_iters[b] = s.alm_iters;
        out.evals[b] = s.evals;
        out.cost[b] = s.cost;
        out.tail_s[b] = w.x[2 * (N - 1)];
        out.alg_bytes[b] = s.alg_bytes;
        out.iters[b] = s.iters;
      }
      double* oi = out.inner_pts + 2 * (size_t)(p0 - b);
      for (int i = lane; i < 2 * (N - 1); i += 32) oi[i] = w.x[i];
      for (int i = lane; i < N; i += 32) out.piece_T[p0 + i] = T1g[i];
      for (int i = lane; i < 12 * N; i += 32) out.coeffs[12 * (size_t)p0 + i] = w.cf[i];
      s.phase = PH_DONE;
      break;
    }
  }
  __syncwarp();
  if (lane == 0) *sp = s;
  __syncwarp();
  return s.phase != PH_DONE;
}

__global__ void __launch_bounds__(32, 16)
wave_step_kernel(const __grid_constant__ WParams kp, BatchDev bt, ResultDev out, WaveDev wd, int cur, double* slabs) {
  extern __shared__ __align__(16) double smem[];
  double* slab = slabs + (size_t)blockIdx.x * kp.L.total;
  const int lane = threadIdx.x;
  const int* list = cur ? wd.list1 : wd.list0;
  int* nlist = cur ? wd.list0 : wd.list1;
  const int nact = wd.count[cur];
  {
    double* q = smem + kp.Nmax + kp.Nmax + 1 + 3;
    q = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(q) + 15) & ~uintptr_t(15));
    two_loop_tma_init(q);                            // the mbarriers of the history pipeline (same carve as step_candidate)
  }
#pragma unroll 1
  for (int slot = blockIdx.x; slot < nact; slot += gridDim.x) {
    const int b = list[slot];
    const long long ts0 = clock64();
    const bool alive = step_candidate(kp, bt, out, wd, b, smem, slab);
    WDBG_ADD(10, clock64() - ts0); WDBG_ADD(11, 1);
    if (alive && lane == 0) nlist[atomicAdd(&wd.count[cur ^ 1], 1)] = b;
    __syncwarp();
  }
}

// One evaluation at caller-supplied x for every candidate (alore_cost_batch): prepares the state the round kernels read.
__global__ void wave_cost_prepare_kernel(const __grid_constant__ WParams kp, BatchDev bt, WaveDev wd, int stage, const double* xs,
                                         const double* gs, const double* lam, const double* rho, const double* safe_dis) {
  const int b = blockIdx.x, lane = threadIdx.x;
  const int p0 = bt.piece_off[b], N = bt.piece_off[b + 1] - p0, n = 3 * N - 1;
  double* x = wd.x + 3 * (size_t)p0;
  double* g = wd.g + 3 * (size_t)p0;
  const size_t xo = 3 * (size_t)p0 - b;
  for (int i = lane; i < n; i += 32) { x[i] = xs[xo + i]; g[i] = gs[xo + i]; }
  __syncwarp();
  const double* tau = x + 2 * (N - 1) + 1;
  for (int i = lane; i < N; i += 32) {
    const double t = tau[i];
    wd.T1[p0 + i] = t > 0.0 ? ((0.5 * t + 1.0) * t + 1.0) : 1.0 / ((0.5 * t - 1.0) * t + 1.0);
  }
  const double ss = wdot(x, x, n, lane);
  if (lane == 0) {
    CandState s{};
    s.phase = PH_INIT; s.stage = stage; s.skip = sqrt(ss) > g_norm_guard ? 1 : 0;
    for (int d = 0; d < 2; d++) {
      s.lam[d] = lam ? lam[2 * b + d] : kp.P.EqualLambda[d];
      s.rho[d] = rho ? rho[2 * b + d] : kp.P.EqualRho[d];
    }
    s.safeDis = safe_dis ? safe_dis[b] : kp.P.safeDis;
    s.time_weight = kp.P.pw_time;
    wd.st[b] = s;
    wd.list0[b] = b;
    if (b == 0) { wd.count[0] = wd.B; wd.count[1] = 0; }
  }
}
__global__ void wave_cost_finish_kernel(const __grid_constant__ WParams kp, BatchDev bt, WaveDev wd, double* cost, double* gs, double* err) {
  const int b = blockIdx.x, lane = threadIdx.x;
  const int p0 = bt.piece_off[b], N = bt.piece_off[b + 1] - p0, n = 3 * N - 1;
  const CandState s = wd.st[b];
  Warp w;
  w.lane = lane; w.N = N; w.n = n; w.n6 = 6 * N;
  w.x = wd.x + 3 * (size_t)p0; w.g = wd.g + 3 * (size_t)p0;
  w.cf = wd.cf + 12 * (size_t)p0; w.gC = wd.gC + 12 * (size_t)p0;
  double f = 0.0;
  if (!s.skip) f = assemble_gradient(w, kp.P, s.stage, wd.T1 + p0, wd.gT + p0, s.f, s.tsum, s.time_weight);
  const size_t xo = 3 * (size_t)p0 - b;
  for (int i = lane; i < n; i += 32) gs[xo + i] = w.g[i];
  if (lane == 0) {
    cost[b] = f;
    if (err) { err[2 * b] = s.err[0]; err[2 * b + 1] = s.err[1]; }
  }
}

// attachPenaltyFunctional on given coefficients (BASELINE configs[2]), one CTA per trajectory, reading the caller's
// coefficient / duration arrays and accumulating straight into the caller's gradient arrays.
template <int NT, int MINB, bool SH>
__global__ void __launch_bounds__(NT, MINB)
penalty_cta_kernel(const __grid_constant__ WParams kp, int B, const int* piece_off, const double* coeffs, const double* Ts,
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
    pen_carve<SH>(w, kp.L, smem, slab, kp.Nmax, N, kp.P.sparseResolution);
    w.cf = const_cast<double*>(coeffs) + 12 * (size_t)p0;
    w.gC = gradC + 12 * (size_t)p0;
    w.sx = start_xy[2 * b]; w.sy = start_xy[2 * b + 1];
    w.fx = final_xy[2 * b]; w.fy = final_xy[2 * b + 1];
    for (int d = 0; d < 2; d++) { w.lam[d] = kp.P.EqualLambda[d]; w.rho[d] = kp.P.EqualRho[d]; }
    w.safeDis = kp.P.safeDis;
    w.init_pos = nullptr;
    tsync<NT>();
    for (int i = tid; i < 12 * N; i += NT) w.gC[i] = 0.0;
    for (int i = tid; i < N; i += NT) { w.T1[i] = Ts[p0 + i]; w.gT[i] = 0.0; }
    tsync<NT>();
    const double f = penalty_passes_t<NT, SH>(w, kp.P, kp.map, 1, 0.0);
    for (int i = tid; i < N; i += NT) gradT[p0 + i] = w.gT[i];
    if (tid == 0) { cost[b] = f; err[2 * b] = w.err[0]; err[2 * b + 1] = w.err[1]; }
  }
}

}  // namespace wave
