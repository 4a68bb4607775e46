// esdf.cu — occupancy grid -> signed ESDF, integer-exact separable squared EDT (sm_100a).
//
// Replaces the body of SDFmap::updateESDF2d / fillESDF
// (reference: planning_ddr_opt/utils/plan_env/src/sdf_map.cpp:618-715).
//
// Data flow (window of NX x NY cells, y contiguous):
//   K1  esdf_row_pass   uint8 occupancy -> int16 SIGNED row distance R(x,y):
//                         free/unknown cell : +d to the nearest Occupied cell in its row (+32767: none)
//                         Occupied cell     : -d to the nearest non-Occupied cell in its row (-32767: none)
//                       One value encodes both of the reference's first passes because a cell is a seed of
//                       exactly one of the two transforms (sdf_map.cpp:635 vs :655-657).
//   K2  esdf_col_pass   exact column transform  val(X) = min_x' (X-x')^2 + g(x')^2 :
//                         main sweep  — per thread a register window of its column (tile + halo staged in shared
//                                       memory): the first 8 search steps without loads or branches;
//                         deferred    — cells that need more (Occupied cells, longer searches) are compacted in
//                                       shared memory and finished with full lanes: expanding search inside the
//                                       32-row halo with the t*t >= best cut-off;
//                         far         — cells whose search leaves the halo (and 32-row bands that deferred every
//                                       cell) are handed to K2e through one mask word per (band, column) and one flag
//                                       per tile;
//                       then dist = gi*sqrt(val) and the reference's pos/neg combine (sdf_map.cpp:671-679).
//   K1b esdf_block_min  per (32-row block, column) minima of g+ and g- (candidate selection of K2e), only in the
//                       128-column tiles where K2 left far cells;
//   K2e esdf_band_kernel  FAR cells: one thread per (32- or 64-row band, column) streams the band's candidate rows
//                       (selected with the block minima) through Felzenszwalb's stack restricted to what the band can
//                       see, then answers the band's rows by a pointer walk — O(reach + band) per band instead of
//                       O(reach) per cell; exact integer tests evaluated in FP64 (all products < 2^53).
//   K2q esdf_quirk_col  ref_compat: window-local column 0 is recomputed from the aliased input the
//                       reference actually reads (SURVEY.md section 8a-E1 / Appendix B2); side stream.
// All arithmetic on squared distances is int32 (exact); the only FP ops are sqrt.rn.f64, mul.rn.f64 and
// add.rn.f64, IEEE-identical to the CPU.  Traffic: 1 B/cell in, 2+2 B/cell intermediate (L2-resident at 4096^2),
// 8 B/cell out; on cluttered maps the kernels are ALU-issue bound at 0.37 of the 13 B/cell HBM roofline, on maps
// with large empty / solid regions K2e dominates (DESIGN.md section 6).
#include <algorithm>
#include <vector>
#include <cstdio>
#include <cfloat>
#include <mutex>
#include <type_traits>

#include "common.cuh"

namespace {

constexpr int SENT = 32767;
constexpr int SQ_SENT = SENT * SENT;  // 1073676289: anything >= this is "no seed" (DBL_MAX in the reference)
constexpr int BLK = 32;               // rows per pruning block
constexpr int TX = 64, TY = 128, HALO = 32;   // halo rows >= W + U - 1 of the register window
constexpr int ROW_THREADS = 256;

__device__ __forceinline__ int excl_scan_max(int v, int* s_warp, int ident) {
  // exclusive max-scan over the CTA in thread order; s_warp has blockDim/32 slots
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc = max(inc, t);
  }
  if (lane == 31) s_warp[w] = inc;
  __syncthreads();
  int carry = ident;
  for (int i = 0; i < w; i++) carry = max(carry, s_warp[i]);
  int ex = __shfl_up_sync(0xffffffffu, inc, 1);
  if (lane == 0) ex = ident;
  __syncthreads();
  (void)nw;
  return max(carry, ex);
}
__device__ __forceinline__ int excl_scan_min_rev(int v, int* s_warp, int ident) {
  // exclusive min-scan from the right (thread t gets min over threads > t)
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_down_sync(0xffffffffu, inc, o);
    if (lane + o < 32) inc = min(inc, t);
  }
  if (lane == 0) s_warp[w] = inc;
  __syncthreads();
  int carry = ident;
  for (int i = w + 1; i < nw; i++) carry = min(carry, s_warp[i]);
  int ex = __shfl_down_sync(0xffffffffu, inc, 1);
  if (lane == 31) ex = ident;
  __syncthreads();
  return min(carry, ex);
}

// K1: one CTA per window row.  Dynamic smem: [NY+32 bytes occupancy][NY int16 forward distances].
__global__ void __launch_bounds__(ROW_THREADS)
esdf_row_pass(const uint8_t* __restrict__ occ, size_t occ_total, int gly, int min_x, int min_y, int NX, int NY,
              int16_t* __restrict__ R, int pitch) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ int s_warp[ROW_THREADS / 32];
  const int X = blockIdx.x;
  const size_t row0 = (size_t)(X + min_x) * gly + min_y;
  const uint8_t* src = occ + row0;
  const int shift = (int)((uintptr_t)src & 15);
  const int nvec = (shift + NY + 15) >> 4;
  uint8_t* s_raw = smem;
  const int occ_bytes = ((NY + 31 + 15) >> 4) << 4;
  int16_t* s_d = reinterpret_cast<int16_t*>(smem + occ_bytes);
  {
    const bool aligned_ok = (((uintptr_t)occ & 15) == 0);  // then src - shift never precedes occ
    const long long off0 = (long long)row0 - shift;        // byte offset in occ of vector 0
    for (int v = threadIdx.x; v < nvec; v += ROW_THREADS) {
      const long long off = off0 + (long long)v * 16;
      if (aligned_ok && off + 16 <= (long long)occ_total) {
        reinterpret_cast<uint4*>(s_raw)[v] = *reinterpret_cast<const uint4*>(occ + off);
      } else {
        for (int b = 0; b < 16; b++) {
          const long long o = off + b;
          s_raw[v * 16 + b] = (o >= 0 && o < (long long)occ_total) ? occ[o] : 0;
        }
      }
    }
  }
  __syncthreads();
  const uint8_t* s_occ = s_raw + shift;

  const int CH = (NY + ROW_THREADS - 1) / ROW_THREADS;
  const int c0 = min(threadIdx.x * CH, NY), c1 = min(c0 + CH, NY);
  const int BIG = 1 << 29;
  int lastOcc = -1, lastFree = -1, firstOcc = BIG, firstFree = BIG;
  for (int y = c0; y < c1; y++) {
    if (s_occ[y] == ALORE_OCCUPIED) { lastOcc = y; if (firstOcc == BIG) firstOcc = y; }
    else { lastFree = y; if (firstFree == BIG) firstFree = y; }
  }
  int lo = excl_scan_max(lastOcc, s_warp, -1);
  int lf = excl_scan_max(lastFree, s_warp, -1);
  int no = excl_scan_min_rev(firstOcc, s_warp, BIG);
  int nf = excl_scan_min_rev(firstFree, s_warp, BIG);
  for (int y = c0; y < c1; y++) {
    int d;
    if (s_occ[y] == ALORE_OCCUPIED) { lo = y; d = (lf < 0) ? SENT : y - lf; }
    else { lf = y; d = (lo < 0) ? SENT : y - lo; }
    s_d[y] = (int16_t)d;
  }
  for (int y = c1 - 1; y >= c0; y--) {
    int d2;
    if (s_occ[y] == ALORE_OCCUPIED) {
      no = y;
      d2 = (nf == BIG) ? SENT : nf - y;
      s_d[y] = (int16_t)(-min((int)s_d[y], d2));
    } else {
      nf = y;
      d2 = (no == BIG) ? SENT : no - y;
      s_d[y] = (int16_t)min((int)s_d[y], d2);
    }
  }
  __syncthreads();
  // coalesced store (row start of R is 16-byte aligned: pitch % 8 == 0)
  int16_t* dst = R + (size_t)X * pitch;
  const int nv = NY >> 3;
  for (int v = threadIdx.x; v < nv; v += ROW_THREADS)
    reinterpret_cast<uint4*>(dst)[v] = reinterpret_cast<const uint4*>(s_d)[v];
  for (int y = (nv << 3) + threadIdx.x; y < NY; y += ROW_THREADS) dst[y] = s_d[y];
}

// Four block-wide exclusive scans in one pass (K1 fast path): max-scans from the left of a, b; min-scans from the
// right of c, d.  Warp-level shuffles, then the 8 warp aggregates of all four quantities are scanned together by
// warp 0 (lane = 8 * quantity + warp), two barriers in total.
__device__ __forceinline__ void excl_scan4(int& a, int& b, int& c, int& d, int (*s_agg)[ROW_THREADS / 32], int identMax, int identMin) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int ia = a, ib = b, ic = c, id = d;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int ta = __shfl_up_sync(0xffffffffu, ia, o), tb = __shfl_up_sync(0xffffffffu, ib, o);
    const int tc = __shfl_down_sync(0xffffffffu, ic, o), td = __shfl_down_sync(0xffffffffu, id, o);
    if (lane >= o) { ia = max(ia, ta); ib = max(ib, tb); }
    if (lane + o < 32) { ic = min(ic, tc); id = min(id, td); }
  }
  if (lane == 31) { s_agg[0][w] = ia; s_agg[1][w] = ib; }
  if (lane == 0) { s_agg[2][w] = ic; s_agg[3][w] = id; }
  if (w == 0 && (lane & 7) >= (int)(blockDim.x >> 5))                // CTAs of fewer than 8 warps (short rows): identities
    s_agg[lane >> 3][lane & 7] = (lane >> 3) < 2 ? identMax : identMin;
  // exclusive within the warp
  int ea = __shfl_up_sync(0xffffffffu, ia, 1), eb = __shfl_up_sync(0xffffffffu, ib, 1);
  int ec = __shfl_down_sync(0xffffffffu, ic, 1), ed = __shfl_down_sync(0xffffffffu, id, 1);
  if (lane == 0) { ea = identMax; eb = identMax; }
  if (lane == 31) { ec = identMin; ed = identMin; }
  __syncthreads();
  if (w == 0) {
    const int q = lane >> 3, i = lane & 7;            // quantity, warp index
    const bool isMax = q < 2;
    int v = s_agg[q][i];
    int inc = v;
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
      const int tu = __shfl_up_sync(0xffffffffu, inc, o), td2 = __shfl_down_sync(0xffffffffu, inc, o);
      if (isMax) { if (i >= o) inc = max(inc, tu); }
      else { if (i + o < 8) inc = min(inc, td2); }
    }
    const int xu = __shfl_up_sync(0xffffffffu, inc, 1), xd = __shfl_down_sync(0xffffffffu, inc, 1);   // both by all lanes
    int ex = isMax ? xu : xd;
    if (isMax && i == 0) ex = identMax;
    if (!isMax && i == 7) ex = identMin;
    s_agg[q][i] = ex;                                  // carry entering warp i
  }
  __syncthreads();
  a = max(s_agg[0][w], ea);
  b = max(s_agg[1][w], eb);
  c = min(s_agg[2][w], ec);
  d = min(s_agg[3][w], ed);
}

// K1 (fast path): rows that start on a 16-byte boundary.  Each thread owns GP consecutive groups of 16 cells;
// a group is one 16-byte load turned into two 16-bit masks (Occupied / not Occupied), nearest seeds inside the
// group come from clz/ffs on the masks, nearest seeds outside from block-wide scans of per-thread extremes.
constexpr int ROW_GP_MAX = 8;
__device__ __forceinline__ unsigned occ_mask4(unsigned w) {   // 4 cells -> 4 bits (bit i = byte i == Occupied)
  const unsigned e = __vcmpeq4(w, 0x02020202u) & 0x01010101u;
  return (e & 1u) | ((e >> 7) & 2u) | ((e >> 14) & 4u) | ((e >> 21) & 8u);
}
template <int GP>
__global__ void __launch_bounds__(ROW_THREADS)
esdf_row_pass16(const uint8_t* __restrict__ occ, size_t occ_total, int gly, int min_x, int min_y, int NX, int NY,
                int16_t* __restrict__ R, int pitch) {
  __shared__ int s_agg[4][ROW_THREADS / 32];
  const int X = blockIdx.x;
  const size_t row0 = (size_t)(X + min_x) * gly + min_y;
  const int G = (NY + 15) >> 4;
  const int g0 = threadIdx.x * GP;
  unsigned om[GP], fm[GP];
  const int BIG = 1 << 20;
  int lastOcc = -BIG, lastFree = -BIG, firstOcc = BIG, firstFree = BIG;
#pragma unroll
  for (int q = 0; q < GP; q++) {
    om[q] = 0u; fm[q] = 0u;
    const int g = g0 + q;
    if (g < G) {
      const size_t off = row0 + (size_t)g * 16;
      uint4 v;
      if (off + 16 <= occ_total) v = *reinterpret_cast<const uint4*>(occ + off);
      else {
        __align__(16) unsigned char b[16];
        for (int t = 0; t < 16; t++) b[t] = (off + t < occ_total) ? occ[off + t] : 0;
        v = *reinterpret_cast<uint4*>(b);
      }
      const unsigned o = occ_mask4(v.x) | (occ_mask4(v.y) << 4) | (occ_mask4(v.z) << 8) | (occ_mask4(v.w) << 12);
      const int rem = NY - g * 16;
      const unsigned valid = rem >= 16 ? 0xffffu : ((1u << rem) - 1u);
      om[q] = o & valid;
      fm[q] = ~o & valid;
      if (om[q]) { lastOcc = g * 16 + 31 - __clz(om[q]); if (firstOcc == BIG) firstOcc = g * 16 + __ffs(om[q]) - 1; }
      if (fm[q]) { lastFree = g * 16 + 31 - __clz(fm[q]); if (firstFree == BIG) firstFree = g * 16 + __ffs(fm[q]) - 1; }
    }
  }
  int lo = lastOcc, lf = lastFree, no = firstOcc, nf = firstFree;
  excl_scan4(lo, lf, no, nf, s_agg, -BIG, BIG);
  // nearest seed to the right of each owned group (suffix over the thread's own groups)
  int ro[GP], rf[GP];
  {
    int co = no, cf = nf;
#pragma unroll
    for (int q = GP - 1; q >= 0; q--) {
      ro[q] = co; rf[q] = cf;
      const int g = g0 + q;
      if (om[q]) co = g * 16 + __ffs(om[q]) - 1;
      if (fm[q]) cf = g * 16 + __ffs(fm[q]) - 1;
    }
  }
#pragma unroll
  for (int q = 0; q < GP; q++) {
    const int g = g0 + q;
    if (g < G) {
      // free/unknown cells: two running-distance recurrences (nearest Occupied from the left / from the right);
      // Occupied cells (few): nearest free cell by bit scans over the group's masks, patched in afterwards
      const int y0 = g * 16;
      int dl_o[16];
      {
        int eo = y0 - 1 - lo;                       // distance of cell -1 to the nearest Occupied cell on its left
#pragma unroll
        for (int i = 0; i < 16; i++) {
          eo = ((om[q] >> i) & 1u) ? 0 : eo + 1;
          dl_o[i] = eo;
        }
      }
      unsigned outw[8];
      {
        int eo = ro[q] - (y0 + 16);                 // distance of cell 16 to the nearest Occupied cell on its right
#pragma unroll
        for (int i = 15; i >= 0; i--) {
          eo = ((om[q] >> i) & 1u) ? 0 : eo + 1;
          const int v = min(min(dl_o[i], eo), SENT);        // 0 at Occupied cells (patched below)
          if (i & 1) outw[i >> 1] = (unsigned)v << 16;
          else outw[i >> 1] |= (unsigned)v;
        }
      }
      int16_t* dst = R + (size_t)X * pitch + y0;
      reinterpret_cast<uint4*>(dst)[0] = make_uint4(outw[0], outw[1], outw[2], outw[3]);
      reinterpret_cast<uint4*>(dst)[1] = make_uint4(outw[4], outw[5], outw[6], outw[7]);
      if (__popc(om[q]) <= 3) {                       // cluttered maps: a few bit scans
        for (unsigned m = om[q]; m; m &= m - 1) {
          const int i = __ffs(m) - 1;
          const unsigned fl = fm[q] & ((1u << i) - 1u), fr = fm[q] >> (i + 1);
          const int dl = fl ? i - (31 - __clz(fl)) : (y0 + i) - lf;      // lf = -BIG when the row has no free cell to the left
          const int dr = fr ? __ffs(fr) : rf[q] - (y0 + i);              // rf = BIG when none to the right
          dst[i] = (int16_t)(-min(min(dl, dr), SENT));
        }
      } else {                                        // solid regions: the same two recurrences, towards the nearest FREE cell
        int dl_f[16];
        int ef = min(y0 - 1 - lf, 2 * SENT);          // distance of cell -1 to the nearest free cell on its left
#pragma unroll
        for (int i = 0; i < 16; i++) {
          ef = ((fm[q] >> i) & 1u) ? 0 : ef + 1;
          dl_f[i] = ef;
        }
        ef = min(rf[q] - (y0 + 16), 2 * SENT);
#pragma unroll
        for (int i = 15; i >= 0; i--) {
          ef = ((fm[q] >> i) & 1u) ? 0 : ef + 1;
          if ((om[q] >> i) & 1u) {
            const unsigned v = (unsigned)(-min(min(dl_f[i], ef), SENT)) & 0xffffu;
            if (i & 1) outw[i >> 1] = (outw[i >> 1] & 0x0000ffffu) | (v << 16);
            else outw[i >> 1] = (outw[i >> 1] & 0xffff0000u) | v;
          }
        }
        reinterpret_cast<uint4*>(dst)[0] = make_uint4(outw[0], outw[1], outw[2], outw[3]);
        reinterpret_cast<uint4*>(dst)[1] = make_uint4(outw[4], outw[5], outw[6], outw[7]);
      }
      // carries for the next owned group
      if (om[q]) lo = y0 + 31 - __clz(om[q]);
      if (fm[q]) lf = y0 + 31 - __clz(fm[q]);
    }
  }
}

// K1b: block minima for K2e's candidate selection.  Four lanes share one group of 8 columns, each taking 8 of the block's 32
// rows (16-byte loads); minima of max(r,0) and max(-r,0) are kept as packed int16 pairs and combined by two xor
// shuffles.  grid (ceil(pitch/8/32), ceil(NX/BLK)), 128 threads = 32 column groups x 4 row quarters.
__device__ __forceinline__ unsigned max0_s2(unsigned v) { return __vmaxs2(v, 0u); }
__global__ void __launch_bounds__(128)
esdf_block_min(const int16_t* __restrict__ R, int pitch, int NX, int NY, uint32_t* __restrict__ blk, int blk_pitch,
               const int* __restrict__ colflag, int ncol, int epoch) {
  // runs after K2: only the 128-column tiles that left FAR cells need their minima (colflag == this run's epoch)
  if (colflag[min(2 * (int)blockIdx.x, ncol - 1)] != epoch && colflag[min(2 * (int)blockIdx.x + 1, ncol - 1)] != epoch) return;
  const int rq = threadIdx.x & 3;
  const int y0 = (blockIdx.x * 32 + (threadIdx.x >> 2)) * 8;
  const bool in = y0 < pitch;
  const int x0 = blockIdx.y * BLK + rq * (BLK / 4), x1 = min(x0 + BLK / 4, NX);
  const unsigned big = (unsigned)SENT | ((unsigned)SENT << 16);
  unsigned mp[4] = {big, big, big, big}, mn[4] = {big, big, big, big};
  if (in) {
#pragma unroll
    for (int x = x0; x < x0 + BLK / 4; x++) {
      if (x < x1) {
        const uint4 v = *reinterpret_cast<const uint4*>(R + (size_t)x * pitch + y0);
        const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 4; q++) {
          mp[q] = __vmins2(mp[q], max0_s2(w[q]));
          mn[q] = __vmins2(mn[q], max0_s2(__vnegss2(w[q])));
        }
      }
    }
  }
#pragma unroll
  for (int o = 1; o <= 2; o <<= 1)
#pragma unroll
    for (int q = 0; q < 4; q++) {
      mp[q] = __vmins2(mp[q], __shfl_xor_sync(0xffffffffu, mp[q], o));
      mn[q] = __vmins2(mn[q], __shfl_xor_sync(0xffffffffu, mn[q], o));
    }
  if (in && rq == 0) {
    uint32_t* dst = blk + (size_t)blockIdx.y * blk_pitch + y0;
    uint32_t o[8];
#pragma unroll
    for (int q = 0; q < 4; q++) {
      o[2 * q] = (mp[q] & 0xffffu) | ((mn[q] & 0xffffu) << 16);
      o[2 * q + 1] = (mp[q] >> 16) | (mn[q] & 0xffff0000u);
    }
    reinterpret_cast<uint4*>(dst)[0] = make_uint4(o[0], o[1], o[2], o[3]);
    reinterpret_cast<uint4*>(dst)[1] = make_uint4(o[4], o[5], o[6], o[7]);
  }
}

// sqrt(k) for k < SQRT_TBL, filled once per process by esdf_fill_sqrt_table with the device's own sqrt.rn.f64
// (so looking a value up is bit-identical to computing it); most squared distances of a cluttered map are small.
constexpr int SQRT_TBL = 4096;
__device__ double g_sqrt_tbl[SQRT_TBL];
__global__ void esdf_fill_sqrt_table() {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < SQRT_TBL) g_sqrt_tbl[k] = sqrt((double)k);
}

__device__ __forceinline__ double esdf_value(int best, bool neg, double gi) {
  double root;
  if (best < SQRT_TBL) root = g_sqrt_tbl[best];
  else root = (best >= SQ_SENT) ? sqrt(DBL_MAX) : sqrt((double)best);
  const double dv = __dmul_rn(gi, root);               // grid_interval_ * std::sqrt(val)
  return neg ? __dadd_rn(0.0, __dadd_rn(-dv, gi))      // all = pos(=0); all += (-neg + gi)
             : dv;
}

// Superband envelope (K2e): the exact column transform for the FAR cells of one column and one kind inside a superband
// of 32 * ENV_NJ rows, all at once.
//
// The expanding search pays O(distance to the nearest seed) per cell; in large empty or solid regions every cell
// repeats nearly the same walk.  Here the candidate rows of the whole superband [lo, hi] are selected once with the
// block minima (per 32-row sub-band j an upper bound U_j valid for each of its far rows: a block can matter only if
// d_near(j, block)^2 + min g^2 <= U_j for some j), streamed in ascending order through Felzenszwalb's stack
// (sdf_map.cpp:682-715) — the intersection test done by integer cross-multiplication, exact and division-free:
//     site q is dominated by (p, r)  <=>  (f_q - f_p)(r - q) >= (f_r - f_q)(q - p),   f_x = g(x)^2 + x^2
// — restricted to what the band can see:
//   * a new site is stored only if it beats the current top at X = hi (its range lies right of the top's: a site that
//     loses at hi owns nothing in the band, and neither does any later site it would have shielded),
//   * a stack of ONE site is replaced by a new site that is STRICTLY better at X = lo (the old one then loses on the
//     whole band).  The bottom pair only changes when the second site is the one just pushed, so this is the complete
//     bottom trim, and the stack base never moves.
// Both rules keep the chain convex and keep every owner of a row in [lo, hi] (checked against brute force on 2·10^5
// random columns, ties included); the stack never held more than (hi - lo + 1) + 2 sites.  The top two sites live in
// registers: a row costs no dependent memory access unless it pops.  The far rows are then answered by a pointer walk
// (owners are monotone).  O(candidate rows + band rows) per (superband, column).
// K2e hand-over buffer: [BAND_FLAG_WORDS flags][far-row masks][Occupied masks].  The flags sit at a FIXED place in front of
// the geometry-dependent mask planes, so a word that was a mask under another window shape can never be read as a flag;
// a flag is "set" when it holds the current run's epoch (never cleared, stale values are always older).
constexpr int BAND_FLAG_WORDS = 33024;          // (16384/64) x (16384/128) tiles + 128 tile columns, 256-byte multiple
constexpr int ENV_CAP = 512;                    // stack capacity; (rows of the superband) + 2 is what the band can need
// rows per superband = 32 * ENV_NJ (template parameter: 1 or 2 sub-bands; chosen by the host from the window size)
template <bool SQ>
__device__ __forceinline__ void esdf_store(int best, bool neg, int X, int y, int NY, double* __restrict__ dist, int gly, int min_x,
                                           int min_y, double gi, int32_t* __restrict__ pos_sq, int32_t* __restrict__ neg_sq) {
  if (SQ) {
    const int v = best >= SQ_SENT ? ALORE_SQ_INF : best;
    pos_sq[(size_t)X * NY + y] = neg ? 0 : v;
    neg_sq[(size_t)X * NY + y] = neg ? v : 0;
  } else {
    dist[(size_t)(X + min_x) * gly + y + min_y] = esdf_value(best, neg, gi);
  }
}

// upper bound for every row of [lo, hi] (one kind, one column) from the rows' own in-row distance and the block minima
__device__ __forceinline__ int esdf_band_bound(const uint32_t* __restrict__ blkc, int blk_pitch, int nblk, int NX, int lo, int hi,
                                               bool neg, int own_max) {
  auto mg = [&](int b) -> int {
    const uint32_t m = blkc[(size_t)b * blk_pitch];
    return neg ? (int)(m >> 16) : (int)(m & 0xffffu);
  };
  const int bL = lo / BLK, bH = hi / BLK;
  long long U = own_max < SENT ? (long long)own_max * own_max : (long long)0x7fffffff;   // val(X) <= g(X)^2
  for (int b = bL; b <= bH; b++) {
    const int m = mg(b);
    if (m < SENT) {
      const int b0 = b * BLK, b1 = min(b0 + BLK - 1, NX - 1);
      const int df = max(hi - b0, b1 - lo);
      U = min(U, (long long)df * df + (long long)m * m);
    }
  }
  // outwards, four blocks per side in flight (the minima are the only loads of this loop; reading a few blocks
  // past the last useful one is harmless)
  for (int d0 = 1;; d0 += 4) {
    int ma[4], mb[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int ba = bL - d0 - i, bb = bH + d0 + i;
      ma[i] = ba >= 0 ? mg(ba) : SENT;
      mb[i] = bb < nblk ? mg(bb) : SENT;
    }
    bool any = false;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int ba = bL - d0 - i, bb = bH + d0 + i;
      any = false;
      if (ba >= 0) {
        const int b0 = ba * BLK, b1 = b0 + BLK - 1;
        const int dn = lo - b1;
        if ((long long)dn * dn < U) {
          any = true;
          if (ma[i] < SENT) { const int df = hi - b0; U = min(U, (long long)df * df + (long long)ma[i] * ma[i]); }
        }
      }
      if (bb < nblk) {
        const int b0 = bb * BLK, b1 = min(b0 + BLK - 1, NX - 1);
        const int dn = b0 - hi;
        if ((long long)dn * dn < U) {
          any = true;
          if (mb[i] < SENT) { const int df = b1 - lo; U = min(U, (long long)df * df + (long long)mb[i] * mb[i]); }
        }
      }
      if (!any) break;
    }
    if (!any) break;
  }
  return (int)U;
}

#ifdef ALORE_BAND_STATS
__device__ unsigned long long g_band_dbg[8];   // developer counters: blocks seen / needed, rows seen / past the filter / stored, items
#define BAND_STAT(i, v) atomicAdd(&g_band_dbg[i], (unsigned long long)(v))
#else
#define BAND_STAT(i, v)
#endif
template <bool SQ, int ENV_NJ>
__device__ __noinline__ bool esdf_band_envelope(const int16_t* __restrict__ R, int pitch, const uint32_t* __restrict__ blk, int blk_pitch,
                                                int NX, int NY, const uint32_t* __restrict__ fm, int mpitch, int nbands, int j0, int j1,
                                                unsigned live, bool neg, int y, double* __restrict__ dist, int gly, int min_x, int min_y, double gi,
                                                int32_t* __restrict__ pos_sq, int32_t* __restrict__ neg_sq) {
  const int nblk = (NX + BLK - 1) / BLK;
  const uint32_t* blkc = blk + y;
  const int16_t* Rc = R + y;
  const unsigned flip = neg ? 0u : 0xffffffffu;               // rows of this kind: far & (occupied ^ flip)
  auto rows_of = [&](int j) -> unsigned {                     // masks of a tile without far cells are not written by K2
    if (!((live >> (j - j0)) & 1u)) return 0u;
    return fm[(size_t)j * mpitch] & (fm[(size_t)(nbands + j) * mpitch] ^ flip);
  };
  // 1. per sub-band: its far rows of this kind, their bound U_j; the candidate range is the hull of the reaches
  int Uj[ENV_NJ], loj[ENV_NJ], hij[ENV_NJ];
  int lo = NX, hi = -1, cl = NX, ch = -1;
  for (int j = j0; j < j1; j++) {
    const unsigned mk = rows_of(j);
    int U = -1, l = NX, h = -1;
    if (mk) {
      l = (j << 5) + __ffs(mk) - 1;
      h = (j << 5) + 31 - __clz(mk);
      U = esdf_band_bound(blkc, blk_pitch, nblk, NX, l, h, neg, SENT);
      const int reach = (int)sqrt((double)U) + 1;
      cl = min(cl, l - reach); ch = max(ch, h + reach);
      lo = min(lo, l); hi = h;
    }
    Uj[j - j0] = U; loj[j - j0] = l; hij[j - j0] = h;
  }
  cl = max(cl, 0); ch = min(ch, NX - 1);
  // 2. the stack of the candidate rows, ascending; top two sites in registers.  All products are integers below 2^53,
  //    so the tests are done in FP64 (exact) — one DMUL where the integer pipe needs four IMADs.
  unsigned long long stk[ENV_CAP];               // site: row x in the high word, f = g^2 + x^2 in the low word
  int top = -1;
  double vt = 0.0, vp = 0.0, ft = 0.0, fp = 0.0;
  bool overflow = false;
  const double lo2 = 2.0 * lo, hi2 = 2.0 * hi;
  unsigned Umax = 0u;
#pragma unroll
  for (int j = 0; j < ENV_NJ; j++)
    if (j < j1 - j0 && Uj[j] >= 0) Umax = max(Umax, (unsigned)Uj[j]);
  const int pad = neg ? -SENT : SENT;
  const size_t rstride = (size_t)pitch;
  const int bfirst = cl / BLK, blast = ch / BLK;
  uint32_t mq[8];                                  // block minima, eight blocks in flight
  for (int b = bfirst; b <= blast && !overflow; b++) {
    if (((b - bfirst) & 7) == 0) {
#pragma unroll
      for (int i = 0; i < 8; i++) mq[i] = blkc[(size_t)min(b + i, blast) * blk_pitch];
    }
    uint32_t mm = mq[0];
#pragma unroll
    for (int i = 0; i < 7; i++) mq[i] = mq[i + 1];
    const int b0 = b * BLK, b1 = min(b0 + BLK - 1, NX - 1);
    const int m = neg ? (int)(mm >> 16) : (int)(mm & 0xffffu);
    BAND_STAT(0, 1);
    if (m >= SENT) continue;
    bool need = false;
    for (int j = 0; j < j1 - j0 && !need; j++) {
      if (Uj[j] < 0) continue;
      const int dn = b1 < loj[j] ? loj[j] - b1 : (b0 > hij[j] ? b0 - hij[j] : 0);
      need = (long long)dn * dn + (long long)m * m <= (long long)Uj[j];
    }
    if (!need) continue;
    BAND_STAT(1, 1);
    const int16_t* rp = Rc + (size_t)b0 * rstride;          // walks down the column, 8 rows in flight
    int rr[8], rn[8];
#pragma unroll
    for (int i = 0; i < 8; i++) rr[i] = (b0 + i <= b1) ? (int)rp[i * rstride] : pad;
#pragma unroll 1
    for (int xb = b0; xb <= b1; xb += 8) {
      rp += 8 * rstride;
#pragma unroll
      for (int i = 0; i < 8; i++) rn[i] = (xb + 8 + i <= b1) ? (int)rp[i * rstride] : pad;   // next batch in flight
      const double xbd = (double)xb;
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int x = xb + i;
        const int g = neg ? max(-rr[i], 0) : max(rr[i], 0);    // a row of the other kind is a seed itself
        const int dnr = max(max(lo - x, x - hi), 0);
        // no seed of this kind in the row, or a site that cannot reach any far row of the band: never an owner
        BAND_STAT(2, 1);
        if (g >= SENT || (unsigned)(dnr * dnr) + (unsigned)(g * g) > Umax) continue;
        BAND_STAT(3, 1);
        const unsigned fi = (unsigned)(g * g) + (unsigned)(x * x);
        const double f = (double)fi, xd = xbd + (double)i;
        double bx = xd - vt, cf = f - ft;
        while (top >= 1 && (ft - fp) * bx >= cf * (vt - vp)) {
          top--;
          vt = vp; ft = fp;
          if (top >= 1) { const unsigned long long e = stk[top - 1]; vp = (double)(int)(e >> 32); fp = (double)(unsigned)e; }
          bx = xd - vt; cf = f - ft;
        }
        if (top >= 0 && cf >= hi2 * bx) continue;              // loses to the top at X = hi
        const unsigned long long site = ((unsigned long long)(unsigned)x << 32) | fi;
        if (top == 0 && cf < lo2 * bx) {                         // the only site loses the whole band
          stk[0] = site;
          vt = xd; ft = f;
          continue;
        }
        if (top + 1 >= ENV_CAP) { overflow = true; break; }
        BAND_STAT(4, 1);
        ++top;
        stk[top] = site;
        vp = vt; fp = ft; vt = xd; ft = f;
      }
#pragma unroll
      for (int i = 0; i < 8; i++) rr[i] = rn[i];
      if (overflow) break;
    }
  }
  if (overflow) return false;
  BAND_STAT(5, 1);
  BAND_STAT(6, hi - lo + 1);
  BAND_STAT(7, ch - cl + 1);
  // 3. the far rows of this kind, ascending, pointer walk
  int k = 0;
  double vk = 0.0, fk = 0.0, vn = 0.0, fn = 0.0;
  if (top >= 0) { vk = (double)(int)(stk[0] >> 32); fk = (double)(unsigned)stk[0]; }
  if (top >= 1) { vn = (double)(int)(stk[1] >> 32); fn = (double)(unsigned)stk[1]; }
  for (int j = j0; j < j1; j++) {
    unsigned mk = rows_of(j);
    while (mk) {
      const int X = (j << 5) + __ffs(mk) - 1;
      mk &= mk - 1;
      int best = SQ_SENT;
      if (top >= 0) {
        const double X2 = 2.0 * X;
        double ck = fk - X2 * vk;                              // cost_k(X) = f_k - 2 X v_k + X^2
        while (k < top) {
          const double cn = fn - X2 * vn;
          if (cn > ck) break;
          ck = cn; k++;
          vk = vn; fk = fn;
          if (k < top) { const unsigned long long e = stk[k + 1]; vn = (double)(int)(e >> 32); fn = (double)(unsigned)e; }
        }
        const double v = ck + (double)X * (double)X;
        best = v < (double)SQ_SENT ? (int)v : SQ_SENT;
      }
      esdf_store<SQ>(best, neg, X, y, NY, dist, gly, min_x, min_y, gi, pos_sq, neg_sq);
    }
  }
  return true;
}

// K2e: one thread per (superband of 32 * ENV_NJ rows, column).  far_mask[X / 32][y] holds the rows K2 left for this kernel,
// far_mask[nbands + X / 32][y] the Occupied ones among them.
template <bool SQ, int ENV_NJ>
__global__ void __launch_bounds__(128)
esdf_band_kernel(const int16_t* __restrict__ R, int pitch, const uint32_t* __restrict__ blk, int blk_pitch, int NX, int NY,
                 const uint32_t* __restrict__ far_mask, int mpitch, int nbands, int epoch, double* __restrict__ dist, int gly, int min_x,
                 int min_y, double gi, int32_t* __restrict__ pos_sq, int32_t* __restrict__ neg_sq) {
  const int y = blockIdx.x * 128 + threadIdx.x;
  if (y >= NY) return;
  const uint32_t* fm = far_mask + y;
  const int j0 = blockIdx.y * ENV_NJ, j1 = min(j0 + ENV_NJ, (NX + 31) / 32);
  // tiles of K2 (64 rows x 128 columns) that left nothing this run (flag != epoch): their masks are not even written
  const int* flag = reinterpret_cast<const int*>(far_mask) - BAND_FLAG_WORDS + blockIdx.x;
  unsigned live = 0u;
#pragma unroll
  for (int i = 0; i < ENV_NJ; i++)
    if (j0 + i < j1 && flag[(size_t)((j0 + i) >> 1) * gridDim.x] == epoch) live |= 1u << i;
  if (!live) return;
  unsigned any_p = 0u, any_n = 0u;
#pragma unroll
  for (int i = 0; i < ENV_NJ; i++) {
    if (!((live >> i) & 1u)) continue;
    const unsigned f = fm[(size_t)(j0 + i) * mpitch], o = fm[(size_t)(nbands + j0 + i) * mpitch];
    any_p |= f & ~o;
    any_n |= f & o;
  }
  bool ok_p = true, ok_n = true;
  if (any_p) ok_p = esdf_band_envelope<SQ, ENV_NJ>(R, pitch, blk, blk_pitch, NX, NY, fm, mpitch, nbands, j0, j1, live, false, y, dist, gly, min_x, min_y, gi, pos_sq, neg_sq);
  if (any_n) ok_n = esdf_band_envelope<SQ, ENV_NJ>(R, pitch, blk, blk_pitch, NX, NY, fm, mpitch, nbands, j0, j1, live, true, y, dist, gly, min_x, min_y, gi, pos_sq, neg_sq);
  if (ok_p && ok_n) return;
  // a stack that outgrew its array (never seen): plain exact search for the rows of that kind
  for (int j = j0; j < j1; j++) {
    unsigned mk = ((live >> (j - j0)) & 1u) ? fm[(size_t)j * mpitch] : 0u;
    while (mk) {
      const int X = (j << 5) + __ffs(mk) - 1;
      mk &= mk - 1;
      const int r0 = R[(size_t)X * pitch + y];
      const bool neg = r0 < 0;
      if (neg ? ok_n : ok_p) continue;
      int best = r0 * r0;
      for (int t = 1; t * t < best && (X - t >= 0 || X + t < NX); t++) {
        if (X - t >= 0) { const int r = R[(size_t)(X - t) * pitch + y]; const int g = neg ? max(-r, 0) : max(r, 0); best = min(best, g * g + t * t); }
        if (X + t < NX) { const int r = R[(size_t)(X + t) * pitch + y]; const int g = neg ? max(-r, 0) : max(r, 0); best = min(best, g * g + t * t); }
      }
      esdf_store<SQ>(best, neg, X, y, NY, dist, gly, min_x, min_y, gi, pos_sq, neg_sq);
    }
  }
}

// K2: column pass.  grid (ceil(NY/TY), ceil(NX/TX)), 256 threads = 128 columns x 2 row halves.
// A probe of row x' contributes t^2 + g(x')^2 where g is the row distance of the SAME kind as the query cell
// (0 for the other kind).  Free/unknown query cells (the overwhelming majority) take the fast path: g = max(R, 0),
// the tile is padded with +SENT outside the window so the loop carries no bounds checks, both sides of a step share
// one square (min(max(a,0), max(b,0)) = max(min(a,b), 0)), t^2 is a running sum.  Occupied query cells (g = max(-R, 0))
// take the general path.  sqrt of small squared distances comes from a shared-memory copy of the table.
constexpr int SQRT_SMEM = 128;    // the register-window path only looks up squared distances <= (W+1)^2 = 81
template <bool SQ>
__global__ void __launch_bounds__(256)
esdf_col_pass(const int16_t* __restrict__ R, int pitch, int NX, int NY, double* __restrict__ dist, int gly, int min_x, int min_y,
              double gi, int ref_compat, int32_t* __restrict__ pos_sq, int32_t* __restrict__ neg_sq, uint32_t* __restrict__ far_mask,
              int epoch) {
  __shared__ __align__(16) int16_t S[TX + 2 * HALO][TY];
  __shared__ unsigned s_far[256], s_farneg[256];                 // per thread: rows of its 32-row band left to K2e / the Occupied ones
  __shared__ int s_anyfar;
  s_far[threadIdx.x] = 0u;
  s_farneg[threadIdx.x] = 0u;
  if (threadIdx.x == 0) s_anyfar = 0;
  __shared__ double s_sqrt[SQ ? 1 : SQRT_SMEM];
  constexpr int DEF_CAP = 2048;                                  // deferred cells held in the list (25 % of a tile)
  __shared__ unsigned short s_list[DEF_CAP];
  __shared__ int s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  const int X0 = blockIdx.y * TX, Y0 = blockIdx.x * TY;
  const int rlo = X0 - HALO;
  const unsigned padw = (unsigned)SENT | ((unsigned)SENT << 16);
  {
    constexpr int NV = (TX + 2 * HALO) * (TY / 8) / 256;         // 16-byte vectors per thread: all loads first, then all stores
    uint4 val[NV];
#pragma unroll
    for (int q = 0; q < NV; q++) {
      const int idx = threadIdx.x + q * 256;
      const int row = idx / (TY / 8), v = idx % (TY / 8);
      const int xr = rlo + row, y = Y0 + v * 8;
      val[q] = make_uint4(padw, padw, padw, padw);
      if (xr >= 0 && xr < NX && y < pitch) val[q] = *reinterpret_cast<const uint4*>(R + (size_t)xr * pitch + y);
    }
#pragma unroll
    for (int q = 0; q < NV; q++) {
      const int idx = threadIdx.x + q * 256;
      *reinterpret_cast<uint4*>(&S[idx / (TY / 8)][(idx % (TY / 8)) * 8]) = val[q];
    }
  }
  if (!SQ)
    for (int k = threadIdx.x; k < SQRT_SMEM; k += 256) s_sqrt[k] = g_sqrt_tbl[k];
  __syncthreads();
  const int ty = threadIdx.x & (TY - 1), half = threadIdx.x / TY;
  const int y = Y0 + ty;
  const bool skip_thread = !SQ && ref_compat && y == NY - 1;     // the reference never writes the window's last column
  const int Xb = X0 + half * (TX / 2);
  int Xe = min(Xb + TX / 2, NX);
  if (!SQ && ref_compat) {
    Xe = min(Xe, NX - 1);                                        // ... nor its last row
    if (y == 0) Xe = min(Xe, 1);                                 // column 0, rows >= 1: esdf_quirk_col
  }
  double* out = dist + (size_t)(Xb + min_x) * gly + y + min_y;
  const int16_t* colp = &S[Xb - rlo][ty];
  // Register window of the column: g[i] = max(R, 0) of row X - W + i.  The first W steps of every search read it with
  // static indices (no loads, no branches: extra candidates cannot lower an exact minimum); four query rows share one
  // window position, then the window slides by four rows.  Cells that need more — Occupied query cells (g == 0) and
  // free cells whose search is not finished after W steps — are DEFERRED: each thread keeps a 32-bit mask of its rows,
  // the CTA compacts all deferred cells into a list and works it off with full lanes after the main sweep.
  constexpr int W = 8, U = 4;
  unsigned defer = 0u;
  if (y < NY && !skip_thread) {
    int g[2 * W + U];
#pragma unroll
    for (int i = 0; i < 2 * W + U; i++) g[i] = max((int)colp[(i - W) * TY], 0);
#define ALORE_K2_CELL(u)                                                                         \
    {                                                                                            \
      const int gc = g[W + (u)];                                                                 \
      int best = gc * gc;                                                                        \
      _Pragma("unroll") for (int k = 1; k <= W; k++) {                                           \
        const int m = min(g[W + (u) - k], g[W + (u) + k]);                                       \
        best = min(best, m * m + k * k);                                                         \
      }                                                                                          \
      if (gc == 0 || best > (W + 1) * (W + 1)) {                                                 \
        defer |= 1u << (X + (u) - Xb);                                                           \
      } else if (SQ) {                                                                           \
        pos_sq[(size_t)(X + (u)) * NY + y] = best;                                               \
        neg_sq[(size_t)(X + (u)) * NY + y] = 0;                                                  \
      } else {                                                                                   \
        out[(size_t)(u) * gly] = __dmul_rn(gi, s_sqrt[best]); /* best <= 81: gi * sqrt(val) */   \
      }                                                                                          \
    }
#pragma unroll 1
    for (int X = Xb; X < Xe; X += U, out += (size_t)U * gly, colp += U * TY) {
      if (X + U <= Xe) {                                   // whole group inside the tile: no per-cell guards
        ALORE_K2_CELL(0) ALORE_K2_CELL(1) ALORE_K2_CELL(2) ALORE_K2_CELL(3)
      } else {
        if (X + 0 < Xe) ALORE_K2_CELL(0)
        if (X + 1 < Xe) ALORE_K2_CELL(1)
        if (X + 2 < Xe) ALORE_K2_CELL(2)
      }
#pragma unroll
      for (int i = 0; i < 2 * W; i++) g[i] = g[i + U];
#pragma unroll
      for (int i = 0; i < U; i++) g[2 * W + i] = max((int)colp[(W + U + i) * TY], 0);
    }
#undef ALORE_K2_CELL
  }
  // ---- a band that defers all of its cells lies in a large empty / solid region: straight to K2e; so do the bands
  //      that do not fit the CTA's list (tiles with more than 25 % deferred cells) ------------------------------------
  constexpr int BAND_MIN = 32;
  auto band_to_far = [&]() {
    unsigned occm = 0u;                                               // the Occupied rows among them
    const int16_t* cs = &S[Xb - rlo][ty];
#pragma unroll
    for (int r = 0; r < 32; r++) occm |= (unsigned)(cs[r * TY] < 0) << r;
    s_far[threadIdx.x] = defer;                                       // own slot; the list below only ORs into it
    s_farneg[threadIdx.x] = occm & defer;
    s_anyfar = 1;
    defer = 0u;
  };
  if (__popc(defer) >= BAND_MIN) band_to_far();
  // ---- deferred cells: compact (thread, row) pairs into shared memory, then one cell per thread per round -----------
  {
    const int cntme = __popc(defer);
    int base = DEF_CAP;
    if (cntme) base = atomicAdd(&s_cnt, cntme);
    if (base + cntme <= DEF_CAP) {
      unsigned mk = defer;
      while (mk) {
        const int r = __ffs(mk) - 1;
        mk &= mk - 1;
        s_list[base++] = (unsigned short)((threadIdx.x << 5) | r);    // thread (8 bits) : row offset (5 bits)
      }
      defer = 0u;
    } else {                                                          // list full
      for (int i = base; i < min(base + cntme, DEF_CAP); i++) s_list[i] = 0xffffu;   // reserved but unused slots
      band_to_far();                                                  // ... K2e takes the band
    }
  }
  __syncthreads();
  const int ndef = min(s_cnt, DEF_CAP);
  // A thread's cells sit next to each other in the list and share ONE shared-memory bank (same column, row stride of
  // 64 words): the lanes of a warp walk the list 33 entries apart (odd multiplier modulo a power of two: a bijection),
  // i.e. in different columns.
  int lmod = 256;
  while (lmod < ndef) lmod <<= 1;
  for (int idx = threadIdx.x; idx < lmod; idx += 256) {
    const int slot = (idx * 33) & (lmod - 1);
    if (slot >= ndef) continue;
    const unsigned e = s_list[slot];
    if ((e >> 5) >= 256) continue;                                    // slot reserved by a thread that did not fit
    const int th = e >> 5, r = e & 31;
    const int cty = th & (TY - 1), chalf = th / TY;
    const int X = X0 + chalf * (TX / 2) + r, yy = Y0 + cty;
    const int16_t* col = &S[X - rlo][cty];
    const int r0 = col[0];
    const bool neg = r0 < 0;
    int best = r0 * r0;
    int t = 1;
    // Row by row inside the halo while the running bound is small; a cell whose bound is still far beyond the halo
    // after TSW rows (deep inside a large solid / empty region) goes to K2e right away instead of walking all 32 halo
    // rows first.
    constexpr int TSW = 6, FAR2 = (HALO + 1) * (HALO + 1);
    if (!neg) {
      for (; t <= HALO; ++t) {
        const int tt = t * t;
        if (tt >= best || (t > TSW && best > FAR2)) break;
        const int m = max(min((int)col[-t * TY], (int)col[t * TY]), 0);
        best = min(best, m * m + tt);
      }
    } else {
      for (; t <= HALO; ++t) {
        const int tt = t * t;
        if (tt >= best || (t > TSW && best > FAR2)) break;
        if (X - t >= 0) { const int a = max(-(int)col[-t * TY], 0); best = min(best, a * a + tt); }
        if (X + t < NX) { const int b = max(-(int)col[t * TY], 0); best = min(best, b * b + tt); }
      }
    }
    if (t * t < best && (X - t >= 0 || X + t < NX)) {    // rows left to look at: a FAR cell, left to K2e
      atomicOr(&s_far[th], 1u << r);
      if (neg) atomicOr(&s_farneg[th], 1u << r);
      s_anyfar = 1;
      continue;
    }
    if (SQ) {
      const int v = best >= SQ_SENT ? ALORE_SQ_INF : best;
      pos_sq[(size_t)X * NY + yy] = neg ? 0 : v;
      neg_sq[(size_t)X * NY + yy] = neg ? v : 0;
    } else {
      double root;
      if (best < SQRT_SMEM) root = s_sqrt[best];
      else if (best < SQRT_TBL) root = g_sqrt_tbl[best];
      else root = (best >= SQ_SENT) ? sqrt(DBL_MAX) : sqrt((double)best);
      const double dv = __dmul_rn(gi, root);                     // grid_interval_ * std::sqrt(val)
      dist[(size_t)(X + min_x) * gly + yy + min_y] = neg ? __dadd_rn(0.0, __dadd_rn(-dv, gi)) : dv;   // all = pos(=0); all += (-neg + gi)
    }
  }
  __syncthreads();                                       // dense: every (32-row band, column) of the tile is written
  const int anyfar = s_anyfar;
  if (anyfar && y < pitch) {
    far_mask[(size_t)(blockIdx.y * 2 + half) * pitch + y] = s_far[threadIdx.x];
    far_mask[(size_t)(gridDim.y * 2 + blockIdx.y * 2 + half) * pitch + y] = s_farneg[threadIdx.x];
  }
  if (anyfar && threadIdx.x == 0) {                      // flags in front of the mask planes: one per tile, one per tile column;
    int* flags = reinterpret_cast<int*>(far_mask) - BAND_FLAG_WORDS;                   // "set" = this run's epoch, never cleared
    flags[blockIdx.y * gridDim.x + blockIdx.x] = epoch;
    flags[gridDim.y * gridDim.x + blockIdx.x] = epoch;
  }
}

// K2q: the reference's aliased column (ref_compat).  Window-local column 0, rows X = 1..NX-1, is the 1-D
// transform over the virtual column W(j), j in [1, NX]:  W(j) = R(j, 0) for j <= NX-1, W(NX) = R(NX-1, NY-1),
// evaluated at j = X  (sdf_map.cpp:639-650: index x*update_Y_SIZE + y with y == update_Y_SIZE aliases row x+1).
template <bool SQ>
__global__ void __launch_bounds__(256)
esdf_quirk_col(const int16_t* __restrict__ R, int pitch, int NX, int NY, double* __restrict__ dist, int gly,
               int min_x, int min_y, double gi, int32_t* __restrict__ pos_sq, int32_t* __restrict__ neg_sq) {
  // one WARP per cell: lane l probes the steps t0 + l of the expanding search, the cut-off t^2 >= best is applied per
  // chunk of 32 steps (extra probes cannot lower an exact minimum)
  const int lane = threadIdx.x & 31;
  const int X = 1 + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (X > NX - 1) return;
  if (!SQ && X > NX - 2) return;
  auto W = [&](int j) -> int { return j <= NX - 1 ? R[(size_t)j * pitch] : R[(size_t)(NX - 1) * pitch + (NY - 1)]; };
  const int r0 = W(X);
  const bool neg = r0 < 0;
  int best = r0 * r0;
  for (int t0 = 1; t0 * t0 < best; t0 += 32) {
    const int t = t0 + lane, tt = t * t;
    const bool lo_ok = X - t >= 1, hi_ok = X + t <= NX;
    int loc = 0x7fffffff;
    if (lo_ok) { const int r = W(X - t); loc = min(loc, tt + (((r < 0) == neg) ? r * r : 0)); }
    if (hi_ok) { const int r = W(X + t); loc = min(loc, tt + (((r < 0) == neg) ? r * r : 0)); }
    best = min(best, __reduce_min_sync(0xffffffffu, loc));
    if (!__any_sync(0xffffffffu, lo_ok || hi_ok)) break;
  }
  if (lane) return;
  if (SQ) {
    const int v = best >= SQ_SENT ? ALORE_SQ_INF : best;
    pos_sq[(size_t)X * NY] = neg ? 0 : v;
    neg_sq[(size_t)X * NY] = neg ? v : 0;
  } else {
    dist[(size_t)(X + min_x) * gly + min_y] = esdf_value(best, neg, gi);
  }
}

}  // namespace

// Runs K1..K2q on `st`.  d_pos_sq/d_neg_sq != NULL: squared-distance dump of the retained row pass of the
// last update instead of writing distances (parity tests).
int alore_esdf_run(alore_ctx* ctx, const alore_map_geom_t* geom, const uint8_t* d_occ, double* d_dist, int min_x, int min_y, int max_x,
                   int max_y, int ref_compat, cudaStream_t st, int32_t* d_pos_sq, int32_t* d_neg_sq) {
  const int NX = max_x - min_x + 1, NY = max_y - min_y + 1;
  const alore_map_geom_t& g = *geom;
  if (NX <= 0 || NY <= 0 || min_x < 0 || min_y < 0 || max_x >= g.glx || max_y >= g.gly)
    return alore_fail(ctx, ALORE_EINVAL, "esdf window [%d,%d]x[%d,%d] outside the %dx%d grid", min_x, max_x, min_y, max_y, g.glx, g.gly);
  if (NX > 16384 || NY > 16384)
    return alore_fail(ctx, ALORE_EINVAL, "esdf window %dx%d exceeds the int16/int32 exactness limit 16384", NX, NY);
  const bool sq = d_pos_sq != nullptr;
  {
    // the sqrt table is per device and filled once; guarded because contexts of several devices may be driven by several host threads
    static std::mutex tbl_mu;
    static bool tbl_ready[64] = {false};
    std::lock_guard<std::mutex> lk(tbl_mu);
    if (ctx->device < 64 && !tbl_ready[ctx->device]) {
      esdf_fill_sqrt_table<<<SQRT_TBL / 256, 256, 0, st>>>();
      ALORE_CUDA(ctx, cudaStreamSynchronize(st));   // other streams / contexts may use the table next
      ctx->launches++;
      tbl_ready[ctx->device] = true;
    }
  }
  const int pitch = ((NY + TY - 1) / TY) * TY;
  const int nblk = (NX + BLK - 1) / BLK;
  // far-cell masks of the superband envelope kernel (K2e): one word per (32-row band, column), rewritten by every K2;
  // flags (fixed size, in front), then per (32-row band, column) the far rows and the Occupied ones among them
  const size_t need_band = ((size_t)BAND_FLAG_WORDS + (size_t)(4 * ((NX + TX - 1) / TX)) * pitch) * sizeof(uint32_t);
  if (need_band > ctx->band_cap) {
    if (ctx->d_band) { cudaDeviceSynchronize(); cudaFree(ctx->d_band); }
    ctx->d_band = nullptr; ctx->band_cap = 0;
    ALORE_CUDA(ctx, cudaMalloc(&ctx->d_band, need_band));
    // flags compare against a per-run epoch >= 1; zeroed on `st`, ahead of the K2 that reads them (a caller stream
    // created non-blocking is not ordered after work on the legacy default stream)
    ALORE_CUDA(ctx, cudaMemsetAsync(ctx->d_band, 0, need_band, st));
    ctx->band_cap = need_band;
    ctx->band_epoch = 0;
  }
  uint32_t* const far_mask = static_cast<uint32_t*>(ctx->d_band) + BAND_FLAG_WORDS;
  const int epoch = ++ctx->band_epoch;
  const int ncol_tiles = (NY + TY - 1) / TY;
  const int* colflag = reinterpret_cast<const int*>(far_mask) - BAND_FLAG_WORDS + (size_t)((NX + TX - 1) / TX) * ncol_tiles;

  if (!sq) {
    const size_t need_row = (size_t)NX * pitch, need_blk = (size_t)nblk * pitch;
    if (need_row > ctx->row_cap) {
      if (ctx->d_row) cudaFree(ctx->d_row);
      ctx->d_row = nullptr;
      ALORE_CUDA(ctx, cudaMalloc(&ctx->d_row, need_row * sizeof(int16_t)));
      // columns NY..pitch-1 travel through K2's 16-byte tile loads but no output depends on them.  They are defined
      // here once, as "far from any seed"; after that they hold whatever was last stored there: the fast row pass
      // writes whole 16-cell groups (finite distances up to column 16*ceil(NY/16)-1), and an earlier, wider window of
      // the same pitch leaves its own (also negative) values.  Zeroed on `st`, ahead of the row pass.
      ALORE_CUDA(ctx, cudaMemsetAsync(ctx->d_row, 0x7f, need_row * sizeof(int16_t), st));
      ctx->row_cap = need_row;
    }
    if (need_blk > ctx->blk_cap) {
      if (ctx->d_blk) cudaFree(ctx->d_blk);
      ctx->d_blk = nullptr;
      ALORE_CUDA(ctx, cudaMalloc(&ctx->d_blk, need_blk * sizeof(uint32_t)));
      ctx->blk_cap = need_blk;
    }
    ctx->row_pitch = pitch;
    ctx->win[0] = min_x; ctx->win[1] = min_y; ctx->win[2] = max_x; ctx->win[3] = max_y;
    ctx->win_geom = g;
    ctx->last_ref_compat = ref_compat;
    const size_t smem = (size_t)(((NY + 31 + 15) >> 4) << 4) + (size_t)NY * 2 + 16;
    if (smem > 48 * 1024)
      ALORE_CUDA(ctx, cudaFuncSetAttribute(esdf_row_pass, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int G16 = (NY + 15) / 16;
    const int GP = (G16 + ROW_THREADS - 1) / ROW_THREADS;
    const bool fast = (((uintptr_t)d_occ & 15) == 0) && (g.gly % 16 == 0) && (min_y % 16 == 0) && GP <= ROW_GP_MAX;
    const size_t occ_total = (size_t)g.glx * g.gly;
    if (fast && GP <= 1)                               // one 16-cell group per thread: no idle warps on short rows
      esdf_row_pass16<1><<<NX, std::min(ROW_THREADS, ((G16 + 31) / 32) * 32), 0, st>>>(d_occ, occ_total, g.gly, min_x, min_y, NX, NY, ctx->d_row, pitch);
    else if (fast && GP <= 2)
      esdf_row_pass16<2><<<NX, ROW_THREADS, 0, st>>>(d_occ, occ_total, g.gly, min_x, min_y, NX, NY, ctx->d_row, pitch);
    else if (fast && GP <= 4)
      esdf_row_pass16<4><<<NX, ROW_THREADS, 0, st>>>(d_occ, occ_total, g.gly, min_x, min_y, NX, NY, ctx->d_row, pitch);
    else if (fast)
      esdf_row_pass16<8><<<NX, ROW_THREADS, 0, st>>>(d_occ, occ_total, g.gly, min_x, min_y, NX, NY, ctx->d_row, pitch);
    else
      esdf_row_pass<<<NX, ROW_THREADS, smem, st>>>(d_occ, (size_t)g.glx * g.gly, g.gly, min_x, min_y, NX, NY, ctx->d_row, pitch);
    if (ref_compat && NX >= 3 && NY >= 2) ALORE_CUDA(ctx, cudaEventRecord(ctx->ev_fork, st));   // the aliased column forks here
    ctx->launches++;
  } else if (ctx->row_pitch != pitch || !ctx->d_row) {
    return alore_fail(ctx, ALORE_EINVAL, "no retained row pass for this window");
  }
  const dim3 grid((NY + TY - 1) / TY, (NX + TX - 1) / TX);
  const bool quirk = ref_compat && NX >= 2 && NY >= 2;
  if (ref_compat && !quirk && !sq) return ALORE_OK;  // update_X_SIZE or update_Y_SIZE == 0: the reference writes nothing
  // superband height: tall bands amortise the candidate scan (O(reach + band) per thread), short ones give more threads
  const int band_nj = (size_t)NX * NY < ((size_t)8 << 20) ? 1 : 2;    // measured: 32 rows on 2048^2 (more threads), 64 on 16 Mcells
  const dim3 band_grid((NY + 127) / 128, (NX + 32 * band_nj - 1) / (32 * band_nj));
  // K2, then the block minima of the tile columns where it left far cells (K1b), then those cells (K2e)
  auto column_pass = [&](auto sq_tag, double* dist, int32_t* pos_sq, int32_t* neg_sq) {
    constexpr bool SQ = decltype(sq_tag)::value;
    esdf_col_pass<SQ><<<grid, 256, 0, st>>>(ctx->d_row, pitch, NX, NY, dist, g.gly, min_x, min_y, g.grid_interval, ref_compat,
                                            pos_sq, neg_sq, far_mask, epoch);
    esdf_block_min<<<dim3((pitch / 8 + 31) / 32, nblk), 128, 0, st>>>(ctx->d_row, pitch, NX, NY, ctx->d_blk, pitch, colflag, ncol_tiles, epoch);
    auto* band = band_nj == 1 ? esdf_band_kernel<SQ, 1> : esdf_band_kernel<SQ, 2>;
    band<<<band_grid, 128, 0, st>>>(ctx->d_row, pitch, ctx->d_blk, pitch, NX, NY, far_mask, pitch, 2 * ((NX + TX - 1) / TX), epoch, dist,
                                    g.gly, min_x, min_y, g.grid_interval, pos_sq, neg_sq);
    ctx->launches += 3;
  };
  if (sq) {
    column_pass(std::true_type{}, d_dist, d_pos_sq, d_neg_sq);
    if (quirk) {
      esdf_quirk_col<true><<<(NX + 7) / 8, 256, 0, st>>>(ctx->d_row, pitch, NX, NY, d_dist, g.gly, min_x, min_y,
                                                             g.grid_interval, d_pos_sq, d_neg_sq);
      ctx->launches++;
    }
  } else {
    // the aliased column only needs the row pass: it runs on the side stream beside K2 / K1b / K2e (disjoint output cells)
    const bool side = quirk && NX >= 3;
    if (side) {
      ALORE_CUDA(ctx, cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
      esdf_quirk_col<false><<<(NX + 7) / 8, 256, 0, ctx->stream2>>>(ctx->d_row, pitch, NX, NY, d_dist, g.gly, min_x, min_y,
                                                                       g.grid_interval, nullptr, nullptr);
      ALORE_CUDA(ctx, cudaEventRecord(ctx->ev_join, ctx->stream2));
      ctx->launches++;
    }
    column_pass(std::false_type{}, d_dist, nullptr, nullptr);
    if (side) ALORE_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_join, 0));
  }
  ALORE_CUDA(ctx, cudaGetLastError());
#ifdef ALORE_BAND_STATS
  {
    cudaDeviceSynchronize();
    unsigned long long h[8], z[8] = {0};
    cudaMemcpyFromSymbol(h, g_band_dbg, sizeof(h));
    cudaMemcpyToSymbol(g_band_dbg, z, sizeof(z));
    fprintf(stderr, "[band] blocks seen %llu needed %llu | rows seen %llu past filter %llu stored %llu | items %llu band rows %llu range rows %llu\n",
            h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7]);
  }
#endif
  return ALORE_OK;
}
