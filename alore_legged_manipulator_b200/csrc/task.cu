// task.cu — task plan on the device: the leg cost matrix of the optimised candidates and the exact visiting-order x
// assignment search over it (alore_task_plan, alore_batch_task_plan; contract in include/alore_b200.h).
//
// Kernels, in launch order on the context's stream:
//   task_leg_key_kernel    atomicMin of an order-preserving 64-bit key of every counted candidate's cost, per leg
//   task_leg_index_kernel  atomicMin of the candidate index over the candidates whose key equals the leg's minimum
//   task_leg_final_kernel  D[i][j] = cost[best[i][j]] (exact bits), +inf / -1 for a leg without a counted candidate
//   task_pick_kernel<F>    DP layer A_k (k = 1..n), one thread per state, interleaved with
//   task_place_kernel<F>   DP layer B_k
//   task_backtrack_kernel  final minimum over B_n and the backtrack of the parents, one thread
// F = fixed assignment: the same state indexing with the target set's rank dropped (T is the image of O).
//
// State index of a layer (combinatorial number system, colex ranks of bit masks over the n objects / n targets):
//   A_k: (rank(O) * C(n, k-1) + rank(T)) * k + position of j among the bits of O        |O| = k, |T| = k-1
//   B_k: (rank(O) * C(n, k)   + rank(T)) * k + position of u among the bits of T        |O| = |T| = k
//   fixed mode: rank(O) * k + position.
// The predecessors a state scans are contiguous in the previous layer (same O', T' ranks, consecutive positions), and
// they are scanned in ascending point index, so the tie rule (strict <, lowest index first) needs no atomics.
#include <algorithm>
#include <climits>
#include <cmath>

#include "common.cuh"

namespace {

constexpr int kMaxN = ALORE_TASK_MAX_FIXED;
constexpr int kMaxP = 2 * kMaxN + 1;
constexpr int kThreads = 256;
static_assert(ALORE_TASK_MAX_FREE <= ALORE_TASK_MAX_FIXED, "one binomial table serves both modes");

struct TaskDP {
  int n, P;
  const double* D;                 // [P*P] leg matrix
  double* val;                     // every DP layer's values: A_1, B_1, A_2, B_2, ..., B_n
  int8_t* par;                     // parents, same offsets: A -> local target index t, B -> local object index j
  long long off[2 * kMaxN];        // element offset of layer A_k at [2k-2], of B_k at [2k-1]
  int8_t tgt[kMaxN];               // fixed mode: local target of local object a
  int8_t obj[kMaxN];               // fixed mode: local object of local target u
};

using Binom = uint32_t[kMaxN + 1][kMaxN + 1];

__device__ void stage_binom(Binom& c) {
  for (int i = threadIdx.x; i < (kMaxN + 1) * (kMaxN + 1); i += blockDim.x) {
    const int n = i / (kMaxN + 1), k = i % (kMaxN + 1);
    unsigned long long v = k > n ? 0 : 1;
    for (int t = 1; t <= k && k <= n; t++) v = v * (n - k + t) / t;   // exact at every step
    c[n][k] = (uint32_t)v;
  }
}

// colex unrank: the k-subset of {0..n-1} with rank r
__device__ __forceinline__ uint32_t unrank(uint32_t r, int k, int n, const Binom& c) {
  uint32_t m = 0;
  int e = n - 1;
  for (int i = k; i >= 1; i--) {
    while (c[e][i] > r) e--;
    m |= 1u << e;
    r -= c[e][i];
    e--;
  }
  return m;
}

__device__ __forceinline__ uint32_t rank_of(uint32_t m, const Binom& c) {
  uint32_t r = 0;
  for (int i = 1; m; m &= m - 1, i++) r += c[__ffs(m) - 1][i];
  return r;
}

__device__ __forceinline__ int nth_bit(uint32_t m, int p) {
  for (; p > 0; p--) m &= m - 1;
  return __ffs(m) - 1;
}

__device__ __forceinline__ int pos_of(uint32_t m, int b) { return __popc(m & ((1u << b) - 1u)); }

__device__ __forceinline__ uint32_t image(uint32_t objs, const int8_t* tgt) {
  uint32_t t = 0;
  for (; objs; objs &= objs - 1) t |= 1u << tgt[__ffs(objs) - 1];
  return t;
}

__device__ __forceinline__ unsigned long long cost_key(double c) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(c == 0.0 ? 0.0 : c);   // -0 shares +0's key
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

__device__ __forceinline__ bool counted(const double* cost, const int32_t* ok, int b) {
  return ok[b] == 1 && isfinite(cost[b]);
}

__global__ void task_leg_key_kernel(int B, int P, const int32_t* from, const int32_t* to, const double* cost, const int32_t* ok,
                                    unsigned long long* keymin) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x)
    if (from[b] >= 0 && counted(cost, ok, b)) atomicMin(&keymin[from[b] * P + to[b]], cost_key(cost[b]));
}

__global__ void task_leg_index_kernel(int B, int P, const int32_t* from, const int32_t* to, const double* cost, const int32_t* ok,
                                      const unsigned long long* keymin, int32_t* best) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x)
    if (from[b] >= 0 && counted(cost, ok, b)) {
      const int l = from[b] * P + to[b];
      if (cost_key(cost[b]) == keymin[l]) atomicMin(&best[l], b);
    }
}

__global__ void task_leg_final_kernel(int B, int P, const double* cost, int32_t* best, double* D) {
  for (int l = blockIdx.x * blockDim.x + threadIdx.x; l < P * P; l += gridDim.x * blockDim.x) {
    const int b = best[l];
    const bool none = b < 0 || b >= B;         // still the INT_MAX-like fill: no counted candidate
    best[l] = none ? -1 : b;
    D[l] = none ? INFINITY : cost[b];
  }
}

struct Shared {
  double D[kMaxP * kMaxP];
  Binom c;
  int8_t tgt[kMaxN], obj[kMaxN];
};

__device__ void stage(const TaskDP& p, Shared& s) {
  stage_binom(s.c);
  for (int i = threadIdx.x; i < p.P * p.P; i += blockDim.x) s.D[i] = p.D[i];
  for (int i = threadIdx.x; i < kMaxN; i += blockDim.x) { s.tgt[i] = p.tgt[i]; s.obj[i] = p.obj[i]; }
  __syncthreads();
}

// A_k[O, T, j]: object j just picked
template <bool FIXED>
__global__ void __launch_bounds__(kThreads) task_pick_kernel(TaskDP p, int k) {
  __shared__ Shared s;
  stage(p, s);
  const int n = p.n, P = p.P;
  const uint32_t CT = FIXED ? 1u : s.c[n][k - 1];
  const uint32_t count = s.c[n][k] * CT * (uint32_t)k;
  double* cur = p.val + p.off[2 * k - 2];
  int8_t* cpar = p.par + p.off[2 * k - 2];
  const double* prev = p.val + (k > 1 ? p.off[2 * k - 3] : 0);
  for (uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x; idx < count; idx += gridDim.x * blockDim.x) {
    const uint32_t q = idx / k, rT = FIXED ? 0u : q % CT, rO = FIXED ? q : q / CT;
    const uint32_t O = unrank(rO, k, n, s.c);
    const int j = nth_bit(O, idx - q * k);
    double best = INFINITY;
    int arg = -1;
    if (k == 1) {
      best = s.D[1 + j];                                     // D[0][j]
    } else {
      const uint32_t O1 = O & ~(1u << j);
      const uint32_t T = FIXED ? image(O1, s.tgt) : unrank(rT, k - 1, n, s.c);
      const uint32_t base = (FIXED ? rank_of(O1, s.c) : rank_of(O1, s.c) * s.c[n][k - 1] + rT) * (uint32_t)(k - 1);
      int i = 0;
      for (uint32_t m = T; m; m &= m - 1, i++) {             // ascending target index
        const int t = __ffs(m) - 1;
        const double v = prev[base + i] + s.D[(n + 1 + t) * P + 1 + j];
        if (v < best) { best = v; arg = t; }
      }
    }
    cur[idx] = best;
    cpar[idx] = (int8_t)arg;
  }
}

// B_k[O, T, u]: target u just filled
template <bool FIXED>
__global__ void __launch_bounds__(kThreads) task_place_kernel(TaskDP p, int k) {
  __shared__ Shared s;
  stage(p, s);
  const int n = p.n, P = p.P;
  const uint32_t CT = FIXED ? 1u : s.c[n][k];
  const uint32_t count = s.c[n][k] * CT * (uint32_t)k;
  double* cur = p.val + p.off[2 * k - 1];
  int8_t* cpar = p.par + p.off[2 * k - 1];
  const double* prev = p.val + p.off[2 * k - 2];
  for (uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x; idx < count; idx += gridDim.x * blockDim.x) {
    const uint32_t q = idx / k, rT = FIXED ? 0u : q % CT, rO = FIXED ? q : q / CT;
    const uint32_t O = unrank(rO, k, n, s.c);
    const uint32_t T = FIXED ? image(O, s.tgt) : unrank(rT, k, n, s.c);
    const int u = nth_bit(T, idx - q * k);
    double best = INFINITY;
    int arg = -1;
    if (FIXED) {
      const int j = s.obj[u];
      const double v = prev[rO * (uint32_t)k + pos_of(O, j)] + s.D[(1 + j) * P + n + 1 + u];
      if (v < best) { best = v; arg = j; }
    } else {
      const uint32_t base = (rO * s.c[n][k - 1] + rank_of(T & ~(1u << u), s.c)) * (uint32_t)k;
      int i = 0;
      for (uint32_t m = O; m; m &= m - 1, i++) {             // ascending object index
        const int j = __ffs(m) - 1;
        const double v = prev[base + i] + s.D[(1 + j) * P + n + 1 + u];
        if (v < best) { best = v; arg = j; }
      }
    }
    cur[idx] = best;
    cpar[idx] = (int8_t)arg;
  }
}

// out_cost[0] = optimum; ints = [feasible, order[n], target[n], leg_cand[2n]]
template <bool FIXED>
__global__ void task_backtrack_kernel(TaskDP p, const int32_t* best, double* out_cost, int32_t* ints) {
  __shared__ Binom c;
  __shared__ int8_t tgt[kMaxN];
  stage_binom(c);
  for (int i = threadIdx.x; i < kMaxN; i += blockDim.x) tgt[i] = p.tgt[i];
  __syncthreads();
  if (threadIdx.x != 0) return;
  const int n = p.n, P = p.P;
  int32_t *order = ints + 1, *target = ints + 1 + n, *leg = ints + 1 + 2 * n;
  const double* Bn = p.val + p.off[2 * n - 1];               // O = T = all: index = position of u = u
  double opt = INFINITY;
  int u = -1;
  for (int s = 0; s < n; s++) {                              // free: ascending u; fixed: ascending j, u = assign(j)
    const int us = FIXED ? tgt[s] : s;
    if (Bn[us] < opt) { opt = Bn[us]; u = us; }
  }
  out_cost[0] = opt;
  ints[0] = opt < INFINITY;
  if (!(opt < INFINITY)) {
    for (int i = 1; i < 1 + 4 * n; i++) ints[i] = -1;
    return;
  }
  uint32_t O = (1u << n) - 1u, T = O;
  for (int k = n; k >= 1; k--) {
    const uint32_t rO = rank_of(O, c);
    const uint32_t Tk = FIXED ? image(O, tgt) : T;
    const uint32_t iB = (FIXED ? rO : rO * c[n][k] + rank_of(Tk, c)) * (uint32_t)k + pos_of(Tk, u);
    const int j = p.par[p.off[2 * k - 1] + iB];
    order[k - 1] = 1 + j;
    target[k - 1] = n + 1 + u;
    const uint32_t T1 = Tk & ~(1u << u);
    int t = -1;
    if (k > 1) {
      const uint32_t iA = (FIXED ? rO : rO * c[n][k - 1] + rank_of(T1, c)) * (uint32_t)k + pos_of(O, j);
      t = p.par[p.off[2 * k - 2] + iA];
    }
    O &= ~(1u << j);
    T = T1;
    u = t;
  }
  int prev = 0;
  for (int k = 0; k < n; k++) {
    leg[2 * k] = best[prev * P + order[k]];
    leg[2 * k + 1] = best[order[k] * P + target[k]];
    prev = target[k];
  }
}

// ---- bounded-width layered search (alore_task_plan_beam) ------------------------------------------------------------
// Layer l = 1..2n is A_k (l = 2k-1) or B_k (l = 2k); layer 0 is the robot.  Per layer, on the device counts only:
//   task_beam_expand_kernel<F,1>  every (kept state, next point) successor: claim its (O,T) slot in table 1 and its
//                                 (slot, last) slot in table 2, atomicMin of cost_key(value) there
//   task_beam_expand_kernel<F,2>  the same successors again: atomicMin of (predecessor's last << 32 | its kept index)
//                                 among those whose key equals the minimum (the exact DP's tie rule, order-free)
//   task_beam_merge_kernel        table 2 -> dense list of merged states (value recomputed from the parent: the exact
//                                 bits of the winning record); resets table 2
//   task_beam_select_kernel       17 launches of a radix select (8-bit digits, MSB first) of the width-th state in
//                                 the order (cost_key, O, T, last); a no-op when the layer fits or the digit is settled
//   task_beam_keep_kernel         the states at or below the selected prefix -> kept list, last point and parent per
//                                 layer for the backtrack; resets table 1
// then task_beam_backtrack_kernel.  Kept lists are stored in any order; the contract speaks of sets and parents.
constexpr int kBeamN = ALORE_TASK_MAX_BEAM_N;
constexpr int kBeamP = 2 * kBeamN + 1;
constexpr int kBeamL = 2 * kBeamN;
constexpr unsigned long long kFree = 0;                     // an empty hash slot (a state's O is never empty)

// digits of the order (cost_key 8, O 4, T 4, last 1).  T stays in fixed mode too: an A-state's T is the image of O
// without its last object, so states of one O differ in T, and T ranks before last.
constexpr int kBeamDigits = 17;

struct BeamCtl {
  int merged[kBeamL + 1];            // merged states of layer l
  int kept[kBeamL + 1];              // kept states of layer l
  int need[kBeamL + 1];              // rank still to find among the states matching the selected prefix
  int depth[kBeamL + 1];             // digits of the prefix selected so far
  int done[kBeamL + 1];              // the prefix holds exactly the states still needed
  uint8_t thr[kBeamL + 1][20];       // the selected digits
  unsigned hist[256];                // the pass's global histogram, cleared by its last block
  unsigned ticket;
  int truncated;                     // some layer had more merged states than the width
};

struct TaskBeam {
  int n, P, W, H;                    // H: capacity of both hash tables, a power of two >= 2 W n
  const double* D;
  unsigned long long *key1, *key2;   // table 1: O << 32 | T; table 2: (table-1 slot << 8 | last) + 1
  unsigned long long *vkey, *pred;   // table 2's minimum cost key and winning (pred last << 32 | pred kept index)
  unsigned long long* mkey;          // merged list [W n]
  uint32_t *mO, *mT;
  int32_t* mpar;
  int8_t* mlast;
  double* mval;
  uint32_t *kO[2], *kT[2];           // kept list of layer l at parity l & 1 [W]
  int8_t* klast[2];
  double* kval[2];
  int8_t* blast;                     // [2n][W] last point (local index) of kept state i of layer l at (l-1) W + i
  int32_t* bpar;                     // [2n][W] its parent: index into layer l-1's kept list
  BeamCtl* ctl;
  int8_t tgt[kBeamN];
};

__device__ __forceinline__ uint32_t hash_slot(unsigned long long k, int H) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull;
  k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull;
  k ^= k >> 33;
  return (uint32_t)k & (uint32_t)(H - 1);
}

// linear probing; keys only go kFree -> k within a layer and the load stays <= 1/2, so this ends
__device__ uint32_t find_or_insert(unsigned long long* keys, unsigned long long k, int H) {
  for (uint32_t s = hash_slot(k, H);; s = (s + 1) & (uint32_t)(H - 1)) {
    const unsigned long long cur = *(volatile unsigned long long*)&keys[s];
    if (cur == k) return s;
    if (cur == kFree) {
      const unsigned long long was = atomicCAS(&keys[s], kFree, k);
      if (was == kFree || was == k) return s;
    }
  }
}

// a slot of `counter` per lane with pred set; every lane of the warp calls it
__device__ __forceinline__ int warp_append(bool pred, int* counter) {
  const unsigned m = __ballot_sync(0xffffffffu, pred);
  const int lane = threadIdx.x & 31;
  int base = 0;
  if (lane == 0 && m) base = atomicAdd(counter, __popc(m));
  base = __shfl_sync(0xffffffffu, base, 0);
  return base + __popc(m & ((1u << lane) - 1u));
}

__device__ __forceinline__ int beam_digit(unsigned long long vk, uint32_t O, uint32_t T, int last, int d) {
  if (d < 8) return (int)(vk >> (56 - 8 * d)) & 0xff;
  if (d < 12) return (int)(O >> (88 - 8 * d)) & 0xff;
  if (d < 16) return (int)(T >> (120 - 8 * d)) & 0xff;
  return last;
}

// the state's first `depth` digits against the selected prefix: < 0, 0, > 0
__device__ __forceinline__ int beam_cmp(unsigned long long vk, uint32_t O, uint32_t T, int last, const uint8_t* thr, int depth) {
  for (int d = 0; d < depth; d++) {
    const int a = beam_digit(vk, O, T, last, d);
    if (a != thr[d]) return a < thr[d] ? -1 : 1;
  }
  return 0;
}

template <bool FIXED, int PASS>
__global__ void __launch_bounds__(kThreads) task_beam_expand_kernel(TaskBeam p, int l) {
  __shared__ double sD[kBeamP * kBeamP];
  __shared__ int8_t stgt[kBeamN];
  const int n = p.n, P = p.P, pb = (l - 1) & 1;
  const int cnt = l == 1 ? 1 : p.ctl->kept[l - 1];
  const int total = cnt * n;
  if ((int)(blockIdx.x * blockDim.x) >= total) return;       // whole block: nothing to expand
  for (int i = threadIdx.x; i < P * P; i += blockDim.x) sD[i] = p.D[i];
  for (int i = threadIdx.x; i < n; i += blockDim.x) stgt[i] = p.tgt[i];
  __syncthreads();
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int s = idx / n, q = idx - s * n;
    uint32_t O = 0, T = 0;
    int last = 0;
    double v = 0.0;
    if (l > 1) { O = p.kO[pb][s]; T = p.kT[pb][s]; last = p.klast[pb][s]; v = p.kval[pb][s]; }
    double nv;
    if (l & 1) {                                            // pick object q, from the robot or target `last`
      if (O >> q & 1) continue;
      nv = l == 1 ? sD[1 + q] : v + sD[(n + 1 + last) * P + 1 + q];
      O |= 1u << q;
    } else {                                                // put object `last` on target q
      if ((T >> q & 1) || (FIXED && stgt[last] != q)) continue;
      nv = v + sD[(1 + last) * P + n + 1 + q];
      T |= 1u << q;
    }
    if (!(nv < INFINITY)) continue;                         // +inf and NaN are dropped
    const uint32_t s1 = find_or_insert(p.key1, (unsigned long long)O << 32 | T, p.H);
    const uint32_t s2 = find_or_insert(p.key2, ((unsigned long long)s1 << 8 | (unsigned)q) + 1, p.H);
    const unsigned long long ck = cost_key(nv);
    if (PASS == 1) atomicMin(&p.vkey[s2], ck);
    else if (ck == p.vkey[s2]) atomicMin(&p.pred[s2], (unsigned long long)last << 32 | (unsigned)s);
  }
}

__global__ void __launch_bounds__(kThreads) task_beam_merge_kernel(TaskBeam p, int l) {
  const int n = p.n, P = p.P, pb = (l - 1) & 1;
  const double* D = p.D;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < p.H; i += gridDim.x * blockDim.x) {   // H % 256 == 0
    const unsigned long long k2 = p.key2[i];
    const bool full = k2 != kFree;
    const int at = warp_append(full, &p.ctl->merged[l]);
    if (!full) continue;
    const uint32_t s1 = (uint32_t)((k2 - 1) >> 8);
    const int last = (int)((k2 - 1) & 0xff);
    const unsigned long long k1 = p.key1[s1], pr = p.pred[i];
    const int par = (int)(uint32_t)pr, plast = (int)(pr >> 32);
    double v;
    if (l & 1) v = l == 1 ? D[1 + last] : p.kval[pb][par] + D[(n + 1 + plast) * P + 1 + last];
    else v = p.kval[pb][par] + D[(1 + plast) * P + n + 1 + last];
    p.mkey[at] = p.vkey[i];
    p.mO[at] = (uint32_t)(k1 >> 32);
    p.mT[at] = (uint32_t)k1;
    p.mlast[at] = (int8_t)last;
    p.mpar[at] = par;
    p.mval[at] = v;
    p.key2[i] = kFree;
    p.vkey[i] = ~0ull;
    p.pred[i] = ~0ull;
  }
}

// digit d of the radix select; the last of the participating blocks picks the digit and clears the histogram
__global__ void __launch_bounds__(kThreads) task_beam_select_kernel(TaskBeam p, int l, int d) {
  __shared__ unsigned h[256];
  __shared__ int last_block;
  BeamCtl* c = p.ctl;
  const int M = c->merged[l];
  if (M <= p.W || c->done[l]) return;                        // grid-uniform
  const int nb = min((int)gridDim.x, (M + kThreads - 1) / kThreads);
  if ((int)blockIdx.x >= nb) return;
  for (int i = threadIdx.x; i < 256; i += blockDim.x) h[i] = 0;
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < M; i += nb * blockDim.x) {
    const unsigned long long vk = p.mkey[i];
    const uint32_t O = p.mO[i], T = p.mT[i];
    const int last = p.mlast[i];
    if (beam_cmp(vk, O, T, last, c->thr[l], d) == 0) atomicAdd(&h[beam_digit(vk, O, T, last, d)], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 256; i += blockDim.x)
    if (h[i]) atomicAdd(&c->hist[i], h[i]);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last_block = atomicAdd(&c->ticket, 1u) == (unsigned)nb - 1;
  __syncthreads();
  if (!last_block) return;
  __threadfence();
  for (int i = threadIdx.x; i < 256; i += blockDim.x) h[i] = atomicExch(&c->hist[i], 0u);
  __syncthreads();
  if (threadIdx.x == 0) {
    int need = d == 0 ? p.W : c->need[l];
    int b = 0;
    while ((int)h[b] < need) need -= (int)h[b++];            // b < 256: the prefix holds >= need states
    c->thr[l][d] = (uint8_t)b;
    c->need[l] = need;
    c->depth[l] = d + 1;
    c->done[l] = (int)h[b] == need;
    c->ticket = 0;
  }
}

__global__ void __launch_bounds__(kThreads) task_beam_keep_kernel(TaskBeam p, int l) {
  BeamCtl* c = p.ctl;
  const int M = c->merged[l], depth = c->depth[l], cb = l & 1;
  const bool all = M <= p.W;
  if (!all && blockIdx.x == 0 && threadIdx.x == 0) c->truncated = 1;
  for (int base = blockIdx.x * blockDim.x; base < M; base += gridDim.x * blockDim.x) {
    const int i = base + threadIdx.x;
    bool keep = false;
    if (i < M) keep = all || beam_cmp(p.mkey[i], p.mO[i], p.mT[i], p.mlast[i], c->thr[l], depth) <= 0;
    const int at = warp_append(keep, &c->kept[l]);
    if (!keep) continue;
    p.kO[cb][at] = p.mO[i];
    p.kT[cb][at] = p.mT[i];
    p.klast[cb][at] = p.mlast[i];
    p.kval[cb][at] = p.mval[i];
    p.blast[(size_t)(l - 1) * p.W + at] = p.mlast[i];
    p.bpar[(size_t)(l - 1) * p.W + at] = p.mpar[i];
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < p.H; i += gridDim.x * blockDim.x) p.key1[i] = kFree;
}

// out_cost[0] = result; ints = [feasible, order[n], target[n], leg_cand[2n], exact]
template <bool FIXED>
__global__ void task_beam_backtrack_kernel(TaskBeam p, const int32_t* best, double* out_cost, int32_t* ints) {
  if (threadIdx.x != 0) return;
  const int n = p.n, P = p.P, L = 2 * n, cnt = p.ctl->kept[L];
  int32_t *order = ints + 1, *target = ints + 1 + n, *leg = ints + 1 + 2 * n;
  ints[1 + 4 * n] = !p.ctl->truncated;
  double opt = INFINITY;
  int at = -1;
  for (int s = 0; s < n; s++) {                              // free: ascending u; fixed: ascending j, u = assign(j)
    const int us = FIXED ? p.tgt[s] : s;
    for (int i = 0; i < cnt; i++)                            // B_n: O = T = all, so at most one state per u
      if (p.klast[L & 1][i] == us && p.kval[L & 1][i] < opt) { opt = p.kval[L & 1][i]; at = i; }
  }
  out_cost[0] = opt;
  ints[0] = opt < INFINITY;
  if (!(opt < INFINITY)) {
    for (int i = 1; i < 1 + 4 * n; i++) ints[i] = -1;
    return;
  }
  for (int l = L; l >= 1; l--) {
    const int last = p.blast[(size_t)(l - 1) * p.W + at];
    if (l & 1) order[l / 2] = 1 + last;
    else target[l / 2 - 1] = n + 1 + last;
    at = p.bpar[(size_t)(l - 1) * p.W + at];
  }
  int prev = 0;
  for (int k = 0; k < n; k++) {
    leg[2 * k] = best[prev * P + order[k]];
    leg[2 * k + 1] = best[order[k] * P + target[k]];
    prev = target[k];
  }
}

unsigned long long binom_host(int n, int k) {
  if (k < 0 || k > n) return 0;
  unsigned long long v = 1;
  for (int t = 1; t <= k; t++) v = v * (n - k + t) / t;
  return v;
}

// width = 0: the exact solver's limits; width != 0: the bounded-width search's
int validate(alore_ctx* ctx, const alore_task_t* task, int B, const alore_task_plan_t* out, int width = 0) {
  if (!task || !out) return alore_fail(ctx, ALORE_EINVAL, "task plan: null task or plan");
  const int fixed = task->fixed_assignment, n = task->n_objects;
  if (fixed != 0 && fixed != 1) return alore_fail(ctx, ALORE_EINVAL, "task plan: fixed_assignment must be 0 or 1, not %d", fixed);
  const int nmax = width ? ALORE_TASK_MAX_BEAM_N : fixed ? ALORE_TASK_MAX_FIXED : ALORE_TASK_MAX_FREE;
  if (n < 1 || n > nmax)
    return alore_fail(ctx, ALORE_EINVAL, "task plan: n_objects %d outside [1, %d] in %s mode", n, nmax, fixed ? "fixed" : "free");
  if (width && (width < 1 || width > ALORE_TASK_MAX_WIDTH))
    return alore_fail(ctx, ALORE_EINVAL, "task plan: width %d outside [1, %d]", width, ALORE_TASK_MAX_WIDTH);
  if (!out->order || !out->target || !out->leg_cand) return alore_fail(ctx, ALORE_EINVAL, "task plan: null order/target/leg_cand");
  if (B < 0) return alore_fail(ctx, ALORE_EINVAL, "task plan: negative batch size");
  if (B > 0 && (!task->leg_from || !task->leg_to)) return alore_fail(ctx, ALORE_EINVAL, "task plan: null leg labels");
  const int P = 2 * n + 1;
  for (int b = 0; b < B; b++) {
    const int f = task->leg_from[b];
    if (f < -1 || f >= P) return alore_fail(ctx, ALORE_EINVAL, "task plan: leg_from[%d] = %d outside [-1, %d)", b, f, P);
    if (f < 0) continue;
    const int t = task->leg_to[b];
    if (t < 0 || t >= P) return alore_fail(ctx, ALORE_EINVAL, "task plan: leg_to[%d] = %d outside [0, %d)", b, t, P);
    if (t == f) return alore_fail(ctx, ALORE_EINVAL, "task plan: candidate %d is labelled with the leg %d -> %d", b, f, t);
  }
  if (fixed && task->assign) {
    uint32_t seen = 0;
    for (int i = 0; i < n; i++) {
      const int a = task->assign[i];
      if (a < n + 1 || a > 2 * n) return alore_fail(ctx, ALORE_EINVAL, "task plan: assign[%d] = %d is not a target in [%d, %d]", i, a, n + 1, 2 * n);
      if (seen & (1u << (a - n - 1))) return alore_fail(ctx, ALORE_EINVAL, "task plan: assign is not a bijection (target %d twice)", a);
      seen |= 1u << (a - n - 1);
    }
  }
  return ALORE_OK;
}

// Carves aligned pieces from the context's task arena.
struct Carve {
  size_t at = 0;
  template <class T>
  size_t take(size_t n) {
    const size_t o = (at + 255) & ~size_t(255);
    at = o + n * sizeof(T);
    return o;
  }
};

// The one device path.  d_cost/d_ok: device results (batch entry), or NULL with h_cost/h_ok to upload (host entry).
// width = 0: the exact DP; width >= 1: the bounded-width search, its `exact` flag to *exact (may be NULL).
int task_plan_run(alore_ctx* ctx, const alore_task_t* task, int B, const double* d_cost, const int32_t* d_ok,
                  const double* h_cost, const int32_t* h_ok, alore_task_plan_t* out, int width = 0, int32_t* exact = nullptr) {
  const int n = task->n_objects, P = 2 * n + 1, PP = P * P;
  const bool fixed = task->fixed_assignment == 1;
  int8_t tgt[kBeamN];
  for (int i = 0; i < n; i++) tgt[i] = (int8_t)((fixed && task->assign ? task->assign[i] : n + 1 + i) - n - 1);
  TaskDP dp{};
  long long S = 0;
  if (!width) {
    dp.n = n;
    dp.P = P;
    for (int k = 1; k <= n; k++) {
      const unsigned long long cO = binom_host(n, k);
      dp.off[2 * k - 2] = S;
      S += (long long)(cO * (fixed ? 1 : binom_host(n, k - 1)) * k);
      dp.off[2 * k - 1] = S;
      S += (long long)(cO * (fixed ? 1 : cO) * k);
    }
    for (int i = 0; i < n; i++) {
      dp.tgt[i] = tgt[i];
      dp.obj[tgt[i]] = (int8_t)i;
    }
  }
  // bounded-width search: at most W n successors per layer, hash tables at load <= 1/2
  TaskBeam bm{};
  bm.n = n;
  bm.P = P;
  bm.W = width;
  const size_t E = (size_t)width * n;
  bm.H = 256;
  while (width && (size_t)bm.H < 2 * E) bm.H *= 2;
  std::memcpy(bm.tgt, tgt, sizeof(tgt));
  // output block (one contiguous download): [D PP][cost][feasible, order n, target n, leg_cand 2n, (exact)][best PP]
  const size_t n_ints = 1 + 4 * (size_t)n + (width ? 1 : 0);
  const size_t block_bytes = 8 * (size_t)PP + 8 + 4 * (n_ints + PP);
  Carve cv;
  const size_t o_block = cv.take<char>(block_bytes);
  const size_t o_key = cv.take<unsigned long long>(PP);
  const size_t o_from = cv.take<int32_t>(B), o_to = cv.take<int32_t>(B);
  const size_t o_cost = h_cost ? cv.take<double>(B) : 0, o_ok = h_cost ? cv.take<int32_t>(B) : 0;
  const size_t o_val = cv.take<double>(S), o_par = cv.take<int8_t>(S);
  size_t o_tab = 0, o_m[6] = {}, o_k[2][4] = {}, o_blast = 0, o_bpar = 0, o_ctl = 0;
  if (width) {
    const size_t W = width;
    o_tab = cv.take<unsigned long long>(4 * (size_t)bm.H);   // key1, key2 (cleared to 0), vkey, pred (set to ~0)
    o_m[0] = cv.take<unsigned long long>(E);
    o_m[1] = cv.take<uint32_t>(E);
    o_m[2] = cv.take<uint32_t>(E);
    o_m[3] = cv.take<int32_t>(E);
    o_m[4] = cv.take<int8_t>(E);
    o_m[5] = cv.take<double>(E);
    for (int b = 0; b < 2; b++) {
      o_k[b][0] = cv.take<uint32_t>(W);
      o_k[b][1] = cv.take<uint32_t>(W);
      o_k[b][2] = cv.take<int8_t>(W);
      o_k[b][3] = cv.take<double>(W);
    }
    o_blast = cv.take<int8_t>(2 * n * W);
    o_bpar = cv.take<int32_t>(2 * n * W);
    o_ctl = cv.take<BeamCtl>(1);
  }
  const size_t need = cv.at;

  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  if (need > ctx->task_pool_bytes) {
    ALORE_CUDA(ctx, cudaStreamSynchronize(st));
    if (ctx->task_pool) cudaFree(ctx->task_pool);
    ctx->task_pool = nullptr;
    ctx->task_pool_bytes = 0;
    if (cudaMalloc(&ctx->task_pool, need) != cudaSuccess) {
      (void)cudaGetLastError();
      return alore_fail(ctx, ALORE_ENOMEM, "task plan: cudaMalloc of %zu bytes of scratch failed", need);
    }
    ctx->task_pool_bytes = need;
  }
  char* base = static_cast<char*>(ctx->task_pool);
  double* d_D = reinterpret_cast<double*>(base + o_block);
  double* d_opt = d_D + PP;
  int32_t* d_ints = reinterpret_cast<int32_t*>(d_opt + 1);
  int32_t* d_best = d_ints + n_ints;
  auto* d_key = reinterpret_cast<unsigned long long*>(base + o_key);
  auto* d_from = reinterpret_cast<int32_t*>(base + o_from);
  auto* d_to = reinterpret_cast<int32_t*>(base + o_to);
  if (h_cost) {
    d_cost = reinterpret_cast<double*>(base + o_cost);
    d_ok = reinterpret_cast<int32_t*>(base + o_ok);
  }
  dp.D = d_D;
  dp.val = reinterpret_cast<double*>(base + o_val);
  dp.par = reinterpret_cast<int8_t*>(base + o_par);
  if (width) {
    bm.D = d_D;
    auto* tab = reinterpret_cast<unsigned long long*>(base + o_tab);
    bm.key1 = tab;
    bm.key2 = tab + bm.H;
    bm.vkey = tab + 2 * (size_t)bm.H;
    bm.pred = tab + 3 * (size_t)bm.H;
    bm.mkey = reinterpret_cast<unsigned long long*>(base + o_m[0]);
    bm.mO = reinterpret_cast<uint32_t*>(base + o_m[1]);
    bm.mT = reinterpret_cast<uint32_t*>(base + o_m[2]);
    bm.mpar = reinterpret_cast<int32_t*>(base + o_m[3]);
    bm.mlast = reinterpret_cast<int8_t*>(base + o_m[4]);
    bm.mval = reinterpret_cast<double*>(base + o_m[5]);
    for (int b = 0; b < 2; b++) {
      bm.kO[b] = reinterpret_cast<uint32_t*>(base + o_k[b][0]);
      bm.kT[b] = reinterpret_cast<uint32_t*>(base + o_k[b][1]);
      bm.klast[b] = reinterpret_cast<int8_t*>(base + o_k[b][2]);
      bm.kval[b] = reinterpret_cast<double*>(base + o_k[b][3]);
    }
    bm.blast = reinterpret_cast<int8_t*>(base + o_blast);
    bm.bpar = reinterpret_cast<int32_t*>(base + o_bpar);
    bm.ctl = reinterpret_cast<BeamCtl*>(base + o_ctl);
    ALORE_CUDA(ctx, cudaMemsetAsync(bm.key1, 0, 2 * (size_t)bm.H * sizeof(unsigned long long), st));
    ALORE_CUDA(ctx, cudaMemsetAsync(bm.vkey, 0xFF, 2 * (size_t)bm.H * sizeof(unsigned long long), st));
    ALORE_CUDA(ctx, cudaMemsetAsync(bm.ctl, 0, sizeof(BeamCtl), st));
  }

  ALORE_CUDA(ctx, cudaMemsetAsync(d_key, 0xFF, PP * sizeof(unsigned long long), st));   // key = max
  ALORE_CUDA(ctx, cudaMemsetAsync(d_best, 0x7F, PP * sizeof(int32_t), st));            // index = 0x7F7F7F7F
  if (B > 0) {
    ALORE_CUDA(ctx, cudaMemcpyAsync(d_from, task->leg_from, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    ALORE_CUDA(ctx, cudaMemcpyAsync(d_to, task->leg_to, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (h_cost) {
      ALORE_CUDA(ctx, cudaMemcpyAsync(const_cast<double*>(d_cost), h_cost, B * sizeof(double), cudaMemcpyHostToDevice, st));
      ALORE_CUDA(ctx, cudaMemcpyAsync(const_cast<int32_t*>(d_ok), h_ok, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    }
    const int g = std::min((B + kThreads - 1) / kThreads, ctx->sm_count * 8);
    task_leg_key_kernel<<<g, kThreads, 0, st>>>(B, P, d_from, d_to, d_cost, d_ok, d_key);
    task_leg_index_kernel<<<g, kThreads, 0, st>>>(B, P, d_from, d_to, d_cost, d_ok, d_key, d_best);
    ctx->launches += 2;
  }
  task_leg_final_kernel<<<(PP + kThreads - 1) / kThreads, kThreads, 0, st>>>(B, P, d_cost, d_best, d_D);
  ctx->launches++;
  if (width) {
    const long long cap = ctx->sm_count * 8LL;
    const int gE = (int)std::min<long long>(((long long)E + kThreads - 1) / kThreads, cap);
    const int gH = (int)std::min<long long>(bm.H / kThreads, cap);
    for (int l = 1; l <= 2 * n; l++) {
      if (fixed) {
        task_beam_expand_kernel<true, 1><<<gE, kThreads, 0, st>>>(bm, l);
        task_beam_expand_kernel<true, 2><<<gE, kThreads, 0, st>>>(bm, l);
      } else {
        task_beam_expand_kernel<false, 1><<<gE, kThreads, 0, st>>>(bm, l);
        task_beam_expand_kernel<false, 2><<<gE, kThreads, 0, st>>>(bm, l);
      }
      task_beam_merge_kernel<<<gH, kThreads, 0, st>>>(bm, l);
      for (int d = 0; d < kBeamDigits; d++) task_beam_select_kernel<<<gE, kThreads, 0, st>>>(bm, l, d);
      task_beam_keep_kernel<<<gH, kThreads, 0, st>>>(bm, l);
      ctx->launches += 4 + kBeamDigits;
    }
    if (fixed) task_beam_backtrack_kernel<true><<<1, 32, 0, st>>>(bm, d_best, d_opt, d_ints);
    else task_beam_backtrack_kernel<false><<<1, 32, 0, st>>>(bm, d_best, d_opt, d_ints);
    ctx->launches++;
  }
  for (int k = 1; k <= n && !width; k++) {
    const long long nA = dp.off[2 * k - 1] - dp.off[2 * k - 2];
    const long long nB = (k < n ? dp.off[2 * k] : S) - dp.off[2 * k - 1];
    const int gA = (int)std::min<long long>((nA + kThreads - 1) / kThreads, ctx->sm_count * 8LL);
    const int gB = (int)std::min<long long>((nB + kThreads - 1) / kThreads, ctx->sm_count * 8LL);
    if (fixed) {
      task_pick_kernel<true><<<gA, kThreads, 0, st>>>(dp, k);
      task_place_kernel<true><<<gB, kThreads, 0, st>>>(dp, k);
    } else {
      task_pick_kernel<false><<<gA, kThreads, 0, st>>>(dp, k);
      task_place_kernel<false><<<gB, kThreads, 0, st>>>(dp, k);
    }
    ctx->launches += 2;
  }
  if (!width) {
    if (fixed) task_backtrack_kernel<true><<<1, 32, 0, st>>>(dp, d_best, d_opt, d_ints);
    else task_backtrack_kernel<false><<<1, 32, 0, st>>>(dp, d_best, d_opt, d_ints);
    ctx->launches++;
  }
  ALORE_CUDA(ctx, cudaGetLastError());

  // download the plan, and the matrix only when it is asked for
  const bool with_matrix = out->leg_cost || out->leg_best;
  std::vector<char> h(block_bytes);
  const size_t lo = with_matrix ? 0 : 8 * (size_t)PP, hi = with_matrix ? block_bytes : 8 * (size_t)PP + 8 + 4 * n_ints;
  ALORE_CUDA(ctx, cudaMemcpyAsync(h.data() + lo, base + o_block + lo, hi - lo, cudaMemcpyDeviceToHost, st));
  ALORE_CUDA(ctx, cudaStreamSynchronize(st));
  const double* hD = reinterpret_cast<const double*>(h.data());
  const int32_t* hi32 = reinterpret_cast<const int32_t*>(hD + PP + 1);
  std::memcpy(&out->cost, hD + PP, sizeof(double));
  out->feasible = hi32[0];
  std::memcpy(out->order, hi32 + 1, n * sizeof(int32_t));
  std::memcpy(out->target, hi32 + 1 + n, n * sizeof(int32_t));
  std::memcpy(out->leg_cand, hi32 + 1 + 2 * n, 2 * n * sizeof(int32_t));
  if (out->leg_cost) std::memcpy(out->leg_cost, hD, PP * sizeof(double));
  if (out->leg_best) std::memcpy(out->leg_best, hi32 + n_ints, PP * sizeof(int32_t));
  if (width && exact) *exact = hi32[1 + 4 * n];
  return ALORE_OK;
}

}  // namespace

extern "C" {

int alore_task_plan(alore_ctx* ctx, const alore_task_t* task, int B, const double* cost, const int32_t* ok,
                    alore_task_plan_t* out) {
  if (!ctx) return ALORE_EINVAL;
  int rc = validate(ctx, task, B, out);
  if (rc) return rc;
  if (B > 0 && (!cost || !ok)) return alore_fail(ctx, ALORE_EINVAL, "task plan: null cost/ok");
  return task_plan_run(ctx, task, B, nullptr, nullptr, cost, ok, out);
}

int alore_batch_task_plan(alore_ctx* ctx, alore_batch* batch, const alore_task_t* task, alore_task_plan_t* out) {
  if (!ctx || !batch) return ALORE_EINVAL;
  int B = 0, runs = 0;
  const double* d_cost = nullptr;
  const int32_t* d_ok = nullptr;
  batch_result_view(batch, &B, &runs, &d_cost, &d_ok);
  int rc = validate(ctx, task, B, out);
  if (rc) return rc;
  if (runs == 0) return alore_fail(ctx, ALORE_EINVAL, "task plan: the batch has not been run");
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  ALORE_CUDA(ctx, cudaDeviceSynchronize());                 // the run may have been enqueued on a caller stream
  return task_plan_run(ctx, task, B, d_cost, d_ok, nullptr, nullptr, out);
}

int alore_task_plan_beam(alore_ctx* ctx, const alore_task_t* task, int width, int B, const double* cost, const int32_t* ok,
                         alore_task_plan_t* out, int32_t* exact) {
  if (!ctx) return ALORE_EINVAL;
  if (width < 1 || width > ALORE_TASK_MAX_WIDTH)
    return alore_fail(ctx, ALORE_EINVAL, "task plan: width %d outside [1, %d]", width, ALORE_TASK_MAX_WIDTH);
  int rc = validate(ctx, task, B, out, width);
  if (rc) return rc;
  if (B > 0 && (!cost || !ok)) return alore_fail(ctx, ALORE_EINVAL, "task plan: null cost/ok");
  return task_plan_run(ctx, task, B, nullptr, nullptr, cost, ok, out, width, exact);
}

int alore_batch_task_plan_beam(alore_ctx* ctx, alore_batch* batch, const alore_task_t* task, int width,
                               alore_task_plan_t* out, int32_t* exact) {
  if (!ctx || !batch) return ALORE_EINVAL;
  if (width < 1 || width > ALORE_TASK_MAX_WIDTH)
    return alore_fail(ctx, ALORE_EINVAL, "task plan: width %d outside [1, %d]", width, ALORE_TASK_MAX_WIDTH);
  int B = 0, runs = 0;
  const double* d_cost = nullptr;
  const int32_t* d_ok = nullptr;
  batch_result_view(batch, &B, &runs, &d_cost, &d_ok);
  int rc = validate(ctx, task, B, out, width);
  if (rc) return rc;
  if (runs == 0) return alore_fail(ctx, ALORE_EINVAL, "task plan: the batch has not been run");
  ALORE_CUDA(ctx, cudaSetDevice(ctx->device));
  ALORE_CUDA(ctx, cudaDeviceSynchronize());                 // the run may have been enqueued on a caller stream
  return task_plan_run(ctx, task, B, d_cost, d_ok, nullptr, nullptr, out, width, exact);
}

}  // extern "C"
