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

unsigned long long binom_host(int n, int k) {
  if (k < 0 || k > n) return 0;
  unsigned long long v = 1;
  for (int t = 1; t <= k; t++) v = v * (n - k + t) / t;
  return v;
}

int validate(alore_ctx* ctx, const alore_task_t* task, int B, const alore_task_plan_t* out) {
  if (!task || !out) return alore_fail(ctx, ALORE_EINVAL, "task plan: null task or plan");
  const int fixed = task->fixed_assignment, n = task->n_objects;
  if (fixed != 0 && fixed != 1) return alore_fail(ctx, ALORE_EINVAL, "task plan: fixed_assignment must be 0 or 1, not %d", fixed);
  const int nmax = fixed ? ALORE_TASK_MAX_FIXED : ALORE_TASK_MAX_FREE;
  if (n < 1 || n > nmax)
    return alore_fail(ctx, ALORE_EINVAL, "task plan: n_objects %d outside [1, %d] in %s mode", n, nmax, fixed ? "fixed" : "free");
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
int task_plan_run(alore_ctx* ctx, const alore_task_t* task, int B, const double* d_cost, const int32_t* d_ok,
                  const double* h_cost, const int32_t* h_ok, alore_task_plan_t* out) {
  const int n = task->n_objects, P = 2 * n + 1, PP = P * P;
  const bool fixed = task->fixed_assignment == 1;
  TaskDP dp{};
  dp.n = n;
  dp.P = P;
  long long S = 0;
  for (int k = 1; k <= n; k++) {
    const unsigned long long cO = binom_host(n, k);
    dp.off[2 * k - 2] = S;
    S += (long long)(cO * (fixed ? 1 : binom_host(n, k - 1)) * k);
    dp.off[2 * k - 1] = S;
    S += (long long)(cO * (fixed ? 1 : cO) * k);
  }
  for (int i = 0; i < n; i++) {
    const int a = fixed && task->assign ? task->assign[i] : n + 1 + i;
    dp.tgt[i] = (int8_t)(a - n - 1);
    dp.obj[a - n - 1] = (int8_t)i;
  }
  // output block (one contiguous download): [D PP][cost][feasible, order n, target n, leg_cand 2n][best PP]
  const size_t n_ints = 1 + 4 * (size_t)n;
  const size_t block_bytes = 8 * (size_t)PP + 8 + 4 * (n_ints + PP);
  Carve cv;
  const size_t o_block = cv.take<char>(block_bytes);
  const size_t o_key = cv.take<unsigned long long>(PP);
  const size_t o_from = cv.take<int32_t>(B), o_to = cv.take<int32_t>(B);
  const size_t o_cost = h_cost ? cv.take<double>(B) : 0, o_ok = h_cost ? cv.take<int32_t>(B) : 0;
  const size_t o_val = cv.take<double>(S), o_par = cv.take<int8_t>(S);
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
  for (int k = 1; k <= n; k++) {
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
  if (fixed) task_backtrack_kernel<true><<<1, 32, 0, st>>>(dp, d_best, d_opt, d_ints);
  else task_backtrack_kernel<false><<<1, 32, 0, st>>>(dp, d_best, d_opt, d_ints);
  ctx->launches++;
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

}  // extern "C"
