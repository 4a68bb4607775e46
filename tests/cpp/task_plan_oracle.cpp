// task_plan_oracle.cpp — sequential reference of the task plan (alore_task_plan, include/alore_b200.h) for the tests.
// Test infrastructure only: tests/task_plan_util.py compiles it into a temporary directory; the product never loads it.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <vector>

#include "../../include/alore_b200.h"

extern "C" {

// Task plan (include/alore_b200.h, alore_task_plan): the leg matrix by one ascending scan of the candidates, then the
// layered DP over (objects picked O, targets filled T) in plain loops over bit masks.  A state of layer A_k / B_k sits at
// (rank(O) * #T-sets + rank(T)) * k + position of j in O / of u in T, ranks counted in ascending mask order (which is
// colex order among masks of one size).  Same tie rule: ascending point index, replace on strict <.
int orc_task_plan(const alore_task_t* task, int B, const double* cost, const int32_t* ok, alore_task_plan_t* out) {
  const int n = task->n_objects, P = 2 * n + 1;
  const bool fixed = task->fixed_assignment != 0;
  if (n < 1 || n > (fixed ? ALORE_TASK_MAX_FIXED : ALORE_TASK_MAX_FREE)) return -1;
  const double inf = std::numeric_limits<double>::infinity();
  std::vector<double> D(size_t(P) * P, inf);
  std::vector<int32_t> best(size_t(P) * P, -1);
  for (int b = 0; b < B; b++) {
    const int f = task->leg_from[b];
    if (f < 0 || ok[b] != 1 || !std::isfinite(cost[b])) continue;
    const size_t l = size_t(f) * P + task->leg_to[b];
    if (best[l] < 0 || cost[b] < D[l]) { D[l] = cost[b]; best[l] = b; }
  }
  auto d = [&](int i, int j) { return D[size_t(i) * P + j]; };
  std::vector<int> tgt(n), obj(n);                                   // local indices 0..n-1
  for (int i = 0; i < n; i++) {
    tgt[i] = (fixed && task->assign ? task->assign[i] : n + 1 + i) - n - 1;
    obj[tgt[i]] = i;
  }
  const uint32_t full = (1u << n) - 1u;
  std::vector<uint32_t> rank(size_t(1) << n);
  std::vector<uint32_t> count(n + 1, 0);
  std::vector<std::vector<uint32_t>> of_size(n + 1);                 // masks of each size, ascending
  for (uint32_t m = 0; m <= full; m++) {
    rank[m] = count[__builtin_popcount(m)]++;
    of_size[__builtin_popcount(m)].push_back(m);
  }
  auto image = [&](uint32_t objs) {
    uint32_t t = 0;
    for (int a = 0; a < n; a++) if (objs >> a & 1) t |= 1u << tgt[a];
    return t;
  };
  auto pos = [](uint32_t m, int b) { return __builtin_popcount(m & ((1u << b) - 1u)); };
  // A[k], B[k]: values and parents of layers k = 1..n
  std::vector<std::vector<double>> Av(n + 1), Bv(n + 1);
  std::vector<std::vector<int8_t>> Ap(n + 1), Bp(n + 1);
  auto idxA = [&](uint32_t O, uint32_t T, int k, int j) {
    return size_t(fixed ? rank[O] : size_t(rank[O]) * count[k - 1] + rank[T]) * k + pos(O, j);
  };
  auto idxB = [&](uint32_t O, uint32_t T, int k, int u) {
    return size_t(fixed ? rank[O] : size_t(rank[O]) * count[k] + rank[T]) * k + pos(T, u);
  };
  for (int k = 1; k <= n; k++) {
    const size_t nT_A = fixed ? 1 : count[k - 1], nT_B = fixed ? 1 : count[k];
    Av[k].assign(count[k] * nT_A * k, inf); Ap[k].assign(Av[k].size(), -1);
    Bv[k].assign(count[k] * nT_B * k, inf); Bp[k].assign(Bv[k].size(), -1);
    for (uint32_t O : of_size[k]) {
      for (uint32_t T : fixed ? std::vector<uint32_t>{0} : of_size[k - 1]) {   // A_k: |T| = k-1
        for (int j = 0; j < n; j++) {
          if (!(O >> j & 1)) continue;
          const uint32_t O1 = O & ~(1u << j);
          const uint32_t Tr = fixed ? image(O1) : T;
          double v = inf;
          int arg = -1;
          if (k == 1) v = d(0, 1 + j);
          else
            for (int t = 0; t < n; t++) {
              if (!(Tr >> t & 1)) continue;
              const double c = Bv[k - 1][idxB(O1, Tr, k - 1, t)] + d(n + 1 + t, 1 + j);
              if (c < v) { v = c; arg = t; }
            }
          Av[k][idxA(O, Tr, k, j)] = v;
          Ap[k][idxA(O, Tr, k, j)] = int8_t(arg);
        }
      }
      for (uint32_t T : fixed ? std::vector<uint32_t>{image(O)} : of_size[k]) {   // B_k: |T| = k
        for (int u = 0; u < n; u++) {
          if (!(T >> u & 1)) continue;
          const uint32_t T1 = T & ~(1u << u);
          double v = inf;
          int arg = -1;
          for (int j = 0; j < n; j++) {
            if (!(O >> j & 1) || (fixed && tgt[j] != u)) continue;
            const double c = Av[k][idxA(O, T1, k, j)] + d(1 + j, n + 1 + u);
            if (c < v) { v = c; arg = j; }
          }
          Bv[k][idxB(O, T, k, u)] = v;
          Bp[k][idxB(O, T, k, u)] = int8_t(arg);
        }
      }
    }
  }
  double opt = inf;
  int u = -1;
  for (int s = 0; s < n; s++) {
    const int us = fixed ? tgt[s] : s;
    const double v = Bv[n][idxB(full, full, n, us)];
    if (v < opt) { opt = v; u = us; }
  }
  out->cost = opt;
  out->feasible = opt < inf;
  if (out->leg_cost) std::memcpy(out->leg_cost, D.data(), D.size() * sizeof(double));
  if (out->leg_best) std::memcpy(out->leg_best, best.data(), best.size() * sizeof(int32_t));
  if (!out->feasible) {
    for (int i = 0; i < n; i++) out->order[i] = out->target[i] = -1;
    for (int i = 0; i < 2 * n; i++) out->leg_cand[i] = -1;
    return 0;
  }
  uint32_t O = full, T = full;
  for (int k = n; k >= 1; k--) {
    const int j = Bp[k][idxB(O, T, k, u)];
    out->order[k - 1] = 1 + j;
    out->target[k - 1] = n + 1 + u;
    const uint32_t T1 = T & ~(1u << u);
    const int t = k > 1 ? Ap[k][idxA(O, T1, k, j)] : -1;
    O &= ~(1u << j);
    T = T1;
    u = t;
  }
  int prev = 0;
  for (int k = 0; k < n; k++) {
    out->leg_cand[2 * k] = best[size_t(prev) * P + out->order[k]];
    out->leg_cand[2 * k + 1] = best[size_t(out->order[k]) * P + out->target[k]];
    prev = out->target[k];
  }
  return 0;
}

}  // extern "C"
