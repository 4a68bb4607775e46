// task_plan_oracle.cpp — sequential reference of the task plan (alore_task_plan and alore_task_plan_beam,
// include/alore_b200.h) for the tests.  Test infrastructure only: tests/task_plan_util.py compiles it into a temporary
// directory; the product never loads it.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <map>
#include <tuple>
#include <vector>

#include "../../include/alore_b200.h"

namespace {

const double inf = std::numeric_limits<double>::infinity();

// What both solvers share: the leg matrix by one ascending scan of the candidates, the local target of every local
// object (indices 0..n-1), and the plan written from a search's optimum and backtrack.
struct Legs {
  int n, P;
  std::vector<double> D;
  std::vector<int32_t> best;
  std::vector<int> tgt;
  Legs(const alore_task_t* task, int B, const double* cost, const int32_t* ok)
      : n(task->n_objects), P(2 * n + 1), D(size_t(P) * P, inf), best(size_t(P) * P, -1), tgt(n) {
    for (int b = 0; b < B; b++) {
      const int f = task->leg_from[b];
      if (f < 0 || ok[b] != 1 || !std::isfinite(cost[b])) continue;
      const size_t l = size_t(f) * P + task->leg_to[b];
      if (best[l] < 0 || cost[b] < D[l]) { D[l] = cost[b]; best[l] = b; }
    }
    const bool fixed = task->fixed_assignment != 0;
    for (int i = 0; i < n; i++) tgt[i] = (fixed && task->assign ? task->assign[i] : n + 1 + i) - n - 1;
  }
  // The optimum, the matrix when asked for, and the tour `backtrack` writes into order / target with its leg
  // candidates; every plan entry -1 when infeasible.
  template <class F>
  int plan(alore_task_plan_t* out, double opt, F backtrack) const {
    out->cost = opt;
    out->feasible = opt < inf;
    if (out->leg_cost) std::memcpy(out->leg_cost, D.data(), D.size() * sizeof(double));
    if (out->leg_best) std::memcpy(out->leg_best, best.data(), best.size() * sizeof(int32_t));
    if (!out->feasible) {
      for (int i = 0; i < n; i++) out->order[i] = out->target[i] = -1;
      for (int i = 0; i < 2 * n; i++) out->leg_cand[i] = -1;
      return 0;
    }
    backtrack();
    int prev = 0;
    for (int k = 0; k < n; k++) {
      out->leg_cand[2 * k] = best[size_t(prev) * P + out->order[k]];
      out->leg_cand[2 * k + 1] = best[size_t(out->order[k]) * P + out->target[k]];
      prev = out->target[k];
    }
    return 0;
  }
};

}  // namespace

extern "C" {

// Task plan (include/alore_b200.h, alore_task_plan): the leg matrix, then the layered DP over (objects picked O,
// targets filled T) in plain loops over bit masks.  A state of layer A_k / B_k sits at (rank(O) * #T-sets + rank(T)) * k
// + position of j in O / of u in T, ranks counted in ascending mask order (which is colex order among masks of one
// size).  Same tie rule: ascending point index, replace on strict <.
int orc_task_plan(const alore_task_t* task, int B, const double* cost, const int32_t* ok, alore_task_plan_t* out) {
  const int n = task->n_objects;
  const bool fixed = task->fixed_assignment != 0;
  if (n < 1 || n > (fixed ? ALORE_TASK_MAX_FIXED : ALORE_TASK_MAX_FREE)) return -1;
  const Legs legs(task, B, cost, ok);
  const std::vector<int>& tgt = legs.tgt;
  auto d = [&](int i, int j) { return legs.D[size_t(i) * legs.P + j]; };
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
  return legs.plan(out, opt, [&] {
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
  });
}

// Bounded-width task plan (include/alore_b200.h, alore_task_plan_beam): the leg matrix as orc_task_plan builds it, then
// the half-step layers held in a std::map keyed by (O, T, last) with the merge rule, truncated to `width` by a sort in
// the contract's total order.  Parents are indices into the previous layer's kept list.
int orc_task_plan_beam(const alore_task_t* task, int width, int B, const double* cost, const int32_t* ok,
                       alore_task_plan_t* out, int32_t* exact) {
  const int n = task->n_objects;
  const bool fixed = task->fixed_assignment != 0;
  if (n < 1 || n > ALORE_TASK_MAX_BEAM_N || width < 1 || width > ALORE_TASK_MAX_WIDTH) return -1;
  const Legs legs(task, B, cost, ok);
  const std::vector<int>& tgt = legs.tgt;
  auto d = [&](int i, int j) { return legs.D[size_t(i) * legs.P + j]; };
  struct State { uint32_t O, T; int last; double v; int pred_last, parent; };
  using Key = std::tuple<uint32_t, uint32_t, int>;
  std::vector<std::vector<State>> layers(2 * n + 1);
  layers[0].push_back({0, 0, -1, 0.0, -1, -1});                     // the robot
  bool truncated = false;
  for (int l = 1; l <= 2 * n; l++) {
    const bool pick = l % 2 == 1;
    std::map<Key, State> merged;
    const std::vector<State>& prev = layers[l - 1];
    for (int s = 0; s < int(prev.size()); s++) {
      const State& p = prev[s];
      for (int q = 0; q < n; q++) {
        State c{p.O, p.T, q, 0.0, p.last, s};
        if (pick) {                                                  // next object q, from the robot or target p.last
          if (p.O >> q & 1) continue;
          c.O |= 1u << q;
          c.v = l == 1 ? d(0, 1 + q) : p.v + d(n + 1 + p.last, 1 + q);
        } else {                                                     // object p.last onto target q
          if ((p.T >> q & 1) || (fixed && tgt[p.last] != q)) continue;
          c.T |= 1u << q;
          c.v = p.v + d(1 + p.last, n + 1 + q);
        }
        if (!(c.v < inf)) continue;
        auto it = merged.find(Key{c.O, c.T, q});
        if (it == merged.end()) merged.emplace(Key{c.O, c.T, q}, c);
        else if (c.v < it->second.v || (c.v == it->second.v && c.pred_last < it->second.pred_last)) it->second = c;
      }
    }
    std::vector<State>& cur = layers[l];
    for (auto& kv : merged) cur.push_back(kv.second);
    if (int(cur.size()) > width) {
      truncated = true;
      std::sort(cur.begin(), cur.end(), [](const State& a, const State& b) {
        if (a.v < b.v) return true;
        if (b.v < a.v) return false;                                 // -0 == +0
        return std::make_tuple(a.O, a.T, a.last) < std::make_tuple(b.O, b.T, b.last);
      });
      cur.resize(width);
    }
  }
  double opt = inf;
  int arg = -1;
  for (int s = 0; s < n; s++) {
    const int us = fixed ? tgt[s] : s;
    for (int i = 0; i < int(layers[2 * n].size()); i++)
      if (layers[2 * n][i].last == us && layers[2 * n][i].v < opt) { opt = layers[2 * n][i].v; arg = i; }
  }
  if (exact) *exact = !truncated;
  return legs.plan(out, opt, [&] {
    for (int l = 2 * n, i = arg; l >= 1; l--) {
      const State& s = layers[l][i];
      if (l % 2 == 0) out->target[l / 2 - 1] = n + 1 + s.last;
      else out->order[l / 2] = 1 + s.last;
      i = s.parent;
    }
  });
}

}  // extern "C"
