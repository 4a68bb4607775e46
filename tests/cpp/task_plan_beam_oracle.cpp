// task_plan_beam_oracle.cpp — sequential reference of the bounded-width task plan (alore_task_plan_beam,
// include/alore_b200.h) for the tests.  Test infrastructure only: tests/task_plan_beam_util.py compiles it into a
// temporary directory; the product never loads it.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <map>
#include <tuple>
#include <vector>

#include "../../include/alore_b200.h"

extern "C" {

// Bounded-width task plan (include/alore_b200.h, alore_task_plan_beam): the leg matrix as orc_task_plan builds it, then the half-step layers
// held in a std::map keyed by (O, T, last) with the merge rule, truncated to `width` by a sort in the contract's total
// order.  Parents are indices into the previous layer's kept list.
int orc_task_plan_beam(const alore_task_t* task, int width, int B, const double* cost, const int32_t* ok,
                       alore_task_plan_t* out, int32_t* exact) {
  const int n = task->n_objects, P = 2 * n + 1;
  const bool fixed = task->fixed_assignment != 0;
  if (n < 1 || n > ALORE_TASK_MAX_BEAM_N || width < 1 || width > ALORE_TASK_MAX_WIDTH) return -1;
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
  std::vector<int> tgt(n), obj(n);
  for (int i = 0; i < n; i++) {
    tgt[i] = (fixed && task->assign ? task->assign[i] : n + 1 + i) - n - 1;
    obj[tgt[i]] = i;
  }
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
  out->cost = opt;
  out->feasible = opt < inf;
  if (exact) *exact = !truncated;
  if (out->leg_cost) std::memcpy(out->leg_cost, D.data(), D.size() * sizeof(double));
  if (out->leg_best) std::memcpy(out->leg_best, best.data(), best.size() * sizeof(int32_t));
  if (!out->feasible) {
    for (int i = 0; i < n; i++) out->order[i] = out->target[i] = -1;
    for (int i = 0; i < 2 * n; i++) out->leg_cand[i] = -1;
    return 0;
  }
  for (int l = 2 * n, i = arg; l >= 1; l--) {
    const State& s = layers[l][i];
    if (l % 2 == 0) out->target[l / 2 - 1] = n + 1 + s.last;
    else out->order[l / 2] = 1 + s.last;
    i = s.parent;
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
