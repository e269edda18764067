// CPU restatement of the SSSP tree contract (include/essentials_b200.h, ess_sssp_tree) for the tests: rules 1-4 and
// the validation, written out plainly over a host CSR. Built on first use by tests/sssp_tree_ref.py.
#include <cfloat>
#include <cstdint>
#include <vector>

using i32 = int32_t;
using i64 = int64_t;

extern "C" {

enum { TREE_OK = 0, TREE_INVALID_ENTRY = 1, TREE_SOURCE_NOT_ZERO = 2, TREE_RELAXABLE_EDGE = 3, TREE_ORPHAN = 4 };

// Fills pred (n entries) and returns TREE_OK, or returns the first kind of violation found in the order above
// (pred is then unspecified).
int sssp_tree_ref(i64 n, const i64* off, const i32* col, const float* w, i32 src, const float* d, i32* pred) {
  const float unreached = FLT_MAX;
  auto weight = [&](i64 e) { return w ? w[e] : 1.0f; };
  for (i64 v = 0; v < n; ++v)
    if (!(d[v] >= 0.0f && d[v] <= unreached)) return TREE_INVALID_ENTRY;
  if (d[src] != 0.0f) return TREE_SOURCE_NOT_ZERO;
  for (i64 u = 0; u < n; ++u) {
    if (d[u] == unreached) continue;
    for (i64 e = off[u]; e < off[u + 1]; ++e) {
      const float through = d[u] + weight(e);
      if (through < d[col[e]]) return TREE_RELAXABLE_EDGE;
    }
  }
  // rule 3: the smallest tail of a strict tight in-edge
  const i32 none = INT32_MAX;
  for (i64 v = 0; v < n; ++v) pred[v] = none;
  for (i64 u = 0; u < n; ++u) {
    if (d[u] == unreached) continue;
    for (i64 e = off[u]; e < off[u + 1]; ++e) {
      const i32 v = col[e];
      const float through = d[u] + weight(e);
      if (through == d[v] && d[u] < d[v] && i32(u) < pred[v]) pred[v] = i32(u);
    }
  }
  pred[src] = src;  // rule 1
  // rule 4: breadth-first over flat tight edges from the anchors (rules 1 and 3), level by level
  std::vector<i64> level(n, -1);
  std::vector<i32> frontier;
  for (i64 v = 0; v < n; ++v)
    if (d[v] != unreached && pred[v] != none) {
      level[v] = 0;
      frontier.push_back(i32(v));
    }
  for (i64 k = 0; !frontier.empty(); ++k) {
    std::vector<i32> next;
    for (i32 u : frontier)
      for (i64 e = off[u]; e < off[u + 1]; ++e) {
        const i32 v = col[e];
        const bool flat = v != u && d[v] == d[u] && d[u] + weight(e) == d[v];
        if (!flat || (level[v] != -1 && level[v] != k + 1)) continue;
        if (level[v] == -1) {
          level[v] = k + 1;
          next.push_back(v);
        }
        if (u < pred[v]) pred[v] = u;
      }
    frontier.swap(next);
  }
  for (i64 v = 0; v < n; ++v) {
    if (d[v] == unreached)
      pred[v] = -1;  // rule 2
    else if (level[v] == -1)
      return TREE_ORPHAN;
  }
  return TREE_OK;
}
}
