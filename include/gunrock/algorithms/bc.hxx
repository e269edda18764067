/**
 * @file bc.hxx
 * @brief Betweenness centrality: Brandes' algorithm over the depths of the direction-optimised BFS (DESIGN.md §3.5).
 *
 * The graph is taken unweighted (hops; edge weights are ignored, as in the reference's bc). A path is a sequence of CSR
 * edges, so parallel edges are distinct paths; a self-loop is never on a shortest path. For a source s, σ_s(v) is the
 * number of shortest s -> v paths and δ_s(v) = Σ_{v->w, d(w) = d(v)+1} σ_s(v)/σ_s(w) · (1 + δ_s(w)) (Brandes'
 * dependency). For a host list S of sources run() writes
 *   bc[v] = float(scale · Σ_{s ∈ S, s != v} δ_s(v))
 * into every entry of bc; a source listed twice counts twice, unreached vertices contribute 0. scale = 1 is the raw sum,
 * 0.5 the undirected convention (each unordered pair once) and the reference's single-source output; a normalisation
 * such as 1/((n-1)(n-2)) may be passed as well. σ, δ and the accumulator are double; the output is rounded once.
 *
 * The result is a pure function of (graph, S, scale): byte-identical between runs and for every way the same CSR is
 * handed over (32- or 64-bit offsets, host arrays, misaligned arrays). Every per-vertex sum walks the vertex's list in
 * an order fixed by its degree (one thread in list order, or lane/thread strides reduced by a fixed tree), sums over
 * sources run in list order, and no float or double atomic touches a value. Products and sums are explicitly rounded
 * (no FMA contraction), so sources = {s, s} gives exactly twice sources = {s}.
 *
 * Per source, all on the context's stream:
 *   depths    bfs::run<merge_path, optimized>, unchanged;
 *   order     counting sort of the reached vertices by bucket = depth · 9 + 3 · bin(in-degree) + bin(out-degree),
 *             bin = b200::degree_bin: [0, 8) one thread, [8, 4096) one warp, [4096, ∞) one CTA per row:
 *             level_histogram_kernel, level_scan_kernel, level_scatter_kernel, then one read-back of the bucket
 *             offsets, which sizes the launches;
 *   forward   levels 1..D, rows binned by in-degree: σ(v) = Σ_{u->v, d(u) = d(v)-1} σ(u) over the CSC, σ(s) = 1;
 *   backward  levels D..0, rows binned by out-degree: δ(v) = σ(v) · Σ_{v->w, d(w) = d(v)+1} c(w) over the CSR, then
 *             c(v) = (1 + δ(v)) / σ(v) and acc[v] += δ(v) for v != s (at level D the sum is empty: c = 1/σ).
 * Both gathers are b200::row_gather with level_sum_t, which reads the 4-byte depth of a neighbour before its 8-byte
 * value, so an edge into another level costs 4 bytes. After the last source one streaming kernel writes bc. Scratch:
 * depth, level order (int32), σ, c, acc (double) — 32 bytes per vertex from the device pool, once per call — and 9
 * counters per level.
 *
 * Needs a CSC view (a symmetric graph or a caller transpose), like direction-optimised BFS. σ is a double: it
 * overflows past ~1.8e308 shortest paths (e.g. grids with more than about 1000 hops between corners), and the
 * result is then not finite. Not available on a partitioned context.
 *
 * This header is not included by algorithms.hxx: the reference's own bc.hxx also declares gunrock::bc.
 */
#pragma once

#include <cmath>
#include <limits>
#include <string>
#include <vector>

#include <gunrock/algorithms/bfs.hxx>
#include <gunrock/b200/row_gather.cuh>

namespace gunrock {
namespace bc {
namespace detail {
using b200::counter_t;

constexpr int buckets_per_level = 9;

/// Bucket of vertex v (-1 when unreached), and the edges the two gathers walk for it (in-edges except at the source's
/// level, out-edges always). `bad` counts depths at or beyond `levels`, which a BFS result never has.
template <typename vertex_t, typename edge_t>
__device__ __forceinline__ long long bucket_of(std::size_t v, std::size_t n, const vertex_t* __restrict__ depth,
                                               const edge_t* __restrict__ in_offsets,
                                               const edge_t* __restrict__ out_offsets, vertex_t levels,
                                               unsigned long long& edges, unsigned& bad) {
  if (v >= n) return -1;
  const vertex_t d = depth[v];
  if (d == std::numeric_limits<vertex_t>::max()) return -1;
  if (d < 0 || d >= levels) {
    ++bad;
    return -1;
  }
  const long long in_deg = (long long)(in_offsets[v + 1] - in_offsets[v]);
  const long long out_deg = (long long)(out_offsets[v + 1] - out_offsets[v]);
  edges += (unsigned long long)((d > 0 ? in_deg : 0) + out_deg);
  return (long long)d * buckets_per_level + 3 * b200::degree_bin(in_deg) + b200::degree_bin(out_deg);
}

/// hist[bucket] += vertices in it (one atomic per distinct bucket per warp); stats[0] += edges both gathers will
/// walk, stats[1] += depths out of range.
template <typename vertex_t, typename edge_t>
__global__ void __launch_bounds__(256)
    level_histogram_kernel(const vertex_t* __restrict__ depth, const edge_t* __restrict__ in_offsets,
                           const edge_t* __restrict__ out_offsets, vertex_t n, vertex_t levels, counter_t* hist,
                           counter_t* stats) {
  unsigned long long edges = 0;
  unsigned bad = 0;
  const unsigned lane = b200::lane_id();
  for (std::size_t base = std::size_t(blockIdx.x) * blockDim.x; base < std::size_t(n);
       base += std::size_t(gridDim.x) * blockDim.x) {
    const long long key =
        bucket_of(base + threadIdx.x, std::size_t(n), depth, in_offsets, out_offsets, levels, edges, bad);
    const unsigned peers = __match_any_sync(b200::full_mask, (unsigned long long)key);
    if (key >= 0 && int(lane) == __ffs(peers) - 1) atomicAdd(hist + key, counter_t(__popc(peers)));
  }
  edges = b200::warp_sum(edges);
  bad = b200::warp_sum(bad);
  if (lane == 0) {
    if (edges) atomicAdd(stats + 0, counter_t(edges));
    if (bad) atomicAdd(stats + 1, counter_t(bad));
  }
}

/// One CTA: offsets[k] = Σ_{j<k} hist[j] for k in [0, buckets], and hist becomes the scatter cursors (= offsets).
__global__ void __launch_bounds__(1024) level_scan_kernel(counter_t* hist, counter_t* offsets, std::size_t buckets) {
  __shared__ counter_t warp_totals[1024 / 32 + 1];
  counter_t carry = 0;
  for (std::size_t base = 0; base < buckets; base += 1024) {
    const std::size_t k = base + threadIdx.x;
    const counter_t x = k < buckets ? hist[k] : counter_t(0);
    counter_t total;
    const counter_t before = b200::cta_exclusive_sum<1024, counter_t>(x, total, warp_totals);
    if (k < buckets) hist[k] = offsets[k] = carry + before;
    carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) offsets[buckets] = carry;
}

/// order[cursor[bucket]++] = v for every reached v (one atomic per distinct bucket per warp). The order inside a
/// bucket is whatever the atomics give; no result depends on it.
template <typename vertex_t, typename edge_t>
__global__ void __launch_bounds__(256)
    level_scatter_kernel(const vertex_t* __restrict__ depth, const edge_t* __restrict__ in_offsets,
                         const edge_t* __restrict__ out_offsets, vertex_t n, vertex_t levels, counter_t* cursor,
                         vertex_t* __restrict__ order) {
  unsigned long long edges = 0;
  unsigned bad = 0;
  const unsigned lane = b200::lane_id();
  for (std::size_t base = std::size_t(blockIdx.x) * blockDim.x; base < std::size_t(n);
       base += std::size_t(gridDim.x) * blockDim.x) {
    const std::size_t v = base + threadIdx.x;
    const long long key = bucket_of(v, std::size_t(n), depth, in_offsets, out_offsets, levels, edges, bad);
    const unsigned peers = __match_any_sync(b200::full_mask, (unsigned long long)key);
    const int leader = __ffs(peers) - 1;
    counter_t at = 0;
    if (key >= 0 && int(lane) == leader) at = atomicAdd(cursor + key, counter_t(__popc(peers)));
    at = __shfl_sync(b200::full_mask, at, leader);
    if (key >= 0) order[at + __popc(peers & b200::lanes_below(lane))] = vertex_t(v);
  }
}

/// Σ value[x] over the list entries x of [first, end) (stride `step`) with depth[x] == want; depth is read first.
template <typename vertex_t, typename edge_t>
struct level_sum_t {
  const vertex_t* indices;
  const vertex_t* depth;
  vertex_t want;
  const double* value;
  __device__ __forceinline__ double operator()(edge_t first, edge_t end, edge_t step) const {
    double acc = 0;
    for (edge_t e = first; e < end; e += step) {
      const vertex_t x = __ldg(indices + e);
      if (__ldg(depth + x) == want) acc = __dadd_rn(acc, __ldg(value + x));
    }
    return acc;
  }
};

/// Forward finish: σ(v) = the sum over the in-edges from the previous level.
template <typename vertex_t>
struct forward_t {
  double* sigma;
  __device__ __forceinline__ void start() {}
  __device__ __forceinline__ void operator()(vertex_t v, double sum) const { sigma[v] = sum; }
  __device__ __forceinline__ void flush() {}
};

/// Backward finish: δ(v) = σ(v) · Σ c(w), c(v) = (1 + δ(v)) / σ(v), acc[v] += δ(v) unless v is the source.
template <typename vertex_t>
struct backward_t {
  const double* sigma;
  double* c;
  double* acc;
  vertex_t source;
  __device__ __forceinline__ void start() {}
  __device__ __forceinline__ void operator()(vertex_t v, double sum) const {
    const double s = sigma[v];
    const double delta = __dmul_rn(s, sum);
    c[v] = __ddiv_rn(__dadd_rn(1.0, delta), s);
    if (v != source) acc[v] = __dadd_rn(acc[v], delta);
  }
  __device__ __forceinline__ void flush() {}
};

template <typename weight_t>
__global__ void __launch_bounds__(256)
    bc_output_kernel(const double* __restrict__ acc, std::size_t n, double scale, weight_t* __restrict__ out) {
  for (std::size_t v = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; v < n;
       v += std::size_t(gridDim.x) * blockDim.x)
    out[v] = weight_t(__dmul_rn(scale, acc[v]));
}

}  // namespace detail

/**
 * @brief bc[v] = scale · Σ_{s ∈ sources, s != v} δ_s(v) (file comment) for the `count` host-array source ids, in list
 * order; sources == nullptr with count == 0 means every vertex in id order (exact BC). `bc_values`: n entries, every one
 * written. Returns the CUDA-event ms of the whole call. `stats` (optional, 3 entries) receives Σ levels, Σ reached
 * vertices and Σ edges gathered by both passes over all sources. Throws, before any launch, on a source out of range,
 * a non-finite scale, a graph without a CSC view, or a partitioned context.
 */
template <typename graph_t>
float run(graph_t& G, const typename graph_t::vertex_type* sources, std::size_t count, double scale,
          typename graph_t::weight_type* bc_values, std::shared_ptr<gcuda::multi_context_t> context,
          long long* stats = nullptr) {
  using vertex_t = typename graph_t::vertex_type;
  using edge_t = typename graph_t::edge_type;
  using detail::counter_t;
  using runs_t = b200::row_runs_t<vertex_t>;
  constexpr int B = detail::buckets_per_level;

  error::throw_if_exception(bc_values == nullptr, "bc::run: bc_values is required");
  error::throw_if_exception((sources == nullptr) != (count == 0),
                            "bc::run: sources == nullptr (every vertex) goes with count == 0, and only with it");
  error::throw_if_exception(!std::isfinite(scale), "bc::run: scale must be finite");
  error::throw_if_exception(context->partition && context->partition->world > 1,
                            "bc::run: betweenness centrality is not available on a partitioned context");
  const auto out_view = graph::adjacency_of<false>(G);
  const auto in_view = graph::adjacency_of<true>(G);
  error::throw_if_exception(in_view.offsets == nullptr || (in_view.m > 0 && in_view.indices == nullptr),
                            "CSR and CSC sparse-matrix representations required for direction-optimized advance.");
  const vertex_t n = G.get_number_of_vertices();
  for (std::size_t i = 0; i < count; ++i)
    error::throw_if_exception(sources[i] < 0 || sources[i] >= n, "bc::run: source out of range");
  const std::size_t total = sources ? count : std::size_t(n);

  auto* ctx = context->get_context(0);
  auto stream = ctx->stream();
  const std::size_t un = std::size_t(n);
  memory::device_array_t<vertex_t> depth(un), order(un);
  memory::device_array_t<double> sigma(un), c(un), acc(un);
  memory::device_array_t<counter_t> levels_buf;  // [0, K) cursors | [K, 2K] offsets | edges | bad depths
  std::vector<counter_t> h;
  long long sum_levels = 0, sum_reached = 0, sum_edges = 0;

  util::timer_t timer(stream);
  timer.begin();
  cudaMemsetAsync(acc.data(), 0, un * sizeof(double), stream);
  for (std::size_t i = 0; i < total; ++i) {
    vertex_t s = sources ? sources[i] : vertex_t(i);
    int iterations = 0;
    bfs::run<operators::load_balance_t::merge_path, operators::advance_direction_t::optimized>(
        G, s, depth.data(), (vertex_t*)nullptr, context, enactor_properties_t(), nullptr, &iterations);
    // every depth lies in [0, iterations]: each BFS iteration settles one more level
    const vertex_t levels = vertex_t(iterations + 1);
    const std::size_t K = std::size_t(levels) * B;
    levels_buf.reserve(2 * K + 3, false);  // the old contents are never needed
    levels_buf.resize(2 * K + 3);
    counter_t* cursor = levels_buf.data();
    counter_t* offsets = cursor + K;
    counter_t* counts = offsets + K + 1;
    cudaMemsetAsync(levels_buf.data(), 0, levels_buf.size() * sizeof(counter_t), stream);
    const unsigned grid = b200::stream_grid(*ctx, un);
    detail::level_histogram_kernel<<<grid, 256, 0, stream>>>(depth.data(), in_view.offsets, out_view.offsets, n,
                                                             levels, cursor, counts);
    detail::level_scan_kernel<<<1, 1024, 0, stream>>>(cursor, offsets, K);
    detail::level_scatter_kernel<<<grid, 256, 0, stream>>>(depth.data(), in_view.offsets, out_view.offsets, n, levels,
                                                           cursor, order.data());
    ctx->profiler().launches_total += 3;
    error::check_last("bc::run level order");
    h.resize(K + 3);
    error::throw_if_exception(
        cudaMemcpyAsync(h.data(), offsets, h.size() * sizeof(counter_t), cudaMemcpyDeviceToHost, stream),
        "bc::run offsets read-back");
    ctx->synchronize();
    error::throw_if_exception(h[K + 2] != 0, "bc::run: BFS returned a depth beyond its level count");
    int deepest = 0;
    for (int d = 0; d < int(levels); ++d)
      if (h[std::size_t(d + 1) * B] > h[std::size_t(d) * B]) deepest = d;
    sum_levels += deepest + 1;
    sum_reached += (long long)h[K];
    sum_edges += (long long)h[K + 1];

    b200::set_one(*ctx, sigma.data() + s, 1.0);
    const auto bucket = [&](int d, int k) { return h[std::size_t(d) * B + k]; };
    for (int d = 1; d <= deepest; ++d) {  // rows of one in-degree bin: one run of three buckets
      runs_t rows[3];
      for (int t = 0; t < 3; ++t)
        rows[t] = runs_t{{order.data() + bucket(d, 3 * t)}, {bucket(d, 3 * t + 3) - bucket(d, 3 * t)}};
      const detail::level_sum_t<vertex_t, edge_t> sum{in_view.indices, depth.data(), vertex_t(d - 1), sigma.data()};
      b200::row_gather(*ctx, in_view.offsets, rows, sum, detail::forward_t<vertex_t>{sigma.data()});
    }
    for (int d = deepest; d >= 0; --d) {  // rows of one out-degree bin: one bucket per in-degree bin
      runs_t rows[3];
      for (int t = 0; t < 3; ++t)
        for (int k = 0; k < 3; ++k) {
          rows[t].begin[k] = order.data() + bucket(d, 3 * k + t);
          rows[t].size[k] = bucket(d, 3 * k + t + 1) - bucket(d, 3 * k + t);
        }
      const detail::level_sum_t<vertex_t, edge_t> sum{out_view.indices, depth.data(), vertex_t(d + 1), c.data()};
      b200::row_gather(*ctx, out_view.offsets, rows, sum,
                       detail::backward_t<vertex_t>{sigma.data(), c.data(), acc.data(), s});
    }
    error::check_last("bc::run gathers");
  }
  if (un)
    detail::bc_output_kernel<<<b200::stream_grid(*ctx, un), 256, 0, stream>>>(acc.data(), un, scale, bc_values);
  error::check_last("bc::run output");
  const float ms = timer.end();
  if (stats) {
    stats[0] = sum_levels;
    stats[1] = sum_reached;
    stats[2] = sum_edges;
  }
  return ms;
}

/// The reference's signature (gunrock::bc::run(G, single_source, bc_values, context)): scale 0.5 over the one source,
/// so bc_values[single_source] == 0.
template <typename graph_t>
float run(graph_t& G, typename graph_t::vertex_type single_source, typename graph_t::weight_type* bc_values,
          std::shared_ptr<gcuda::multi_context_t> context =
              std::shared_ptr<gcuda::multi_context_t>(new gcuda::multi_context_t(0))) {
  return run(G, &single_source, 1, 0.5, bc_values, context);
}

}  // namespace bc
}  // namespace gunrock
