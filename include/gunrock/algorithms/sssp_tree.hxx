/**
 * @file sssp_tree.hxx
 * @brief Shortest-path tree from finished SSSP distances: sssp::build_tree (DESIGN.md §3.5).
 *
 * The parent cannot be recorded while SSSP relaxes (the float atomic::min and a parent store are not one atomic
 * step), so the tree is a pass over the distance array that run(), run<…, near_far>() or run_delta() returned. It is a
 * pure function of the graph, `d` and the source, so the three engines, which return bit-identical distances, give
 * byte-identical trees. With fl(a + w) the single-precision add every SSSP kernel uses, an edge u -> v of weight w is
 * tight when u is reached (d[u] < FLT_MAX) and d[v] == fl(d[u] + w); tight edges are strict when d[u] < d[v] and flat
 * when d[u] == d[v] and u != v (zero weights, or weights the rounding absorbs: fl(1e8 + 1) == 1e8).
 *   1. pred[source] = source;
 *   2. pred[v] = -1 exactly where d[v] == FLT_MAX;
 *   3. a reached v with a strict tight in-edge takes the smallest such tail;
 *   4. every other reached v has only flat tight in-edges. With the vertices of rules 1 and 3 as anchors and L(v)
 *      the number of flat hops from the nearest anchor, v takes the smallest u with a flat edge u -> v and
 *      L(u) == L(v) - 1.
 * Along a chain of parents (d, L) strictly decreases, so there are no cycles. When `d` is the SSSP fixed point every
 * reached vertex gets a parent; the pass checks that, and rejects anything that is not that fixed point: NaN,
 * negative or infinite entries, d[source] != 0, an edge that still relaxes (fl(d[u] + w) < d[v] with u reached), or
 * a reached vertex left without a parent (e.g. a zero-weight cycle the source does not reach, given equal finite
 * distances). Parent chains then show d >= the float shortest-path value, and "nothing relaxes" shows d <= it.
 *
 * The pass reads CSR out-edges and CSR weights only (the weights SSSP relaxed), so directed graphs without a CSC work.
 *   fill      pred = INT32_MAX ("no strict parent yet");
 *   sweep     one balanced advance over the whole graph (tree_sweep_t): strict tight edges atomic::min the parent,
 *             flat tight edges mark their tail in an n/32-word bitmap, relaxable edges are counted;
 *   finalize  one streaming pass over the vertices (tree_finalize_kernel): validate d, write -1 and the source,
 *             count the vertices still without a parent, and queue the anchors that have a flat out-edge;
 *   rounds    only when some vertex is unresolved: round k advances from the vertices with L == k - 1 and settles
 *             the unresolved heads of their flat edges (tree_flat_t), until every vertex is settled or a round
 *             settles none.
 * Graphs without flat edges (all weights >= 1, as the hash and grid weights) cost a fill, the sweep and one pass.
 */
#pragma once

#include <limits>
#include <string>

#include <gunrock/algorithms/algorithms.hxx>

namespace gunrock {
namespace sssp {
namespace detail {

/// The sweep's per-edge operator: atomic::min of the parent on strict tight edges (after a plain read that skips the
/// atomic when `u` cannot win), the tail's flat bit on flat tight edges, and a warp-aggregated count of the edges that
/// still relax. Never emits.
template <typename vertex_t, typename edge_t, typename weight_t>
struct tree_sweep_t {
  const weight_t* dist;
  vertex_t* pred;
  unsigned* flat_tail;
  b200::counter_t* relaxable;

  __device__ __forceinline__ bool operator()(vertex_t const& u, vertex_t const& v, edge_t const& edge,
                                             weight_t const& weight) const {
    const weight_t du = dist[u];
    if (!(du < std::numeric_limits<weight_t>::max())) return false;  // unreached (NaN and inf are finalize's)
    const weight_t dv = dist[v];
    const weight_t through = du + weight;
    if (through == dv) {
      if (du < dv) {
        if (u < pred[v]) math::atomic::min(&pred[v], u);
      } else if (du == dv && u != v) {
        unsigned* word = flat_tail + (unsigned(u) >> 5);
        const unsigned bit = 1u << (unsigned(u) & 31u);
        if (!(*word & bit)) atomicOr(word, bit);
      }
    } else if (through < dv) {
      const unsigned peers = __activemask();  // the lanes counting this edge together: one atomic for all of them
      if (int(b200::lane_id()) == __ffs(peers) - 1) atomicAdd(relaxable, b200::counter_t(__popc(peers)));
    }
    return false;
  }
};

/// Round `round` of the flat rounds: a flat tight edge u -> v into a vertex not settled before this round lowers its
/// parent to u. Returns true for the one call that settles v (its stamp leaves INT32_MAX), so v enters the next
/// frontier once. Anchors carry stamp 0 and are never touched.
template <typename vertex_t, typename edge_t, typename weight_t>
struct tree_flat_t {
  const weight_t* dist;
  vertex_t* pred;
  vertex_t* stamp;
  vertex_t round;

  __device__ __forceinline__ bool operator()(vertex_t const& u, vertex_t const& v, edge_t const& edge,
                                             weight_t const& weight) const {
    if (stamp[v] < round) return false;
    const weight_t dv = dist[v];
    if (u == v || !(dist[u] == dv) || !(dist[u] + weight == dv)) return false;
    if (u < pred[v]) math::atomic::min(&pred[v], u);
    return math::atomic::min(&stamp[v], round) == std::numeric_limits<vertex_t>::max();
  }
};

/// build_tree's pass over the vertices, after the sweep. Counters (gcuda::scratch_t): out_count anchors queued,
/// aux0 entries of `dist` that are NaN, negative or +inf, aux1 relaxable edges (copied from the sweep's counter so
/// that one read-back reports everything), aux2 reached vertices without a strict parent, aux3 1 if dist[source] != 0.
template <typename vertex_t, typename weight_t>
__global__ void __launch_bounds__(256)
    tree_finalize_kernel(const weight_t* __restrict__ dist, vertex_t* __restrict__ pred,
                         const unsigned* __restrict__ flat_tail, vertex_t n, vertex_t source,
                         vertex_t* __restrict__ anchors, const b200::counter_t* relaxable, b200::counter_t* counters) {
  __shared__ b200::counter_t sm[256 / 32 + 4];
  constexpr vertex_t no_parent = std::numeric_limits<vertex_t>::max();
  constexpr weight_t unreached = std::numeric_limits<weight_t>::max();
  unsigned invalid = 0, unresolved = 0;
  for (std::size_t base = std::size_t(blockIdx.x) * 256; base < std::size_t(n); base += std::size_t(gridDim.x) * 256) {
    const std::size_t i = base + threadIdx.x;
    vertex_t ids[1] = {vertex_t(i)};
    unsigned keep = 0;
    if (i < std::size_t(n)) {
      const vertex_t v = vertex_t(i);
      const weight_t d = dist[i];
      invalid += !(d >= weight_t(0) && d <= unreached);
      bool anchor = false;
      if (v == source) {
        if (!(d == weight_t(0))) counters[gcuda::scratch_t::aux3] = 1;
        pred[i] = source;
        anchor = true;
      } else if (d == unreached) {
        pred[i] = vertex_t(-1);
      } else {
        anchor = pred[i] != no_parent;
        unresolved += !anchor;
      }
      keep = anchor && ((flat_tail[i >> 5] >> (i & 31u)) & 1u);
    }
    b200::cta_append<256, 1>(ids, keep, anchors, counters + gcuda::scratch_t::out_count, b200::counter_t(n), sm);
  }
  invalid = b200::warp_sum(invalid);
  unresolved = b200::warp_sum(unresolved);
  if (b200::lane_id() == 0) {
    if (invalid) atomicAdd(counters + gcuda::scratch_t::aux0, b200::counter_t(invalid));
    if (unresolved) atomicAdd(counters + gcuda::scratch_t::aux2, b200::counter_t(unresolved));
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) counters[gcuda::scratch_t::aux1] = *relaxable;
}

/// stamp[v] = INT32_MAX for the vertices the flat rounds must settle (no parent yet), 0 for all others.
template <typename vertex_t>
__global__ void __launch_bounds__(256)
    tree_stamp_kernel(const vertex_t* __restrict__ pred, vertex_t n, vertex_t* __restrict__ stamp) {
  constexpr vertex_t no_parent = std::numeric_limits<vertex_t>::max();
  for (std::size_t i = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < std::size_t(n);
       i += std::size_t(gridDim.x) * blockDim.x)
    stamp[i] = pred[i] == no_parent ? no_parent : vertex_t(0);
}

}  // namespace detail

/**
 * @brief The shortest-path tree of `distances` (the result of an SSSP run from `source`, any engine) into
 * `predecessors` (n entries; every one is written). See the file comment for the contract. Returns the CUDA-event ms
 * of the pass. `rounds` (optional) receives the number of flat rounds, `stats[0]` (optional) the number of vertices
 * parented over a flat edge. Throws when `distances` is not the SSSP fixed point for `source`, naming the violation
 * and its count; `predecessors` is then unspecified. Not available on a partitioned context.
 */
template <typename graph_t>
float build_tree(graph_t& G, typename graph_t::vertex_type source, const typename graph_t::weight_type* distances,
                 typename graph_t::vertex_type* predecessors, std::shared_ptr<gcuda::multi_context_t> context,
                 int* rounds = nullptr, long long* stats = nullptr) {
  using vertex_t = typename graph_t::vertex_type;
  using edge_t = typename graph_t::edge_type;
  using weight_t = typename graph_t::weight_type;
  using frontier_type = frontier::frontier_t<vertex_t, edge_t>;
  using counter_t = b200::counter_t;
  using gcuda::scratch_t;
  namespace adv = operators::advance;
  constexpr auto merge_path = operators::load_balance_t::merge_path;
  constexpr auto forward = operators::advance_direction_t::forward;
  constexpr auto graph_io = operators::advance_io_type_t::graph;
  constexpr auto vertices = operators::advance_io_type_t::vertices;
  constexpr auto none = operators::advance_io_type_t::none;

  error::throw_if_exception(distances == nullptr || predecessors == nullptr,
                            "sssp::build_tree: distances and predecessors are required");
  error::throw_if_exception(context->partition && context->partition->world > 1,
                            "sssp::build_tree: the SSSP tree is not available on a partitioned context");
  const vertex_t n = G.get_number_of_vertices();
  error::throw_if_exception(source < 0 || source >= n, "sssp::build_tree: source out of range");
  auto* ctx = context->get_context(0);
  auto stream = ctx->stream();
  auto& scratch = ctx->scratch();
  auto& prof = ctx->profiler();

  // one buffer, one memset: [0] the sweep's relaxable-edge counter, then the flat-tail bitmap (n/32 words)
  const std::size_t words = (std::size_t(n) + 31) / 32;
  memory::device_array_t<counter_t> marks{1 + (words + 1) / 2};
  counter_t* relaxable = marks.data();
  auto* flat_tail = reinterpret_cast<unsigned*>(marks.data() + 1);
  frontier_type frontier{std::size_t(n)}, next, none_frontier;
  memory::device_array_t<edge_t> segments;

  auto& timer = ctx->timer();
  timer.begin();
  cudaMemsetAsync(marks.data(), 0, marks.size() * sizeof(counter_t), stream);
  b200::fill(*ctx, predecessors, std::size_t(n), std::numeric_limits<vertex_t>::max());
  {
    struct restore_t {
      bool& flag;
      bool was;
      ~restore_t() { flag = was; }
    } restore{scratch.async_when_no_output, scratch.async_when_no_output};
    scratch.async_when_no_output = true;  // the finalize read-back below is the pass's one host round trip
    adv::execute<merge_path, forward, graph_io, none>(
        G, detail::tree_sweep_t<vertex_t, edge_t, weight_t>{distances, predecessors, flat_tail, relaxable},
        &none_frontier, &none_frontier, segments, *context);
  }
  scratch.zero(stream);
  prof.begin(gcuda::profiler_t::dense_state, stream);
  detail::tree_finalize_kernel<<<gcuda::persistent_grid(*ctx, (std::size_t(n) + 255) / 256, 8), 256, 0, stream>>>(
      distances, predecessors, flat_tail, n, source, frontier.data(), relaxable, scratch.d);
  prof.end(stream);
  error::check_last("sssp::build_tree finalize");
  scratch.fetch(stream);
  const long long invalid = (long long)scratch.h[scratch_t::aux0];
  const long long relaxing = (long long)scratch.h[scratch_t::aux1];
  const long long unresolved = (long long)scratch.h[scratch_t::aux2];
  const bool bad_source = scratch.h[scratch_t::aux3] != 0;
  const std::size_t anchors = std::size_t(scratch.h[scratch_t::out_count]);
  if (invalid || bad_source || relaxing) {
    std::string what = "sssp::build_tree: the distances are not the SSSP result for this source:";
    if (invalid) what += " " + std::to_string(invalid) + " entries are NaN, negative or infinite;";
    if (bad_source) what += " the source's distance is not 0;";
    if (relaxing) what += " " + std::to_string(relaxing) + " relaxable edges;";
    what.pop_back();
    error::throw_if_exception(true, what);
  }

  long long settled = 0;
  int round = 0;
  if (unresolved) {
    memory::device_array_t<vertex_t> stamp{std::size_t(n)};
    prof.begin(gcuda::profiler_t::dense_state, stream);
    detail::tree_stamp_kernel<<<b200::stream_grid(*ctx, std::size_t(n)), 256, 0, stream>>>(predecessors, n,
                                                                                            stamp.data());
    prof.end(stream);
    error::check_last("sssp::build_tree stamps");
    next.reserve(std::size_t(n));
    frontier.set_number_of_elements(anchors);
    while (frontier.get_number_of_elements() && settled < unresolved) {
      ++round;
      adv::execute<merge_path, forward, vertices, vertices>(
          G, detail::tree_flat_t<vertex_t, edge_t, weight_t>{distances, predecessors, stamp.data(), vertex_t(round)},
          &frontier, &next, segments, *context);
      settled += (long long)next.get_number_of_elements();
      std::swap(frontier, next);
    }
  }
  const float ms = timer.end();
  error::throw_if_exception(settled != unresolved,
                            "sssp::build_tree: the distances are not the SSSP result for this source: " +
                                std::to_string(unresolved - settled) +
                                " reached vertices have no tight path from the source");
  if (rounds) *rounds = round;
  if (stats) stats[0] = settled;
  return ms;
}

}  // namespace sssp
}  // namespace gunrock
