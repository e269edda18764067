/**
 * @file bfs.hxx
 * @brief Breadth-first search client of the frontier operators.
 *
 * Same problem/enactor/run shape and the same per-edge operator as the reference
 * (include/gunrock/algorithms/bfs.hxx:80-132: old = atomic::min(&dist[nbr], iter+1); keep iff iter+1 < old;
 * reset :53-60 fills INT_MAX and zeroes the source). run() keeps the reference signature (:151-159); the
 * two leading template parameters are additive and select the load balancer and the direction, so
 *   bfs::run(G, src, dist, pred)                                   == reference behaviour (block_mapped push)
 *   bfs::run<load_balance_t::merge_path, advance_direction_t::optimized>(...)  = push/pull switching
 * Depths are an order-independent fixed point, so every variant returns the same array.
 * run_tree() takes the same arguments and also writes the BFS tree into `predecessors` (DESIGN.md §3.5); run() never
 * touches that array, so callers that size it arbitrarily (the reference's drivers pass a 1-element vector) stay safe.
 * With a partitioned context (gcuda::partition_t, one process per GPU) the same loop body runs on the owned rows and
 * operators::exchange::execute routes each level's discoveries to their owners: `distances` is then a full-length
 * array whose owned slice is the result.
 */
#pragma once

#include <gunrock/algorithms/algorithms.hxx>

namespace gunrock {
namespace bfs {

template <typename vertex_t>
struct param_t {
  vertex_t single_source;
  param_t(vertex_t _single_source) : single_source(_single_source) {}
};

template <typename vertex_t>
struct result_t {
  vertex_t* distances;
  vertex_t* predecessors;  ///< written by run_tree() only; run() accepts it for signature parity and leaves it alone
  result_t(vertex_t* _distances, vertex_t* _predecessors) : distances(_distances), predecessors(_predecessors) {}
};

/// `tree`: also record each reached vertex's parent in result.predecessors (run_tree). The depth-only problem and its
/// enactor instantiate exactly the operators they always had.
template <typename graph_t, typename param_type, typename result_type, bool tree = false>
struct problem_t : gunrock::problem_t<graph_t> {
  static constexpr bool record_tree = tree;
  param_type param;
  result_type result;
  using vertex_t = typename graph_t::vertex_type;
  using edge_t = typename graph_t::edge_type;
  using weight_t = typename graph_t::weight_type;

  /// One bit per vertex: "already has its depth". The push operator looks here before it touches the 4-byte label:
  /// ~97 % of the edges of a Kronecker BFS lead to a settled vertex, the map (n/8 bytes: 2 MiB at scale-24) stays in
  /// L2 while the streaming column indices keep evicting the 64 MiB label array (ncu: 35 % of the label gathers of the
  /// heavy level went to DRAM, 4.7 GB for 1.6 GB of column indices). Purely an accelerator: a clear bit only means
  /// "ask the label", so the depths are the same fixed point.
  memory::device_array_t<unsigned> settled;

  problem_t(graph_t& G, param_type& _param, result_type& _result, std::shared_ptr<gcuda::multi_context_t> _context)
      : gunrock::problem_t<graph_t>(G, _context), param(_param), result(_result) {}

  void init() override { settled.resize((this->label_count() + 31) / 32 + 1); }
  void reset() override {
    auto* ctx = this->get_single_context();
    const std::size_t n = this->label_count();  // global length in a partitioned run
    b200::fill(*ctx, result.distances, n, std::numeric_limits<vertex_t>::max());
    b200::set_one(*ctx, result.distances + param.single_source, vertex_t(0));
    cudaMemsetAsync(settled.data(), 0, settled.size() * sizeof(unsigned), ctx->stream());
    b200::set_one(*ctx, settled.data() + (std::size_t(param.single_source) >> 5),
                  1u << (unsigned(param.single_source) & 31u));
    if constexpr (tree) {  // -1 = unreached; the source is its own parent
      b200::fill(*ctx, result.predecessors, n, vertex_t(-1));
      b200::set_one(*ctx, result.predecessors + param.single_source, param.single_source);
    }
  }
};

/// A BFS operator that also records the parent: it returns true for exactly one call per vertex (push: the caller whose
/// atomic::min lowered the depth from INT_MAX; bottom-up and claim-first top-down: the thread that owns the vertex), so
/// that call stores `source` as the vertex's parent with a plain store and no other call touches it.
template <typename op_t, typename vertex_t>
struct record_parent_t {
  op_t op;
  vertex_t* predecessors;
  template <typename edge_t, typename weight_t>
  __host__ __device__ __forceinline__ bool operator()(vertex_t const& source, vertex_t const& neighbor,
                                                      edge_t const& edge, weight_t const& weight) const {
    if (!op(source, neighbor, edge, weight)) return false;
    predecessors[neighbor] = source;
    return true;
  }
};

template <typename problem_t, operators::load_balance_t lb, operators::advance_direction_t direction>
struct enactor_t : gunrock::enactor_t<problem_t> {
  using base_t = gunrock::enactor_t<problem_t>;
  using vertex_t = typename problem_t::vertex_t;
  using edge_t = typename problem_t::edge_t;
  using weight_t = typename problem_t::weight_t;
  using frontier_t = typename base_t::frontier_t;

  enactor_t(problem_t* _problem, std::shared_ptr<gcuda::multi_context_t> _context,
            enactor_properties_t _properties = enactor_properties_t())
      : base_t(_problem, _context, _properties) {
    if constexpr (direction == operators::advance_direction_t::optimized)  // bitmaps sized outside the timed loop
      this->direction.allocate(std::size_t(_problem->get_graph().get_number_of_vertices()),
                               _context->get_context(0)->stream());
  }

  void prepare_frontier(frontier_t* f, gcuda::multi_context_t& context) override {
    // partitioned run: only the owner starts with the source (as a local row id)
    const vertex_t row = this->get_problem()->local_row(this->get_problem()->param.single_source);
    if (util::limits::is_valid(row)) f->push_back(row);
  }

  void loop(gcuda::multi_context_t& context) override {
    auto E = this->get_enactor();
    auto P = this->get_problem();
    auto G = P->get_graph();
    auto distances = P->result.distances;
    // the depth-only problem gets its operators back unchanged
    auto with_parent = [P](auto op) {
      if constexpr (problem_t::record_tree)
        return record_parent_t<decltype(op), vertex_t>{op, P->result.predecessors};
      else
        return op;
    };
    const vertex_t next_depth = vertex_t(this->iteration + 1);

    unsigned* settled = P->settled.data();
    auto search = [distances, next_depth, settled] __host__ __device__(vertex_t const& source, vertex_t const& neighbor,
                                                                       edge_t const& edge,
                                                                       weight_t const& weight) -> bool {
      // same decision as the reference's unconditional atomicMin (bfs.hxx:96-99): a set bit or a label at or below
      // next_depth means the atomic could not lower it; the plain reads keep the ~97 % of edges that lead to an
      // already-settled vertex off the L2 atomic units and, through the 1-bit map, off the 4-byte label array
      const unsigned bit = 1u << (unsigned(neighbor) & 31u);
      if (thread::load(&settled[unsigned(neighbor) >> 5]) & bit) return false;
      const bool won = next_depth < math::atomic::min(&distances[neighbor], next_depth);
#ifdef __CUDA_ARCH__
      atomicOr(&settled[unsigned(neighbor) >> 5], bit);
#else
      settled[unsigned(neighbor) >> 5] |= bit;
#endif
      return won;
    };
    if constexpr (direction == operators::advance_direction_t::optimized) {
      // bottom-up form: the destination is unvisited and owned by the calling thread, so the same update
      // (depth := next_depth, always an improvement over INT_MAX) is a plain store.
      auto adopt = [distances, next_depth] __host__ __device__(vertex_t const& source, vertex_t const& neighbor,
                                                              edge_t const& edge, weight_t const& weight) -> bool {
        distances[neighbor] = next_depth;
        return true;
      };
      operators::advance::execute<lb, direction>(
          G, E, operators::advance::directional(with_parent(search), with_parent(adopt)), context);
    } else {
      operators::advance::execute<lb, direction>(G, E, with_parent(search), context);
    }
    if (context.partition && context.partition->world > 1) {
      // 1-D partitioned run: discovered vertices go to their owners, who keep min(depth) and de-duplicate
      error::throw_if_exception(direction == operators::advance_direction_t::optimized,
                                "partitioned direction-optimized BFS is driven by ess_dist_bfs");
      operators::exchange::execute(G, E, distances, context);
    }
  }
};

namespace detail {
template <bool tree, operators::load_balance_t lb, operators::advance_direction_t direction, typename graph_t>
float run(graph_t& G, typename graph_t::vertex_type& single_source, typename graph_t::vertex_type* distances,
          typename graph_t::vertex_type* predecessors, std::shared_ptr<gcuda::multi_context_t> context,
          enactor_properties_t properties, int* pull_steps, int* iterations, long long* work_stats) {
  using vertex_t = typename graph_t::vertex_type;
  using param_type = param_t<vertex_t>;
  using result_type = result_t<vertex_t>;
  using problem_type = problem_t<graph_t, param_type, result_type, tree>;
  using enactor_type = enactor_t<problem_type, lb, direction>;

  param_type param(single_source);
  result_type result(distances, predecessors);
  problem_type problem(G, param, result, context);
  problem.init();
  problem.reset();
  enactor_type enactor(&problem, context, properties);
  float ms = enactor.enact();
  if (pull_steps) *pull_steps = enactor.direction.pull_steps;
  if (iterations) *iterations = enactor.iteration;
  if (work_stats) {  // [0] pull vertices walked, [1] pull in-edges read, [2] push vertices, [3] push edges
    work_stats[0] = enactor.direction.pull_vertices_scanned;
    work_stats[1] = enactor.direction.pull_edges_inspected;
    work_stats[2] = enactor.direction.push_vertices_expanded;
    work_stats[3] = enactor.direction.push_edges_expanded;
    work_stats[4] = enactor.direction.pull_hint_misses;     // [4] bottom-up hint misses (lists walked)
    work_stats[5] = enactor.direction.pull_vertices_found;  // [5] vertices adopted bottom-up
    work_stats[6] = enactor.direction.push_vertices_found;  // [6] vertices claimed top-down
  }
  return ms;
}
}  // namespace detail

/// Depths only: `predecessors` is accepted for signature parity with the reference and never read or written.
template <operators::load_balance_t lb = operators::load_balance_t::block_mapped,
          operators::advance_direction_t direction = operators::advance_direction_t::forward, typename graph_t>
float run(graph_t& G, typename graph_t::vertex_type& single_source, typename graph_t::vertex_type* distances,
          typename graph_t::vertex_type* predecessors,
          std::shared_ptr<gcuda::multi_context_t> context =
              std::shared_ptr<gcuda::multi_context_t>(new gcuda::multi_context_t(0)),
          enactor_properties_t properties = enactor_properties_t(), int* pull_steps = nullptr, int* iterations = nullptr,
          long long* work_stats = nullptr) {
  return detail::run<false, lb, direction>(G, single_source, distances, predecessors, context, properties, pull_steps,
                                           iterations, work_stats);
}

/**
 * @brief run() plus the BFS tree. `distances` are the same as run()'s; `predecessors` (n entries, required, not
 * aliasing `distances`) receives predecessors[source] = source, -1 for every unreached vertex, and for every other
 * reached v an in-neighbour u (an edge u -> v of the CSR) with distances[u] == distances[v] - 1. Which of several such
 * parents is chosen depends on scheduling. Every entry is written, whatever the array held before. Not available on a
 * partitioned context: the exchange carries (vertex, depth) records only, so the parent would be lost at the owner.
 */
template <operators::load_balance_t lb = operators::load_balance_t::block_mapped,
          operators::advance_direction_t direction = operators::advance_direction_t::forward, typename graph_t>
float run_tree(graph_t& G, typename graph_t::vertex_type& single_source, typename graph_t::vertex_type* distances,
               typename graph_t::vertex_type* predecessors,
               std::shared_ptr<gcuda::multi_context_t> context =
                   std::shared_ptr<gcuda::multi_context_t>(new gcuda::multi_context_t(0)),
               enactor_properties_t properties = enactor_properties_t(), int* pull_steps = nullptr,
               int* iterations = nullptr, long long* work_stats = nullptr) {
  error::throw_if_exception(predecessors == nullptr, "bfs::run_tree: predecessors is required");
  error::throw_if_exception(predecessors == distances, "bfs::run_tree: predecessors must not alias distances");
  error::throw_if_exception(context->partition && context->partition->world > 1,
                            "bfs::run_tree: the BFS tree is not available on a partitioned context");
  return detail::run<true, lb, direction>(G, single_source, distances, predecessors, context, properties, pull_steps,
                                          iterations, work_stats);
}

}  // namespace bfs
}  // namespace gunrock
