/**
 * @file sssp.hxx
 * @brief Single-source shortest paths (label-correcting) client of the frontier operators.
 *
 * Same operators-level recipe as the reference (include/gunrock/algorithms/sssp.hxx:98-151): advance with
 * `d = dist[src] + w; old = atomic::min(&dist[nbr], d); keep iff d < old`, then a bypass filter that drops
 * a vertex already seen in this iteration (`visited[v] == iteration`, benign race). reset (:61-78): FLT_MAX
 * everywhere, 0 at the source, visited = -1. The single float add per relaxation is rounded exactly like
 * the CPU reference's, and min over monotone relaxations has a unique fixed point, so distances are
 * bit-identical to sssp_cpu for non-negative weights. run() keeps the reference signature (:155-163); the
 * leading template parameter picks the balancer (default block_mapped as in the reference).
 *
 * `near_far = true` (additive): the same relaxation operator driven by operators::advance::execute_near_far —
 * Davidson et al.'s near/far ordering inside one persistent kernel (advance/near_far.cuh) — for high-diameter
 * graphs where the level-per-launch loop above is latency- and rework-bound. `delta` is the bucket width
 * (<= 0: 64 x mean edge weight / mean degree — the mean weight on a degree-64 graph, narrower buckets for denser
 * ones, wider for sparse ones such as grids and road networks). Same distances, bit for bit.
 *
 * `run_delta` (additive): the same relaxation with a DENSE active set and a distance threshold, for low-diameter
 * graphs with big frontiers (Kronecker/RMAT). Per round one streaming pass over (dist, expanded-at) picks the
 * vertices whose distance dropped since they were last expanded and lies below the threshold T (duplicates are
 * impossible by construction: no output frontier, no de-duplication filter), the balanced merge-path advance
 * relaxes their out-edges, and T advances by `delta` only when nothing below it is left. Expanding near vertices
 * first halves the relaxations of plain label-correcting on scale-24 (1.2 G -> 0.6 G). Same fixed point, so the
 * distances are bit-identical again. Not for high-diameter graphs (an n-length pass per round): use near_far.
 */
#pragma once

#include <cmath>

#include <gunrock/algorithms/algorithms.hxx>

namespace gunrock {
namespace sssp {

template <typename vertex_t>
struct param_t {
  vertex_t single_source;
  param_t(vertex_t _single_source) : single_source(_single_source) {}
};

template <typename vertex_t, typename weight_t>
struct result_t {
  weight_t* distances;
  vertex_t* predecessors;
  result_t(weight_t* _distances, vertex_t* _predecessors, vertex_t) : distances(_distances), predecessors(_predecessors) {}
};

template <typename graph_t, typename param_type, typename result_type>
struct problem_t : gunrock::problem_t<graph_t> {
  param_type param;
  result_type result;
  using vertex_t = typename graph_t::vertex_type;
  using edge_t = typename graph_t::edge_type;
  using weight_t = typename graph_t::weight_type;

  memory::device_array_t<vertex_t> visited;

  problem_t(graph_t& G, param_type& _param, result_type& _result, std::shared_ptr<gcuda::multi_context_t> _context)
      : gunrock::problem_t<graph_t>(G, _context), param(_param), result(_result) {}

  void init() override { visited.resize(std::size_t(this->get_graph().get_number_of_vertices())); }
  void reset() override {
    auto* ctx = this->get_single_context();
    const std::size_t n = std::size_t(this->get_graph().get_number_of_vertices());
    b200::fill(*ctx, result.distances, this->label_count(), std::numeric_limits<weight_t>::max());
    b200::set_one(*ctx, result.distances + param.single_source, weight_t(0));
    b200::fill(*ctx, visited.data(), n, vertex_t(-1));
  }
};

/// Knob (ess_tune "sssp_fused_unique", default on): the level loop uses operators::advance::execute_unique (fused
/// advance + uniquify) instead of the reference's advance -> bypass-filter pair (0 selects that pair). Same
/// distances; 5-15 % faster on Kronecker scale-24 (profiles/r01h_probe_sssp_kron24.log).
inline int& fused_unique() {
  static int on = 1;
  return on;
}

template <typename problem_t, operators::load_balance_t lb, bool near_far = false>
struct enactor_t : gunrock::enactor_t<problem_t> {
  using base_t = gunrock::enactor_t<problem_t>;
  using vertex_t = typename problem_t::vertex_t;
  using edge_t = typename problem_t::edge_t;
  using weight_t = typename problem_t::weight_t;
  using frontier_t = typename base_t::frontier_t;

  float delta = 0.f;                               ///< near-far bucket width
  operators::advance::near_far_result_t near_far_stats;  ///< filled by the near-far path

  enactor_t(problem_t* _problem, std::shared_ptr<gcuda::multi_context_t> _context) : base_t(_problem, _context) {}

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
    auto visited = P->visited.data();
    const vertex_t iteration = vertex_t(this->iteration);
    if (context.partition && context.partition->world > 1) {
      // 1-D partitioned run: relax the owned rows against the full-length label array, then route every improved
      // neighbour to its owner, who keeps the minimum and de-duplicates (operators::exchange); the bypass filter
      // / fused uniquify of the single-GPU loop is subsumed by the owner-side de-duplication
      static_assert(!near_far || true, "");
      error::throw_if_exception(near_far, "partitioned SSSP uses the level loop, not the near-far kernel");
      auto shortest = [distances] __host__ __device__(vertex_t const& source, vertex_t const& neighbor,
                                                      edge_t const& edge, weight_t const& weight) -> bool {
        const weight_t candidate = thread::load(&distances[source]) + weight;
        return candidate < math::atomic::min(&distances[neighbor], candidate);
      };
      operators::advance::execute<lb>(G, E, shortest, context);
      operators::exchange::execute(G, E, distances, context);
      return;
    }

    // near-far form of the same relaxation: inside the persistent kernel the labels are read through L2
    auto relax = [distances] __host__ __device__(vertex_t const& source, vertex_t const& neighbor,
                                                 edge_t const& edge, weight_t const& weight) -> bool {
      const weight_t candidate = thread::load<thread::cache_t::global>(&distances[source]) + weight;
      return candidate < math::atomic::min(&distances[neighbor], candidate);
    };
    auto tentative = [distances] __host__ __device__(vertex_t const& v) -> float {
      return float(thread::load<thread::cache_t::global>(&distances[v]));
    };
    if constexpr (near_far) {
      // the same relaxation split at the atomic (advance::two_phase): the kernel keeps a lane's edges in flight together
      auto relax_issue = [distances] __host__ __device__(vertex_t const& source, vertex_t const& neighbor,
                                                         edge_t const& edge, weight_t const& weight) -> float2 {
        const weight_t candidate = thread::load<thread::cache_t::global>(&distances[source]) + weight;
        return make_float2(float(candidate), float(math::atomic::min(&distances[neighbor], candidate)));
      };
      auto relax_resolve = [] __host__ __device__(float2 const& token) -> bool { return token.x < token.y; };
      (void)relax;
      // (a per-source prologue — two_phase(prepare, issue, resolve), one label read per vertex — measured the same
      // time on the 4900^2 grid but 30 % more relaxations, because a staler source label is used for later edges)
      near_far_stats = operators::advance::execute_near_far(
          G, E, operators::advance::two_phase(relax_issue, relax_resolve), tentative, delta, context);
      this->iteration += near_far_stats.levels > 0 ? near_far_stats.levels - 1 : 0;  // enact() adds the last one
      (void)visited;
      (void)iteration;
      return;
    }

    auto shortest_path = [distances] __host__ __device__(vertex_t const& source, vertex_t const& neighbor,
                                                         edge_t const& edge, weight_t const& weight) -> bool {
      const weight_t candidate = thread::load(&distances[source]) + weight;
      return candidate < math::atomic::min(&distances[neighbor], candidate);
    };
    auto drop_repeats = [visited, iteration] __host__ __device__(vertex_t const& vertex) -> bool {
      if (visited[vertex] == iteration) return false;
      visited[vertex] = iteration;
      return true;
    };
    if (fused_unique()) {  // one pass: repeats are dropped at emission, no holes reach the next advance
      operators::advance::execute_unique<lb>(G, E, shortest_path, context);
      (void)drop_repeats;
    } else {
      operators::advance::execute<lb>(G, E, shortest_path, context);
      operators::filter::execute<operators::filter_algorithm_t::bypass>(G, E, drop_repeats, context);
    }
  }
};

template <operators::load_balance_t lb = operators::load_balance_t::block_mapped, bool near_far = false,
          typename graph_t>
float run(graph_t& G, typename graph_t::vertex_type& single_source, typename graph_t::weight_type* distances,
          typename graph_t::vertex_type* predecessors,
          std::shared_ptr<gcuda::multi_context_t> context =
              std::shared_ptr<gcuda::multi_context_t>(new gcuda::multi_context_t(0)),
          int* iterations = nullptr, float delta = 0.f, long long* work_stats = nullptr) {
  using vertex_t = typename graph_t::vertex_type;
  using weight_t = typename graph_t::weight_type;
  using param_type = param_t<vertex_t>;
  using result_type = result_t<vertex_t, weight_t>;
  using problem_type = problem_t<graph_t, param_type, result_type>;
  using enactor_type = enactor_t<problem_type, lb, near_far>;

  param_type param(single_source);
  result_type result(distances, predecessors, G.get_number_of_vertices());
  problem_type problem(G, param, result, context);
  problem.init();
  problem.reset();
  enactor_type enactor(&problem, context);
  if constexpr (near_far) {
    if (!(delta > 0.f)) {  // default bucket width: 64 x mean edge weight / mean degree (Davidson et al.'s rule of thumb)
      auto* ctx = context->get_context(0);
      const auto weights = graph::adjacency_of<false>(G).values;
      const auto m = G.get_number_of_edges();
      delta = 1.f;
      if (weights && m > 0) {
        memory::device_array_t<double> sum(1);
        cudaMemsetAsync(sum.data(), 0, sizeof(double), ctx->stream());
        b200::kernels::sum_kernel<<<b200::stream_grid(*ctx, std::size_t(m)), 256, 0, ctx->stream()>>>(
            weights, std::size_t(m), sum.data());
        double h = 0;
        cudaMemcpyAsync(&h, sum.data(), sizeof(double), cudaMemcpyDeviceToHost, ctx->stream());
        ctx->synchronize();
        if (h > 0) delta = float(h / double(m));
      }
      const double mean_degree = double(m) / double(G.get_number_of_vertices() > 0 ? G.get_number_of_vertices() : 1);
      delta = float(double(delta) * 64.0 / (mean_degree > 1.0 ? mean_degree : 1.0));
    }
    enactor.delta = delta;
  }
  float ms = enactor.enact();
  if (iterations) *iterations = enactor.iteration;
  if (work_stats) {  // [0] near levels, [1] far splits, [2] relaxations (near-far path only)
    work_stats[0] = enactor.near_far_stats.levels;
    work_stats[1] = enactor.near_far_stats.splits;
    work_stats[2] = (long long)enactor.near_far_stats.relaxations;
  }
  return ms;
}


namespace detail {

/// Mean edge weight of the graph (1 when it has no values): one streaming pass.
template <typename graph_t>
float mean_edge_weight(graph_t& G, gcuda::standard_context_t& ctx) {
  const auto weights = graph::adjacency_of<false>(G).values;
  const auto m = G.get_number_of_edges();
  if (!weights || m <= 0) return 1.f;
  memory::device_array_t<double> sum(1);
  cudaMemsetAsync(sum.data(), 0, sizeof(double), ctx.stream());
  b200::kernels::sum_kernel<<<b200::stream_grid(ctx, std::size_t(m)), 256, 0, ctx.stream()>>>(weights, std::size_t(m),
                                                                                            sum.data());
  double h = 0;
  cudaMemcpyAsync(&h, sum.data(), sizeof(double), cudaMemcpyDeviceToHost, ctx.stream());
  ctx.synchronize();
  return h > 0 ? float(h / double(m)) : 1.f;
}

/// run_delta's per-round selection. A vertex is due when dist[v] < expanded[v]; due vertices below `threshold`
/// are appended to `active` (expanded[v] = dist[v]); the others are counted (aux2) and the smallest of their
/// distances is kept (aux3, as 0x7f800000 - float bits so that zero means "none" under atomicMax).
template <typename vertex_t, typename weight_t>
__global__ void __launch_bounds__(256)
    delta_collect_kernel(const weight_t* __restrict__ dist, weight_t* __restrict__ expanded, vertex_t n,
                         weight_t threshold, vertex_t* __restrict__ active, b200::counter_t* counters) {
  __shared__ b200::counter_t sm[256 / 32 + 4];
  unsigned pending = 0, nearest = 0;
  const std::size_t per_cta = 256 * 4;
  const bool vector_dist = (reinterpret_cast<std::uintptr_t>(dist) & 15u) == 0;
  for (std::size_t base = std::size_t(blockIdx.x) * per_cta; base < std::size_t(n);
       base += std::size_t(gridDim.x) * per_cta) {
    const std::size_t first = base + std::size_t(threadIdx.x) * 4;
    vertex_t ids[4];
    weight_t d[4], e[4];
    // `dist` is the caller's output array, possibly a tensor view at any 4-byte offset; `expanded` is run_delta's
    // own n-length cudaMalloc'd array, 256-byte aligned
    if (vector_dist && first + 4 <= std::size_t(n) && sizeof(weight_t) == 4) {
      const float4 a = *reinterpret_cast<const float4*>(dist + first);
      const float4 b = *reinterpret_cast<const float4*>(expanded + first);
      d[0] = a.x, d[1] = a.y, d[2] = a.z, d[3] = a.w;
      e[0] = b.x, e[1] = b.y, e[2] = b.z, e[3] = b.w;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool in = first + i < std::size_t(n);
        d[i] = in ? dist[first + i] : weight_t(0);
        e[i] = in ? expanded[first + i] : weight_t(0);
      }
    }
    unsigned keep = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      ids[i] = vertex_t(first + i);
      if (first + i < std::size_t(n) && d[i] < e[i]) {
        if (d[i] < threshold) {
          keep |= 1u << i;
          expanded[first + i] = d[i];
        } else {
          ++pending;
          const unsigned key = 0x7f800000u - __float_as_uint(float(d[i]));
          nearest = key > nearest ? key : nearest;
        }
      }
    }
    b200::cta_append<256, 4>(ids, keep, active, counters + gcuda::scratch_t::out_count, b200::counter_t(n), sm);
  }
  pending = b200::warp_sum(pending);
  nearest = b200::warp_max(nearest);
  if (b200::lane_id() == 0 && pending) {
    atomicAdd(counters + gcuda::scratch_t::aux2, b200::counter_t(pending));
    atomicMax(counters + gcuda::scratch_t::aux3, b200::counter_t(nearest));
  }
}

}  // namespace detail

/**
 * @brief SSSP with a dense active set and delta thresholds (see the file comment). `delta` <= 0 picks half
 * the mean edge weight; +inf degenerates to plain label-correcting. stats (optional): [0] rounds that expanded,
 * [1] threshold advances, [2] vertices expanded (with repeats), [3] selection passes.
 */
template <typename graph_t>
float run_delta(graph_t& G, typename graph_t::vertex_type single_source, typename graph_t::weight_type* distances,
                std::shared_ptr<gcuda::multi_context_t> context, float delta = 0.f, int* iterations = nullptr,
                long long* stats = nullptr) {
  using vertex_t = typename graph_t::vertex_type;
  using edge_t = typename graph_t::edge_type;
  using weight_t = typename graph_t::weight_type;
  static_assert(sizeof(weight_t) == 4, "run_delta keys distances as IEEE-754 binary32");
  auto* ctx = context->get_context(0);
  auto stream = ctx->stream();
  auto& scratch = ctx->scratch();
  const vertex_t n = G.get_number_of_vertices();
  if (!(delta > 0.f)) delta = detail::mean_edge_weight(G, *ctx) / 2.f;

  memory::device_array_t<weight_t> expanded{std::size_t(n)};  // distance each vertex was last expanded at
  using frontier_type = frontier::frontier_t<vertex_t, edge_t>;
  frontier_type active{std::size_t(n)}, none;
  memory::device_array_t<edge_t> segments;
  b200::fill(*ctx, distances, std::size_t(n), std::numeric_limits<weight_t>::max());
  b200::fill(*ctx, expanded.data(), std::size_t(n), std::numeric_limits<weight_t>::max());
  b200::set_one(*ctx, distances + single_source, weight_t(0));

  auto relax = [distances] __host__ __device__(vertex_t const& source, vertex_t const& neighbor, edge_t const& edge,
                                               weight_t const& weight) -> bool {
    const weight_t candidate = distances[source] + weight;
    if (candidate < distances[neighbor]) math::atomic::min(&distances[neighbor], candidate);  // plain read prunes
    return false;
  };

  auto& timer = ctx->timer();
  timer.begin();
  float threshold = delta;
  long long rounds = 0, advances = 0, expanded_vertices = 0, passes = 0;
  const bool was_async = scratch.async_when_no_output;
  scratch.async_when_no_output = true;  // the selection pass that follows is the round's one host round trip
  const unsigned grid = gcuda::persistent_grid(*ctx, (std::size_t(n) + 1023) / 1024, 8);
  for (;;) {
    scratch.zero(stream);
    ctx->profiler().begin(gcuda::profiler_t::filter_op, stream);
    detail::delta_collect_kernel<<<grid, 256, 0, stream>>>(distances, expanded.data(), n, weight_t(threshold),
                                                           active.data(), scratch.d);
    ctx->profiler().end(stream);
    scratch.fetch(stream);
    ++passes;
    const std::size_t count = std::size_t(scratch.h[gcuda::scratch_t::out_count]);
    const auto pending = scratch.h[gcuda::scratch_t::aux2];
    if (count == 0) {
      if (pending == 0) break;
      // nothing due below the threshold: jump to the bucket of the nearest pending distance
      const unsigned bits = 0x7f800000u - unsigned(scratch.h[gcuda::scratch_t::aux3]);
      float nearest;
      std::memcpy(&nearest, &bits, sizeof(float));
      const float next = (std::floor(nearest / delta) + 1.f) * delta;
      threshold = next > threshold ? next : threshold + delta;
      // strict progress: with distances above ~2^24 * delta both forms can round to <= nearest and the round
      // would select nothing for ever; the selection is `dist < threshold`, so step just past the nearest key
      if (!(threshold > nearest)) threshold = std::nextafter(nearest, std::numeric_limits<float>::infinity());
      if (!(threshold < std::numeric_limits<float>::max())) threshold = std::numeric_limits<float>::max();
      ++advances;
      continue;
    }
    active.set_number_of_elements(count);
    operators::advance::execute<operators::load_balance_t::merge_path, operators::advance_direction_t::forward,
                                operators::advance_io_type_t::vertices, operators::advance_io_type_t::none>(
        G, relax, &active, &none, segments, *context);
    ++rounds;
    expanded_vertices += (long long)count;
  }
  scratch.async_when_no_output = was_async;
  const float ms = timer.end();
  if (iterations) *iterations = int(rounds);
  if (stats) stats[0] = rounds, stats[1] = advances, stats[2] = expanded_vertices, stats[3] = passes;
  return ms;
}

}  // namespace sssp
}  // namespace gunrock
