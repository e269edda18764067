/**
 * @file pr.hxx
 * @brief PageRank client of the frontier operators (whole-graph advance, no output frontier).
 *
 * Follows the reference's iteration (include/gunrock/algorithms/pr.hxx): reset :64-92 (p = 1/n, plast = 0,
 * iweights[v] = alpha / Σw(v), 0 when v has no out-edges); loop :106-153 (plast = p; dangling mass
 * dsum = Σ_{iweights==0} alpha·p; p = (1-alpha+dsum)/n; advance<graph, none> with
 * atomic::add(p+dst, plast[src]·iweights[src]·w)); is_converged :155-178 (after the first iteration, stop
 * when max|p - plast| < tol). Enactor runs with self_manage_frontiers like the reference (:210-211).
 *
 * The n-length passes are fused: one kernel copies p→plast and reduces the dangling mass into a device
 * scalar (double), the next one reads that scalar to refill p — no host round trip between them
 * (the reference blocks on a thrust::transform_reduce, :128-131). `pull = true` replaces the atomic
 * scatter by a CSC gather with a per-vertex double accumulator (deterministic, no atomics): needs
 * a CSC view.
 */
#pragma once

#include <gunrock/algorithms/algorithms.hxx>

namespace gunrock {
namespace pr {

template <typename weight_t>
struct param_t {
  weight_t alpha;
  weight_t tol;
  int max_iterations;
  param_t(weight_t _alpha, weight_t _tol, int _max_iterations = 1000)
      : alpha(_alpha), tol(_tol), max_iterations(_max_iterations) {}
};

template <typename weight_t>
struct result_t {
  weight_t* p;
  result_t(weight_t* _p) : p(_p) {}
};

namespace kernels {
using b200::counter_t;

template <typename graph_t, typename weight_t>
__global__ void __launch_bounds__(256) inverse_weights_kernel(graph_t G, weight_t alpha, weight_t* iweights) {
  using edge_t = typename graph_t::edge_type;
  using vertex_t = typename graph_t::vertex_type;
  const std::size_t n = std::size_t(G.get_number_of_vertices());
  for (std::size_t v = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; v < n;
       v += std::size_t(gridDim.x) * blockDim.x) {
    const edge_t beg = G.get_starting_edge(vertex_t(v)), end = beg + G.get_number_of_neighbors(vertex_t(v));
    weight_t sum = 0;
    for (edge_t e = beg; e < end; ++e) sum += G.get_edge_weight(e);
    iweights[v] = sum != 0 ? alpha / sum : weight_t(0);
  }
}

/// plast = p and dangling += Σ_{iweights==0} alpha·p (double accumulator, one atomic per warp).
template <typename weight_t>
__global__ void __launch_bounds__(256)
    snapshot_kernel(const weight_t* __restrict__ p, weight_t* __restrict__ plast, const weight_t* __restrict__ iweights,
                    std::size_t n, weight_t alpha, double* dangling) {
  double mine = 0;
  for (std::size_t v = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; v < n;
       v += std::size_t(gridDim.x) * blockDim.x) {
    const weight_t x = p[v];
    plast[v] = x;
    if (iweights[v] == 0) mine += double(alpha) * double(x);
  }
  mine = b200::warp_sum(mine);
  if (b200::lane_id() == 0 && mine != 0) atomicAdd(dangling, mine);
}

template <typename weight_t>
__global__ void __launch_bounds__(256)
    teleport_kernel(weight_t* __restrict__ p, std::size_t n, weight_t alpha, const double* dangling) {
  const weight_t base = weight_t((1.0 - double(alpha) + *dangling) / double(n));
  for (std::size_t v = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; v < n;
       v += std::size_t(gridDim.x) * blockDim.x)
    p[v] = base;
}

/// Pull-side snapshot: plast = p, contrib[u] = p[u]·iweights[u] (what every out-edge of u carries), and the
/// dangling mass in double. One pass; the per-edge gather then needs ONE random 4-byte read per edge.
template <typename weight_t>
__global__ void __launch_bounds__(256)
    snapshot_contrib_kernel(const weight_t* __restrict__ p, weight_t* __restrict__ plast,
                            const weight_t* __restrict__ iweights, weight_t* __restrict__ contrib, std::size_t n,
                            weight_t alpha, double* dangling) {
  double mine = 0;
  for (std::size_t v = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; v < n;
       v += std::size_t(gridDim.x) * blockDim.x) {
    const weight_t x = p[v], iw = iweights[v];
    plast[v] = x;
    contrib[v] = x * iw;
    if (iw == 0) mine += double(alpha) * double(x);
  }
  mine = b200::warp_sum(mine);
  if (b200::lane_id() == 0 && mine != 0) atomicAdd(dangling, mine);
}

/// Rows binned once per graph by in-degree: [0, short_degree) one thread each, [short_degree, hub_degree) one
/// warp each, the rest one CTA each. Lists are ascending (stable) so neighbouring threads touch neighbouring rows.
constexpr int short_degree = 8;
constexpr int hub_degree = 4096;

template <typename vertex_t, typename edge_t>
__global__ void __launch_bounds__(256)
    bin_rows_kernel(const edge_t* __restrict__ offsets, vertex_t n, vertex_t* __restrict__ short_rows,
                    vertex_t* __restrict__ warp_rows, vertex_t* __restrict__ hub_rows, counter_t* counts) {
  for (std::size_t base = std::size_t(blockIdx.x) * blockDim.x; base < std::size_t(n);
       base += std::size_t(gridDim.x) * blockDim.x) {
    const std::size_t v = base + threadIdx.x;
    long long d = -1;
    if (v < std::size_t(n)) d = (long long)(offsets[v + 1] - offsets[v]);
    const bool is_short = d >= 0 && d < short_degree, is_hub = d >= hub_degree, is_warp = d >= short_degree && !is_hub;
    counter_t at = b200::warp_append_slot(is_short, counts + 0);
    if (is_short) short_rows[at] = vertex_t(v);
    at = b200::warp_append_slot(is_warp, counts + 1);
    if (is_warp) warp_rows[at] = vertex_t(v);
    at = b200::warp_append_slot(is_hub, counts + 2);
    if (is_hub) hub_rows[at] = vertex_t(v);
  }
}

/// Σ over the in-edges [beg, end) strided by `step` starting at `first`, double accumulator.
template <typename vertex_t, typename edge_t, typename weight_t>
__device__ __forceinline__ double gather_edges(const graph::adjacency_t<vertex_t, edge_t, weight_t>& A,
                                               const weight_t* __restrict__ contrib, edge_t first, edge_t end,
                                               edge_t step) {
  double acc = 0;
  if (A.values) {
    for (edge_t e = first; e < end; e += step) acc += double(__ldg(contrib + __ldg(A.indices + e)) * __ldg(A.values + e));
  } else {
    for (edge_t e = first; e < end; e += step) acc += double(__ldg(contrib + __ldg(A.indices + e)));
  }
  return acc;
}

template <typename weight_t>
__device__ __forceinline__ void finish_row(weight_t* p, const weight_t* plast, std::size_t v, double base, double acc,
                                           float& err) {
  const weight_t x = weight_t(base + acc);
  p[v] = x;
  err = fmaxf(err, fabsf(float(x) - float(plast[v])));
}

/// mode 0: one thread per listed row; 1: one warp per row; 2: one CTA per row. p[v] = base + Σ contrib·w (pull
/// PageRank), and the convergence error max|p - plast| is folded in (no separate pass).
template <int mode, typename vertex_t, typename edge_t, typename weight_t>
__global__ void __launch_bounds__(256)
    gather_rows_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, const vertex_t* __restrict__ rows,
                       std::size_t n_rows, const weight_t* __restrict__ contrib, const weight_t* __restrict__ plast,
                       weight_t* __restrict__ p, weight_t alpha, const double* dangling, unsigned* err_bits) {
  __shared__ double block_acc[256 / 32];
  const double base = (1.0 - double(alpha) + *dangling) / double(A.n);
  const unsigned lane = b200::lane_id();
  float err = 0.f;
  if constexpr (mode == 0) {
    for (std::size_t i = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n_rows;
         i += std::size_t(gridDim.x) * blockDim.x) {
      const vertex_t v = rows[i];
      finish_row(p, plast, std::size_t(v), base, gather_edges(A, contrib, A.offsets[v], A.offsets[v + 1], edge_t(1)), err);
    }
  } else if constexpr (mode == 1) {
    const std::size_t warps = (std::size_t(gridDim.x) * blockDim.x) >> 5;
    for (std::size_t i = (std::size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; i < n_rows; i += warps) {
      const vertex_t v = rows[i];
      double acc = gather_edges(A, contrib, edge_t(A.offsets[v] + lane), A.offsets[v + 1], edge_t(32));
      acc = b200::warp_sum(acc);
      if (lane == 0) finish_row(p, plast, std::size_t(v), base, acc, err);
    }
  } else {
    for (std::size_t i = blockIdx.x; i < n_rows; i += gridDim.x) {
      const vertex_t v = rows[i];
      double acc = gather_edges(A, contrib, edge_t(A.offsets[v] + threadIdx.x), A.offsets[v + 1], edge_t(256));
      acc = b200::warp_sum(acc);
      if (lane == 0) block_acc[threadIdx.x >> 5] = acc;
      __syncthreads();
      if (threadIdx.x == 0) {
        double total = 0;
        for (int k = 0; k < 256 / 32; ++k) total += block_acc[k];
        finish_row(p, plast, std::size_t(v), base, total, err);
      }
      __syncthreads();
    }
  }
  err = b200::warp_max(err);
  if (lane == 0 && err > 0.f) atomicMax(err_bits, __float_as_uint(err));
}
}  // namespace kernels

template <typename graph_t, typename param_type, typename result_type>
struct problem_t : gunrock::problem_t<graph_t> {
  param_type param;
  result_type result;
  using vertex_t = typename graph_t::vertex_type;
  using edge_t = typename graph_t::edge_type;
  using weight_t = typename graph_t::weight_type;

  memory::device_array_t<weight_t> plast;
  memory::device_array_t<weight_t> iweights;
  memory::device_array_t<double> scalars;  ///< [0] dangling mass, [1] (as unsigned) max-abs-diff bits
  // pull path only: per-vertex contribution p·iweights and the rows binned by in-degree (built once in init)
  bool pull = false;
  memory::device_array_t<weight_t> contrib;
  memory::device_array_t<vertex_t> short_rows, warp_rows, hub_rows;
  std::size_t n_short = 0, n_warp = 0, n_hub = 0;

  problem_t(graph_t& G, param_type& _param, result_type& _result, std::shared_ptr<gcuda::multi_context_t> _context)
      : gunrock::problem_t<graph_t>(G, _context), param(_param), result(_result) {}

  void init() override {
    const std::size_t n = std::size_t(this->get_graph().get_number_of_vertices());
    plast.resize(n);
    iweights.resize(n);
    scalars.resize(2);
    if (pull) prepare_pull();
  }

  /// One-time binning of the rows of the CSC view by in-degree (see kernels::bin_rows_kernel).
  void prepare_pull() {
    auto* ctx = this->get_single_context();
    auto g = this->get_graph();
    const auto A = graph::adjacency_of<true>(g);
    // iweights sums the CSR weights and the gather multiplies by the CSC ones: with weights on only one view the
    // ranks would be silently wrong, so refuse the graph.
    error::throw_if_exception(A.m > 0 && (A.values == nullptr) != (graph::adjacency_of<false>(g).values == nullptr),
                              "pr: pull needs edge weights on both the CSR and the CSC view, or on neither");
    const std::size_t n = std::size_t(A.n);
    contrib.resize(n);
    short_rows.resize(n);
    warp_rows.resize(n);
    hub_rows.resize(n);
    memory::device_array_t<b200::counter_t> counts(3);
    cudaMemsetAsync(counts.data(), 0, 3 * sizeof(b200::counter_t), ctx->stream());
    kernels::bin_rows_kernel<<<b200::stream_grid(*ctx, n), 256, 0, ctx->stream()>>>(
        A.offsets, A.n, short_rows.data(), warp_rows.data(), hub_rows.data(), counts.data());
    b200::counter_t h[3] = {0, 0, 0};
    cudaMemcpyAsync(h, counts.data(), sizeof(h), cudaMemcpyDeviceToHost, ctx->stream());
    ctx->synchronize();
    n_short = std::size_t(h[0]), n_warp = std::size_t(h[1]), n_hub = std::size_t(h[2]);
  }
  void reset() override {
    auto* ctx = this->get_single_context();
    auto g = this->get_graph();
    const std::size_t n = std::size_t(g.get_number_of_vertices());
    b200::fill(*ctx, result.p, n, weight_t(1.0 / double(n)));
    b200::fill(*ctx, plast.data(), n, weight_t(0));
    kernels::inverse_weights_kernel<<<b200::stream_grid(*ctx, n), 256, 0, ctx->stream()>>>(g, param.alpha,
                                                                                          iweights.data());
  }
};

template <typename problem_t, operators::load_balance_t lb, bool pull>
struct enactor_t : gunrock::enactor_t<problem_t> {
  using base_t = gunrock::enactor_t<problem_t>;
  using vertex_t = typename problem_t::vertex_t;
  using edge_t = typename problem_t::edge_t;
  using weight_t = typename problem_t::weight_t;

  enactor_t(problem_t* _problem, std::shared_ptr<gcuda::multi_context_t> _context, enactor_properties_t _properties)
      : base_t(_problem, _context, _properties) {}

  void loop(gcuda::multi_context_t& context) override {
    auto E = this->get_enactor();
    auto P = this->get_problem();
    auto G = P->get_graph();
    auto* ctx = context.get_context(0);
    const std::size_t n = std::size_t(G.get_number_of_vertices());
    weight_t* p = P->result.p;
    weight_t* plast = P->plast.data();
    weight_t* iweights = P->iweights.data();
    const weight_t alpha = P->param.alpha;
    double* dangling = P->scalars.data();

    // (extended lambdas may not be defined inside an if-constexpr block, so it is built unconditionally)
    auto spread = [p, plast, iweights] __host__ __device__(vertex_t const& src, vertex_t const& dst,
                                                           edge_t const& edge, weight_t const& weight) -> bool {
      math::atomic::add(p + dst, plast[src] * iweights[src] * weight);
      return false;
    };
    cudaMemsetAsync(P->scalars.data(), 0, 2 * sizeof(double), ctx->stream());
    if constexpr (pull) {
      const auto A = graph::adjacency_of<true>(G);
      weight_t* contrib = P->contrib.data();
      unsigned* err_bits = reinterpret_cast<unsigned*>(P->scalars.data() + 1);
      kernels::snapshot_contrib_kernel<<<b200::stream_grid(*ctx, n), 256, 0, ctx->stream()>>>(p, plast, iweights, contrib,
                                                                                              n, alpha, dangling);
      if (P->n_short)
        kernels::gather_rows_kernel<0><<<b200::stream_grid(*ctx, P->n_short), 256, 0, ctx->stream()>>>(
            A, P->short_rows.data(), P->n_short, contrib, plast, p, alpha, dangling, err_bits);
      if (P->n_warp)
        kernels::gather_rows_kernel<1><<<gcuda::persistent_grid(*ctx, (P->n_warp + 7) / 8, 8), 256, 0, ctx->stream()>>>(
            A, P->warp_rows.data(), P->n_warp, contrib, plast, p, alpha, dangling, err_bits);
      if (P->n_hub)
        kernels::gather_rows_kernel<2><<<gcuda::persistent_grid(*ctx, P->n_hub, 8), 256, 0, ctx->stream()>>>(
            A, P->hub_rows.data(), P->n_hub, contrib, plast, p, alpha, dangling, err_bits);
      error::check_last("pr gather");
      (void)spread;
      (void)E;
    } else {
      kernels::snapshot_kernel<<<b200::stream_grid(*ctx, n), 256, 0, ctx->stream()>>>(p, plast, iweights, n, alpha,
                                                                                      dangling);
      kernels::teleport_kernel<<<b200::stream_grid(*ctx, n), 256, 0, ctx->stream()>>>(p, n, alpha, dangling);
      operators::advance::execute<lb, operators::advance_direction_t::forward, operators::advance_io_type_t::graph,
                                  operators::advance_io_type_t::none>(G, E, spread, context);
    }
  }

  bool is_converged(gcuda::multi_context_t& context) override {
    if (this->iteration == 0) return false;
    auto P = this->get_problem();
    if (this->iteration >= P->param.max_iterations) return true;
    auto* ctx = context.get_context(0);
    const std::size_t n = std::size_t(P->get_graph().get_number_of_vertices());
    unsigned* err_bits = reinterpret_cast<unsigned*>(P->scalars.data() + 1);
    if constexpr (!pull) {  // the pull kernels fold max|p - plast| into the gather
      cudaMemsetAsync(err_bits, 0, sizeof(unsigned), ctx->stream());
      b200::kernels::max_abs_diff_kernel<<<b200::stream_grid(*ctx, n), 256, 0, ctx->stream()>>>(
          P->result.p, P->plast.data(), n, err_bits);
    }
    unsigned h_bits = 0;
    cudaMemcpyAsync(&h_bits, err_bits, sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream());
    ctx->synchronize();
    float err;
    std::memcpy(&err, &h_bits, sizeof(float));
    return err < P->param.tol;
  }
};

template <operators::load_balance_t lb = operators::load_balance_t::block_mapped, bool pull = false, typename graph_t>
float run(graph_t& G, typename graph_t::weight_type alpha, typename graph_t::weight_type tol,
          typename graph_t::weight_type* p,
          std::shared_ptr<gcuda::multi_context_t> context =
              std::shared_ptr<gcuda::multi_context_t>(new gcuda::multi_context_t(0)),
          int* iterations = nullptr, int max_iterations = 1000) {
  using weight_t = typename graph_t::weight_type;
  using param_type = param_t<weight_t>;
  using result_type = result_t<weight_t>;
  using problem_type = problem_t<graph_t, param_type, result_type>;
  using enactor_type = enactor_t<problem_type, lb, pull>;

  param_type param(alpha, tol, max_iterations);
  result_type result(p);
  problem_type problem(G, param, result, context);
  problem.pull = pull;
  problem.init();
  problem.reset();
  enactor_properties_t props;
  props.self_manage_frontiers = true;
  enactor_type enactor(&problem, context, props);
  float ms = enactor.enact();
  if (iterations) *iterations = enactor.iteration;
  return ms;
}

}  // namespace pr
}  // namespace gunrock
