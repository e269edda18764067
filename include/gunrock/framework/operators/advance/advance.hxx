/**
 * @file advance.hxx
 * @brief operators::advance::execute — neighbour expansion of a frontier.
 *
 * Public signatures are the reference's (include/gunrock/framework/operators/advance/advance.hxx:91-104
 * explicit buffers, :192-221 enactor form, default template arguments included):
 *
 *   advance::execute<lb, direction, input_type, output_type>(G, E, op, context, swap_buffers = true)
 *   advance::execute<lb, direction, input_type, output_type>(G, op, input*, output*, segments, context)
 *
 * op is  bool(vertex_t const& src, vertex_t const& nbr, edge_t const& e, weight_t const& w)  invoked with
 * lvalues exactly once per (frontier item, edge). Behavioural contract vs the reference:
 *   - output holds the neighbours for which op returned true. The reference writes one slot per edge and
 *     marks failures with -1 (block_mapped.hxx:143-144); here survivors are compacted, so
 *     get_number_of_elements() is the number of survivors. Slot order is unspecified in both.
 *   - direction::backward walks the CSC view for every balancer (the reference honours it only in
 *     merge_path, merge_path.hxx:59-61).
 *   - direction::optimized (reference: throws, merge_path.hxx:41-43) switches between push over CSR and pull
 *     over CSC with a visited bitmap kept in E->direction; see pull.cuh for its operator contract. Only the
 *     enactor form supports it, and the graph must hold both views.
 *   - load_balance_t::bucketing (reference: empty body, bucketing.hxx:31-36, never dispatched) is implemented.
 *   - warp_mapped / work_stealing / edge frontiers throw "not supported", as the reference does.
 *   - more than one context in `context` throws like the reference (advance.hxx:125-128): multi-GPU runs
 *     are one process per GPU, each with a single-device context (DESIGN.md "multi-GPU").
 * Host cost per call: one counter memset, 1-4 kernel launches, one 128-byte D2H and ONE stream
 * synchronisation (the reference: >=3 syncs + cudaMalloc/cudaFree, SURVEY.md §3.1).
 */
#pragma once

#include <gunrock/cuda/cuda.hxx>
#include <gunrock/error.hxx>
#include <gunrock/util/type_limits.hxx>
#include <gunrock/framework/operators/configs.hxx>
#include <gunrock/framework/operators/advance/kernels.cuh>
#include <gunrock/framework/operators/advance/quad.cuh>
#include <gunrock/framework/operators/advance/pull.cuh>
#include <gunrock/framework/operators/advance/near_far.cuh>

namespace gunrock {
namespace operators {
namespace advance {

namespace detail {

using gcuda::scratch_t;
using kernels::counter_t;
using kernels::visit_t;

/// Max degree of one view of a graph, computed once per (context, graph build, view) and cached. The key is the
/// graph's build serial, not the offsets address: a graph built over recycled memory (the torch caching allocator,
/// the handle's device pool) must not inherit the max degree of the graph that lived there before, because a stale,
/// too small value switches off the output-capacity guard of the thread- and block-mapped kernels. Serial 0 (a graph
/// set() on the device) is never cached.
template <typename vertex_t, typename edge_t>
long long max_degree(gcuda::standard_context_t& ctx, std::uint64_t graph_serial, const edge_t* offsets, vertex_t n) {
  auto& s = ctx.scratch();
  if (graph_serial != 0 && s.max_degree_graph == graph_serial && s.max_degree_offsets == offsets &&
      s.max_degree_val >= 0)
    return s.max_degree_val;
  auto stream = ctx.stream();
  cudaMemsetAsync(s.d + scratch_t::aux3, 0, sizeof(counter_t), stream);
  kernels::max_degree_kernel<<<gcuda::persistent_grid(ctx, (std::size_t(n) + 255) / 256, 8), 256, 0, stream>>>(
      offsets, n, s.d + scratch_t::aux3);
  s.fetch(stream);
  s.max_degree_graph = graph_serial;
  s.max_degree_offsets = offsets;
  s.max_degree_val = (long long)s.h[scratch_t::aux3];
  return s.max_degree_val;
}

/// Raw device pointer of a work-offsets container (our device_array_t or a thrust::device_vector).
template <typename pointer_t>
auto raw_of(pointer_t p) {
  if constexpr (std::is_pointer<pointer_t>::value)
    return p;
  else
    return p.get();
}

template <typename frontier_t>
void grow_output(frontier_t* output, std::size_t needed) {
  if (output->get_capacity() < needed) output->reserve(needed);
}

struct no_epilogue_t {
  template <typename... args_t>
  void operator()(args_t&&...) const {}
};

/// Calls f(std::true_type{}) or f(std::false_type{}), so that a runtime flag picks a kernel's template flag in
/// one launch expression.
template <typename F>
void with_bool(bool b, F&& f) {
  if (b)
    f(std::true_type{});
  else
    f(std::false_type{});
}

/**
 * @brief The push kernels of one expansion attempt, one launcher per balancer. Each launcher chooses once between
 * the quad engine (quad.cuh) and the scalar kernels, and brackets its launches for the profiler.
 */
template <bool graph_input, bool has_output, visit_t policy, typename vertex_t, typename edge_t, typename weight_t,
          typename operator_t>
struct push_launch_t {
  /// 128-bit column / weight loads need 4-byte elements (and 16-byte aligned arrays, checked at run time)
  static constexpr bool quad_types = sizeof(vertex_t) == 4 && sizeof(weight_t) == 4;

  gcuda::standard_context_t& ctx;
  graph::adjacency_t<vertex_t, edge_t, weight_t> A;
  operator_t& op;
  const vertex_t* in;
  std::size_t nf;
  vertex_t* out;
  counter_t* C;
  counter_t capacity;
  unsigned* visited;
  bool quad;  // the quad engine runs (never true without quad_types)
  long long maxdeg;

  gcuda::profiler_t& prof() { return ctx.profiler(); }
  gcuda::stream_t stream() { return ctx.stream(); }
  std::size_t item_ctas() const { return (nf + kernels::cta_threads - 1) / kernels::cta_threads; }

  /// Calls f(std::bool_constant<quad>{}); the quad kernels are only instantiated for quad_types.
  template <typename F>
  void with_engine(F&& f) {
    if constexpr (quad_types) {
      if (quad) return f(std::true_type{});
    }
    f(std::false_type{});
  }

  /// Σdeg of the frontier, needed by the thread- and block-mapped kernels' capacity guard when every item at the
  /// max degree might not fit the output. Returns whether the guard is on.
  bool degree_sum_for_guard() {
    const bool guard = has_output && (long double)(nf) * (long double)(maxdeg) > (long double)(capacity);
    if (guard) {
      prof().begin(gcuda::profiler_t::work_prepare, stream());
      kernels::degree_sum_kernel<graph_input><<<gcuda::persistent_grid(ctx, item_ctas(), 8), 256, 0, stream()>>>(
          A.offsets, in, nf, C);
      prof().end(stream());
    }
    return guard;
  }

  /// The hubs deferred to `big_list` (block_mapped, bucketing), expanded grid-wide. The guard of these kernels
  /// reads Σdeg, which is 0 = "fits" when it was not computed.
  template <bool quad_engine>
  void hubs(vertex_t* big_list) {
    if constexpr (quad_engine) {  // column indices staged through shared memory by the TMA unit
      auto kernel = kernels::big_list_bulk_kernel<has_output, policy, vertex_t, edge_t, weight_t, operator_t>;
      kernel<<<gcuda::full_grid(ctx, kernel), 256, 0, stream()>>>(A, op, big_list, C + scratch_t::big_count, out, C,
                                                                  capacity, visited);
    } else {
      kernels::big_list_kernel<has_output, policy>
          <<<gcuda::persistent_grid(ctx, ~std::size_t(0), 6), 256, 0, stream()>>>(
              A, op, big_list, C + scratch_t::big_count, out, C, capacity, visited);
    }
  }

  void thread_mapped() {
    const bool guard = degree_sum_for_guard();
    prof().begin(gcuda::profiler_t::push_expand, stream());
    with_bool(guard, [&](auto g) {
      kernels::thread_mapped_kernel<graph_input, has_output, decltype(g)::value, policy>
          <<<gcuda::persistent_grid(ctx, item_ctas(), 8), 256, 0, stream()>>>(A, op, in, nf, nullptr, out, C, capacity,
                                                                              visited);
    });
    prof().end(stream());
  }

  void block_mapped() {
    const bool guard = degree_sum_for_guard();
    prof().begin(gcuda::profiler_t::push_expand, stream());
    vertex_t* big_list = nullptr;
    if (maxdeg >= kernels::big_degree) {
      // a frontier may repeat a hub (SSSP), so the only safe bound on deferred items is nf
      big_list = reinterpret_cast<vertex_t*>(ctx.scratch().temp(nf * sizeof(vertex_t)));
    }
    with_engine([&](auto q) {
      with_bool(guard, [&](auto g) {
        constexpr bool guarded = decltype(g)::value;
        if constexpr (decltype(q)::value) {
          auto kernel = kernels::block_mapped_quad_kernel<graph_input, has_output, guarded, policy, vertex_t, edge_t,
                                                          weight_t, operator_t>;
          kernel<<<gcuda::full_grid(ctx, kernel, item_ctas()), 256, 0, stream()>>>(A, op, in, nf, out, C, capacity,
                                                                                   visited, big_list);
        } else {
          kernels::block_mapped_kernel<graph_input, has_output, guarded, policy>
              <<<gcuda::persistent_grid(ctx, item_ctas(), 6), 256, 0, stream()>>>(A, op, in, nf, out, C, capacity,
                                                                                  visited, big_list);
        }
      });
      if (big_list) {
        hubs<decltype(q)::value>(big_list);
        prof().launches_total += 1;
      }
    });
    prof().end(stream());
  }

  template <typename work_tiles_t>
  void merge_path(work_tiles_t& segments) {
    // CTAs the single-launch kernels can use on a tiny level
    const long double bound = (long double)nf * (long double)maxdeg / kernels::tile_edges + 1;
    const std::size_t tiles = bound > 1e9L ? std::size_t(1000000000) : std::size_t(bound);
    with_engine([&](auto q) {
      constexpr bool quad_engine = decltype(q)::value;
      if (nf <= std::size_t(quad_engine ? kernels::small_items : kernels::tile_edges)) {
        // tiny level: one launch, table built per CTA
        prof().begin(gcuda::profiler_t::push_expand, stream());
        if constexpr (quad_engine) {
          auto kernel = kernels::merge_path_small_quad_kernel<graph_input, has_output, policy, vertex_t, edge_t,
                                                              weight_t, operator_t>;
          kernel<<<gcuda::full_grid(ctx, kernel, (tiles + 1) / 2), 256, 0, stream()>>>(A, op, in, int(nf), out, C,
                                                                                       capacity, visited);
        } else {
          kernels::merge_path_small_kernel<graph_input, has_output, policy>
              <<<gcuda::persistent_grid(ctx, tiles, 6), 256, 0, stream()>>>(A, op, in, int(nf), out, C, capacity,
                                                                            visited);
        }
        prof().end(stream());
        return;
      }
      if (segments.size() < nf + 1) segments.resize(nf + 1);
      const std::size_t prep_tiles = (nf + kernels::cta_threads * kernels::prep_items - 1) /
                                     (kernels::cta_threads * kernels::prep_items);
      gcuda::arena_layout_t layout;
      const std::size_t at_src = layout.add((nf + 1) * sizeof(vertex_t));
      const std::size_t at_beg = layout.add((nf + 1) * sizeof(edge_t));
      const std::size_t at_end = layout.add((nf + 1) * sizeof(edge_t));
      const std::size_t at_state = layout.add(2 * prep_tiles * sizeof(b200::tile_word_t));
      unsigned char* base = ctx.scratch().temp(layout.bytes);
      auto* work_src = reinterpret_cast<vertex_t*>(base + at_src);
      auto* work_beg = reinterpret_cast<edge_t*>(base + at_beg);
      auto* work_end = reinterpret_cast<edge_t*>(base + at_end);
      auto* state = reinterpret_cast<b200::tile_word_t*>(base + at_state);
      edge_t* work_seg = raw_of(segments.data());
      const unsigned prep_grid = gcuda::persistent_grid(ctx, prep_tiles, 6);
      prof().begin(gcuda::profiler_t::work_prepare, stream());
      cudaMemsetAsync(state, 0, 2 * prep_tiles * sizeof(b200::tile_word_t), stream());
      if constexpr (quad_engine)
        kernels::prepare_quads_kernel<graph_input><<<prep_grid, 256, 0, stream()>>>(
            A.offsets, in, nf, work_src, work_beg, work_end, work_seg, state, state + prep_tiles, C);
      else
        kernels::prepare_work_kernel<graph_input><<<prep_grid, 256, 0, stream()>>>(
            A.offsets, in, nf, work_src, work_beg, work_seg, state, state + prep_tiles, C);
      prof().end(stream());
      prof().begin(gcuda::profiler_t::push_expand, stream());
      if constexpr (quad_engine) {
        auto kernel = kernels::merge_path_quad_kernel<has_output, policy, vertex_t, edge_t, weight_t, operator_t>;
        kernel<<<gcuda::full_grid(ctx, kernel), 256, 0, stream()>>>(A, op, work_src, work_beg, work_end, work_seg, out,
                                                                    C, capacity, visited);
      } else {
        kernels::merge_path_kernel<has_output, policy>
            <<<gcuda::persistent_grid(ctx, ~std::size_t(0), 6), 256, 0, stream()>>>(A, op, work_src, work_beg,
                                                                                    work_seg, out, C, capacity, visited);
      }
      prof().end(stream());
    });
  }

  void bucketing() {
    gcuda::arena_layout_t layout;
    const std::size_t at_small = layout.add(nf * sizeof(vertex_t));
    const std::size_t at_warp = layout.add(nf * sizeof(vertex_t));
    const std::size_t at_big = layout.add(nf * sizeof(vertex_t));
    unsigned char* base = ctx.scratch().temp(layout.bytes);
    auto* small_list = reinterpret_cast<vertex_t*>(base + at_small);
    auto* warp_list = reinterpret_cast<vertex_t*>(base + at_warp);
    auto* big_list = reinterpret_cast<vertex_t*>(base + at_big);
    prof().begin(gcuda::profiler_t::work_prepare, stream());
    kernels::bin_by_degree_kernel<graph_input><<<gcuda::persistent_grid(ctx, item_ctas(), 8), 256, 0, stream()>>>(
        A.offsets, in, nf, small_list, warp_list, big_list, C);
    prof().end(stream());
    prof().begin(gcuda::profiler_t::push_expand, stream());
    kernels::thread_mapped_kernel<false, has_output, true, policy>
        <<<gcuda::persistent_grid(ctx, item_ctas(), 8), 256, 0, stream()>>>(A, op, small_list, 0, C + scratch_t::aux0,
                                                                            out, C, capacity, visited);
    with_engine([&](auto q) {
      if constexpr (decltype(q)::value) {
        auto kernel = kernels::warp_mapped_quad_kernel<has_output, policy, vertex_t, edge_t, weight_t, operator_t>;
        kernel<<<gcuda::full_grid(ctx, kernel, (nf + 7) / 8), 256, 0, stream()>>>(A, op, warp_list, C + scratch_t::aux1,
                                                                                  out, C, capacity, visited);
      } else {
        kernels::warp_mapped_kernel<has_output, policy>
            <<<gcuda::persistent_grid(ctx, (nf + 7) / 8, 8), 256, 0, stream()>>>(A, op, warp_list, C + scratch_t::aux1,
                                                                                out, C, capacity, visited);
      }
      hubs<decltype(q)::value>(big_list);
    });
    prof().end(stream(), 3);
  }
};

/**
 * @brief Push-direction expansion with one of the balancers. `visited` non-null selects the
 * test-and-set policy (direction-optimised callers); null keeps reference semantics.
 * `epilogue(counters, output)` enqueues extra kernels that consume the device-side output count before the one sync.
 */
template <load_balance_t lb, bool use_csc, advance_io_type_t input_type, advance_io_type_t output_type, visit_t policy,
          typename graph_t, typename operator_t, typename frontier_t, typename work_tiles_t,
          typename epilogue_t = no_epilogue_t>
void expand(graph_t& G, operator_t op, frontier_t* input, frontier_t* output, work_tiles_t& segments,
            gcuda::standard_context_t& ctx, unsigned* visited, epilogue_t epilogue = epilogue_t()) {
  using vertex_t = typename graph_t::vertex_type;
  using edge_t = typename graph_t::edge_type;
  using weight_t = typename graph_t::weight_type;
  constexpr bool graph_input = input_type == advance_io_type_t::graph;
  constexpr bool has_output = output_type != advance_io_type_t::none;
  static_assert(input_type == advance_io_type_t::graph || input_type == advance_io_type_t::vertices,
                "advance input must be `graph` or `vertices`");
  static_assert(output_type == advance_io_type_t::none || output_type == advance_io_type_t::vertices,
                "advance output must be `vertices` or `none`");
  using launch_t = push_launch_t<graph_input, has_output, policy, vertex_t, edge_t, weight_t, operator_t>;

  const auto A = graph::adjacency_of<use_csc>(G);
  const std::size_t nf = graph_input ? std::size_t(A.n) : input->get_number_of_elements();
  if (nf == 0) {
    if constexpr (has_output) output->set_number_of_elements(0);
    return;
  }
  auto& scratch = ctx.scratch();
  auto stream = ctx.stream();
  const bool quad = launch_t::quad_types && kernels::advance_engine() != 0 &&
                    (reinterpret_cast<std::uintptr_t>(A.indices) & 15u) == 0 &&
                    (reinterpret_cast<std::uintptr_t>(A.values) & 15u) == 0;

  // max_degree() may run a kernel and fetch() the counters on its first call per graph: resolve it BEFORE the
  // counters of this call are zeroed, so `clean` never claims a block that kernels of this call have written
  long long maxdeg = 0;
  if constexpr (lb == load_balance_t::thread_mapped || lb == load_balance_t::block_mapped ||
                lb == load_balance_t::merge_path || lb == load_balance_t::merge_path_v2)
    maxdeg = max_degree(ctx, G.get_build_serial(), A.offsets, A.n);
  // merge_path over `input = graph` (PageRank push, SpMV): the frontier is every vertex in id order, so the
  // scan + compaction pass of merge-path (16-24 bytes written and re-read per vertex) buys nothing over
  // block-mapped tiles of 256 consecutive rows with dynamic tickets and hub deferral; same operator calls
  constexpr bool as_block_mapped =
      lb == load_balance_t::block_mapped ||
      ((lb == load_balance_t::merge_path || lb == load_balance_t::merge_path_v2) && graph_input && launch_t::quad_types);
  for (int attempt = 0; attempt < 3; ++attempt) {
    scratch.zero(stream);
    launch_t launch{ctx, A, op, graph_input ? nullptr : input->data(), nf, has_output ? output->data() : nullptr,
                    scratch.d, has_output ? counter_t(output->get_capacity()) : counter_t(0), visited, quad, maxdeg};
    if constexpr (lb == load_balance_t::thread_mapped)
      launch.thread_mapped();
    else if constexpr (as_block_mapped)
      launch.block_mapped();
    else if constexpr (lb == load_balance_t::merge_path || lb == load_balance_t::merge_path_v2)
      launch.merge_path(segments);
    else if constexpr (lb == load_balance_t::bucketing)
      launch.bucketing();
    else
      error::throw_if_exception(cudaErrorUnknown, "Advance type not supported.");
    epilogue(launch.C, launch.out);
    error::check_last("advance launch");
    if constexpr (!has_output)
      if (scratch.async_when_no_output) {  // nothing to report; the next zero() must really clear the counters
        scratch.clean = false;
        return;
      }
    scratch.fetch(stream);
    if constexpr (has_output) {
      if (scratch.h[scratch_t::overflow]) {  // nothing was expanded: grow and go again
        grow_output(output, std::size_t(scratch.h[scratch_t::overflow]));
        continue;
      }
      // every kernel drops stores past `capacity` but keeps counting: a count above it with no overflow flagged means
      // the guard was skipped on a wrong max degree. The operator has run already, so a relaunch would call it twice
      error::throw_if_exception(scratch.h[scratch_t::out_count] > launch.capacity,
                                "advance: output count exceeds the output capacity but no overflow was flagged");
      output->set_number_of_elements(std::size_t(scratch.h[scratch_t::out_count]));
    }
    return;
  }
  error::throw_if_exception(cudaErrorMemoryAllocation, "advance: output frontier could not be sized");
}

/**
 * @brief Direction-optimised advance (Beamer-style push/pull switching) on the enactor's dense state.
 */
template <load_balance_t lb, advance_io_type_t input_type, advance_io_type_t output_type, typename graph_t,
          typename enactor_type, typename operator_t>
void optimized(graph_t& G, enactor_type* E, operator_t op, gcuda::standard_context_t& ctx) {
  using vertex_t = typename graph_t::vertex_type;
  using edge_t = typename graph_t::edge_type;
  static_assert(input_type == advance_io_type_t::vertices && output_type == advance_io_type_t::vertices,
                "direction-optimised advance maps a vertex frontier to a vertex frontier");
  auto& D = E->direction;
  auto& scratch = ctx.scratch();
  auto& prof = ctx.profiler();
  using gcuda::profiler_t;
  auto stream = ctx.stream();
  const auto out_adj = graph::adjacency_of<false>(G);
  auto in_adj = graph::adjacency_of<true>(G);
  if (!kernels::pull_hints_enabled()) in_adj.head = nullptr;
  const vertex_t n = out_adj.n;
  auto* input = E->get_input_frontier();
  auto* output = E->get_output_frontier();

  if (!D.initialised) {
    D.allocate(std::size_t(n), stream);
    const std::size_t nf = input->get_number_of_elements();
    scratch.zero(stream);
    prof.begin(profiler_t::dense_state, stream);
    if (in_adj.isolated)  // cached with the graph's pull hints: 2 MiB copy instead of an n-length pass
      cudaMemcpyAsync(D.visited.data(), in_adj.isolated, ((std::size_t(n) + 31) / 32) * sizeof(unsigned),
                      cudaMemcpyDeviceToDevice, stream);
    else
      kernels::init_visited_kernel<<<gcuda::persistent_grid(ctx, (std::size_t(n) + 255) / 256, 8), 256, 0, stream>>>(
          in_adj.offsets, n, D.visited.data());
    if (nf)
      kernels::mark_frontier_kernel<<<gcuda::persistent_grid(ctx, (nf + 255) / 256, 8), 256, 0, stream>>>(
          out_adj.offsets, input->data(), nf, nullptr, D.visited.data(), scratch.d);
    prof.end(stream);
    scratch.fetch(stream);
    D.frontier_edges = (long long)scratch.h[scratch_t::aux2];
    D.unexplored_edges = (long long)out_adj.m - D.frontier_edges;
    D.frontier_vertices = (long long)nf;
    D.previous_frontier_vertices = 0;
    D.frontier_is_dense = false;
    D.pulling = false;
    D.initialised = true;
  }

  // --- choose the direction for this level (Beamer, Asanovic, Patterson) ---
  const float alpha = E->properties.direction_alpha, beta = E->properties.direction_beta;
  if (!D.pulling) {
    if (double(D.frontier_edges) > double(D.unexplored_edges) / double(alpha) &&
        D.frontier_vertices > D.previous_frontier_vertices)
      D.pulling = true;
  } else {
    if (double(D.frontier_vertices) < double(n) / double(beta) && D.frontier_vertices < D.previous_frontier_vertices)
      D.pulling = false;
  }

  long long next_vertices = 0, next_edges = 0;
  if (D.pulling) {
    if (!D.frontier_is_dense) {  // sparse -> dense
      prof.begin(profiler_t::dense_state, stream);
      frontier::convert(*input, D.dense[D.dense_selector], stream);
      prof.end(stream);
      D.frontier_is_dense = true;
    }
    auto& cur = D.dense[D.dense_selector];
    auto& nxt = D.dense[D.dense_selector ^ 1];
    scratch.zero(stream);
    prof.begin(profiler_t::pull_step, stream);
    const std::size_t chunks = ((std::size_t(n) + 31) / 32 + kernels::pull_chunk_words - 1) / kernels::pull_chunk_words;
    auto kernel = kernels::pull_chunk_kernel<vertex_t, edge_t, typename graph_t::weight_type, operator_t>;
    kernel<<<gcuda::full_grid(ctx, kernel, (chunks + 7) / 8), 256, 0, stream>>>(in_adj, op, cur.data(), nxt.data(),
                                                                                D.visited.data(), scratch.d);
    prof.end(stream);
    error::check_last("pull step");
    scratch.fetch(stream);
    next_vertices = (long long)scratch.h[scratch_t::out_count];
    // the pull kernel does not read row bounds of the vertices it adopts, so Σdeg of the next frontier is
    // unknown while pulling; it is recomputed from the sparse list on the way back to top-down (below)
    next_edges = 0;
    D.pull_vertices_scanned += (long long)scratch.h[scratch_t::aux0];
    D.pull_edges_inspected += (long long)scratch.h[scratch_t::aux1];
    D.pull_hint_misses += (long long)scratch.h[scratch_t::aux2];
    D.pull_vertices_found += next_vertices;
    D.dense_selector ^= 1;
    D.dense[D.dense_selector].set_number_of_elements(std::size_t(next_vertices));
    output->set_number_of_elements(std::size_t(next_vertices));  // contents live in the dense map
    ++D.pull_steps;
  } else {
    if (D.frontier_is_dense) {  // dense -> sparse, and Σdeg of the list (Beamer's m_f) in the same round trip
      prof.begin(profiler_t::dense_state, stream);
      auto& dense = D.dense[D.dense_selector];
      const std::size_t upper = std::size_t(D.frontier_vertices);
      if (input->get_capacity() < upper) input->reserve(upper);
      scratch.zero(stream);
      if (upper) {
        frontier::kernels::gather_bits_kernel<<<gcuda::persistent_grid(ctx, (dense.words() + 255) / 256, 4), 256, 0,
                                                stream>>>(dense.data(), dense.words(), input->data(),
                                                          scratch.d + scratch_t::out_count);
        kernels::mark_frontier_kernel<<<gcuda::persistent_grid(ctx, (upper + 255) / 256, 8), 256, 0, stream>>>(
            out_adj.offsets, input->data(), upper, scratch.d + scratch_t::out_count, nullptr, scratch.d);
      }
      prof.end(stream, 2);
      scratch.fetch(stream);
      input->set_number_of_elements(std::size_t(scratch.h[scratch_t::out_count]));
      D.frontier_edges = (long long)scratch.h[scratch_t::aux2];
      D.frontier_is_dense = false;
    }
    D.push_vertices_expanded += D.frontier_vertices;
    D.push_edges_expanded += D.frontier_edges;
    grow_output(output, std::size_t(n));
    // Σdeg of the new frontier (Beamer's m_f): one parallel pass over the output list, enqueued behind the
    // expansion kernels and in front of the level's single host round trip (it reads the list length from the
    // device counter the expansion just produced). It is not summed inside the expansion kernels: that put two
    // dependent row-bound loads at the end of every discovery's probe -> test-and-set -> operator chain.
    const auto* degree_offsets = out_adj.offsets;
    auto degree_sum = [&](counter_t* C, vertex_t* out) {
      kernels::mark_frontier_kernel<<<gcuda::persistent_grid(ctx, ~std::size_t(0), 4), 256, 0, stream>>>(
          degree_offsets, out, 0, C + scratch_t::out_count, nullptr, C);
      prof.launches_total += 1;
    };
    expand<lb, false, input_type, output_type, visit_t::test_and_set>(G, op, input, output, E->scanned_work_domain, ctx,
                                                                     D.visited.data(), degree_sum);
    next_vertices = (long long)output->get_number_of_elements();
    next_edges = next_vertices ? (long long)scratch.h[scratch_t::aux2] : 0;
    D.push_vertices_found += next_vertices;
    ++D.push_steps;
  }
  D.previous_frontier_vertices = D.frontier_vertices;
  D.frontier_vertices = next_vertices;
  D.frontier_edges = next_edges;
  D.unexplored_edges -= next_edges;
}

}  // namespace detail

/// Pairs a push operator with its bottom-up form for direction-optimised advance (see pull.cuh).
template <typename push_t, typename pull_t>
kernels::directional_operator_t<push_t, pull_t> directional(push_t push, pull_t pull) {
  return kernels::directional_operator_t<push_t, pull_t>{push, pull};
}

/// Splits an operator into issue / resolve halves so batched kernels can overlap the atomics of several edges
/// (see kernels::two_phase_operator_t).
template <typename issue_t, typename resolve_t>
kernels::two_phase_operator_t<issue_t, resolve_t> two_phase(issue_t issue, resolve_t resolve) {
  return kernels::two_phase_operator_t<issue_t, resolve_t>{issue, resolve};
}

template <typename prepare_t, typename issue_t, typename resolve_t>
kernels::staged_operator_t<prepare_t, issue_t, resolve_t> two_phase(prepare_t prepare, issue_t issue, resolve_t resolve) {
  return kernels::staged_operator_t<prepare_t, issue_t, resolve_t>{prepare, issue, resolve};
}

/**
 * @brief Explicit-buffers form (reference advance.hxx:91-129; used by e.g. bc.hxx:140-146).
 */
template <load_balance_t lb, advance_direction_t direction, advance_io_type_t input_type,
          advance_io_type_t output_type, typename graph_t, typename operator_t, typename frontier_t,
          typename work_tiles_t>
void execute(graph_t& G, operator_t op, frontier_t* input, frontier_t* output, work_tiles_t& segments,
             gcuda::multi_context_t& context) {
  error::throw_if_exception(context.size() != 1, "`context.size() != 1` not supported");
  auto* ctx = context.get_context(0);
  if constexpr (direction == advance_direction_t::optimized) {
    error::throw_if_exception(cudaErrorUnknown,
                              "direction-optimized advance needs the enactor form (it keeps dense state in E)");
  } else if constexpr (lb == load_balance_t::warp_mapped || lb == load_balance_t::work_stealing) {
    error::throw_if_exception(cudaErrorUnknown, "Advance type not supported.");
  } else {
    detail::expand<lb, direction == advance_direction_t::backward, input_type, output_type,
                   detail::visit_t::none>(G, op, input, output, segments, *ctx, nullptr);
  }
}

/**
 * @brief Enactor form (reference advance.hxx:192-221): reads E's input frontier, writes E's output
 * frontier, swaps the buffers unless output_type == none or swap_buffers is false.
 */
template <load_balance_t lb = load_balance_t::merge_path,
          advance_direction_t direction = advance_direction_t::forward,
          advance_io_type_t input_type = advance_io_type_t::vertices,
          advance_io_type_t output_type = advance_io_type_t::vertices, typename graph_t, typename enactor_type,
          typename operator_type>
void execute(graph_t& G, enactor_type* E, operator_type op, gcuda::multi_context_t& context, bool swap_buffers = true) {
  if constexpr (direction == advance_direction_t::optimized) {
    error::throw_if_exception(context.size() != 1, "`context.size() != 1` not supported");
    using csr_v = typename graph_t::graph_csr_view_t;
    using csc_v = typename graph_t::graph_csc_view_t;
    static_assert(graph_t::template contains_representation<csr_v>() &&
                      graph_t::template contains_representation<csc_v>(),
                  "CSR and CSC representations are required for direction-optimized advance");
    detail::optimized<lb, input_type, output_type>(G, E, op, *context.get_context(0));
  } else {
    execute<lb, direction, input_type, output_type>(G, op, E->get_input_frontier(), E->get_output_frontier(),
                                                    E->scanned_work_domain, context);
  }
  if (swap_buffers && (output_type != advance_io_type_t::none)) E->swap_frontier_buffers();
}

/**
 * @brief Fused advance + uniquify (the step the reference leaves commented out after its advances, sssp.hxx:146-150,
 * bfs.hxx:128-131). Same call as the enactor form of execute<lb, direction, input, vertices>: `op` runs on every
 * edge exactly once, but each kept neighbour is written to the output frontier ONCE however many edges kept it —
 * the expansion kernels test-and-set a per-enactor bitmap (n/8 bytes, L2 resident) at emission, and an
 * O(|output|) epilogue clears the words again. Replaces advance -> uniquify (or the bypass filter SSSP uses to
 * drop repeats) without the intermediate Σdeg-long frontier.
 */
template <load_balance_t lb, advance_direction_t direction, advance_io_type_t input_type, typename graph_t,
          typename operator_t, typename frontier_t, typename work_tiles_t, typename bitmap_t>
void execute_unique(graph_t& G, operator_t op, frontier_t* input, frontier_t* output, work_tiles_t& segments,
                    bitmap_t& seen, gcuda::multi_context_t& context) {
  static_assert(direction != advance_direction_t::optimized, "execute_unique: forward or backward");
  static_assert(lb != load_balance_t::warp_mapped && lb != load_balance_t::work_stealing,
                "execute_unique: thread_mapped, block_mapped, merge_path or bucketing");
  error::throw_if_exception(context.size() != 1, "`context.size() != 1` not supported");
  auto* ctx = context.get_context(0);
  auto stream = ctx->stream();
  const std::size_t n = std::size_t(G.get_number_of_vertices());
  if (seen.get_universe() != n) {  // (re)sized maps start all clear
    seen.resize(n, stream);
    seen.fill(0, stream);
  }
  detail::expand<lb, direction == advance_direction_t::backward, input_type, advance_io_type_t::vertices,
                 detail::visit_t::unique_output>(G, op, input, output, segments, *ctx, seen.data());
  const std::size_t count = output->get_number_of_elements();
  if (count) {
    ctx->profiler().begin(gcuda::profiler_t::dense_state, stream);
    kernels::clear_emitted_kernel<<<gcuda::persistent_grid(*ctx, (count + 255) / 256, 8), 256, 0, stream>>>(
        output->data(), count, seen.data());
    ctx->profiler().end(stream);
    ctx->synchronize();  // completion contract: the map is clear and the frontier final on return
  }
}

/// Enactor form: E's input frontier -> E's output frontier, E->unique_seen as the bitmap, buffers swapped.
template <load_balance_t lb = load_balance_t::merge_path,
          advance_direction_t direction = advance_direction_t::forward,
          advance_io_type_t input_type = advance_io_type_t::vertices, typename graph_t, typename enactor_type,
          typename operator_type>
void execute_unique(graph_t& G, enactor_type* E, operator_type op, gcuda::multi_context_t& context,
                    bool swap_buffers = true) {
  execute_unique<lb, direction, input_type>(G, op, E->get_input_frontier(), E->get_output_frontier(),
                                            E->scanned_work_domain, E->unique_seen, context);
  if (swap_buffers) E->swap_frontier_buffers();
}

}  // namespace advance
}  // namespace operators
}  // namespace gunrock
