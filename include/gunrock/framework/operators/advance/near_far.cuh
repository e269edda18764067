/**
 * @file near_far.cuh
 * @brief operators::advance::execute_near_far — a whole priority-ordered traversal in ONE persistent kernel.
 *
 * Why it exists. On a high-diameter, low-degree graph (BASELINE config 3: 4900 x 4900 grid, ~10 K levels) the
 * bulk-synchronous recipe of the reference — one advance + one filter per level, each with host round trips
 * (include/gunrock/algorithms/sssp.hxx:98-151) — is bound by launch/sync latency, and plain label-correcting
 * re-relaxes every vertex many times. Both are addressed here:
 *   - work efficiency: the Davidson/Baxter/Garland/Owens "near-far pile" ordering, which the reference's
 *     `load_balance_t::bucketing  // Davidson et al. (SSSP)` enumerator names but never implements
 *     (advance/bucketing.hxx:31-36): vertices whose priority is below a moving threshold are expanded now,
 *     the others wait in the far pile until the threshold reaches them;
 *   - latency: the level loop runs inside a cooperative kernel (all CTAs co-resident); a level costs one grid
 *     barrier instead of two operator calls with host round trips.
 *
 * Contract. `op(src, nbr, e, w)` is an ordinary advance operator (SSSP: relax with atomic::min, true when the
 * neighbour improved) that does not depend on the iteration number. `priority(v)` returns the current key of a
 * vertex as a non-negative float (SSSP: its tentative distance); keys only decrease. A neighbour for which op
 * returned true is queued at most once per level (stamp array) and joins `near` if priority < threshold, else
 * the far pile (at most once, flag array). When `near` empties the threshold jumps to the first multiple of
 * delta above the smallest far priority; far entries below the OLD threshold are stale (they were expanded
 * from `near` when they dropped below it) and are discarded, entries below the new one move to `near`.
 * Ends when both are empty. For an operator with a unique fixed point (SSSP) the result is identical to
 * running the reference's advance/filter loop to convergence — SSSP distances are bit-equal.
 * The grid barrier (cooperative_groups grid sync) carries a device-scope fence, so values written by atomics
 * in one level are visible to plain loads in the next.
 */
#pragma once

#include <climits>
#include <cooperative_groups.h>

#include <gunrock/b200/warp.cuh>
#include <gunrock/framework/operators/advance/directional.cuh>
#include <gunrock/cuda/context.hxx>
#include <gunrock/graph/graph.hxx>

namespace gunrock {
namespace operators {
namespace advance {
namespace kernels {

/// Device-side control block of one near-far run.
struct near_far_state_t {
  unsigned long long near_count[3];  ///< rotating: level k reads [k%3], appends to [(k+1)%3], clears [(k+2)%3]
  unsigned long long far_count[2];   ///< double-buffered far pile lengths
  unsigned long long relaxations;    ///< operator calls (work accounting)
  unsigned far_min_bits;             ///< min priority in the far pile (bit pattern of a non-negative float)
  float threshold;
  int far_selector;
  int levels;    ///< near levels executed
  int splits;    ///< far-pile splits executed
  int overflow;  ///< a queue ran out of capacity (impossible with capacity n thanks to the stamps; checked anyway)
};

constexpr unsigned near_far_inf_bits = 0x7f800000u;

/**
 * @brief One near level of near_far_kernel: every lane takes one vertex of the level's queue; its edges are relaxed
 * 4 per batch so that the column/weight loads, the operators (atomics) and the routing
 * (priority loads, stamp / flag exchanges) of a batch are in flight together — the edge-at-a-time loop this
 * replaces paid one full dependent chain of L2 round trips PER EDGE, most of a level's 13-15 us on the grid. A
 * neighbour the operator improved joins the next near queue (priority < threshold, once per level: stamp) or the
 * far pile (once: flag); the warp claims its slots with ONE atomic per queue and batch. Called by all threads of the
 * kernel.
 */
template <typename vertex_t, typename edge_t, typename weight_t, typename operator_t, typename priority_t>
__device__ __forceinline__ void near_far_expand_level(
    const graph::adjacency_t<vertex_t, edge_t, weight_t>& A, operator_t& op, priority_t& priority,
    const vertex_t* __restrict__ q_in, unsigned long long n_in, vertex_t* __restrict__ q_out,
    unsigned long long* out_count, vertex_t* __restrict__ far_out, unsigned long long* far_count, float threshold,
    int next_level, int* queue_stamp, int* far_flag, unsigned long long capacity, unsigned long long tid,
    unsigned long long threads, unsigned long long& my_relax, bool& overflowed) {
  const unsigned lane = b200::lane_id();
  // Routes up to 4 improved neighbours per lane: priorities, stamps and flags of the batch are in flight
  // together, and the whole warp claims its queue slots with ONE atomic per queue.
  auto route4 = [&](const bool (&improved)[4], const vertex_t (&u)[4]) {  // called by all 32 lanes
    float pri[4];
    int previous[4];
    bool to_near[4], to_far[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) pri[j] = improved[j] ? float(priority(u[j])) : 0.f;
    // all exchanges of the batch are issued before the first result is looked at (in-order issue: a compare in
    // between would make the warp wait for each round trip in turn)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      previous[j] = 0;
      if (improved[j])
        previous[j] = pri[j] < threshold ? atomicExch(queue_stamp + u[j], next_level) : atomicExch(far_flag + u[j], 1);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      to_near[j] = improved[j] && pri[j] < threshold && previous[j] != next_level;
      to_far[j] = improved[j] && !(pri[j] < threshold) && previous[j] == 0;
    }
    unsigned near_votes[4], far_votes[4], n_near = 0, n_far_new = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      near_votes[j] = __ballot_sync(b200::full_mask, to_near[j]);
      far_votes[j] = __ballot_sync(b200::full_mask, to_far[j]);
      n_near += __popc(near_votes[j]);
      n_far_new += __popc(far_votes[j]);
    }
    if ((n_near | n_far_new) == 0) return;  // warp-uniform
    unsigned long long base_near = 0, base_far = 0;
    if (lane == 0) {
      if (n_near) base_near = atomicAdd(out_count, (unsigned long long)n_near);
      if (n_far_new) base_far = atomicAdd(far_count, (unsigned long long)n_far_new);
    }
    base_near = __shfl_sync(b200::full_mask, base_near, 0);
    base_far = __shfl_sync(b200::full_mask, base_far, 0);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (to_near[j]) {
        const unsigned long long at = base_near + __popc(near_votes[j] & b200::lanes_below(lane));
        if (at < capacity) q_out[at] = u[j]; else overflowed = true;
      }
      if (to_far[j]) {
        const unsigned long long at = base_far + __popc(far_votes[j] & b200::lanes_below(lane));
        if (at < capacity) far_out[at] = u[j]; else overflowed = true;
      }
      base_near += __popc(near_votes[j]);
      base_far += __popc(far_votes[j]);
    }
  };

  // Runs the operator on the (up to) 4 live edges of a lane. A two-phase operator has all its issues (atomics) in
  // flight before the first resolve; a plain operator is simply called edge by edge.
  auto apply4 = [&](vertex_t source, const bool (&live)[4], vertex_t (&u)[4], edge_t (&edge)[4], weight_t (&w)[4],
                    bool (&improved)[4]) {
    if constexpr (has_two_phase<operator_t>::value && has_prepare<operator_t>::value) {
      vertex_t s = source;
      const auto state = op.prepare(s);  // once per source (and batch): e.g. its tentative distance
      using token_t = decltype(op.issue(state, s, u[0], edge[0], w[0]));
      token_t token[4];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (live[j]) token[j] = op.issue(state, s, u[j], edge[j], w[j]);
#pragma unroll
      for (int j = 0; j < 4; ++j) improved[j] = live[j] && op.resolve(token[j]);
    } else if constexpr (has_two_phase<operator_t>::value) {
      vertex_t s = source;
      using token_t = decltype(op.issue(s, u[0], edge[0], w[0]));
      token_t token[4];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (live[j]) token[j] = op.issue(s, u[j], edge[j], w[j]);
#pragma unroll
      for (int j = 0; j < 4; ++j) improved[j] = live[j] && op.resolve(token[j]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        vertex_t s = source;
        improved[j] = live[j] && op(s, u[j], edge[j], w[j]);
      }
    }
  };

  for (unsigned long long base = (tid >> 5) << 5; base < n_in; base += threads) {
    const unsigned long long i = base + lane;
    vertex_t v = 0;
    edge_t beg = 0, deg = 0;
    if (i < n_in) {
      v = q_in[i];
      beg = A.offsets[v];
      deg = A.offsets[v + 1] - beg;
    }
    unsigned long_lanes = __ballot_sync(b200::full_mask, deg >= 32);
    while (long_lanes) {  // adjacency lists of >= 32 edges: the whole warp, coalesced, 4 strides per batch
      const int owner = __ffs(long_lanes) - 1;
      long_lanes &= long_lanes - 1;
      const vertex_t src = __shfl_sync(b200::full_mask, v, owner);
      const edge_t b = __shfl_sync(b200::full_mask, beg, owner);
      const edge_t e_end = b + __shfl_sync(b200::full_mask, deg, owner);
      for (edge_t e0 = b; e0 < e_end; e0 += 128) {
        bool improved[4];
        vertex_t u[4];
        edge_t edge[4];
        weight_t w[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          edge[j] = e0 + edge_t(32 * j) + edge_t(lane);
          u[j] = 0, w[j] = weight_t(1);
          if (edge[j] < e_end) {
            u[j] = __ldg(A.indices + edge[j]);
            if (A.values) w[j] = __ldg(A.values + edge[j]);
          }
        }
        bool live[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          live[j] = edge[j] < e_end;
          my_relax += live[j];
        }
        apply4(src, live, u, edge, w, improved);
        route4(improved, u);
      }
    }
    // short lists: every lane walks its own, 4 edges per batch (loads, operators and routing of a batch overlap:
    // the serial edge-at-a-time loop cost one full dependent chain of L2 round trips PER EDGE, which at degree 4
    // was most of a level's 13-15 us on the grid)
    const edge_t short_deg = deg < 32 ? deg : edge_t(0);
    const edge_t trips = b200::warp_max(short_deg);  // warp-uniform trip count keeps the ballots converged
    for (edge_t k0 = 0; k0 < trips; k0 += 4) {
      bool improved[4];
      vertex_t u[4];
      edge_t edge[4];
      weight_t w[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        edge[j] = beg + k0 + edge_t(j);
        u[j] = 0, w[j] = weight_t(1);
        if (k0 + edge_t(j) < short_deg) {
          u[j] = __ldg(A.indices + edge[j]);
          if (A.values) w[j] = __ldg(A.values + edge[j]);
        }
      }
      bool live[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        live[j] = k0 + edge_t(j) < short_deg;
        my_relax += live[j];
      }
      apply4(v, live, u, edge, w, improved);
      route4(improved, u);
    }
  }
}

/**
 * @brief The whole traversal (see file comment): one cooperative launch of 256-thread CTAs, one grid barrier per
 * level. Queue lengths, threshold and selectors live in `state` (global memory, L2). A thread-block-cluster form, whose
 * barrier is cheaper, was measured slower on the 4900 x 4900 grid (DESIGN.md §3.3).
 */
template <typename vertex_t, typename edge_t, typename weight_t, typename operator_t, typename priority_t>
__global__ void __launch_bounds__(256, 2)
    near_far_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op, priority_t priority,
                    float delta, vertex_t* near0, vertex_t* near1, vertex_t* far0, vertex_t* far1, int* queue_stamp,
                    int* far_flag, near_far_state_t* state, unsigned long long capacity, int max_levels) {
  cooperative_groups::grid_group grid = cooperative_groups::this_grid();
  volatile near_far_state_t* st = state;
  const unsigned lane = b200::lane_id();
  const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long threads = (unsigned long long)gridDim.x * blockDim.x;
  vertex_t* near_q[2] = {near0, near1};
  vertex_t* far_q[2] = {far0, far1};
  unsigned long long my_relax = 0;
  int level = 0;
  bool stop = false;
  bool overflowed = false;

  // warp-aggregated append (one atomic per warp and call)
  auto append = [&](bool keep, vertex_t value, vertex_t* queue, unsigned long long* count) {
    const unsigned votes = __ballot_sync(b200::full_mask, keep);
    if (votes == 0) return;
    const int first = __ffs(votes) - 1;
    unsigned long long base = 0;
    if (int(lane) == first) base = atomicAdd(count, (unsigned long long)__popc(votes));
    base = __shfl_sync(b200::full_mask, base, first);
    if (keep) {
      const unsigned long long at = base + __popc(votes & b200::lanes_below(lane));
      if (at < capacity) queue[at] = value; else overflowed = true;
    }
  };

  while (!stop) {
    // ---------------------------- near levels: one barrier each ----------------------------
    for (;;) {
      const unsigned long long n_in = st->near_count[level % 3];
      if (n_in == 0) break;
      if (level >= max_levels) {
        stop = true;
        break;
      }
      const vertex_t* q_in = near_q[level & 1];
      vertex_t* q_out = near_q[(level + 1) & 1];
      unsigned long long* out_count = &state->near_count[(level + 1) % 3];
      const float threshold = st->threshold;
      const int fsel = st->far_selector;
      vertex_t* far_out = far_q[fsel];
      unsigned long long* far_count = &state->far_count[fsel];
      const int next_level = level + 1;
      if (tid == 0) st->near_count[(level + 2) % 3] = 0;  // consumed a level ago; the next level appends to it
      near_far_expand_level(A, op, priority, q_in, n_in, q_out, out_count, far_out, far_count, threshold, next_level,
                            queue_stamp, far_flag, capacity, tid, threads, my_relax, overflowed);
      grid.sync();
      ++level;
    }
    if (stop) break;

    // ---------------------------- far pile: raise the threshold, split ----------------------------
    const int fsel = st->far_selector;
    const unsigned long long n_far = st->far_count[fsel];
    if (n_far == 0) break;
    const vertex_t* far_in = far_q[fsel];
    vertex_t* far_keep = far_q[fsel ^ 1];
    {
      unsigned lowest = near_far_inf_bits;
      for (unsigned long long i = tid; i < n_far; i += threads) {
        const unsigned bits = __float_as_uint(float(priority(far_in[i])));
        lowest = bits < lowest ? bits : lowest;
      }
      for (int d = 16; d > 0; d >>= 1) {
        const unsigned other = __shfl_xor_sync(b200::full_mask, lowest, d);
        lowest = other < lowest ? other : lowest;
      }
      if (lane == 0 && lowest != near_far_inf_bits) atomicMin(&state->far_min_bits, lowest);
    }
    grid.sync();
    const float old_threshold = st->threshold;
    const float far_min = __uint_as_float(st->far_min_bits);
    float new_threshold = (floorf(far_min / delta) + 1.0f) * delta;
    if (!(new_threshold > old_threshold)) new_threshold = old_threshold + delta;
    // strict progress past the smallest pending key: both forms above can round to <= far_min once keys exceed
    // ~2^24 * delta, and a far pile that never drains would spin this persistent kernel for ever
    if (!(new_threshold > far_min)) new_threshold = nextafterf(far_min, __int_as_float(0x7f800000));
    {
      vertex_t* q_in = near_q[level & 1];  // promoted vertices become the input of the next near level
      unsigned long long* in_count = &state->near_count[level % 3];
      unsigned long long* keep_count = &state->far_count[fsel ^ 1];
      for (unsigned long long base = (tid >> 5) << 5; base < n_far; base += threads) {
        const unsigned long long i = base + lane;
        bool promote = false, keep = false;
        vertex_t u = 0;
        if (i < n_far) {
          u = far_in[i];
          const float p = float(priority(u));
          if (p < old_threshold) {
            far_flag[u] = 0;  // stale: it was expanded from `near` when it dropped below the old threshold
          } else if (p < new_threshold) {
            far_flag[u] = 0;
            promote = atomicExch(queue_stamp + u, level) != level;
          } else {
            keep = true;
          }
        }
        append(promote, u, q_in, in_count);
        append(keep, u, far_keep, keep_count);
      }
    }
    grid.sync();
    if (tid == 0) {
      st->threshold = new_threshold;
      st->far_count[fsel] = 0;
      st->far_selector = fsel ^ 1;
      st->far_min_bits = near_far_inf_bits;
      st->splits = st->splits + 1;
    }
    grid.sync();
  }

  my_relax = b200::warp_sum(my_relax);
  if (lane == 0 && my_relax) atomicAdd(&state->relaxations, my_relax);
  if (overflowed) state->overflow = 1;
  if (tid == 0) st->levels = level;
}

}  // namespace kernels

/// Statistics of one execute_near_far call.
struct near_far_result_t {
  int levels = 0;
  int splits = 0;
  unsigned long long relaxations = 0;
  float final_threshold = 0.f;
};

/**
 * @brief Runs the near-far traversal to completion (see file comment). The enactor's input frontier holds the
 * start vertices (unique, valid); on return both frontier buffers are empty.
 * `delta` > 0 is the bucket width in priority units. Needs a device that supports cooperative launches.
 */
template <typename graph_t, typename enactor_type, typename operator_t, typename priority_t>
near_far_result_t execute_near_far(graph_t& G, enactor_type* E, operator_t op, priority_t priority, float delta,
                                   gcuda::multi_context_t& context, int max_levels = INT_MAX) {
  using vertex_t = typename graph_t::vertex_type;
  using edge_t = typename graph_t::edge_type;
  using weight_t = typename graph_t::weight_type;
  using kernels::near_far_state_t;
  error::throw_if_exception(context.size() != 1, "`context.size() != 1` not supported");
  error::throw_if_exception(!(delta > 0.f), "execute_near_far: delta must be positive");
  auto* ctx = context.get_context(0);
  auto stream = ctx->stream();
  const auto A = graph::adjacency_of<false>(G);
  const std::size_t n = std::size_t(A.n);
  auto* in = E->get_input_frontier();
  auto* out = E->get_output_frontier();
  const std::size_t nf = in->get_number_of_elements();
  near_far_result_t result;
  if (nf == 0 || n == 0) return result;
  if (in->get_capacity() < n) in->reserve(n);
  if (out->get_capacity() < n) out->reserve(n);

  memory::device_array_t<vertex_t> far0(n), far1(n);
  memory::device_array_t<int> stamp(n), far_flag(n);
  memory::device_array_t<near_far_state_t> state(1);
  cudaMemsetAsync(stamp.data(), 0xff, n * sizeof(int), stream);
  cudaMemsetAsync(far_flag.data(), 0, n * sizeof(int), stream);
  near_far_state_t h{};
  h.near_count[0] = nf;
  h.threshold = delta;
  h.far_min_bits = kernels::near_far_inf_bits;
  cudaMemcpyAsync(state.data(), &h, sizeof(h), cudaMemcpyHostToDevice, stream);

  auto kernel = kernels::near_far_kernel<vertex_t, edge_t, weight_t, operator_t, priority_t>;
  int per_sm = 0;
  error::throw_if_exception(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0), "occupancy");
  error::throw_if_exception(per_sm < 1, "execute_near_far: kernel does not fit on an SM");
  // one CTA per SM: the fewer CTAs, the cheaper the grid barrier (4900^2 grid: 178 ms at 1 CTA/SM, 192 ms at 2,
  // 232 ms at 4)
  const unsigned grid = unsigned(ctx->sm_count());
  auto adjacency = A;
  vertex_t *near0 = in->data(), *near1 = out->data(), *f0 = far0.data(), *f1 = far1.data();
  int *stamp_ptr = stamp.data(), *flag_ptr = far_flag.data();
  near_far_state_t* state_ptr = state.data();
  unsigned long long capacity = n;
  void* args[] = {&adjacency, &op, &priority, &delta, &near0, &near1, &f0, &f1, &stamp_ptr, &flag_ptr, &state_ptr,
                  &capacity, &max_levels};
  ctx->profiler().begin(gcuda::profiler_t::push_expand, stream);
  error::throw_if_exception(cudaLaunchCooperativeKernel((void*)kernel, dim3(grid), dim3(256), args, 0, stream),
                            "execute_near_far launch");
  cudaMemcpyAsync(&h, state.data(), sizeof(h), cudaMemcpyDeviceToHost, stream);
  ctx->synchronize();
  ctx->profiler().end(stream);
  error::throw_if_exception(h.overflow != 0, "execute_near_far: queue overflow");
  in->set_number_of_elements(0);
  out->set_number_of_elements(0);
  result.levels = h.levels;
  result.splits = h.splits;
  result.relaxations = h.relaxations;
  result.final_threshold = h.threshold;
  return result;
}

}  // namespace advance
}  // namespace operators
}  // namespace gunrock
