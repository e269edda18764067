/**
 * @file kernels.cuh
 * @brief Hand-written sm_100a kernels behind operators::advance (push direction).
 *
 * What the reference does per advance (SURVEY.md §3.1): a Thrust reduce/scan + blocking D2H, a cudaMalloc,
 * one kernel whose threads binary-search 256 shared-memory degrees for every single edge, writes one
 * output slot per edge (mostly -1 holes), a sync and a cudaFree
 * (advance/block_mapped.hxx:38-147,155-205; advance/helpers.hxx:39-146; advance/thread_mapped.hxx:32-96;
 * advance/merge_path.hxx:35-114 = mgpu::transform_lbs).
 *
 * Every balancer of both engines (these scalar kernels and the quad engine of quad.cuh) applies the same
 * visited-bitmap policy (1 bit/vertex, L2 resident), defined below: is_visited / drop_visited probe it,
 * admit() claims a neighbour the operator kept, claim_first() claims a batch before the operator runs.
 * The scalar kernels expand edges through two device routines:
 *   - visit_edge():   probe, call the user operator exactly once with lvalues, admit.
 *   - expand_tile():  a CTA walks a tile of edges described by shared-memory (source, first edge, offset)
 *                     triples; ITEMS independent column loads per thread are issued before any operator
 *                     runs; survivors are compacted with ONE global atomic per CTA round (warp shuffle
 *                     scans), so the output frontier has no holes and the next level reads |F| not Σdeg.
 * The balancers differ only in how tiles are cut:
 *   thread_mapped : one thread per frontier item (warp-uniform trip count, warp-aggregated appends)
 *   block_mapped  : a CTA takes 256 consecutive frontier items, all their edges form its tile; items with
 *                   degree >= big_degree are deferred to a grid-wide kernel (no single-CTA hub tail)
 *   merge_path    : one fused pass scans degrees by decoupled look-back and compacts non-empty items;
 *                   tiles are equal slices of the edge range, located by binary search on the scan
 *   bucketing     : items are binned by degree into thread-, warp- and grid-mapped lists
 * Kernels are persistent (grid = SMs x resident CTAs, grid-stride) and read work sizes from the device
 * counter block, so the host never has to learn Σdeg before launching.
 */
#pragma once

#include <gunrock/b200/warp.cuh>
#include <gunrock/b200/lookback.cuh>
#include <gunrock/framework/operators/advance/directional.cuh>
#include <gunrock/cuda/context.hxx>
#include <gunrock/graph/graph.hxx>
#include <gunrock/util/type_limits.hxx>

namespace gunrock {
namespace operators {
namespace advance {
namespace kernels {

using b200::counter_t;
using gcuda::scratch_t;

constexpr int cta_threads = 256;
constexpr int tile_items = 4;                         // edges per thread per round
constexpr int tile_edges = cta_threads * tile_items;  // 1024 edges per CTA round
constexpr int prep_items = 4;                         // frontier items per thread in the preparation pass
constexpr long long big_degree = 4096;                // adjacency lists this long are expanded grid-wide
constexpr int warp_degree = 32;                       // bucketing: lists at least this long get a warp

/// Visited-bitmap handling of an advance: `none` = reference semantics (operator runs on every edge);
/// `test_and_set` = direction-optimised traversal (neighbours already in the bitmap are skipped, survivors join it);
/// `unique_output` = fused uniquify: the operator still runs on every edge, but a neighbour it keeps is emitted
/// only by the first edge that sets its bit in the (per-call, initially clear) bitmap.
enum class visit_t { none, test_and_set, unique_output };

// ------------------------------------------------------------------------------------------------
// The visited-bitmap policy, shared by the scalar and quad engines.

__device__ __forceinline__ bool is_visited(unsigned* __restrict__ visited, unsigned v) {
  return (visited[v >> 5] >> (v & 31u)) & 1u;
}

/// Sets v's bit; true iff this call set it.
__device__ __forceinline__ bool test_and_set(unsigned* __restrict__ visited, unsigned v) {
  const unsigned bit = 1u << (v & 31u);
  return !(atomicOr(&visited[v >> 5], bit) & bit);
}

/// Clears the live bits of the items whose neighbour is already visited. All probes are issued before any is
/// tested, so their round trips overlap.
template <int N, typename vertex_t>
__device__ __forceinline__ unsigned drop_visited(const vertex_t (&nbr)[N], unsigned live,
                                                 unsigned* __restrict__ visited) {
  unsigned word[N];
#pragma unroll
  for (int i = 0; i < N; ++i)
    if (live & (1u << i)) word[i] = visited[unsigned(nbr[i]) >> 5];
#pragma unroll
  for (int i = 0; i < N; ++i)
    if ((live & (1u << i)) && ((word[i] >> (unsigned(nbr[i]) & 31u)) & 1u)) live &= ~(1u << i);
  return live;
}

/// After the operator: whether a neighbour it kept (`keep`) goes to the output. test_and_set admits the edge that
/// claims the neighbour's bit; unique_output likewise, behind a plain read that keeps repeats off the atomic units.
template <visit_t policy>
__device__ __forceinline__ bool admit(unsigned* __restrict__ visited, unsigned neighbor, bool keep) {
  if constexpr (policy == visit_t::test_and_set) {
    if (keep) keep = test_and_set(visited, neighbor);
  }
  if constexpr (policy == visit_t::unique_output) {
    if (keep) keep = !is_visited(visited, neighbor) && test_and_set(visited, neighbor);
  }
  return keep;
}

/// Claim-first test_and_set of a thread's N edges, for operators with an owner-exclusive (pull) form: probe all,
/// then test-and-set the unvisited, so the dependent memory round trips of the discoveries overlap instead of
/// running one after the other (ncu showed the heavy top-down levels long-scoreboard bound at 19 % issue
/// utilisation with the per-edge chain, profiles/r01c_merge_path_heavy_push.txt). Returns the items whose
/// neighbour this thread claimed; the caller runs the pull form of the operator on exactly those.
template <int N, typename vertex_t>
__device__ __forceinline__ unsigned claim_first(const vertex_t (&nbr)[N], unsigned live,
                                                unsigned* __restrict__ visited) {
  live = drop_visited(nbr, live, visited);
  unsigned claimed = 0;
#pragma unroll
  for (int i = 0; i < N; ++i)
    if ((live & (1u << i)) && test_and_set(visited, unsigned(nbr[i]))) claimed |= 1u << i;
  return claimed;
}

template <visit_t policy, typename vertex_t, typename edge_t, typename weight_t, typename operator_t>
__device__ __forceinline__ bool visit_edge(const graph::adjacency_t<vertex_t, edge_t, weight_t>& A,
                                           operator_t& op, vertex_t source, edge_t edge, vertex_t neighbor,
                                           unsigned* __restrict__ visited) {
  if constexpr (policy == visit_t::test_and_set) {
    if (is_visited(visited, unsigned(neighbor))) return false;
  }
  weight_t weight = A.values ? __ldg(A.values + edge) : weight_t(1);
  source += A.source_offset;  // 1-D partition: operators see global vertex ids
  return admit<policy>(visited, unsigned(neighbor), op(source, neighbor, edge, weight));
}

/// unique_output epilogue: clears the bitmap words of the emitted vertices (only emitted vertices ever set a bit,
/// so storing zero to their words restores the all-clear state in O(|output|)).
template <typename vertex_t>
__global__ void __launch_bounds__(256)
    clear_emitted_kernel(const vertex_t* __restrict__ output, std::size_t count, unsigned* __restrict__ seen) {
  for (std::size_t i = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count;
       i += std::size_t(gridDim.x) * blockDim.x) {
    const vertex_t v = output[i];
    if (util::limits::is_valid(v)) seen[unsigned(v) >> 5] = 0u;
  }
}

/// Shared-memory description of the work a CTA expands in one go.
template <typename vertex_t, typename edge_t>
struct tile_smem_t {
  vertex_t src[tile_edges + 1];
  edge_t beg[tile_edges + 1];
  edge_t seg[tile_edges + 1];               // exclusive offsets of the segments inside the tile
  counter_t append[cta_threads / 32 + 4];   // scratch of b200::cta_append
  edge_t scan_e[cta_threads / 32 + 1];
  unsigned scan_u[cta_threads / 32 + 1];
  long long bcast[4];
};

/**
 * @brief The CTA expands `n_edges` edges spread over `n_seg` non-empty segments held in shared memory.
 * Edge r of the tile belongs to the last segment j with seg[j] <= r and is global edge beg[j] + r - seg[j].
 * Consecutive threads take consecutive edges (coalesced column loads).
 */
template <bool has_output, visit_t policy, typename vertex_t, typename edge_t, typename weight_t, typename operator_t>
__device__ __forceinline__ void expand_tile(const graph::adjacency_t<vertex_t, edge_t, weight_t>& A, operator_t& op,
                                            tile_smem_t<vertex_t, edge_t>& sm, int n_seg, edge_t n_edges,
                                            vertex_t* __restrict__ output, counter_t* counters, counter_t capacity,
                                            unsigned* __restrict__ visited, edge_t edge_base = 0) {
  // edge_base: when the segment table covers more than this tile (small-frontier kernel), tile edge r is
  // edge (edge_base + r) of the table.
  for (edge_t round = 0; round < n_edges; round += tile_edges) {
    vertex_t nbr[tile_items];
    vertex_t src[tile_items];
    edge_t eid[tile_items];
    unsigned live = 0;
#pragma unroll
    for (int i = 0; i < tile_items; ++i) {
      edge_t r = round + edge_t(i * cta_threads + threadIdx.x);
      if (r < n_edges) {
        const edge_t at = r + edge_base;
        int j = n_seg == 1 ? 0 : b200::upper_segment(sm.seg, n_seg, at);
        src[i] = sm.src[j];
        eid[i] = sm.beg[j] + (at - sm.seg[j]);
        live |= 1u << i;
      }
    }
#pragma unroll
    for (int i = 0; i < tile_items; ++i)
      if (live & (1u << i)) nbr[i] = __ldg(A.indices + eid[i]);
    unsigned keep = 0;
    if constexpr (policy == visit_t::test_and_set && has_pull_operator<operator_t>::value) {
      const unsigned claimed = claim_first(nbr, live, visited);
#pragma unroll
      for (int i = 0; i < tile_items; ++i)
        if (claimed & (1u << i)) {
          const weight_t weight = A.values ? __ldg(A.values + eid[i]) : weight_t(1);
          if (call_pull(op, vertex_t(src[i] + A.source_offset), nbr[i], eid[i], weight)) keep |= 1u << i;
        }
    } else {
#pragma unroll
      for (int i = 0; i < tile_items; ++i)
        if (live & (1u << i))
          if (visit_edge<policy>(A, op, src[i], eid[i], nbr[i], visited)) keep |= 1u << i;
    }
    if constexpr (has_output)
      b200::cta_append<cta_threads, tile_items>(nbr, keep, output, counters + scratch_t::out_count, capacity,
                                                sm.append);
  }
}

/// Output-capacity guard shared by the expansion kernels: when the worst case (every edge kept) does not
/// fit, nothing runs and the required size is reported, so the host can grow the buffer and relaunch
/// WITHOUT any operator having been called twice.
__device__ __forceinline__ bool output_fits(counter_t* counters, counter_t capacity) {
  const counter_t worst = counters[scratch_t::work_total];
  if (worst <= capacity) return true;
  if (blockIdx.x == 0 && threadIdx.x == 0) counters[scratch_t::overflow] = worst;
  return false;
}

/// Frontier item i (item i is vertex i when the input is the whole graph) and its row: [beg, end), or beg and the
/// degree when `degree` is set. Past the end of the frontier, and for an invalid id, the vertex is invalid and the
/// row empty.
template <bool graph_input, bool degree = false, typename index_t, typename vertex_t, typename edge_t>
__device__ __forceinline__ void load_row(const edge_t* __restrict__ offsets, const vertex_t* __restrict__ input,
                                         index_t i, index_t input_size, vertex_t& v, edge_t& beg, edge_t& end) {
  v = gunrock::numeric_limits<vertex_t>::invalid();
  beg = 0, end = 0;
  if (i < input_size) {
    v = graph_input ? vertex_t(i) : input[i];
    if (util::limits::is_valid(v)) {
      beg = offsets[v];
      end = degree ? offsets[v + 1] - beg : offsets[v + 1];
    }
  }
}

/// Frontier items [first, first + prep_items) of the preparation passes, invalid past the end.
template <bool graph_input, typename vertex_t>
__device__ __forceinline__ void load_frontier(const vertex_t* __restrict__ input, std::size_t first,
                                              std::size_t input_size, vertex_t (&v)[prep_items]) {
  if constexpr (!graph_input) {
    // the frontier may be a caller's buffer at any 4-byte offset (a tensor view): 128-bit loads need 16 bytes
    const bool vector_input = (reinterpret_cast<std::uintptr_t>(input) & 15u) == 0;
    if (vector_input && first + prep_items <= input_size && prep_items == 4 && sizeof(vertex_t) == 4) {
      const int4 q = *reinterpret_cast<const int4*>(input + first);  // 128-bit frontier load
      v[0] = vertex_t(q.x), v[1] = vertex_t(q.y), v[2] = vertex_t(q.z), v[3] = vertex_t(q.w);
    } else {
#pragma unroll
      for (int k = 0; k < prep_items; ++k)
        v[k] = first + k < input_size ? input[first + k] : gunrock::numeric_limits<vertex_t>::invalid();
    }
  } else {
#pragma unroll
    for (int k = 0; k < prep_items; ++k)
      v[k] = first + k < input_size ? vertex_t(first + k) : gunrock::numeric_limits<vertex_t>::invalid();
  }
}

/// Writes the neighbour of every lane that keeps it to the output, one atomic per warp. Called by all 32 lanes.
template <typename vertex_t>
__device__ __forceinline__ void warp_emit(bool keep, vertex_t nbr, vertex_t* __restrict__ output, counter_t* counters,
                                          counter_t capacity) {
  const unsigned votes = __ballot_sync(b200::full_mask, keep);
  if (votes) {
    counter_t at = b200::warp_append_slot(keep, counters + scratch_t::out_count);
    if (keep && at < capacity) output[at] = nbr;
  }
}

// ------------------------------------------------------------------------------------------------
// Σ degree of a frontier (only launched when nf * max_degree could exceed the output capacity).
template <bool graph_input, typename vertex_t, typename edge_t>
__global__ void __launch_bounds__(cta_threads)
    degree_sum_kernel(const edge_t* __restrict__ offsets, const vertex_t* __restrict__ input, std::size_t input_size,
                      counter_t* counters) {
  counter_t mine = 0;
  for (std::size_t i = std::size_t(blockIdx.x) * cta_threads + threadIdx.x; i < input_size;
       i += std::size_t(gridDim.x) * cta_threads) {
    vertex_t v = graph_input ? vertex_t(i) : input[i];
    if (util::limits::is_valid(v)) mine += counter_t(offsets[v + 1] - offsets[v]);
  }
  mine = b200::warp_sum(mine);
  if (b200::lane_id() == 0 && mine) atomicAdd(counters + scratch_t::work_total, mine);
}

/// Max degree of the graph (once per graph and context; cached by the host).
template <typename vertex_t, typename edge_t>
__global__ void __launch_bounds__(cta_threads)
    max_degree_kernel(const edge_t* __restrict__ offsets, vertex_t n, counter_t* result) {
  counter_t mine = 0;
  for (std::size_t v = std::size_t(blockIdx.x) * cta_threads + threadIdx.x; v < std::size_t(n);
       v += std::size_t(gridDim.x) * cta_threads) {
    counter_t d = counter_t(offsets[v + 1] - offsets[v]);
    mine = d > mine ? d : mine;
  }
  mine = b200::warp_max(mine);
  if (b200::lane_id() == 0) atomicMax(result, mine);
}

// ------------------------------------------------------------------------------------------------
// thread_mapped: one thread per frontier item. `size_ptr` (optional) overrides input_size with a device
// value so the kernel can consume a list another kernel just produced (bucketing's small bin).
template <bool graph_input, bool has_output, bool guard, visit_t policy, typename vertex_t, typename edge_t,
          typename weight_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads)
    thread_mapped_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                         const vertex_t* __restrict__ input, std::size_t input_size, const counter_t* size_ptr,
                         vertex_t* __restrict__ output, counter_t* counters, counter_t capacity,
                         unsigned* __restrict__ visited) {
  if constexpr (has_output && guard)
    if (!output_fits(counters, capacity)) return;
  if (size_ptr) input_size = std::size_t(*size_ptr);
  for (std::size_t base = std::size_t(blockIdx.x) * cta_threads; base < input_size;
       base += std::size_t(gridDim.x) * cta_threads) {
    vertex_t v;
    edge_t beg, deg;
    load_row<graph_input, true>(A.offsets, input, base + threadIdx.x, input_size, v, beg, deg);
    const edge_t trips = b200::warp_max(deg);  // warp-uniform loop so ballots see the whole warp
    for (edge_t k = 0; k < trips; ++k) {
      bool keep = false;
      vertex_t nbr = 0;
      if (k < deg) {
        nbr = __ldg(A.indices + beg + k);
        keep = visit_edge<policy>(A, op, v, edge_t(beg + k), nbr, visited);
      }
      if constexpr (has_output) warp_emit(keep, nbr, output, counters, capacity);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// warp_mapped: one warp per list item, lanes stride the adjacency (coalesced). Used by bucketing's
// medium bin; the list length comes from a device counter.
template <bool has_output, visit_t policy, typename vertex_t, typename edge_t, typename weight_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads)
    warp_mapped_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                       const vertex_t* __restrict__ list, const counter_t* size_ptr, vertex_t* __restrict__ output,
                       counter_t* counters, counter_t capacity, unsigned* __restrict__ visited) {
  if constexpr (has_output)
    if (!output_fits(counters, capacity)) return;
  const std::size_t count = std::size_t(*size_ptr);
  const unsigned lane = b200::lane_id();
  const std::size_t warps = (std::size_t(gridDim.x) * cta_threads) >> 5;
  for (std::size_t item = (std::size_t(blockIdx.x) * cta_threads + threadIdx.x) >> 5; item < count; item += warps) {
    vertex_t v = list[item];
    const edge_t beg = A.offsets[v], end = A.offsets[v + 1];
    for (edge_t e0 = beg; e0 < end; e0 += 32) {
      const edge_t e = e0 + lane;
      bool keep = false;
      vertex_t nbr = 0;
      if (e < end) {
        nbr = __ldg(A.indices + e);
        keep = visit_edge<policy>(A, op, v, e, nbr, visited);
      }
      if constexpr (has_output) warp_emit(keep, nbr, output, counters, capacity);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// block_mapped: a CTA owns 256 consecutive frontier items and every edge under them.
template <bool graph_input, bool has_output, bool guard, visit_t policy, typename vertex_t, typename edge_t,
          typename weight_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads)
    block_mapped_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                        const vertex_t* __restrict__ input, std::size_t input_size, vertex_t* __restrict__ output,
                        counter_t* counters, counter_t capacity, unsigned* __restrict__ visited,
                        vertex_t* __restrict__ big_list) {
  __shared__ tile_smem_t<vertex_t, edge_t> sm;
  if constexpr (has_output && guard)
    if (!output_fits(counters, capacity)) return;
  for (std::size_t base = std::size_t(blockIdx.x) * cta_threads; base < input_size;
       base += std::size_t(gridDim.x) * cta_threads) {
    vertex_t v;
    edge_t beg, deg;
    load_row<graph_input, true>(A.offsets, input, base + threadIdx.x, input_size, v, beg, deg);
    if (big_list && deg >= edge_t(big_degree)) {  // hub: hand it to the grid-wide kernel
      counter_t at = atomicAdd(counters + scratch_t::big_count, counter_t(1));
      big_list[at] = v;
      deg = 0;
    }
    unsigned n_seg;
    edge_t n_edges;
    const unsigned my_seg = b200::cta_exclusive_sum<cta_threads, unsigned>(deg > 0 ? 1u : 0u, n_seg, sm.scan_u);
    const edge_t my_off = b200::cta_exclusive_sum<cta_threads, edge_t>(deg, n_edges, sm.scan_e);
    if (deg > 0) {
      sm.src[my_seg] = v;
      sm.beg[my_seg] = beg;
      sm.seg[my_seg] = my_off;
    }
    __syncthreads();
    if (n_edges > 0)
      expand_tile<has_output, policy>(A, op, sm, int(n_seg), n_edges, output, counters, capacity, visited);
    __syncthreads();
  }
}

/// Grid-wide expansion of the deferred hubs: every CTA strides the 1024-edge tiles of each listed vertex.
template <bool has_output, visit_t policy, typename vertex_t, typename edge_t, typename weight_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads)
    big_list_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                    const vertex_t* __restrict__ big_list, const counter_t* size_ptr, vertex_t* __restrict__ output,
                    counter_t* counters, counter_t capacity, unsigned* __restrict__ visited) {
  __shared__ tile_smem_t<vertex_t, edge_t> sm;
  if constexpr (has_output)
    if (!output_fits(counters, capacity)) return;
  const std::size_t count = std::size_t(*size_ptr);
  for (std::size_t item = 0; item < count; ++item) {
    const vertex_t v = big_list[item];
    const edge_t beg = A.offsets[v], deg = A.offsets[v + 1] - beg;
    for (edge_t t0 = edge_t(blockIdx.x) * tile_edges; t0 < deg; t0 += edge_t(gridDim.x) * tile_edges) {
      if (threadIdx.x == 0) {
        sm.src[0] = v;
        sm.beg[0] = beg + t0;
        sm.seg[0] = 0;
      }
      __syncthreads();
      const edge_t left = deg - t0;
      expand_tile<has_output, policy>(A, op, sm, 1, left < edge_t(tile_edges) ? left : edge_t(tile_edges), output,
                                      counters, capacity, visited);
      __syncthreads();
    }
  }
}

// ------------------------------------------------------------------------------------------------
// merge_path, pass 1: fused validity filter + degree gather + device-wide scan + compaction.
// Produces work_src[k], work_beg[k], work_seg[k] (exclusive Σdeg over the compacted, non-empty items, with
// work_seg[K] = total), counters[items] = K, counters[work_total] = Σdeg. Stable (frontier order kept).
template <bool graph_input, typename vertex_t, typename edge_t>
__global__ void __launch_bounds__(cta_threads)
    prepare_work_kernel(const edge_t* __restrict__ offsets, const vertex_t* __restrict__ input, std::size_t input_size,
                        vertex_t* __restrict__ work_src, edge_t* __restrict__ work_beg, edge_t* __restrict__ work_seg,
                        b200::tile_word_t* state_items, b200::tile_word_t* state_edges, counter_t* counters) {
  constexpr int per_tile = cta_threads * prep_items;
  __shared__ unsigned scan_u[cta_threads / 32 + 1];
  __shared__ unsigned long long scan_e[cta_threads / 32 + 1];
  __shared__ unsigned long long prefix[2];
  __shared__ int s_tile;
  const int n_tiles = int((input_size + per_tile - 1) / per_tile);
  for (;;) {
    if (threadIdx.x == 0) s_tile = int(atomicAdd(counters + scratch_t::ticket, counter_t(1)));
    __syncthreads();
    const int tile = s_tile;
    if (tile >= n_tiles) break;
    const std::size_t first = std::size_t(tile) * per_tile + std::size_t(threadIdx.x) * prep_items;
    vertex_t v[prep_items];
    edge_t beg[prep_items], deg[prep_items];
    load_frontier<graph_input>(input, first, input_size, v);
    unsigned my_items = 0;
    unsigned long long my_edges = 0;
#pragma unroll
    for (int k = 0; k < prep_items; ++k) {
      beg[k] = 0, deg[k] = 0;
      if (util::limits::is_valid(v[k])) {
        beg[k] = offsets[v[k]];
        deg[k] = offsets[v[k] + 1] - beg[k];
      }
      my_items += deg[k] > 0;
      my_edges += (unsigned long long)deg[k];
    }
    unsigned tile_items_total;
    unsigned long long tile_edges_total;
    const unsigned items_before = b200::cta_exclusive_sum<cta_threads, unsigned>(my_items, tile_items_total, scan_u);
    const unsigned long long edges_before =
        b200::cta_exclusive_sum<cta_threads, unsigned long long>(my_edges, tile_edges_total, scan_e);
    if (threadIdx.x < 32) {
      const unsigned long long a = b200::lookback_exclusive(state_items, tile, tile_items_total);
      const unsigned long long b = b200::lookback_exclusive(state_edges, tile, tile_edges_total);
      if (threadIdx.x == 0) {
        prefix[0] = a;
        prefix[1] = b;
      }
    }
    __syncthreads();
    std::size_t at = std::size_t(prefix[0]) + items_before;
    unsigned long long run = prefix[1] + edges_before;
#pragma unroll
    for (int k = 0; k < prep_items; ++k)
      if (deg[k] > 0) {
        work_src[at] = v[k];
        work_beg[at] = beg[k];
        work_seg[at] = edge_t(run);
        ++at;
        run += (unsigned long long)deg[k];
      }
    if (tile == n_tiles - 1 && threadIdx.x == 0) {
      const unsigned long long K = prefix[0] + tile_items_total, T = prefix[1] + tile_edges_total;
      counters[scratch_t::items] = K;
      counters[scratch_t::work_total] = T;
      work_seg[K] = edge_t(T);
    }
    __syncthreads();  // s_tile / prefix reuse
  }
}

// merge_path, pass 2: equal slices of the edge range; each CTA finds its first/last segment by binary
// search on the scanned offsets, stages the slice's segments in shared memory and expands the tile.
template <bool has_output, visit_t policy, typename vertex_t, typename edge_t, typename weight_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads)
    merge_path_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                      const vertex_t* __restrict__ work_src, const edge_t* __restrict__ work_beg,
                      const edge_t* __restrict__ work_seg, vertex_t* __restrict__ output, counter_t* counters,
                      counter_t capacity, unsigned* __restrict__ visited) {
  __shared__ tile_smem_t<vertex_t, edge_t> sm;
  if constexpr (has_output)
    if (!output_fits(counters, capacity)) return;
  const long long total = (long long)counters[scratch_t::work_total];
  const long long n_items = (long long)counters[scratch_t::items];
  // Each CTA takes a CONTIGUOUS run of 1024-edge slices, so only its first slice needs the binary search on
  // the scanned offsets (17 dependent L2 round trips at |F| = 120 K while 254 threads wait); every following
  // slice starts in the segment the previous one ended in and its last segment is found from shared memory.
  const long long n_tiles = (total + tile_edges - 1) / tile_edges;
  const long long per_cta = (n_tiles + gridDim.x - 1) / gridDim.x;
  const long long first_tile = (long long)blockIdx.x * per_cta;
  const long long last_tile = first_tile + per_cta < n_tiles ? first_tile + per_cta : n_tiles;
  long long j0 = 0;
  for (long long tile = first_tile; tile < last_tile; ++tile) {
    const long long g0 = tile * tile_edges;
    const long long g1 = g0 + tile_edges < total ? g0 + tile_edges : total;
    if (tile == first_tile) {
      if (threadIdx.x == 0) {
        long long lo = 0, hi = n_items;  // work_seg[lo] <= g0 < work_seg[hi]
        while (hi - lo > 1) {
          const long long mid = (lo + hi) >> 1;
          if ((long long)work_seg[mid] <= g0)
            lo = mid;
          else
            hi = mid;
        }
        sm.bcast[0] = lo;
      }
      __syncthreads();
      j0 = sm.bcast[0];
    }
    // stage segments j0, j0+1, ... until one starts at or beyond g1 (at most tile_edges + 1 of them: all but the
    // first start inside the slice and are non-empty). Threads load candidates in parallel; the count is the
    // number of staged segments that start before g1.
    int n_seg = 0;
    {
      unsigned mine = 0;
      for (int j = threadIdx.x; j <= tile_edges; j += cta_threads) {
        const long long jj = j0 + j;
        if (jj < n_items) {
          const long long s = (long long)work_seg[jj];
          if (s < g1) {
            sm.src[j] = work_src[jj];
            sm.beg[j] = work_beg[jj] + edge_t(s < g0 ? g0 - s : 0);  // first segment may start before the slice
            sm.seg[j] = edge_t(s < g0 ? 0 : s - g0);
            ++mine;
          }
        }
      }
      unsigned total_seg;
      b200::cta_exclusive_sum<cta_threads, unsigned>(mine, total_seg, sm.scan_u);
      n_seg = int(total_seg);
    }
    __syncthreads();
    expand_tile<has_output, policy>(A, op, sm, n_seg, edge_t(g1 - g0), output, counters, capacity, visited);
    // next slice starts in the last segment of this one if that segment continues past g1, else in the next
    {
      const long long last = j0 + n_seg - 1;
      const long long last_end = (long long)work_seg[last + 1];  // work_seg[n_items] holds the total
      j0 = last_end > g1 ? last : last + 1;
    }
    __syncthreads();
  }
}

// merge_path for small frontiers (nf <= tile_edges items): ONE launch. Every CTA redundantly builds the whole
// (source, first edge, scanned offset) table in shared memory — at most 1024 row-bound pairs, L2 hits — and
// then expands its own equal slices of the edge range straight from that table. Replaces the
// memset + prepare_work_kernel + merge_path_kernel sequence on the many tiny levels of a BFS
// (source level, the first hops, the tail) where launch latency, not bandwidth, is the cost.
template <bool graph_input, bool has_output, visit_t policy, typename vertex_t, typename edge_t, typename weight_t,
          typename operator_t>
__global__ void __launch_bounds__(cta_threads)
    merge_path_small_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                            const vertex_t* __restrict__ input, int input_size, vertex_t* __restrict__ output,
                            counter_t* counters, counter_t capacity, unsigned* __restrict__ visited) {
  __shared__ tile_smem_t<vertex_t, edge_t> sm;
  vertex_t v[tile_items];
  edge_t beg[tile_items], deg[tile_items];
  unsigned my_items = 0;
  edge_t my_edges = 0;
#pragma unroll
  for (int k = 0; k < tile_items; ++k) {
    const int i = int(threadIdx.x) * tile_items + k;  // blocked order keeps the table in frontier order
    load_row<graph_input, true>(A.offsets, input, i, input_size, v[k], beg[k], deg[k]);
    my_items += deg[k] > 0;
    my_edges += deg[k];
  }
  unsigned n_seg;
  edge_t total;
  unsigned at = b200::cta_exclusive_sum<cta_threads, unsigned>(my_items, n_seg, sm.scan_u);
  edge_t run = b200::cta_exclusive_sum<cta_threads, edge_t>(my_edges, total, sm.scan_e);
#pragma unroll
  for (int k = 0; k < tile_items; ++k)
    if (deg[k] > 0) {
      sm.src[at] = v[k];
      sm.beg[at] = beg[k];
      sm.seg[at] = run;
      ++at;
      run += deg[k];
    }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0) counters[scratch_t::work_total] = counter_t(total);
  if constexpr (has_output) {
    if (counter_t(total) > capacity) {  // every CTA computes the same total, so all of them leave
      if (blockIdx.x == 0 && threadIdx.x == 0) counters[scratch_t::overflow] = counter_t(total);
      return;
    }
  }
  for (edge_t g0 = edge_t(blockIdx.x) * tile_edges; g0 < total; g0 += edge_t(gridDim.x) * tile_edges) {
    const edge_t left = total - g0;
    expand_tile<has_output, policy>(A, op, sm, int(n_seg), left < edge_t(tile_edges) ? left : edge_t(tile_edges),
                                    output, counters, capacity, visited, g0);
  }
}

// ------------------------------------------------------------------------------------------------
// bucketing, pass 1: bin valid non-empty items by degree (thread / warp / grid classes) and total Σdeg.
template <bool graph_input, typename vertex_t, typename edge_t>
__global__ void __launch_bounds__(cta_threads)
    bin_by_degree_kernel(const edge_t* __restrict__ offsets, const vertex_t* __restrict__ input,
                         std::size_t input_size, vertex_t* __restrict__ small_list, vertex_t* __restrict__ warp_list,
                         vertex_t* __restrict__ big_list, counter_t* counters) {
  counter_t my_edges = 0;
  for (std::size_t base = std::size_t(blockIdx.x) * cta_threads; base < input_size;
       base += std::size_t(gridDim.x) * cta_threads) {
    const std::size_t i = base + threadIdx.x;
    edge_t deg = 0;
    vertex_t v = 0;
    if (i < input_size) {
      v = graph_input ? vertex_t(i) : input[i];
      if (util::limits::is_valid(v)) deg = offsets[v + 1] - offsets[v];
    }
    my_edges += counter_t(deg);
    const bool is_big = deg >= edge_t(big_degree);
    const bool is_warp = !is_big && deg >= edge_t(warp_degree);
    const bool is_small = deg > 0 && deg < edge_t(warp_degree);
    if (__ballot_sync(b200::full_mask, is_small)) {
      counter_t at = b200::warp_append_slot(is_small, counters + scratch_t::aux0);
      if (is_small) small_list[at] = v;
    }
    if (__ballot_sync(b200::full_mask, is_warp)) {
      counter_t at = b200::warp_append_slot(is_warp, counters + scratch_t::aux1);
      if (is_warp) warp_list[at] = v;
    }
    if (__ballot_sync(b200::full_mask, is_big)) {
      counter_t at = b200::warp_append_slot(is_big, counters + scratch_t::big_count);
      if (is_big) big_list[at] = v;
    }
  }
  my_edges = b200::warp_sum(my_edges);
  if (b200::lane_id() == 0 && my_edges) atomicAdd(counters + scratch_t::work_total, my_edges);
}

}  // namespace kernels
}  // namespace advance
}  // namespace operators
}  // namespace gunrock
