/**
 * @file pull.cuh
 * @brief Bottom-up ("pull") step and dense-state kernels of direction-optimised advance.
 *
 * The reference declares advance_direction_t::optimized but throws when it is requested
 * (advance/merge_path.hxx:41-43) and cannot even hold CSR and CSC together (graph/detail/build.hxx:85-89),
 * so the semantics are defined here (DESIGN.md "direction-optimised advance"):
 * for every vertex v outside the visited set, walk v's IN-edges (CSC); for the first in-neighbour u that is
 * in the current frontier and for which op(u, v, e, w) returns true, v joins the next frontier and the
 * visited set and the walk stops. Frontier, next frontier and visited set are 1-bit-per-vertex maps: at
 * scale-26 each is 8 MiB and stays in the 126 MB L2, so the per-edge membership probe never reaches HBM.
 *
 * Mapping: one warp per 1024-vertex chunk (pull_chunk_kernel); next-frontier and visited words are assembled in
 * shared memory and leave as coalesced stores.
 */
#pragma once

#include <type_traits>
#include <utility>
#include <gunrock/b200/warp.cuh>
#include <gunrock/framework/operators/advance/directional.cuh>
#include <gunrock/cuda/context.hxx>
#include <gunrock/graph/graph.hxx>

namespace gunrock {
namespace operators {
namespace advance {
namespace kernels {

using b200::counter_t;
using gcuda::scratch_t;

/// Hint encoding (graph::build::pull_hints): head[v] >= 0 = highest-degree in-neighbour of v; -1 = v has no
/// in-edges; <= -2 = v has exactly ONE in-edge, from vertex -2 - head[v] (nothing to walk when that hint misses).
template <typename vertex_t>
__device__ __forceinline__ vertex_t hint_vertex(vertex_t h) { return h < -1 ? vertex_t(-2) - h : h; }

/// visited := {isolated vertices} ∪ frontier; also Σdeg(frontier) -> counters[aux2].
template <typename vertex_t, typename edge_t>
__global__ void __launch_bounds__(256)
    init_visited_kernel(const edge_t* __restrict__ offsets, vertex_t n, unsigned* __restrict__ visited) {
  const unsigned lane = b200::lane_id();
  const std::size_t n_words = (std::size_t(n) + 31) / 32;
  const std::size_t warps = (std::size_t(gridDim.x) * blockDim.x) >> 5;
  for (std::size_t w = (std::size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; w < n_words; w += warps) {
    const std::size_t v = w * 32 + lane;
    bool skip = true;  // padding bits count as visited so nobody ever walks them
    if (v < std::size_t(n)) skip = offsets[v + 1] == offsets[v];
    const unsigned word = __ballot_sync(b200::full_mask, skip);
    if (lane == 0) visited[w] = word;
  }
}

/// Frontier vertices enter the visited set; accumulates their degree sum (m_f) into counters[aux2].
template <typename vertex_t, typename edge_t>
__global__ void __launch_bounds__(256)
    mark_frontier_kernel(const edge_t* __restrict__ offsets, const vertex_t* __restrict__ list, std::size_t count,
                         const counter_t* count_ptr, unsigned* __restrict__ visited, counter_t* counters) {
  if (count_ptr) count = std::size_t(*count_ptr);
  counter_t mine = 0;
  for (std::size_t i = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count;
       i += std::size_t(gridDim.x) * blockDim.x) {
    const vertex_t v = list[i];
    if (!util::limits::is_valid(v)) continue;
    if (visited) atomicOr(&visited[unsigned(v) >> 5], 1u << (unsigned(v) & 31u));
    mine += counter_t(offsets[v + 1] - offsets[v]);
  }
  // lanes may have diverged on `continue`; reconverge before the shuffle reduction
  __syncwarp();
  mine = b200::warp_sum(mine);
  if (b200::lane_id() == 0 && mine) atomicAdd(counters + scratch_t::aux2, mine);
}

/// A chunk is 32 words = 1024 vertices: what one warp takes per trip of pull_chunk_kernel.
constexpr int pull_chunk_words = 32;
constexpr int pull_queue_cap = 32 + 4 * 32;  ///< walk queue of a warp: < 32 left over + one 4-batch group of misses
constexpr int pull_long_list = 64;           ///< adjacency lists longer than this are walked by the whole warp

/**
 * @brief One bottom-up level. Counters: counters[out_count] += |next frontier|, counters[aux0] += unvisited vertices
 * probed, counters[aux1] += in-edges read, counters[aux2] += vertices whose adjacency was walked. The row bounds of
 * adopted vertices are not read, so Σdeg of the next frontier is not produced.
 * Semantics: for each unvisited vertex, the hinted in-neighbour is offered to the operator first, then the in-edges
 * in list order, until the operator returns true.
 * `A` is the CSC adjacency (for a symmetric graph it aliases the CSR arrays). It may cover a contiguous row range
 * that starts at a multiple of 32 (a partitioned graph's owned rows): `visited` and `next_bits` then point at that
 * range's words, `frontier_bits` and the neighbour ids stay global, and the operator receives the LOCAL row index as
 * destination.
 *
 * Why it looks as it does: a warp-per-word walk ran most of its instructions with 2-5 busy lanes and read row bounds
 * for every probed vertex, though the head hint alone settles most of them (DESIGN.md §3.2). So the chunk's unvisited
 * vertices are compacted into shared memory (all 32 lanes busy however sparse the level), the hints are probed
 * 4 x 32 at a time without row bounds, and only hint misses with more than one in-edge join a walk queue, drained
 * 32 at a time; lists longer than pull_long_list are walked by the whole warp in coalesced 32-edge strides.
 */
template <typename vertex_t, typename edge_t, typename weight_t, typename operator_t>
__global__ void __launch_bounds__(256, 5)
    pull_chunk_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                      const unsigned* __restrict__ frontier_bits, unsigned* __restrict__ next_bits,
                      unsigned* __restrict__ visited, counter_t* counters) {
  __shared__ unsigned short s_open[8][pull_chunk_words * 32];
  __shared__ unsigned s_queue[8][pull_queue_cap];
  __shared__ unsigned s_fresh[8][pull_chunk_words];
  const unsigned lane = b200::lane_id();
  unsigned short* open_list = s_open[b200::warp_id()];
  unsigned* queue = s_queue[b200::warp_id()];
  unsigned* fresh_words = s_fresh[b200::warp_id()];
  const unsigned n = unsigned(A.n);
  const unsigned n_words = (n + 31u) >> 5;
  const unsigned n_chunks = (n_words + pull_chunk_words - 1) / pull_chunk_words;
  const unsigned warps = (gridDim.x * blockDim.x) >> 5;
  const bool hinted = A.head != nullptr;
  unsigned found_vertices = 0, scanned = 0, inspected = 0, walked = 0;
  unsigned queued = 0;                    // warp-uniform
  unsigned live_chunk = 0xffffffffu;      // chunk whose result words are still in shared memory
  constexpr unsigned tried_flag = 0x80000000u;  // queue entry: the hint was offered to the operator and refused

  // walks the adjacency of up to 32 queued vertices (one per lane), all lanes busy
  auto drain = [&](unsigned take) {  // take <= 32, warp-uniform; consumes queue[queued - take .. queued)
    unsigned entry = 0;
    const bool mine = lane < take;
    if (mine) entry = queue[queued - take + lane];
    queued -= take;
    const bool head_tried = (entry & tried_flag) != 0;
    const vertex_t v = vertex_t(entry & ~tried_flag);
    edge_t beg = 0, end = 0;
    if (mine) {
      beg = A.offsets[v];
      end = A.offsets[v + 1];
      ++walked;
    }
    const vertex_t head = (mine && head_tried) ? hint_vertex(__ldg(A.head + v)) : vertex_t(-1);
    bool found = false;
    const bool is_long = mine && (end - beg) > edge_t(pull_long_list);
    if (mine && !is_long) {
      for (edge_t e = beg; e < end && !found; ++e) {
        ++inspected;
        const vertex_t u = __ldg(A.indices + e);
        if (u == head) continue;  // already offered to the operator
        if ((__ldg(frontier_bits + (unsigned(u) >> 5)) >> (unsigned(u) & 31u)) & 1u) {
          const weight_t weight = A.values ? __ldg(A.values + e) : weight_t(1);
          found = call_pull(op, u, v, e, weight);
        }
      }
    }
    // long lists: the warp strides the list 32 edges at a time; candidates are offered in list order
    unsigned long_lanes = __ballot_sync(b200::full_mask, is_long);
    while (long_lanes) {
      const int owner = __ffs(long_lanes) - 1;
      long_lanes &= long_lanes - 1;
      const vertex_t ov = __shfl_sync(b200::full_mask, v, owner);
      const vertex_t ohead = __shfl_sync(b200::full_mask, head, owner);
      const edge_t ob = __shfl_sync(b200::full_mask, beg, owner);
      const edge_t oe = __shfl_sync(b200::full_mask, end, owner);
      bool done = false;
      for (edge_t e0 = ob; e0 < oe && !done; e0 += 32) {
        const edge_t e = e0 + edge_t(lane);
        vertex_t u = vertex_t(-1);
        bool candidate = false;
        if (e < oe) {
          ++inspected;
          u = __ldg(A.indices + e);
          candidate = u != ohead && ((__ldg(frontier_bits + (unsigned(u) >> 5)) >> (unsigned(u) & 31u)) & 1u);
        }
        unsigned votes = __ballot_sync(b200::full_mask, candidate);
        while (votes && !done) {
          const int first = __ffs(votes) - 1;
          votes &= votes - 1;
          bool ok = false;
          if (int(lane) == first) {
            const weight_t weight = A.values ? __ldg(A.values + e) : weight_t(1);
            ok = call_pull(op, u, ov, e, weight);
          }
          done = __shfl_sync(b200::full_mask, ok, first);
        }
      }
      if (int(lane) == owner) found = done;
    }
    if (found) {
      const unsigned bit = 1u << (unsigned(v) & 31u);
      if ((unsigned(v) >> 10) == live_chunk) {  // result words of this chunk are still in shared memory
        atomicOr(fresh_words + ((unsigned(v) >> 5) & 31u), bit);
      } else {  // older chunk: its words were written back; OR into them
        atomicOr(next_bits + (unsigned(v) >> 5), bit);
        atomicOr(visited + (unsigned(v) >> 5), bit);
        ++found_vertices;
      }
    }
    __syncwarp();
  };

  for (unsigned chunk = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; chunk < n_chunks; chunk += warps) {
    const unsigned w_mine = chunk * pull_chunk_words + lane;
    const unsigned seen_mine = w_mine < n_words ? visited[w_mine] : 0xffffffffu;
    fresh_words[lane] = 0u;
    live_chunk = chunk;
    // compact the chunk's unvisited vertices (ascending) into shared memory
    unsigned open_bits = ~seen_mine;
    const unsigned mine_open = __popc(open_bits);
    const unsigned incl = b200::warp_inclusive_sum(mine_open);
    const unsigned total = __shfl_sync(b200::full_mask, incl, 31);
    {
      unsigned at = incl - mine_open;
      while (open_bits) {
        const unsigned b = __ffs(open_bits) - 1;
        open_bits &= open_bits - 1;
        open_list[at++] = (unsigned short)((lane << 5) | b);
      }
    }
    __syncwarp();
    if (lane == 0) scanned += total;
    for (unsigned base = 0; base < total; base += 128) {
      unsigned loc[4];
      vertex_t hid[4];
      bool single[4];
      unsigned probe[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const unsigned idx = base + 32u * k + lane;
        loc[k] = idx < total ? unsigned(open_list[idx]) : 0xffffffffu;
        vertex_t h = vertex_t(-1);
        if (loc[k] != 0xffffffffu && hinted) h = __ldg(A.head + ((chunk << 10) + loc[k]));
        single[k] = h < vertex_t(-1);
        hid[k] = hint_vertex(h);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) probe[k] = hid[k] >= 0 ? __ldg(frontier_bits + (unsigned(hid[k]) >> 5)) : 0u;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const bool valid = loc[k] != 0xffffffffu;
        const vertex_t v = vertex_t((chunk << 10) + (valid ? loc[k] : 0u));
        bool found = false, tried = false;
        if (valid && hid[k] >= 0 && ((probe[k] >> (unsigned(hid[k]) & 31u)) & 1u)) {
          const edge_t edge = __ldg(A.head_edge + v);
          const weight_t weight = A.values ? __ldg(A.values + edge) : weight_t(1);
          found = call_pull(op, hid[k], v, edge, weight);
          tried = true;
        }
        if (found) atomicOr(fresh_words + (loc[k] >> 5), 1u << (loc[k] & 31u));
        // a vertex with a single in-edge has nothing left to offer once its hint missed or was refused
        const bool miss = valid && !found && !(single[k] && hinted);
        const unsigned misses = __ballot_sync(b200::full_mask, miss);
        if (miss) queue[queued + __popc(misses & b200::lanes_below(lane))] = unsigned(v) | (tried ? tried_flag : 0u);
        queued += __popc(misses);
      }
      __syncwarp();
      while (queued >= 32) drain(32);
    }
    __syncwarp();
    const unsigned fresh_mine = fresh_words[lane];
    if (w_mine < n_words) {
      next_bits[w_mine] = fresh_mine;
      if (fresh_mine) visited[w_mine] = seen_mine | fresh_mine;
    }
    found_vertices += __popc(fresh_mine);
    live_chunk = 0xffffffffu;
    __syncwarp();  // the word stores above precede the atomics of later drains on the same words
  }
  if (queued) drain(queued);

  found_vertices = b200::warp_sum(found_vertices);
  scanned = b200::warp_sum(scanned);
  inspected = b200::warp_sum(inspected);
  walked = b200::warp_sum(walked);
  if (lane == 0) {
    if (found_vertices) atomicAdd(counters + scratch_t::out_count, counter_t(found_vertices));
    if (scanned) atomicAdd(counters + scratch_t::aux0, counter_t(scanned));
    if (inspected) atomicAdd(counters + scratch_t::aux1, counter_t(inspected));
    if (walked) atomicAdd(counters + scratch_t::aux2, counter_t(walked));  // vertices whose adjacency was walked
  }
}

/// Development knob: use the per-vertex head hints when the graph carries them (default on).
inline int& pull_hints_enabled() {
  static int enabled = 1;
  return enabled;
}

}  // namespace kernels
}  // namespace advance
}  // namespace operators
}  // namespace gunrock
