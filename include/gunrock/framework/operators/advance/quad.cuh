/**
 * @file quad.cuh
 * @brief The sm_100a expansion engine of operators::advance (push direction): warp-autonomous rounds over
 * 16-byte-aligned QUADS of the column-index array.
 *
 * What it replaces. The reference's only hand-written advance kernel (advance/block_mapped.hxx:38-147) makes every
 * thread binary-search 256 shared-memory degrees for every single edge (:121), loads column indices and weights
 * with scalar 4-byte loads and claims output slots with a block-wide scan + atomic per 256 edges; merge_path
 * (advance/merge_path.hxx:35-114) is two moderngpu passes. Round 1 of this tree kept the per-edge search and a
 * CTA barrier + one global atomic per 1024 edges; ncu showed that kernel at 20 % issue utilisation, dominated by
 * long-scoreboard and barrier stalls (profiles/r01c_merge_path_full_raw.csv).
 *
 * Design.
 *   - Unit of work = a quad: the 4 column indices at edges [4g, 4g+4). A list [beg, end) covers quads
 *     beg>>2 .. (end-1)>>2; elements of the first/last quad outside the list are masked. Every column (and weight)
 *     access is therefore ONE aligned 128-bit load (LDG.E.128), whatever the list's start.
 *   - The scanned work domain counts quads. A warp owns a contiguous run of 64-quad rounds (256 edges); per round
 *     it stages the <= 65 segments that intersect the round into its own shared-memory table, each lane takes two
 *     quads (lane-consecutive, so a warp instruction reads 512 contiguous bytes), finds their segment with one
 *     short search per QUAD (not per edge), and issues both 128-bit loads before any operator runs.
 *   - No CTA barrier anywhere in the expansion loop: warps run decoupled, so one warp's DRAM miss does not stall
 *     seven others. Survivors go to a per-warp shared-memory staging buffer (shuffle scan, no atomics) that is
 *     flushed with ONE global atomic per >= 256 survivors and fully coalesced stores; the output stays compact.
 *   - Hubs (>= big_degree edges) of block_mapped / bucketing are streamed through shared memory by the TMA unit:
 *     cp.async.bulk global->shared, double buffered on mbarriers (big_list_bulk_kernel), so the next 8 KB of
 *     neighbours arrive while the current tile's random probes are in flight.
 * Requirements checked by the host dispatch (advance.hxx): 4-byte vertex ids and 16-byte aligned index / weight
 * arrays; anything else takes the scalar kernels in kernels.cuh.
 */
#pragma once

#include <climits>
#include <gunrock/framework/operators/advance/kernels.cuh>

namespace gunrock {
namespace operators {
namespace advance {
namespace kernels {

constexpr int quad_warps = cta_threads / 32;        // warps per CTA
constexpr int quads_per_lane = 2;                   // 8 edges per lane per round
constexpr int round_quads = 32 * quads_per_lane;    // 64 quads = 256 edges per warp round
constexpr int round_items = quads_per_lane * 4;     // edges per lane per round
constexpr int warp_table_cap = 96;                  // >= 65 segments can intersect a round; staged 32 at a time
constexpr int stage_cap = 512;                      // per-warp staging entries (flushed above stage_cap - 256)
constexpr int small_items = 512;                    // frontiers up to this size take the single-launch kernel
constexpr int bulk_tile_quads = 512;                // TMA tile of the hub kernel: 2048 edges = 8 KB

/// Development knob (ess_tune "advance_engine"): 1 = quad engine (default), 0 = round-1 scalar kernels.
inline int& advance_engine() {
  static int engine = 1;
  return engine;
}

// ------------------------------------------------------------------------------------------------------------
// 128-bit loads

/// x[0..3] = p[e0..e0+3]; e0 is a multiple of 4 and p is 16-byte aligned. The last quad of an array whose length
/// is not a multiple of 4 is read element-wise (no access past `count`). p is only ever a graph's column indices or
/// values, and expand() takes the quad engine only after checking both on the host; graphs over arrays at another
/// offset run the scalar kernels.
template <typename T, typename index_t>
__device__ __forceinline__ void load_quad(const T* __restrict__ p, index_t e0, index_t count, T (&x)[4]) {
  static_assert(sizeof(T) == 4, "quad loads move four 4-byte elements");
  if (e0 + 4 <= count) {
    const int4 q = __ldg(reinterpret_cast<const int4*>(p + e0));
    x[0] = __builtin_bit_cast(T, q.x);
    x[1] = __builtin_bit_cast(T, q.y);
    x[2] = __builtin_bit_cast(T, q.z);
    x[3] = __builtin_bit_cast(T, q.w);
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) x[i] = e0 + i < count ? __ldg(p + e0 + i) : T(0);
  }
}

// ------------------------------------------------------------------------------------------------------------
// per-warp output staging

template <typename vertex_t, int CAP = stage_cap>
struct warp_stage_t {
  vertex_t buf[CAP];
};

template <typename vertex_t>
__device__ __forceinline__ void stage_flush(vertex_t* buf, unsigned& staged, vertex_t* __restrict__ output,
                                            counter_t* out_count, counter_t capacity) {
  if (staged == 0) return;  // warp-uniform
  __syncwarp();
  counter_t base = 0;
  if (b200::lane_id() == 0) base = atomicAdd(out_count, counter_t(staged));
  base = __shfl_sync(b200::full_mask, base, 0);
  for (unsigned k = b200::lane_id(); k < staged; k += 32)
    if (base + k < capacity) output[base + k] = buf[k];
  __syncwarp();
  staged = 0;
}

/// Appends the kept values of every lane (bit i of `keep` <-> vals[i]) to the warp's staging buffer; flushes it to
/// the global queue when fewer than 32*N free slots remain. Called by all 32 lanes.
template <int CAP, int N, typename vertex_t>
__device__ __forceinline__ void stage_append(const vertex_t (&vals)[N], unsigned keep, vertex_t* buf, unsigned& staged,
                                             vertex_t* __restrict__ output, counter_t* out_count, counter_t capacity) {
  static_assert(CAP >= 2 * 32 * N || CAP > 32 * N, "staging buffer too small");
  if (!__any_sync(b200::full_mask, keep != 0)) return;
  const unsigned mine = __popc(keep);
  const unsigned incl = b200::warp_inclusive_sum(mine);
  const unsigned total = __shfl_sync(b200::full_mask, incl, 31);
  unsigned at = staged + incl - mine;
#pragma unroll
  for (int i = 0; i < N; ++i)
    if (keep & (1u << i)) buf[at++] = vals[i];
  staged += total;
  if (staged > unsigned(CAP - 32 * N)) stage_flush(buf, staged, output, out_count, capacity);
}

// ------------------------------------------------------------------------------------------------------------
// operator invocation on the (up to) 8 edges of a lane

/**
 * @brief Runs the visit policy on the live edges of QPL quads held in registers. Edge i (0 <= i < 4*QPL) belongs
 * to quad q = i/4: source src[q], edge id e0[q] + i%4, neighbour nbr[i]. Returns the keep mask.
 */
template <visit_t policy, int QPL, typename vertex_t, typename edge_t, typename weight_t, typename operator_t>
__device__ __forceinline__ unsigned visit_items(const graph::adjacency_t<vertex_t, edge_t, weight_t>& A, operator_t& op,
                                                const vertex_t (&nbr)[QPL * 4], unsigned live,
                                                const vertex_t (&src)[QPL], const edge_t (&e0)[QPL],
                                                unsigned* __restrict__ visited) {
  constexpr int N = QPL * 4;
  unsigned keep = 0;
  weight_t wt[N];
#pragma unroll
  for (int i = 0; i < N; ++i) wt[i] = weight_t(1);
  auto load_weights = [&](unsigned needed) {
    if (A.values == nullptr) return;
#pragma unroll
    for (int q = 0; q < QPL; ++q)
      if ((needed >> (4 * q)) & 0xfu) {
        weight_t w4[4];
        load_quad(A.values, e0[q], A.m, w4);
#pragma unroll
        for (int i = 0; i < 4; ++i) wt[4 * q + i] = w4[i];
      }
  };

  if constexpr (policy == visit_t::test_and_set && has_pull_operator<operator_t>::value) {
    const unsigned claimed = claim_first(nbr, live, visited);
    if (claimed) {
      load_weights(claimed);
#pragma unroll
      for (int i = 0; i < N; ++i)
        if (claimed & (1u << i))
          if (call_pull(op, vertex_t(src[i >> 2] + A.source_offset), nbr[i], edge_t(e0[i >> 2] + (i & 3)), wt[i]))
            keep |= 1u << i;
    }
  } else {
    // the whole batch is probed before the operator runs on any edge
    if constexpr (policy == visit_t::test_and_set) live = drop_visited(nbr, live, visited);
    load_weights(live);
#pragma unroll
    for (int i = 0; i < N; ++i)
      if (live & (1u << i)) {
        vertex_t s = src[i >> 2] + A.source_offset, d = nbr[i];  // 1-D partition: global source id
        edge_t e = edge_t(e0[i >> 2] + (i & 3));
        weight_t w = wt[i];
        if (admit<policy>(visited, unsigned(d), op(s, d, e, w))) keep |= 1u << i;  // lvalues, once per live edge
      }
  }
  return keep;
}

/// live mask of the QPL quads of a lane: element i of quad q is live iff the quad exists and the edge lies in
/// the list [lo[q], hi[q]).
template <int QPL, typename edge_t>
__device__ __forceinline__ unsigned live_mask(unsigned have, const edge_t (&e0)[QPL], const edge_t (&lo)[QPL],
                                              const edge_t (&hi)[QPL]) {
  unsigned live = 0;
#pragma unroll
  for (int q = 0; q < QPL; ++q)
    if (have & (1u << q)) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const edge_t e = e0[q] + i;
        if (e >= lo[q] && e < hi[q]) live |= 1u << (4 * q + i);
      }
    }
  return live;
}

// ------------------------------------------------------------------------------------------------------------
// one warp round over a segment table in shared memory

/**
 * @brief The warp expands `n_quads` (<= 64) consecutive table positions starting at `pos0`. Table entry j describes
 * a list: it owns positions [rel[j], rel[j+1]) (rel ascending, rel[0] <= pos0), position p maps to global quad
 * qoff[j] + p; beg/end are the list bounds in edges and src its vertex. Lane L takes positions pos0 + L and
 * pos0 + 32 + L.
 */
template <bool has_output, visit_t policy, int CAP, typename vertex_t, typename edge_t, typename weight_t,
          typename operator_t>
__device__ __forceinline__ void expand_round(const graph::adjacency_t<vertex_t, edge_t, weight_t>& A, operator_t& op,
                                             const edge_t* rel, const edge_t* qoff, const edge_t* beg,
                                             const edge_t* end, const vertex_t* src_of, int n_seg, edge_t pos0,
                                             int n_quads, vertex_t* sbuf, unsigned& staged,
                                             vertex_t* __restrict__ output, counter_t* counters, counter_t capacity,
                                             unsigned* __restrict__ visited) {
  const int lane = int(b200::lane_id());
  vertex_t src[quads_per_lane];
  edge_t e0[quads_per_lane], lo[quads_per_lane], hi[quads_per_lane];
  unsigned have = 0;
#pragma unroll
  for (int q = 0; q < quads_per_lane; ++q) {
    src[q] = 0, e0[q] = 0, lo[q] = 0, hi[q] = 0;
    const int k = q * 32 + lane;
    if (k < n_quads) {
      const edge_t pos = pos0 + edge_t(k);
      const int j = n_seg == 1 ? 0 : b200::upper_segment(rel, n_seg, pos);
      e0[q] = (qoff[j] + pos) * 4;
      lo[q] = beg[j];
      hi[q] = end[j];
      src[q] = src_of[j];
      have |= 1u << q;
    }
  }
  vertex_t nbr[round_items];
#pragma unroll
  for (int q = 0; q < quads_per_lane; ++q) {
    vertex_t c[4] = {0, 0, 0, 0};
    if (have & (1u << q)) load_quad(A.indices, e0[q], A.m, c);
#pragma unroll
    for (int i = 0; i < 4; ++i) nbr[4 * q + i] = c[i];
  }
  const unsigned live = live_mask<quads_per_lane>(have, e0, lo, hi);
  const unsigned keep = visit_items<policy, quads_per_lane>(A, op, nbr, live, src, e0, visited);
  if constexpr (has_output)
    stage_append<CAP>(nbr, keep, sbuf, staged, output, counters + scratch_t::out_count, capacity);
}

// ------------------------------------------------------------------------------------------------------------
// merge_path, pass 1: validity filter + bounds gather + device-wide scan of QUAD counts + compaction.
// Produces work_src/work_beg/work_end/work_seg for the K non-empty items (work_seg = exclusive quad scan,
// work_seg[K] = total), counters[items] = K, counters[quads] = total quads, counters[work_total] = Σdeg.
template <bool graph_input, typename vertex_t, typename edge_t>
__global__ void __launch_bounds__(cta_threads)
    prepare_quads_kernel(const edge_t* __restrict__ offsets, const vertex_t* __restrict__ input, std::size_t input_size,
                         vertex_t* __restrict__ work_src, edge_t* __restrict__ work_beg, edge_t* __restrict__ work_end,
                         edge_t* __restrict__ work_seg, b200::tile_word_t* state_items, b200::tile_word_t* state_quads,
                         counter_t* counters) {
  constexpr int per_tile = cta_threads * prep_items;
  __shared__ unsigned scan_u[cta_threads / 32 + 1];
  __shared__ unsigned long long scan_q[cta_threads / 32 + 1];
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
    edge_t beg[prep_items], end[prep_items];
    load_frontier<graph_input>(input, first, input_size, v);
    unsigned my_items = 0;
    unsigned long long my_quads = 0, my_edges = 0;
    unsigned long long nq[prep_items];
#pragma unroll
    for (int k = 0; k < prep_items; ++k) {
      beg[k] = 0, end[k] = 0, nq[k] = 0;
      if (util::limits::is_valid(v[k])) {
        beg[k] = offsets[v[k]];
        end[k] = offsets[v[k] + 1];
      }
      if (end[k] > beg[k]) {
        nq[k] = (unsigned long long)(((end[k] - 1) >> 2) - (beg[k] >> 2) + 1);
        my_items += 1;
        my_edges += (unsigned long long)(end[k] - beg[k]);
      }
      my_quads += nq[k];
    }
    unsigned tile_items_total;
    unsigned long long tile_quads_total;
    const unsigned items_before = b200::cta_exclusive_sum<cta_threads, unsigned>(my_items, tile_items_total, scan_u);
    const unsigned long long quads_before =
        b200::cta_exclusive_sum<cta_threads, unsigned long long>(my_quads, tile_quads_total, scan_q);
    my_edges = b200::warp_sum(my_edges);
    if (b200::lane_id() == 0 && my_edges) atomicAdd(counters + scratch_t::work_total, my_edges);
    if (threadIdx.x < 32) {
      const unsigned long long a = b200::lookback_exclusive(state_items, tile, tile_items_total);
      const unsigned long long b = b200::lookback_exclusive(state_quads, tile, tile_quads_total);
      if (threadIdx.x == 0) {
        prefix[0] = a;
        prefix[1] = b;
      }
    }
    __syncthreads();
    std::size_t at = std::size_t(prefix[0]) + items_before;
    unsigned long long run = prefix[1] + quads_before;
#pragma unroll
    for (int k = 0; k < prep_items; ++k)
      if (nq[k]) {
        work_src[at] = v[k];
        work_beg[at] = beg[k];
        work_end[at] = end[k];
        work_seg[at] = edge_t(run);
        ++at;
        run += nq[k];
      }
    if (tile == n_tiles - 1 && threadIdx.x == 0) {
      const unsigned long long K = prefix[0] + tile_items_total, T = prefix[1] + tile_quads_total;
      counters[scratch_t::items] = K;
      counters[scratch_t::quads] = T;
      work_seg[K] = edge_t(T);
    }
    __syncthreads();  // s_tile / prefix reuse
  }
}

template <typename vertex_t, typename edge_t>
struct warp_table_t {
  edge_t rel[warp_table_cap];
  edge_t qoff[warp_table_cap];
  edge_t beg[warp_table_cap];
  edge_t end[warp_table_cap];
  vertex_t src[warp_table_cap];
};

// merge_path, pass 2: every warp takes a contiguous run of 64-quad rounds of the scanned quad range.
template <bool has_output, visit_t policy, typename vertex_t, typename edge_t, typename weight_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads, 4)
    merge_path_quad_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                           const vertex_t* __restrict__ work_src, const edge_t* __restrict__ work_beg,
                           const edge_t* __restrict__ work_end, const edge_t* __restrict__ work_seg,
                           vertex_t* __restrict__ output, counter_t* counters, counter_t capacity,
                           unsigned* __restrict__ visited) {
  __shared__ warp_table_t<vertex_t, edge_t> tables[quad_warps];
  __shared__ warp_stage_t<vertex_t> stages[has_output ? quad_warps : 1];
  if constexpr (has_output)
    if (!output_fits(counters, capacity)) return;
  const long long total = (long long)counters[scratch_t::quads];
  const long long n_items = (long long)counters[scratch_t::items];
  const unsigned lane = b200::lane_id(), warp = b200::warp_id();
  auto& T = tables[warp];
  vertex_t* sbuf = stages[has_output ? warp : 0].buf;
  unsigned staged = 0;

  const long long n_rounds = (total + round_quads - 1) / round_quads;
  const long long n_warps = (long long)gridDim.x * quad_warps;
  const long long per_warp = (n_rounds + n_warps - 1) / n_warps;
  const long long first_round = ((long long)blockIdx.x * quad_warps + warp) * per_warp;
  long long last_round = first_round + per_warp;
  if (last_round > n_rounds) last_round = n_rounds;

  if (first_round < last_round) {
    // segment holding the warp's first quad: largest j with work_seg[j] <= p0, by a 32-way search (each step is
    // ONE round trip for the whole warp: 5 steps at 2^25 items instead of 25 dependent loads)
    const long long p0 = first_round * round_quads;
    long long lo = 0, hi = n_items;  // work_seg[lo] <= p0 < work_seg[hi]   (work_seg[n_items] = total > p0)
    while (hi - lo > 1) {
      const long long step = (hi - lo + 31) / 32;
      const long long idx = lo + (long long)(lane + 1) * step;
      const bool le = idx < hi && (long long)work_seg[idx] <= p0;
      const int cnt = __popc(__ballot_sync(b200::full_mask, le));  // true for a prefix of the lanes
      lo += (long long)cnt * step;
      hi = lo + step < hi ? lo + step : hi;
    }
    long long j0 = lo;
    for (long long round = first_round; round < last_round; ++round) {
      const long long r = round * round_quads;
      const long long rend = r + round_quads < total ? r + round_quads : total;
      int n_seg = 0;
#pragma unroll 1
      for (int k = 0; k < warp_table_cap; k += 32) {
        const long long jj = j0 + k + lane;
        long long s = LLONG_MAX;
        if (jj < n_items) s = (long long)work_seg[jj];
        const bool in = s < rend;
        if (in) {
          const edge_t b = work_beg[jj];
          const int slot = k + int(lane);
          T.rel[slot] = edge_t(s > r ? s - r : 0);
          T.qoff[slot] = edge_t((long long)(b >> 2) - (s - r));
          T.beg[slot] = b;
          T.end[slot] = work_end[jj];
          T.src[slot] = work_src[jj];
        }
        const unsigned votes = __ballot_sync(b200::full_mask, in);
        n_seg += __popc(votes);
        if (votes != b200::full_mask) break;
      }
      __syncwarp();
      expand_round<has_output, policy, stage_cap>(A, op, T.rel, T.qoff, T.beg, T.end, T.src, n_seg, edge_t(0),
                                                  int(rend - r), sbuf, staged, output, counters, capacity, visited);
      {  // the next round starts in this round's last list when that list continues past rend
        const int last = n_seg - 1;
        const long long last_stop = r - (long long)T.qoff[last] + (long long)((T.end[last] - 1) >> 2) + 1;
        j0 += last_stop > rend ? last : last + 1;
      }
      __syncwarp();  // table reuse
    }
  }
  if constexpr (has_output) stage_flush(sbuf, staged, output, counters + scratch_t::out_count, capacity);
}

// ------------------------------------------------------------------------------------------------------------
// CTA-wide segment table (block_mapped tiles and the single-launch small-frontier kernel)

template <typename vertex_t, typename edge_t, int ITEMS>
struct cta_table_t {
  edge_t rel[ITEMS + 1];
  edge_t qoff[ITEMS];
  edge_t beg[ITEMS];
  edge_t end[ITEMS];
  vertex_t src[ITEMS];
  edge_t scan_e[cta_threads / 32 + 1];
  unsigned scan_u[cta_threads / 32 + 1];
  int ticket;
};

/// Builds the table from PER_THREAD (vertex, beg, end) triples held in blocked order by the CTA's threads.
/// Returns (uniform) the number of segments and quads. Ends with a barrier.
template <int PER_THREAD, int ITEMS, typename vertex_t, typename edge_t>
__device__ __forceinline__ void build_cta_table(cta_table_t<vertex_t, edge_t, ITEMS>& T, const vertex_t (&v)[PER_THREAD],
                                                const edge_t (&beg)[PER_THREAD], const edge_t (&end)[PER_THREAD],
                                                unsigned& n_seg, edge_t& n_quads) {
  unsigned my_items = 0;
  edge_t my_quads = 0;
  edge_t nq[PER_THREAD];
#pragma unroll
  for (int k = 0; k < PER_THREAD; ++k) {
    nq[k] = end[k] > beg[k] ? ((end[k] - 1) >> 2) - (beg[k] >> 2) + 1 : edge_t(0);
    my_items += nq[k] > 0;
    my_quads += nq[k];
  }
  unsigned at = b200::cta_exclusive_sum<cta_threads, unsigned>(my_items, n_seg, T.scan_u);
  edge_t run = b200::cta_exclusive_sum<cta_threads, edge_t>(my_quads, n_quads, T.scan_e);
#pragma unroll
  for (int k = 0; k < PER_THREAD; ++k)
    if (nq[k] > 0) {
      T.rel[at] = run;
      T.qoff[at] = (beg[k] >> 2) - run;
      T.beg[at] = beg[k];
      T.end[at] = end[k];
      T.src[at] = v[k];
      ++at;
      run += nq[k];
    }
  __syncthreads();
}

// block_mapped: a CTA owns 256 consecutive frontier items (dynamic tickets) and every quad under them; its warps
// take the tile's rounds round-robin. Items with degree >= big_degree go to the TMA-staged hub kernel.
template <bool graph_input, bool has_output, bool guard, visit_t policy, typename vertex_t, typename edge_t,
          typename weight_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads, 4)
    block_mapped_quad_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                             const vertex_t* __restrict__ input, std::size_t input_size, vertex_t* __restrict__ output,
                             counter_t* counters, counter_t capacity, unsigned* __restrict__ visited,
                             vertex_t* __restrict__ big_list) {
  __shared__ cta_table_t<vertex_t, edge_t, cta_threads> T;
  __shared__ warp_stage_t<vertex_t> stages[has_output ? quad_warps : 1];
  if constexpr (has_output && guard)
    if (!output_fits(counters, capacity)) return;
  const unsigned warp = b200::warp_id();
  vertex_t* sbuf = stages[has_output ? warp : 0].buf;
  unsigned staged = 0;
  const std::size_t n_tiles = (input_size + cta_threads - 1) / cta_threads;
  for (;;) {
    if (threadIdx.x == 0) T.ticket = int(atomicAdd(counters + scratch_t::ticket, counter_t(1)));
    __syncthreads();
    const std::size_t tile = std::size_t(T.ticket);
    if (tile >= n_tiles) break;
    vertex_t v[1];
    edge_t beg[1], end[1];
    load_row<graph_input>(A.offsets, input, tile * cta_threads + threadIdx.x, input_size, v[0], beg[0], end[0]);
    if (big_list && end[0] - beg[0] >= edge_t(big_degree)) {  // hub: hand it to the grid-wide kernel
      const counter_t at = atomicAdd(counters + scratch_t::big_count, counter_t(1));
      big_list[at] = v[0];
      end[0] = beg[0];
    }
    unsigned n_seg;
    edge_t n_quads;
    build_cta_table<1>(T, v, beg, end, n_seg, n_quads);
    const edge_t rounds = (n_quads + round_quads - 1) / round_quads;
    for (edge_t round = edge_t(warp); round < rounds; round += quad_warps) {
      const edge_t pos0 = round * round_quads;
      const edge_t left = n_quads - pos0;
      expand_round<has_output, policy, stage_cap>(A, op, T.rel, T.qoff, T.beg, T.end, T.src, int(n_seg), pos0,
                                                  int(left < edge_t(round_quads) ? left : edge_t(round_quads)), sbuf,
                                                  staged, output, counters, capacity, visited);
    }
    __syncthreads();  // table and ticket reuse
  }
  if constexpr (has_output) stage_flush(sbuf, staged, output, counters + scratch_t::out_count, capacity);
}

// merge_path for small frontiers (nf <= small_items): ONE launch. Every CTA builds the whole table in shared
// memory (row bounds are L2 hits) and the grid's warps take the rounds round-robin.
template <bool graph_input, bool has_output, visit_t policy, typename vertex_t, typename edge_t, typename weight_t,
          typename operator_t>
__global__ void __launch_bounds__(cta_threads, 4)
    merge_path_small_quad_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                                 const vertex_t* __restrict__ input, int input_size, vertex_t* __restrict__ output,
                                 counter_t* counters, counter_t capacity, unsigned* __restrict__ visited) {
  constexpr int per_thread = small_items / cta_threads;
  __shared__ cta_table_t<vertex_t, edge_t, small_items> T;
  __shared__ warp_stage_t<vertex_t> stages[has_output ? quad_warps : 1];
  __shared__ unsigned long long s_edges;
  if (threadIdx.x == 0) s_edges = 0;
  __syncthreads();
  vertex_t v[per_thread];
  edge_t beg[per_thread], end[per_thread];
  unsigned long long my_edges = 0;
#pragma unroll
  for (int k = 0; k < per_thread; ++k) {
    const int i = int(threadIdx.x) * per_thread + k;  // blocked order keeps the table in frontier order
    load_row<graph_input>(A.offsets, input, i, input_size, v[k], beg[k], end[k]);
    my_edges += (unsigned long long)(end[k] - beg[k]);
  }
  my_edges = b200::warp_sum(my_edges);
  if (b200::lane_id() == 0 && my_edges) atomicAdd(&s_edges, my_edges);
  unsigned n_seg;
  edge_t n_quads;
  build_cta_table<per_thread>(T, v, beg, end, n_seg, n_quads);  // ends with a barrier: s_edges is complete
  const counter_t total_edges = counter_t(s_edges);
  if (blockIdx.x == 0 && threadIdx.x == 0) counters[scratch_t::work_total] = total_edges;
  if constexpr (has_output) {
    if (total_edges > capacity) {  // every CTA computes the same total, so all of them leave
      if (blockIdx.x == 0 && threadIdx.x == 0) counters[scratch_t::overflow] = total_edges;
      return;
    }
  }
  const unsigned warp = b200::warp_id();
  vertex_t* sbuf = stages[has_output ? warp : 0].buf;
  unsigned staged = 0;
  const edge_t rounds = (n_quads + round_quads - 1) / round_quads;
  for (edge_t round = edge_t(blockIdx.x) * quad_warps + edge_t(warp); round < rounds;
       round += edge_t(gridDim.x) * quad_warps) {
    const edge_t pos0 = round * round_quads;
    const edge_t left = n_quads - pos0;
    expand_round<has_output, policy, stage_cap>(A, op, T.rel, T.qoff, T.beg, T.end, T.src, int(n_seg), pos0,
                                                int(left < edge_t(round_quads) ? left : edge_t(round_quads)), sbuf,
                                                staged, output, counters, capacity, visited);
  }
  if constexpr (has_output) stage_flush(sbuf, staged, output, counters + scratch_t::out_count, capacity);
}

// warp_mapped over quads: one warp per list item (bucketing's medium bin), lanes stride the list's quads.
template <bool has_output, visit_t policy, typename vertex_t, typename edge_t, typename weight_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads, 4)
    warp_mapped_quad_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                            const vertex_t* __restrict__ list, const counter_t* size_ptr, vertex_t* __restrict__ output,
                            counter_t* counters, counter_t capacity, unsigned* __restrict__ visited) {
  __shared__ warp_stage_t<vertex_t> stages[has_output ? quad_warps : 1];
  if constexpr (has_output)
    if (!output_fits(counters, capacity)) return;
  const std::size_t count = std::size_t(*size_ptr);
  const unsigned lane = b200::lane_id(), warp = b200::warp_id();
  const std::size_t warps = std::size_t(gridDim.x) * quad_warps;
  vertex_t* sbuf = stages[has_output ? warp : 0].buf;
  unsigned staged = 0;
  for (std::size_t item = std::size_t(blockIdx.x) * quad_warps + warp; item < count; item += warps) {
    const vertex_t v = list[item];
    const edge_t beg = A.offsets[v], end = A.offsets[v + 1];
    if (end <= beg) continue;  // warp-uniform
    const edge_t q_first = beg >> 2, q_stop = ((end - 1) >> 2) + 1;
    for (edge_t q0 = q_first; q0 < q_stop; q0 += round_quads) {
      vertex_t src[quads_per_lane];
      edge_t e0[quads_per_lane], lo[quads_per_lane], hi[quads_per_lane];
      unsigned have = 0;
      vertex_t nbr[round_items];
#pragma unroll
      for (int q = 0; q < quads_per_lane; ++q) {
        const edge_t g = q0 + edge_t(q * 32 + int(lane));
        src[q] = v, e0[q] = g * 4, lo[q] = beg, hi[q] = end;
        if (g < q_stop) have |= 1u << q;
      }
#pragma unroll
      for (int q = 0; q < quads_per_lane; ++q) {
        vertex_t c[4] = {0, 0, 0, 0};
        if (have & (1u << q)) load_quad(A.indices, e0[q], A.m, c);
#pragma unroll
        for (int i = 0; i < 4; ++i) nbr[4 * q + i] = c[i];
      }
      const unsigned live = live_mask<quads_per_lane>(have, e0, lo, hi);
      const unsigned keep = visit_items<policy, quads_per_lane>(A, op, nbr, live, src, e0, visited);
      if constexpr (has_output)
        stage_append<stage_cap>(nbr, keep, sbuf, staged, output, counters + scratch_t::out_count, capacity);
    }
  }
  if constexpr (has_output) stage_flush(sbuf, staged, output, counters + scratch_t::out_count, capacity);
}

// ------------------------------------------------------------------------------------------------------------
// TMA (cp.async.bulk) + mbarrier helpers

__device__ __forceinline__ unsigned smem_address(const void* p) { return unsigned(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbarrier_init(unsigned long long* bar, unsigned arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_address(bar)), "r"(arrivals) : "memory");
}
/// Makes the barrier initialisation visible to the async (TMA) proxy.
__device__ __forceinline__ void mbarrier_init_fence() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbarrier_arrive_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_address(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbarrier_wait(unsigned long long* bar, unsigned parity) {
  unsigned done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_address(bar)), "r"(parity)
        : "memory");
  } while (!done);
}
/// 1-D bulk copy global -> shared through the TMA unit; completion is signalled on `bar` as `bytes` of transaction
/// count. dst, src and bytes are multiples of 16.
__device__ __forceinline__ void bulk_copy_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_address(dst)),
               "l"(src), "r"(bytes), "r"(smem_address(bar))
               : "memory");
}

/**
 * @brief Grid-wide expansion of the deferred hubs. Each hub's quad range is cut into 512-quad tiles; the tiles of
 * all hubs form one global sequence that is dealt round-robin to the CTAs (tile g -> CTA g mod grid), so the grid
 * stays balanced whatever the degree mix. Hubs are taken 256 at a time: their bounds are loaded by the CTA in
 * parallel and scanned into tile prefixes in shared memory. A tile's 8 KB of column indices are brought into shared
 * memory by ONE cp.async.bulk issued by thread 0 (double buffered: tile k+1 is in flight while tile k is expanded),
 * consumers wait on the stage's mbarrier and read their two quads with 128-bit shared loads.
 */
template <bool has_output, visit_t policy, typename vertex_t, typename edge_t, typename weight_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads, 4)
    big_list_bulk_kernel(const graph::adjacency_t<vertex_t, edge_t, weight_t> A, operator_t op,
                         const vertex_t* __restrict__ big_list, const counter_t* size_ptr,
                         vertex_t* __restrict__ output, counter_t* counters, counter_t capacity,
                         unsigned* __restrict__ visited) {
  static_assert(sizeof(vertex_t) == 4, "bulk tiles hold 4-byte ids");
  __shared__ __align__(128) vertex_t s_col[2][bulk_tile_quads * 4];
  __shared__ __align__(8) unsigned long long s_bar[2];
  __shared__ warp_stage_t<vertex_t> stages[has_output ? quad_warps : 1];
  __shared__ vertex_t s_v[cta_threads];
  __shared__ edge_t s_beg[cta_threads], s_end[cta_threads];
  __shared__ unsigned long long s_first[cta_threads + 1];  // first global tile of each hub of the batch
  __shared__ unsigned long long s_scan[cta_threads / 32 + 1];
  if constexpr (has_output)
    if (!output_fits(counters, capacity)) return;
  const std::size_t count = std::size_t(*size_ptr);
  if (count == 0) return;
  const unsigned warp = b200::warp_id();
  vertex_t* sbuf = stages[has_output ? warp : 0].buf;
  unsigned staged = 0;
  if (threadIdx.x == 0) {
    mbarrier_init(&s_bar[0], 1);
    mbarrier_init(&s_bar[1], 1);
    mbarrier_init_fence();
  }
  __syncthreads();

  struct tile_t {
    vertex_t v;
    edge_t beg, end;    // list bounds (edges)
    edge_t q_first;     // first global quad of the tile
    int n_quads;        // quads in the tile (<= 512)
    int covered;        // elements of the tile delivered by the bulk copy (the array's ragged last quad is not)
  };
  unsigned parity[2] = {0u, 0u};
  unsigned long long tiles_before = 0;  // global tiles of the batches already done
  for (std::size_t batch = 0; batch < count; batch += cta_threads) {
    const int in_batch = int(count - batch < std::size_t(cta_threads) ? count - batch : std::size_t(cta_threads));
    {  // hubs of the batch: bounds in parallel, tile counts scanned
      vertex_t v = 0;
      edge_t b = 0, e = 0;
      if (int(threadIdx.x) < in_batch) {
        v = big_list[batch + threadIdx.x];
        b = A.offsets[v];
        e = A.offsets[v + 1];
      }
      const unsigned long long nq = e > b ? (unsigned long long)(((e - 1) >> 2) - (b >> 2) + 1) : 0ull;
      const unsigned long long tiles = (nq + bulk_tile_quads - 1) / bulk_tile_quads;
      unsigned long long batch_tiles;
      const unsigned long long before = b200::cta_exclusive_sum<cta_threads, unsigned long long>(tiles, batch_tiles, s_scan);
      s_v[threadIdx.x] = v;
      s_beg[threadIdx.x] = b;
      s_end[threadIdx.x] = e;
      s_first[threadIdx.x] = tiles_before + before;
      if (threadIdx.x == cta_threads - 1) s_first[cta_threads] = tiles_before + batch_tiles;
    }
    __syncthreads();
    const unsigned long long batch_end = s_first[cta_threads];
    // this CTA's tiles of the batch: g = first id >= tiles_before congruent to blockIdx.x, then += gridDim.x
    unsigned long long g = tiles_before + (blockIdx.x + gridDim.x - unsigned(tiles_before % gridDim.x)) % gridDim.x;
    auto describe = [&](unsigned long long id, tile_t& out) {
      const int i = b200::upper_segment(s_first, cta_threads, id);  // hub of the batch owning tile `id`
      const long long t = (long long)(id - s_first[i]);
      out.v = s_v[i], out.beg = s_beg[i], out.end = s_end[i];
      const long long item_quads = (long long)(((out.end - 1) >> 2) - (out.beg >> 2) + 1);
      out.q_first = (out.beg >> 2) + edge_t(t * bulk_tile_quads);
      const long long left = item_quads - t * bulk_tile_quads;
      out.n_quads = int(left < bulk_tile_quads ? left : bulk_tile_quads);
      long long avail = ((long long)A.m - (long long)out.q_first * 4) & ~3ll;  // whole quads left in the array
      const long long want = (long long)out.n_quads * 4;
      out.covered = int(want < avail ? want : avail);
    };
    auto issue = [&](const tile_t& tile, int stage) {  // thread 0 only
      const unsigned bytes = unsigned(tile.covered) * 4u;
      mbarrier_arrive_expect_tx(&s_bar[stage], bytes);
      if (bytes) bulk_copy_g2s(&s_col[stage][0], A.indices + (long long)tile.q_first * 4, bytes, &s_bar[stage]);
    };
    tile_t cur, nxt;
    bool have_cur = g < batch_end;
    int stage = 0;
    if (have_cur) {
      describe(g, cur);
      if (threadIdx.x == 0) issue(cur, 0);
    }
    while (have_cur) {
      g += gridDim.x;
      const bool have_nxt = g < batch_end;
      if (have_nxt) {
        describe(g, nxt);
        if (threadIdx.x == 0) issue(nxt, stage ^ 1);
      }
      mbarrier_wait(&s_bar[stage], parity[stage]);
      parity[stage] ^= 1u;

      vertex_t src[quads_per_lane];
      edge_t e0[quads_per_lane], lo[quads_per_lane], hi[quads_per_lane];
      unsigned have = 0;
      vertex_t nbr[round_items];
#pragma unroll
      for (int q = 0; q < quads_per_lane; ++q) {
        const int k = q * cta_threads + int(threadIdx.x);  // thread-consecutive quads: conflict-free 128-bit LDS
        src[q] = cur.v, lo[q] = cur.beg, hi[q] = cur.end;
        e0[q] = (cur.q_first + edge_t(k)) * 4;
        vertex_t c[4] = {0, 0, 0, 0};
        if (k < cur.n_quads) {
          have |= 1u << q;
          if (4 * k + 4 <= cur.covered) {
            const int4 x = *reinterpret_cast<const int4*>(&s_col[stage][4 * k]);  // shared-memory stage, 16-B aligned
            c[0] = vertex_t(x.x), c[1] = vertex_t(x.y), c[2] = vertex_t(x.z), c[3] = vertex_t(x.w);
          } else {
            load_quad(A.indices, e0[q], A.m, c);  // ragged last quad of the array
          }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) nbr[4 * q + i] = c[i];
      }
      const unsigned live = live_mask<quads_per_lane>(have, e0, lo, hi);
      const unsigned keep = visit_items<policy, quads_per_lane>(A, op, nbr, live, src, e0, visited);
      if constexpr (has_output)
        stage_append<stage_cap>(nbr, keep, sbuf, staged, output, counters + scratch_t::out_count, capacity);
      __syncthreads();  // everyone is done with s_col[stage] before it is refilled two tiles from now
      cur = nxt;
      have_cur = have_nxt;
      stage ^= 1;
    }
    tiles_before = batch_end;
    __syncthreads();  // batch tables are rewritten by the next iteration
  }
  if constexpr (has_output) stage_flush(sbuf, staged, output, counters + scratch_t::out_count, capacity);
}

}  // namespace kernels
}  // namespace advance
}  // namespace operators
}  // namespace gunrock
