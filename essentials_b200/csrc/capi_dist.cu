/**
 * @file capi_dist.cu
 * @brief C ABI, multi-GPU: per-level kernels of the 1-D partitioned BFS / SSSP, the peer-memory exchange kernels,
 * and the native drivers (ess_dist_bfs, ess_dist_sssp) that run the whole loop in C++ with one process per GPU.
 */
#include "capi_dispatch.hxx"
#include "capi_frontier.hxx"
#include <gunrock/algorithms/bfs.hxx>
#include <gunrock/algorithms/sssp.hxx>

#include <dlfcn.h>
#include <nccl.h>
#include <vector>

using namespace gunrock;
using gcuda::scratch_t;
using ess::borrowed_frontier_t;

namespace {

// ---- multi-GPU BFS level kernels (bitmaps are global, rows are local) -------------------------------

/// Owner side: candidate word = OR of `n_slices` contributions (stride `slice_stride` words); fresh =
/// candidate & ~visited over the owned words; depth, visited, next-frontier slice, sparse list of fresh local
/// ids, and the two Beamer counters (|fresh|, Σdeg fresh) accumulated into `counts` (device, caller-zeroed).
template <typename edge_t>
__global__ void __launch_bounds__(256)
    absorb_kernel(const edge_t* __restrict__ offsets, unsigned n_local, unsigned first_word, int level,
                  unsigned* candidates, int n_slices, unsigned slice_stride, unsigned* __restrict__ visited_bits,
                  unsigned* __restrict__ next_slice, int* __restrict__ depth_local, int* __restrict__ fresh_list,
                  b200::counter_t* counts, bool consume) {
  // consume: zero every non-zero candidate word after reading it — the peer-memory exchange only stores non-zero
  // words into this inbox, so it must be all-zero again before the next level's senders arrive
  // one THREAD per 32-vertex word (coalesced word streams; a warp-per-word version spent 140 us per level on
  // 1 M mostly empty words at scale-26), one warp-aggregated slot claim per warp trip
  const unsigned n_words = (n_local + 31u) >> 5;
  const unsigned stride = gridDim.x * blockDim.x;
  b200::counter_t edges = 0;
  for (unsigned base = blockIdx.x * blockDim.x; base < n_words; base += stride) {
    const unsigned w = base + threadIdx.x;
    unsigned fresh = 0, seen = 0;
    if (w < n_words) {
      seen = visited_bits[first_word + w];
      unsigned cand = 0;
      for (int p = 0; p < n_slices; ++p) {
        const unsigned x = candidates[std::size_t(p) * slice_stride + w];
        if (consume && x) candidates[std::size_t(p) * slice_stride + w] = 0;
        cand |= x;
      }
      fresh = cand & ~seen;
      next_slice[w] = fresh;
      if (fresh) visited_bits[first_word + w] = seen | fresh;
    }
    const unsigned mine = __popc(fresh);
    const unsigned incl = b200::warp_inclusive_sum(mine);
    const unsigned total = __shfl_sync(b200::full_mask, incl, 31);
    if (total == 0) continue;  // warp-uniform
    b200::counter_t at = 0;
    if (b200::lane_id() == 0) at = atomicAdd(counts, b200::counter_t(total));
    at = __shfl_sync(b200::full_mask, at, 0) + (incl - mine);
    while (fresh) {
      const unsigned b = __ffs(fresh) - 1;
      fresh &= fresh - 1;
      const unsigned v = (w << 5) + b;
      if (v < n_local) {
        depth_local[v] = level;
        fresh_list[at] = int(v);
        edges += b200::counter_t(offsets[v + 1] - offsets[v]);
      }
      ++at;
    }
  }
  edges = b200::warp_sum(edges);
  if (b200::lane_id() == 0 && edges) atomicAdd(counts + 1, edges);
}

/// After the per-level all_gather: unpack the P rows of (next-frontier slice | 2 x int64 counters) into the
/// replicated frontier bitmap, fold it into the visited bitmap and collect the counters in one small array.
static __global__ void __launch_bounds__(256)
    merge_gathered_kernel(unsigned* gathered, int world, unsigned slice_words, unsigned* __restrict__ frontier_bits,
                          unsigned* __restrict__ visited_bits, long long* __restrict__ counts_out, bool consume) {
  const unsigned row = slice_words + 4;
  const std::size_t total = std::size_t(world) * slice_words;
  for (std::size_t w = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; w < total;
       w += std::size_t(gridDim.x) * blockDim.x) {
    const unsigned r = unsigned(w / slice_words), k = unsigned(w % slice_words);
    const unsigned bits = gathered[std::size_t(r) * row + k];
    if (consume && bits) gathered[std::size_t(r) * row + k] = 0;  // see absorb_kernel
    frontier_bits[w] = bits;
    if (bits) visited_bits[w] |= bits;
  }
  if (blockIdx.x == 0 && threadIdx.x < 2 * world) {
    const int r = threadIdx.x / 2, c = threadIdx.x % 2;
    long long* cell = reinterpret_cast<long long*>(gathered + std::size_t(r) * row + slice_words) + c;
    counts_out[threadIdx.x] = *cell;
    if (consume) *cell = 0;
  }
}

inline int fail_pull_via_step() {
  return ess::fail("ess_bfs_partition_step: bottom-up levels go through ess_bfs_partition_pull");
}

/// Adds out_count of the operator counter block to the caller's counts[0] and re-zeroes the block. counts[1] (Σdeg
/// of the vertices found) is left alone: the pull kernel does not read row bounds of the vertices it adopts, and only
/// the top-down rule uses Beamer's m_f, which absorb_kernel supplies there.
static __global__ void export_counts_kernel(b200::counter_t* counters, b200::counter_t* counts) {
  if (threadIdx.x == 0) counts[0] += counters[scratch_t::out_count];
  if (threadIdx.x < scratch_t::n_slots) counters[threadIdx.x] = 0;
}

template <typename graph_t>
int partition_pull(ess_context_t ctx, graph_t& G, int64_t row_begin, int32_t level, const uint32_t* d_frontier_bits,
                   uint32_t* d_visited_bits, uint32_t* d_next_slice, int32_t* d_depth_local, int64_t* d_counts) {
  auto* c = ctx->single();
  auto stream = c->stream();
  auto& scratch = c->scratch();
  auto A = graph::adjacency_of<true>(G);  // symmetric graph: the CSC view aliases the owned CSR rows (+ hints)
  int32_t* depth = d_depth_local;
  using edge_t = typename graph_t::edge_type;
  // the destination is an owned, unvisited vertex handled by exactly one thread: adopting it is a plain store
  auto adopt = [depth, level] __device__(int32_t const& src, int32_t const& dst_local, edge_t const& e,
                                         float const& w) -> bool {
    depth[dst_local] = level;
    return true;
  };
  scratch.zero(stream);
  c->profiler().begin(gcuda::profiler_t::pull_step, stream);
  namespace k = operators::advance::kernels;
  // same kernel as the single-GPU bottom-up level: rows, visited and next words are the owned range
  auto kernel = k::pull_chunk_kernel<int32_t, edge_t, float, decltype(adopt)>;
  const std::size_t chunks = ((std::size_t(A.n) + 31) / 32 + k::pull_chunk_words - 1) / k::pull_chunk_words;
  kernel<<<gcuda::full_grid(*c, kernel, (chunks + 7) / 8), 256, 0, stream>>>(
      A, adopt, d_frontier_bits, d_next_slice, d_visited_bits + (row_begin >> 5), scratch.d);
  export_counts_kernel<<<1, 32, 0, stream>>>(scratch.d, reinterpret_cast<b200::counter_t*>(d_counts));
  c->profiler().end(stream, 2);
  scratch.clean = true;  // export_counts_kernel re-zeroed the block
  error::check_last("partition pull");
  return 0;
}

template <typename graph_t>
int partition_step(ess_context_t ctx, graph_t& G, int64_t row_begin, int64_t n_global, int pull,
                   const uint32_t* d_frontier_bits, const uint32_t* d_visited_bits, uint32_t* d_candidate_bits,
                   const int32_t* d_frontier_list, int64_t frontier_count) {
  using edge_t = typename graph_t::edge_type;
  auto* c = ctx->single();
  auto stream = c->stream();
  const auto A = graph::adjacency_of<false>(G);
  const std::size_t n_local = std::size_t(A.n);
  if (pull) return fail_pull_via_step();
  // push: balanced advance over this rank's sparse frontier (local row ids); the operator ORs unvisited
  // neighbours into the global-length candidate bitmap. No host round trip: the caller synchronises once per
  // level through the all_gather that follows.
  cudaMemsetAsync(d_candidate_bits, 0, ((std::size_t(n_global) + 31) / 32) * sizeof(uint32_t), stream);
  if (frontier_count <= 0) return 0;
  borrowed_frontier_t<edge_t> in, out;
  in.ptr = const_cast<int32_t*>(d_frontier_list);
  in.count = in.cap = std::size_t(frontier_count);
  static thread_local memory::device_array_t<edge_t> segments;  // merge-path work offsets, reused across levels
  const unsigned* visited = d_visited_bits;
  unsigned* candidate = d_candidate_bits;
  auto op = [visited, candidate] __device__(int32_t const& src, int32_t const& nbr, edge_t const& e,
                                            float const& w) -> bool {
    const unsigned u = unsigned(nbr), bit = 1u << (u & 31u);
    if (!(visited[u >> 5] & bit) && !(candidate[u >> 5] & bit)) atomicOr(candidate + (u >> 5), bit);
    return false;
  };
  // owner-only visited set (peer-memory driver): every neighbour is a candidate, its owner filters (absorb_kernel)
  auto op_unfiltered = [candidate] __device__(int32_t const& src, int32_t const& nbr, edge_t const& e,
                                              float const& w) -> bool {
    const unsigned u = unsigned(nbr), bit = 1u << (u & 31u);
    if (!(candidate[u >> 5] & bit)) atomicOr(candidate + (u >> 5), bit);
    return false;
  };
  using namespace operators;
  auto& scratch = c->scratch();
  const bool was_async = scratch.async_when_no_output;
  scratch.async_when_no_output = true;
  if (visited)
    advance::execute<load_balance_t::merge_path, advance_direction_t::forward, advance_io_type_t::vertices,
                     advance_io_type_t::none>(G, op, &in, &out, segments, *ctx->ctx);
  else
    advance::execute<load_balance_t::merge_path, advance_direction_t::forward, advance_io_type_t::vertices,
                     advance_io_type_t::none>(G, op_unfiltered, &in, &out, segments, *ctx->ctx);
  scratch.async_when_no_output = was_async;
  return 0;
}


// ---- 1-D partitioned SSSP ------------------------------------------------------------------------
// Every rank keeps a full-length `replica` of tentative distances. Owned entries are exact after each exchange;
// the others are only this rank's best candidates so far (a pruning bound: a candidate that does not beat it
// was already sent). A relaxation round = relax (atomic min into the replica) -> reduce_scatter(min) so each
// owner receives the best candidate for its rows -> collect (owned rows whose distance dropped form the next
// active list).

/// Relax the out-edges of this rank's active rows (LOCAL row ids): replica[nbr] = min(replica[nbr], dist[src] + w).
template <typename graph_t>
int partition_relax(ess_context_t ctx, graph_t& G, const int32_t* d_active_list, int64_t active_count,
                    const float* d_dist_local, float* d_replica, unsigned* d_dirty_chunks = nullptr) {
  using edge_t = typename graph_t::edge_type;
  if (active_count <= 0) return 0;
  auto* c = ctx->single();
  borrowed_frontier_t<edge_t> in, out;
  in.ptr = const_cast<int32_t*>(d_active_list);
  in.count = in.cap = std::size_t(active_count);
  static thread_local memory::device_array_t<edge_t> segments;
  const float* dist_local = d_dist_local;
  float* replica = d_replica;
  // dirty (optional): one word per 1024 replica entries, raised when an entry of the chunk was lowered — the
  // owners' fused reduce+collect only fetches chunks a peer actually touched
  unsigned* dirty = d_dirty_chunks;
  auto op = [dist_local, replica, dirty] __device__(int32_t const& src, int32_t const& nbr, edge_t const& e,
                                                    float const& w) -> bool {
    const float nd = dist_local[src] + w;
    if (nd < replica[nbr]) {  // the plain read only prunes
      const float old = math::atomic::min(replica + nbr, nd);
      if (dirty && nd < old && !dirty[unsigned(nbr) >> 10]) dirty[unsigned(nbr) >> 10] = 1u;
    }
    return false;
  };
  using namespace operators;
  auto& scratch = c->scratch();
  const bool was_async = scratch.async_when_no_output;
  scratch.async_when_no_output = true;
  advance::execute<load_balance_t::merge_path, advance_direction_t::forward, advance_io_type_t::vertices,
                   advance_io_type_t::none>(G, op, &in, &out, segments, *ctx->ctx);
  scratch.async_when_no_output = was_async;
  return 0;
}

/// Owner side after the exchange: rows whose reduced candidate beats the stored distance adopt it and join the
/// next active list; counts[0] += rows, counts[1] += their out-degrees. 4 rows per thread, one atomic per CTA.
template <typename edge_t>
static __global__ void __launch_bounds__(256)
    sssp_collect_kernel(const edge_t* __restrict__ offsets, unsigned n_local, const float* __restrict__ reduced,
                        float* __restrict__ dist_local, int* __restrict__ active_list, b200::counter_t* counts) {
  __shared__ b200::counter_t sm[256 / 32 + 4];
  b200::counter_t edges = 0;
  const unsigned per_cta = 256 * 4;
  for (unsigned base = blockIdx.x * per_cta; base < n_local; base += gridDim.x * per_cta) {
    const unsigned first = base + threadIdx.x * 4;
    int rows[4];
    unsigned keep = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const unsigned v = first + i;
      rows[i] = int(v);
      if (v < n_local) {
        const float r = reduced[v];
        if (r < dist_local[v]) {
          dist_local[v] = r;
          keep |= 1u << i;
          edges += b200::counter_t(offsets[v + 1] - offsets[v]);
        }
      }
    }
    b200::cta_append<256, 4>(rows, keep, active_list, counts, b200::counter_t(n_local), sm);
  }
  edges = b200::warp_sum(edges);
  if (b200::lane_id() == 0 && edges) atomicAdd(counts + 1, edges);
}

template <typename graph_t>
int partition_collect(ess_context_t ctx, graph_t& G, const float* d_reduced, float* d_dist_local,
                      int32_t* d_active_list, int64_t* d_counts) {
  auto* c = ctx->single();
  const unsigned n_local = unsigned(G.get_number_of_vertices());
  if (n_local == 0) return 0;
  c->profiler().begin(gcuda::profiler_t::dense_state, c->stream());
  sssp_collect_kernel<<<gcuda::persistent_grid(*c, (std::size_t(n_local) + 1023) / 1024, 8), 256, 0, c->stream()>>>(
      graph::adjacency_of<false>(G).offsets, n_local, d_reduced, d_dist_local, d_active_list,
      reinterpret_cast<b200::counter_t*>(d_counts));
  c->profiler().end(c->stream(), 1);
  error::check_last("partition collect");
  return 0;
}

}  // namespace

extern "C" {

int ess_bfs_partition_step(ess_context_t ctx, ess_graph_t g, int64_t row_begin, int64_t n_global, int pull,
                           const uint32_t* d_frontier_bits, const uint32_t* d_visited_bits,
                           uint32_t* d_candidate_bits, const int32_t* d_frontier_list, int64_t frontier_count) {
  ESS_TRY
  if (!ctx || !g) return ess::fail("ess_bfs_partition_step: null argument");
  if (row_begin % 32) return ess::fail("ess_bfs_partition_step: row_begin must be a multiple of 32");
  ESS_WITH_GRAPH(g, G, {
    return partition_step(ctx, G, row_begin, n_global, pull, d_frontier_bits, d_visited_bits, d_candidate_bits,
                          d_frontier_list, frontier_count);
  })
  ESS_CATCH
}

int ess_bfs_partition_pull(ess_context_t ctx, ess_graph_t g, int64_t row_begin, int32_t level,
                           const uint32_t* d_frontier_bits, uint32_t* d_visited_bits, uint32_t* d_next_slice,
                           int32_t* d_depth_local, int64_t* d_counts) {
  ESS_TRY
  if (!ctx || !g || !d_counts) return ess::fail("ess_bfs_partition_pull: null argument");
  if (row_begin % 32) return ess::fail("ess_bfs_partition_pull: row_begin must be a multiple of 32");
  if (!g->has_csc) return ess::fail("ess_bfs_partition_pull: the partition must be created symmetric (CSC view)");
  ESS_WITH_GRAPH(g, G, {
    return partition_pull(ctx, G, row_begin, level, d_frontier_bits, d_visited_bits, d_next_slice, d_depth_local,
                          d_counts);
  })
  ESS_CATCH
}

int ess_bfs_merge_gathered(ess_context_t ctx, const uint32_t* d_gathered, int32_t world, int64_t slice_words,
                           uint32_t* d_frontier_bits, uint32_t* d_visited_bits, int64_t* d_counts_out) {
  ESS_TRY
  if (!ctx || !d_gathered || !d_counts_out) return ess::fail("ess_bfs_merge_gathered: null argument");
  if (world < 1 || world > 128) return ess::fail("ess_bfs_merge_gathered: world size out of range");
  auto* c = ctx->single();
  const std::size_t total = std::size_t(world) * std::size_t(slice_words);
  merge_gathered_kernel<<<gcuda::persistent_grid(*c, (total + 255) / 256, 8), 256, 0, c->stream()>>>(
      const_cast<uint32_t*>(d_gathered), world, unsigned(slice_words), d_frontier_bits, d_visited_bits,
      reinterpret_cast<long long*>(d_counts_out), false);
  error::check_last("merge gathered");
  return 0;
  ESS_CATCH
}

int ess_bfs_absorb(ess_context_t ctx, ess_graph_t g, int64_t row_begin, int32_t level, const uint32_t* d_candidates,
                   int32_t n_slices, int64_t slice_stride_words, uint32_t* d_visited_bits, uint32_t* d_next_slice,
                   int32_t* d_depth_local, int32_t* d_fresh_list, int64_t* d_counts) {
  ESS_TRY
  if (!ctx || !g || !d_candidates || !d_counts) return ess::fail("ess_bfs_absorb: null argument");
  auto* c = ctx->single();
  auto stream = c->stream();
  const unsigned n_local = unsigned(g->n);
  const unsigned grid = gcuda::persistent_grid(*c, ((std::size_t(n_local) + 31) / 32 + 255) / 256, 8);
  auto* counts = reinterpret_cast<b200::counter_t*>(d_counts);
  c->profiler().begin(gcuda::profiler_t::dense_state, stream);
  if (g->offset_bits == 64)
    absorb_kernel<int64_t><<<grid, 256, 0, stream>>>(g->g64.get_row_offsets(), n_local, unsigned(row_begin >> 5), level,
                                                      const_cast<uint32_t*>(d_candidates), n_slices,
                                                      unsigned(slice_stride_words), d_visited_bits, d_next_slice,
                                                      d_depth_local, d_fresh_list, counts, false);
  else
    absorb_kernel<int32_t><<<grid, 256, 0, stream>>>(g->g32.get_row_offsets(), n_local, unsigned(row_begin >> 5), level,
                                                      const_cast<uint32_t*>(d_candidates), n_slices,
                                                      unsigned(slice_stride_words), d_visited_bits, d_next_slice,
                                                      d_depth_local, d_fresh_list, counts, false);
  c->profiler().end(stream);
  error::check_last("absorb");
  return 0;
  ESS_CATCH
}

}  // extern "C"

// =====================================================================================================
// Native multi-GPU BFS driver: the whole level loop of the 1-D partitioned, direction-optimising BFS runs in
// C++ with NCCL called directly (one process per GPU). Same logic, step for step, as
// essentials_b200/dist.py::PartitionedBFS (which stays the gloo-testable statement of the host logic); this
// removes the Python/torch dispatch from the per-level critical path (~150 us -> ~50 us per level).
// NCCL is resolved at run time from the libnccl the process already loaded (torch's), so the library has no
// link-time dependency on it.
// =====================================================================================================
namespace {

struct nccl_api_t {
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*ReduceScatter)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t,
                                cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
};

nccl_api_t& nccl() {
  static nccl_api_t api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL | RTLD_NOLOAD);  // already loaded by torch
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    auto sym = [&](const char* name) { return h ? dlsym(h, name) : dlsym(RTLD_DEFAULT, name); };
    api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
    api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
    api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
    api.ReduceScatter = (decltype(api.ReduceScatter))sym("ncclReduceScatter");
    api.Send = (decltype(api.Send))sym("ncclSend");
    api.Recv = (decltype(api.Recv))sym("ncclRecv");
    api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
    api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
    api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
    api.ok = api.CommInitRank && api.CommDestroy && api.AllGather && api.AllReduce && api.ReduceScatter && api.Send &&
             api.Recv &&
             api.GroupStart && api.GroupEnd && api.GetUniqueId && api.GetErrorString;
  }
  return api;
}

void nccl_check(ncclResult_t r, const char* what) {
  if (r != ncclSuccess)
    throw error::exception_t(std::string(what) + ": " + (nccl().GetErrorString ? nccl().GetErrorString(r) : "NCCL error"));
}

/// isolated (degree-0) vertices of the owned range as a bitmap slice.
template <typename edge_t>
__global__ void __launch_bounds__(256)
    isolated_slice_kernel(const edge_t* __restrict__ offsets, unsigned n_local, unsigned* __restrict__ slice) {
  const unsigned lane = b200::lane_id();
  const unsigned n_words = (n_local + 31u) >> 5;
  const unsigned warps = (gridDim.x * blockDim.x) >> 5;
  for (unsigned w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_words; w += warps) {
    const unsigned v = (w << 5) + lane;
    const bool iso = v >= n_local || offsets[v + 1] == offsets[v];
    const unsigned bits = __ballot_sync(b200::full_mask, iso);
    if (lane == 0) slice[w] = bits;
  }
}

/// Start state of one BFS: frontier = {source}; visited = isolated ∪ {source}; owner seeds depth and its list.
template <typename edge_t>
__global__ void seed_kernel(const edge_t* __restrict__ offsets, long long source, long long row_begin,
                            unsigned n_local, unsigned* frontier_bits, unsigned* visited_bits, int* depth_local,
                            int* fresh_list, long long* seed_counts) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const unsigned bit = 1u << (unsigned(source) & 31u);
  frontier_bits[source >> 5] = bit;
  visited_bits[source >> 5] |= bit;
  seed_counts[0] = 0;
  seed_counts[1] = 0;
  const long long local = source - row_begin;
  if (local >= 0 && local < (long long)n_local) {
    depth_local[local] = 0;
    fresh_list[0] = int(local);
    seed_counts[0] = 1;
    seed_counts[1] = (long long)(offsets[local + 1] - offsets[local]);
  }
}


// ---- peer-memory exchange (NVLink loads/stores instead of NCCL collectives) --------------------------
// Every rank exposes one IPC-mapped window: [inbox: P candidate slices][gather 0 | gather 1: P rows of
// (next-frontier slice | counters)][flags A: P words][flags B: P words]. A sender copies its data straight
// into the receivers' windows with 8-byte stores (only the non-zero ones: receivers clear what they consume, so
// sparse levels cost almost no NVLink traffic) and then raises flag[sender] = epoch in each of them (last
// CTA, after a system-scope fence); the receiver's stream waits on its own flags before the consuming kernel.
// Epochs only grow, so flags are never reset; the gather area is double-buffered by level parity because a
// fast peer may already deliver level L+1 while this rank still merges level L.
constexpr int max_peers = 16;
struct peers_t {
  unsigned* base[max_peers];
};

/// After this thread's stores: fence, count the CTA in; the last CTA publishes `epoch` to every peer's flag word.
__device__ __forceinline__ void raise_flags_when_grid_done(const peers_t& peers, int world, int rank,
                                                           std::size_t flag_off, unsigned epoch, unsigned* done) {
  __shared__ bool last;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(done, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence_system();
  if (threadIdx.x < unsigned(world)) {
    volatile unsigned* flag = peers.base[threadIdx.x] + flag_off + rank;
    *flag = epoch;
  }
  if (threadIdx.x == 0) *done = 0;
}

/// all_to_all: slice p (slice_words words) of `src` lands in peer p's inbox row `rank`.
static __global__ void __launch_bounds__(256)
    peer_scatter_kernel(const unsigned* __restrict__ src, peers_t peers, int world, int rank, unsigned slice_words,
                        std::size_t inbox_off, std::size_t flag_off, unsigned epoch, unsigned* done) {
  const std::size_t pairs_per_slice = slice_words / 2, total = pairs_per_slice * world;
  const uint2* in = reinterpret_cast<const uint2*>(src);
  for (std::size_t i = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += std::size_t(gridDim.x) * blockDim.x) {
    const int p = int(i / pairs_per_slice);
    const std::size_t k = i - std::size_t(p) * pairs_per_slice;
    const uint2 v = in[i];
    if (v.x | v.y)  // receivers keep their inbox all-zero between levels (absorb_kernel, consume)
      reinterpret_cast<uint2*>(peers.base[p] + inbox_off + std::size_t(rank) * slice_words)[k] = v;
  }
  raise_flags_when_grid_done(peers, world, rank, flag_off, epoch, done);
}

static unsigned long long peer_timeout_ns() {
  return (unsigned long long)(ess::dist_peer_timeout_ms() > 0 ? ess::dist_peer_timeout_ms() : 4000) * 1000000ull;
}

/// Wall-clock nanoseconds (independent of the SM clock, unlike clock64).
static __device__ __forceinline__ unsigned long long wall_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

/// Stream-side wait: returns once every peer's flag reached `epoch`; gives up after `timeout_ns` (ess_tune
/// "dist_peer_timeout_ms", default 4 s: a dead peer must not hang the box) and reports through *timed_out (mapped
/// host memory) — the host then poisons the handle, see ess_dist_s::poisoned.
static __global__ void peer_wait_kernel(const unsigned* flags, int world, unsigned epoch, unsigned* timed_out,
                                        unsigned long long timeout_ns) {
  if (threadIdx.x >= unsigned(world)) return;
  const volatile unsigned* flag = flags + threadIdx.x;
  const unsigned long long start = wall_ns();
  while (int(*flag - epoch) < 0) {
    if (wall_ns() - start > timeout_ns) {
      *timed_out = 1u + threadIdx.x;
      break;
    }
    __nanosleep(64);
  }
  __threadfence_system();
}


/// Flag-only signal (no payload pushed): "my kernels before this point are done for epoch".
static __global__ void peer_signal_kernel(peers_t peers, int world, int rank, std::size_t flag_off, unsigned epoch) {
  if (threadIdx.x < unsigned(world)) {
    __threadfence_system();
    volatile unsigned* flag = peers.base[threadIdx.x] + flag_off + rank;
    *flag = epoch;
  }
}

/// all_gather of the level's result, second form: the slice goes into row `rank` of the peers' BITS area (rows of
/// exactly slice_words, so the area IS the replicated next-frontier bitmap — no unpacking pass) and the two Beamer
/// counters into row `rank` of their COUNTS area. Zero words / counters are skipped (receivers keep both all-zero).
static __global__ void __launch_bounds__(256)
    peer_publish_level_kernel(const unsigned* __restrict__ slice, const unsigned* __restrict__ counters4, peers_t peers,
                              int world, int rank, unsigned slice_words, std::size_t bits_off, std::size_t cnt_off,
                              std::size_t flag_off, unsigned epoch, unsigned* done) {
  const std::size_t pairs = slice_words / 2, total = pairs * world;
  const uint2* in = reinterpret_cast<const uint2*>(slice);
  for (std::size_t i = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += std::size_t(gridDim.x) * blockDim.x) {
    const int p = int(i / pairs);
    const std::size_t k = i - std::size_t(p) * pairs;
    const uint2 v = in[k];
    if (v.x | v.y) reinterpret_cast<uint2*>(peers.base[p] + bits_off + std::size_t(rank) * slice_words)[k] = v;
  }
  if (blockIdx.x == 0 && threadIdx.x < unsigned(world) * 4u) {
    const int p = threadIdx.x >> 2, k = threadIdx.x & 3;
    const unsigned v = counters4[k];
    if (v) peers.base[p][cnt_off + std::size_t(rank) * 4 + k] = v;
  }
  raise_flags_when_grid_done(peers, world, rank, flag_off, epoch, done);
}

/// Stream-side wait for every peer's level data, then the level's ONE host hand-off: the P x 2 counters go to
/// mapped pinned host memory (and are cleared in the window), followed by the sequence word the host spins on —
/// a PCIe write instead of cudaMemcpyAsync(D2H) + cudaStreamSynchronize.
static __global__ void peer_wait_publish_kernel(const unsigned* flags, int world, unsigned epoch, unsigned* timed_out,
                                                unsigned* cnt_area, volatile long long* host_counts,
                                                unsigned long long sequence, unsigned long long timeout_ns) {
  if (threadIdx.x < unsigned(world)) {
    const volatile unsigned* flag = flags + threadIdx.x;
    const unsigned long long start = wall_ns();
    while (int(*flag - epoch) < 0) {
      if (wall_ns() - start > timeout_ns) {
        *timed_out = 1u + threadIdx.x;
        break;
      }
      __nanosleep(32);
    }
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < unsigned(world) * 2u) {
    volatile long long* cell = reinterpret_cast<volatile long long*>(cnt_area) + threadIdx.x;
    host_counts[threadIdx.x] = *cell;
    *cell = 0;
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) host_counts[2 * max_peers] = (long long)sequence;
}

struct replicas_t {
  const float* value[max_peers];     ///< every rank's full-length replica of tentative distances
  const unsigned* dirty[max_peers];  ///< its per-1024-entry dirty words
};

/// Partitioned SSSP, owner side, exchange and filter in ONE kernel over peer memory: a CTA takes a 1024-row chunk
/// of the owned range, looks at each peer's dirty word for it, fetches the chunk only from the peers that touched
/// it (float4 loads over NVLink), takes the minimum with the local candidates, and the rows whose distance dropped
/// adopt it and join the next active list. Replaces reduce_scatter(min) + sssp_collect_kernel; late rounds, where
/// few chunks are dirty, move almost nothing.
template <typename edge_t>
static __global__ void __launch_bounds__(256)
    sssp_peer_reduce_collect_kernel(const edge_t* __restrict__ offsets, unsigned n_local, long long row_begin,
                                    replicas_t reps, int world, int rank, float* replica_self,
                                    float* __restrict__ dist_local, int* __restrict__ active_list,
                                    b200::counter_t* counts) {
  __shared__ unsigned s_dirty[max_peers];
  __shared__ b200::counter_t sm[256 / 32 + 4];
  const unsigned chunks = n_local >> 10;  // the caller guarantees n_local % 1024 == 0
  b200::counter_t edges = 0, fetched = 0;
  for (unsigned c = blockIdx.x; c < chunks; c += gridDim.x) {
    const std::size_t global_chunk = std::size_t(row_begin >> 10) + c;
    if (threadIdx.x < unsigned(world))
      s_dirty[threadIdx.x] = int(threadIdx.x) == rank ? 0u : reps.dirty[threadIdx.x][global_chunk];
    __syncthreads();
    // float4 accesses: the replicas and dist_local are allocated by the dist handle itself (the peers' replicas
    // through IPC), never by a caller, and row_begin and v0 are multiples of 1024 and 4
    const unsigned v0 = (c << 10) + threadIdx.x * 4;
    float4 best = *reinterpret_cast<const float4*>(replica_self + row_begin + v0);
    for (int p0 = 0; p0 < world; p0 += 8) {  // all fetches of a batch in flight before the first min
      float4 got[8];
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (p0 + k < world && s_dirty[p0 + k])
          got[k] = *reinterpret_cast<const float4*>(reps.value[p0 + k] + row_begin + v0);
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (p0 + k < world && s_dirty[p0 + k]) {
          best.x = fminf(best.x, got[k].x), best.y = fminf(best.y, got[k].y);
          best.z = fminf(best.z, got[k].z), best.w = fminf(best.w, got[k].w);
          if (threadIdx.x == 0) ++fetched;
        }
    }
    const float4 cur = *reinterpret_cast<const float4*>(dist_local + v0);
    const float b[4] = {best.x, best.y, best.z, best.w}, o[4] = {cur.x, cur.y, cur.z, cur.w};
    int rows[4];
    unsigned keep = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      rows[i] = int(v0 + i);
      if (b[i] < o[i]) {
        keep |= 1u << i;
        edges += b200::counter_t(offsets[v0 + i + 1] - offsets[v0 + i]);
      }
    }
    if (keep) {
      *reinterpret_cast<float4*>(dist_local + v0) = best;                 // best <= cur in every lane
      *reinterpret_cast<float4*>(replica_self + row_begin + v0) = best;   // owned replica entries stay exact
    }
    b200::cta_append<256, 4>(rows, keep, active_list, counts, b200::counter_t(n_local), sm);
  }
  edges = b200::warp_sum(edges);
  if (b200::lane_id() == 0 && edges) atomicAdd(counts + 1, edges);
  if (threadIdx.x == 0 && fetched) atomicAdd(counts + 4, fetched * 4096);  // bytes pulled over NVLink
}

}  // namespace

struct ess_dist_s {
  ess_context_t ctx = nullptr;
  ess_graph_t graph = nullptr;
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1;
  long long n_global = 0, per = 0, m_global = 0, row_begin = 0;
  unsigned wper = 0, words = 0;
  memory::device_array_t<unsigned> frontier_bits, visited_bits, candidate_bits, isolated_bits, send, recv, a2a_recv;
  memory::device_array_t<int> depth_local, fresh_list;
  memory::device_array_t<float> replica, dist_local;  // SSSP state, allocated by the first ess_dist_sssp
  memory::device_array_t<long long> counts_dev;
  long long* counts_host = nullptr;  // pinned
  int levels = 0, pull_levels = 0;
  long long bytes_exchanged = 0;
  // peer-memory window (see peers_t): own allocation + the mapped windows of the other ranks
  unsigned* window = nullptr;
  peers_t peers{};
  bool peer_ready = false;
  std::size_t inbox_off = 0, gather_off[2] = {0, 0}, flag_off[2] = {0, 0};
  std::size_t bits_off[2] = {0, 0}, cnt_off[2] = {0, 0};  // replicated next-frontier bitmap + counters, by parity
  long long* level_counts = nullptr;   // mapped pinned: [2 * max_peers] counters + sequence word
  unsigned long long level_sequence = 0;
  unsigned epoch = 0;
  // SSSP over peer memory: replica + dirty words in one IPC-mapped allocation per rank
  float* replica_window = nullptr;
  replicas_t replicas{};
  bool sssp_peer_tried = false, sssp_peer_ready = false;
  unsigned* done_counter = nullptr;  // device word of raise_flags_when_grid_done
  unsigned* timed_out = nullptr;     // pinned, mapped
  // A peer that missed a level leaves this rank's windows, epochs and counters in an unknown state (the consuming
  // kernels ran on partial data, later flags may still arrive): every later call on the handle fails fast instead of
  // computing on it or waiting on ranks that have moved on. Destroy the handle on every rank and create a new one.
  bool poisoned = false;
  std::shared_ptr<gunrock::gcuda::partition_t> partition;  // NCCL bound to the operator-API partition descriptor
  ~ess_dist_s() {
    for (int p = 0; p < world && p < max_peers; ++p)
      if (p != rank && peers.base[p]) cudaIpcCloseMemHandle(peers.base[p]);
    for (int p = 0; p < world && p < max_peers; ++p)
      if (p != rank && replicas.value[p]) cudaIpcCloseMemHandle(const_cast<float*>(replicas.value[p]));
    if (replica_window) cudaFree(replica_window);
    if (window) cudaFree(window);
    if (done_counter) cudaFree(done_counter);
    if (timed_out) cudaFreeHost(timed_out);
    if (level_counts) cudaFreeHost(level_counts);
    if (counts_host) cudaFreeHost(counts_host);
    if (comm && nccl().CommDestroy) nccl().CommDestroy(comm);
  }
};

extern "C" {

int ess_sssp_partition_relax(ess_context_t ctx, ess_graph_t g, const int32_t* d_active_list, int64_t active_count,
                             const float* d_dist_local, float* d_replica) {
  ESS_TRY
  if (!ctx || !g || !d_dist_local || !d_replica) return ess::fail("ess_sssp_partition_relax: null argument");
  ESS_WITH_GRAPH(g, G, { return partition_relax(ctx, G, d_active_list, active_count, d_dist_local, d_replica); })
  ESS_CATCH
}

int ess_sssp_partition_collect(ess_context_t ctx, ess_graph_t g, const float* d_reduced, float* d_dist_local,
                               int32_t* d_active_list, int64_t* d_counts) {
  ESS_TRY
  if (!ctx || !g || !d_reduced || !d_dist_local || !d_active_list || !d_counts)
    return ess::fail("ess_sssp_partition_collect: null argument");
  ESS_WITH_GRAPH(g, G, { return partition_collect(ctx, G, d_reduced, d_dist_local, d_active_list, d_counts); })
  ESS_CATCH
}

}  // extern "C"

extern "C" {

int ess_nccl_unique_id(void* out_128_bytes) {
  ESS_TRY
  if (!nccl().ok) return ess::fail("NCCL is not loaded in this process");
  ncclUniqueId id;
  nccl_check(nccl().GetUniqueId(&id), "ncclGetUniqueId");
  std::memcpy(out_128_bytes, &id, sizeof(id));
  return 0;
  ESS_CATCH
}

int ess_dist_create(ess_context_t ctx, ess_graph_t g, int rank, int world, int64_t n_global, const void* unique_id,
                    ess_dist_t* out) {
  ESS_TRY
  if (!ctx || !g || !out || !unique_id) return ess::fail("ess_dist_create: null argument");
  if (!nccl().ok) return ess::fail("NCCL is not loaded in this process");
  if (world < 1 || rank < 0 || rank >= world) return ess::fail("ess_dist_create: bad rank/world");
  if (n_global % (64LL * world)) return ess::fail("ess_dist_create: n_global must be a multiple of 64*world");
  if (!g->has_csc) return ess::fail("ess_dist_create: the partition must be created symmetric");
  auto d = std::make_unique<ess_dist_s>();
  d->ctx = ctx;
  d->graph = g;
  d->rank = rank;
  d->world = world;
  d->n_global = n_global;
  d->per = n_global / world;
  if (g->n != d->per) return ess::fail("ess_dist_create: the graph must hold exactly n_global/world rows");
  d->row_begin = d->per * rank;
  d->wper = unsigned(d->per / 32);
  d->words = unsigned(n_global / 32);
  auto* c = ctx->single();
  auto stream = c->stream();
  ncclUniqueId id;
  std::memcpy(&id, unique_id, sizeof(id));
  nccl_check(nccl().CommInitRank(&d->comm, world, id, rank), "ncclCommInitRank");
  d->frontier_bits.resize(d->words);
  d->visited_bits.resize(d->words + 1);
  d->candidate_bits.resize(d->words + 1);
  d->isolated_bits.resize(d->words);
  d->send.resize(d->wper + 4);
  d->recv.resize(std::size_t(world) * (d->wper + 4));
  d->a2a_recv.resize(d->words);
  d->depth_local.resize(std::size_t(d->per));
  d->fresh_list.resize(std::size_t(d->per));
  d->counts_dev.resize(2 * std::size_t(world) + 2);
  error::throw_if_exception(cudaMallocHost(&d->counts_host, (2 * std::size_t(world) + 2) * sizeof(long long)),
                            "pinned counters");
  // replicated map of isolated vertices + global edge count
  const unsigned grid = gcuda::persistent_grid(*c, (std::size_t(d->per) + 255) / 256, 8);
  if (g->offset_bits == 64)
    isolated_slice_kernel<int64_t><<<grid, 256, 0, stream>>>(g->g64.get_row_offsets(), unsigned(d->per), d->send.data());
  else
    isolated_slice_kernel<int32_t><<<grid, 256, 0, stream>>>(g->g32.get_row_offsets(), unsigned(d->per), d->send.data());
  nccl_check(nccl().AllGather(d->send.data(), d->isolated_bits.data(), d->wper, ncclUint32, d->comm, stream), "allgather");
  d->counts_host[0] = g->m;
  cudaMemcpyAsync(d->counts_dev.data(), d->counts_host, sizeof(long long), cudaMemcpyHostToDevice, stream);
  nccl_check(nccl().AllReduce(d->counts_dev.data(), d->counts_dev.data(), 1, ncclInt64, ncclSum, d->comm, stream),
             "allreduce");
  cudaMemcpyAsync(d->counts_host, d->counts_dev.data(), sizeof(long long), cudaMemcpyDeviceToHost, stream);
  c->synchronize();
  d->m_global = d->counts_host[0];
  // peer-memory window: allocate, exchange IPC handles through the communicator, map the peers
  if (world <= max_peers) {
    const std::size_t row = std::size_t(d->wper) + 4;
    d->inbox_off = 0;
    d->gather_off[0] = std::size_t(d->words);
    d->gather_off[1] = d->gather_off[0] + row * world;
    d->flag_off[0] = d->gather_off[1] + row * world;
    d->flag_off[1] = d->flag_off[0] + 32;
    d->bits_off[0] = d->flag_off[1] + 32;
    d->bits_off[1] = d->bits_off[0] + std::size_t(d->words);
    d->cnt_off[0] = d->bits_off[1] + std::size_t(d->words);
    d->cnt_off[1] = d->cnt_off[0] + 4 * std::size_t(max_peers);
    const std::size_t window_words = d->cnt_off[1] + 4 * std::size_t(max_peers);
    cudaIpcMemHandle_t mine;
    bool ok = cudaMalloc(&d->window, window_words * sizeof(unsigned)) == cudaSuccess &&
              cudaMemsetAsync(d->window, 0, window_words * sizeof(unsigned), stream) == cudaSuccess &&
              cudaIpcGetMemHandle(&mine, d->window) == cudaSuccess &&
              cudaMalloc(&d->done_counter, sizeof(unsigned)) == cudaSuccess &&
              cudaMemsetAsync(d->done_counter, 0, sizeof(unsigned), stream) == cudaSuccess &&
              cudaHostAlloc(&d->timed_out, sizeof(unsigned), cudaHostAllocMapped) == cudaSuccess &&
              cudaHostAlloc(&d->level_counts, (2 * max_peers + 1) * sizeof(long long), cudaHostAllocMapped) ==
                  cudaSuccess;
    if (d->level_counts) std::memset(d->level_counts, 0, (2 * max_peers + 1) * sizeof(long long));
    memory::device_array_t<unsigned char> handles(std::size_t(world + 1) * sizeof(cudaIpcMemHandle_t));
    std::vector<cudaIpcMemHandle_t> all(world);
    if (!ok) std::memset(&mine, 0, sizeof(mine));
    cudaMemcpyAsync(handles.data() + std::size_t(world) * sizeof(mine), &mine, sizeof(mine), cudaMemcpyHostToDevice, stream);
    nccl_check(nccl().AllGather(handles.data() + std::size_t(world) * sizeof(mine), handles.data(), sizeof(mine), ncclUint8,
                                d->comm, stream), "allgather ipc handles");
    cudaMemcpyAsync(all.data(), handles.data(), std::size_t(world) * sizeof(mine), cudaMemcpyDeviceToHost, stream);
    c->synchronize();
    for (int p = 0; p < world && ok; ++p) {
      if (p == rank) {
        d->peers.base[p] = d->window;
        continue;
      }
      void* mapped = nullptr;
      ok = cudaIpcOpenMemHandle(&mapped, all[p], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
      d->peers.base[p] = ok ? static_cast<unsigned*>(mapped) : nullptr;
    }
    cudaGetLastError();  // a failed mapping only means the NCCL exchange is used
    // every rank must take the same path: agree on the outcome
    d->counts_host[0] = ok ? 1 : 0;
    cudaMemcpyAsync(d->counts_dev.data(), d->counts_host, sizeof(long long), cudaMemcpyHostToDevice, stream);
    nccl_check(nccl().AllReduce(d->counts_dev.data(), d->counts_dev.data(), 1, ncclInt64, ncclMin, d->comm, stream),
               "allreduce peer window");
    cudaMemcpyAsync(d->counts_host, d->counts_dev.data(), sizeof(long long), cudaMemcpyDeviceToHost, stream);
    c->synchronize();
    d->peer_ready = d->counts_host[0] == 1;
    if (d->timed_out) *d->timed_out = 0;
  }
  // the operator-API form of the partitioned run (operators::exchange, enactor_t::enact): bind NCCL to the context
  {
    auto part = std::make_shared<gcuda::partition_t>();
    part->rank = rank;
    part->world = world;
    part->n_global = n_global;
    part->per = d->per;
    ncclComm_t comm = d->comm;
    part->all_gather = [comm](const void* send, void* recv, std::size_t bytes, cudaStream_t st) {
      nccl_check(nccl().AllGather(send, recv, bytes, ncclUint8, comm, st), "partition all_gather");
    };
    part->all_reduce_sum = [comm](long long* values, std::size_t count, cudaStream_t st) {
      nccl_check(nccl().AllReduce(values, values, count, ncclInt64, ncclSum, comm, st), "partition all_reduce");
    };
    part->all_to_all_v = [comm, rank, world](const void* send, const std::size_t* send_bytes,
                                             const std::size_t* send_off, void* recv, const std::size_t* recv_bytes,
                                             const std::size_t* recv_off, cudaStream_t st) {
      const auto* s8 = static_cast<const unsigned char*>(send);
      auto* r8 = static_cast<unsigned char*>(recv);
      if (send_bytes[rank])  // own records never touch the network
        cudaMemcpyAsync(r8 + recv_off[rank], s8 + send_off[rank], send_bytes[rank], cudaMemcpyDeviceToDevice, st);
      nccl_check(nccl().GroupStart(), "group");
      for (int p = 0; p < world; ++p) {
        if (p == rank) continue;
        if (send_bytes[p]) nccl_check(nccl().Send(s8 + send_off[p], send_bytes[p], ncclUint8, p, comm, st), "send");
        if (recv_bytes[p]) nccl_check(nccl().Recv(r8 + recv_off[p], recv_bytes[p], ncclUint8, p, comm, st), "recv");
      }
      nccl_check(nccl().GroupEnd(), "group");
    };
    d->partition = part;
  }
  *out = d.release();
  return 0;
  ESS_CATCH
}

}  // extern "C"

namespace {
/// gunrock::bfs::run / sssp::run on the owned rows with the partitioned context: the SAME enactor loop as on one GPU
/// (prepare_frontier -> while(!is_converged) loop()), operators::exchange routing each level's frontier to the owners.
template <typename graph_t, typename body_t>
int run_partitioned(ess_dist_t d, graph_t view, body_t body) {
  view.get_properties().row_offset = d->row_begin;
  view.get_properties().global_vertices = d->n_global;
  auto& mc = *d->ctx->ctx;
  mc.set_partition(d->partition);
  try {
    body(view);
  } catch (...) {
    mc.set_partition(nullptr);
    throw;
  }
  mc.set_partition(nullptr);
  return 0;
}
}  // namespace

extern "C" {

int ess_dist_bfs_enactor(ess_dist_t d, int64_t source, int lb, int32_t* d_depth_global, ess_run_info* info) {
  ESS_TRY
  if (!d || !d_depth_global) return ess::fail("ess_dist_bfs_enactor: null argument");
  if (source < 0 || source >= d->n_global) return ess::fail("ess_dist_bfs_enactor: source out of range");
  return ess::with_load_balance(lb, [&](auto lbc) -> int {
    constexpr auto LB = decltype(lbc)::value;
    ESS_WITH_GRAPH(d->graph, G, {
      return run_partitioned(d, G, [&](auto& view) {
        int32_t src = int32_t(source);
        int iters = 0;
        const float ms = bfs::run<LB, operators::advance_direction_t::forward>(
            view, src, d_depth_global, (int32_t*)nullptr, d->ctx->ctx, enactor_properties_t(), nullptr, &iters);
        ess::fill_info(info, ms, iters);
      });
    })
  });
  ESS_CATCH
}

int ess_dist_sssp_enactor(ess_dist_t d, int64_t source, int lb, float* d_dist_global, ess_run_info* info) {
  ESS_TRY
  if (!d || !d_dist_global) return ess::fail("ess_dist_sssp_enactor: null argument");
  if (source < 0 || source >= d->n_global) return ess::fail("ess_dist_sssp_enactor: source out of range");
  return ess::with_load_balance(lb, [&](auto lbc) -> int {
    constexpr auto LB = decltype(lbc)::value;
    ESS_WITH_GRAPH(d->graph, G, {
      return run_partitioned(d, G, [&](auto& view) {
        int32_t src = int32_t(source);
        int iters = 0;
        const float ms = sssp::run<LB>(view, src, d_dist_global, (int32_t*)nullptr, d->ctx->ctx, &iters);
        ess::fill_info(info, ms, iters);
      });
    })
  });
  ESS_CATCH
}

int ess_dist_destroy(ess_dist_t d) {
  delete d;
  return 0;
}

int ess_dist_bfs(ess_dist_t d, int64_t source, float alpha, float beta, ess_run_info* info) {
  ESS_TRY
  if (!d) return ess::fail("ess_dist_bfs: null handle");
  if (d->poisoned) return ess::fail("ess_dist_bfs: an earlier peer exchange on this handle timed out; destroy and recreate it");
  if (source < 0 || source >= d->n_global) return ess::fail("ess_dist_bfs: source out of range");
  if (!(alpha > 0)) alpha = 14.f;
  if (!(beta > 0)) beta = 24.f;
  auto* c = d->ctx->single();
  auto stream = c->stream();
  auto& api = nccl();
  ess_graph_t g = d->graph;
  const unsigned wper = d->wper, words = d->words;
  const int world = d->world, rank = d->rank;
  const unsigned first_word = unsigned(d->row_begin >> 5);
  unsigned* next_slice = d->send.data();
  long long* counts = reinterpret_cast<long long*>(d->send.data() + wper);  // 8-byte aligned: wper is even
  cudaEvent_t t0, t1;
  cudaEventCreate(&t0);
  cudaEventCreate(&t1);
  cudaEventRecord(t0, stream);

  // ---- start state ----
  cudaMemcpyAsync(d->visited_bits.data(), d->isolated_bits.data(), words * sizeof(unsigned), cudaMemcpyDeviceToDevice, stream);
  cudaMemsetAsync(d->frontier_bits.data(), 0, words * sizeof(unsigned), stream);
  b200::kernels::fill_kernel<<<gcuda::persistent_grid(*c, (std::size_t(d->per) + 255) / 256, 8), 256, 0, stream>>>(
      d->depth_local.data(), std::size_t(d->per), 2147483647);
  long long* seed = d->counts_dev.data() + 2 * world;
  if (g->offset_bits == 64)
    seed_kernel<int64_t><<<1, 32, 0, stream>>>(g->g64.get_row_offsets(), source, d->row_begin, unsigned(d->per),
                                                d->frontier_bits.data(), d->visited_bits.data(), d->depth_local.data(),
                                                d->fresh_list.data(), seed);
  else
    seed_kernel<int32_t><<<1, 32, 0, stream>>>(g->g32.get_row_offsets(), source, d->row_begin, unsigned(d->per),
                                                d->frontier_bits.data(), d->visited_bits.data(), d->depth_local.data(),
                                                d->fresh_list.data(), seed);
  nccl_check(api.AllReduce(seed, seed, 2, ncclInt64, ncclSum, d->comm, stream), "allreduce seed");
  cudaMemcpyAsync(d->counts_host, seed, 2 * sizeof(long long), cudaMemcpyDeviceToHost, stream);
  c->synchronize();
  long long n_f = d->counts_host[0], m_f = d->counts_host[1];
  long long m_u = d->m_global - m_f, prev_n_f = 0;
  long long my_count = (source >= d->row_begin && source < d->row_begin + d->per) ? 1 : 0;
  bool pulling = false, list_is_current = true;
  int level = 0, pulls = 0;
  long long exchanged = 0;

  const bool peer = d->peer_ready && ess::dist_peer_exchange() != 0;
  // replicated frontier bitmap the level kernels read: the seed array at level 1, then (peer-memory driver) the
  // window area the previous level's slices landed in
  unsigned* cur_frontier = d->frontier_bits.data();
  // ess_tune("dist_trace", 1): CUDA events between the phases of every level, summed and printed by rank 0
  const bool trace = ess::dist_trace() != 0;
  static const char* phase_names[] = {"local(push|pull)", "candidates->owners", "absorb", "slice->all", "merge", "host"};
  std::vector<std::pair<int, cudaEvent_t>> marks;
  auto mark = [&](int phase) {
    if (!trace) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, stream);
    marks.emplace_back(phase, e);
  };
  while (n_f > 0) {
    ++level;
    mark(-1);
    const unsigned epoch = ++d->epoch;  // same sequence on every rank: one epoch per level of every run
    if (!pulling) {
      if (double(m_f) > double(m_u) / double(alpha) && n_f > prev_n_f) pulling = true;
    } else if (double(n_f) < double(d->n_global) / double(beta) && n_f < prev_n_f) {
      pulling = false;
    }
    cudaMemsetAsync(counts, 0, 2 * sizeof(long long), stream);
    if (pulling) {
      ++pulls;
      ESS_WITH_GRAPH(g, G, {
        partition_pull(d->ctx, G, d->row_begin, level, cur_frontier, d->visited_bits.data(), next_slice,
                       d->depth_local.data(), reinterpret_cast<int64_t*>(counts));
      })
      list_is_current = false;
      mark(0);
    } else {
      if (!list_is_current) {
        auto& scratch = c->scratch();
        scratch.zero(stream);
        frontier::kernels::gather_bits_kernel<<<gcuda::persistent_grid(*c, (std::size_t(wper) + 255) / 256, 8), 256, 0,
                                                stream>>>(cur_frontier + first_word, std::size_t(wper),
                                                          d->fresh_list.data(), scratch.d + scratch_t::out_count);
      }
      ESS_WITH_GRAPH(g, G, {
        // peer-memory driver: the visited set is owner-only (no replicated copy to pre-filter with)
        partition_step(d->ctx, G, d->row_begin, d->n_global, 0, cur_frontier, peer ? nullptr : d->visited_bits.data(),
                       d->candidate_bits.data(), d->fresh_list.data(), my_count);
      })
      list_is_current = true;
      mark(0);
      if (peer) {  // candidate slices go straight into the owners' inboxes over NVLink
        peer_scatter_kernel<<<gcuda::persistent_grid(*c, (std::size_t(words) / 2 + 255) / 256, 4), 256, 0, stream>>>(
            d->candidate_bits.data(), d->peers, world, rank, wper, d->inbox_off, d->flag_off[0], epoch, d->done_counter);
        peer_wait_kernel<<<1, 32, 0, stream>>>(d->window + d->flag_off[0], world, epoch, d->timed_out, peer_timeout_ns());
        c->profiler().launches_total += 2;
      } else {
        nccl_check(api.GroupStart(), "group");
        for (int p = 0; p < world; ++p) {
          nccl_check(api.Send(d->candidate_bits.data() + std::size_t(p) * wper, wper, ncclUint32, p, d->comm, stream), "send");
          nccl_check(api.Recv(d->a2a_recv.data() + std::size_t(p) * wper, wper, ncclUint32, p, d->comm, stream), "recv");
        }
        nccl_check(api.GroupEnd(), "group");
      }
      mark(1);
      unsigned* inbox = peer ? d->window + d->inbox_off : d->a2a_recv.data();
      exchanged += (long long)(world - 1) * wper * 4;
      const unsigned grid = gcuda::persistent_grid(*c, ((std::size_t(d->per) + 31) / 32 + 255) / 256, 8);
      auto* cnt = reinterpret_cast<b200::counter_t*>(counts);
      if (g->offset_bits == 64)
        absorb_kernel<int64_t><<<grid, 256, 0, stream>>>(g->g64.get_row_offsets(), unsigned(d->per), first_word, level,
                                                          inbox, world, wper, d->visited_bits.data(),
                                                          next_slice, d->depth_local.data(), d->fresh_list.data(), cnt,
                                                          peer);
      else
        absorb_kernel<int32_t><<<grid, 256, 0, stream>>>(g->g32.get_row_offsets(), unsigned(d->per), first_word, level,
                                                          inbox, world, wper, d->visited_bits.data(),
                                                          next_slice, d->depth_local.data(), d->fresh_list.data(), cnt,
                                                          peer);
    }
    if (!pulling) mark(2);
    if (peer) {
      // The new frontier slice lands in row `rank` of every rank's BITS area of this epoch's parity: once all flags
      // are up that area IS the replicated next-frontier bitmap (no unpacking pass, no replicated visited set), and
      // the counters reach the host through mapped memory (no D2H copy, no stream synchronisation).
      // The other parity's area — the frontier this level just finished reading — is cleared first: peers write
      // into it one level from now, only after they have seen the flag raised below (senders skip zero words).
      const std::size_t bits = d->bits_off[epoch & 1], cnts = d->cnt_off[epoch & 1];
      if (cur_frontier == d->window + d->bits_off[(epoch & 1) ^ 1])
        cudaMemsetAsync(d->window + d->bits_off[(epoch & 1) ^ 1], 0, std::size_t(words) * sizeof(unsigned), stream);
      peer_publish_level_kernel<<<gcuda::persistent_grid(*c, (std::size_t(wper) / 2 * world + 255) / 256, 4), 256, 0,
                                  stream>>>(next_slice, d->send.data() + wper, d->peers, world, rank, wper, bits, cnts,
                                            d->flag_off[1], epoch, d->done_counter);
      mark(3);
      const unsigned long long sequence = ++d->level_sequence;
      peer_wait_publish_kernel<<<1, 32, 0, stream>>>(d->window + d->flag_off[1], world, epoch, d->timed_out,
                                                     d->window + cnts, d->level_counts, sequence, peer_timeout_ns());
      c->profiler().launches_total += 2;
      mark(4);
      mark(5);
      volatile long long* seq = d->level_counts + 2 * max_peers;
      for (unsigned spins = 0; (unsigned long long)*seq != sequence; ++spins) {
        if ((spins & 0x3ff) == 0x3ff) {  // every ~1k polls make sure the stream is still healthy
          cudaError_t st = cudaStreamQuery(stream);
          if (st != cudaSuccess && st != cudaErrorNotReady) error::throw_if_exception(st, "dist bfs level");
          if (st == cudaSuccess && (unsigned long long)*seq != sequence) {
            error::throw_if_exception(cudaStreamSynchronize(stream), "dist bfs level");
            if ((unsigned long long)*seq != sequence) error::throw_if_exception(cudaErrorUnknown, "level hand-off lost");
          }
        }
      }
      for (int p = 0; p < 2 * world; ++p) d->counts_host[p] = d->level_counts[p];
      cur_frontier = d->window + bits;
      exchanged += (long long)(world - 1) * (wper + 4) * 4;
    } else {
      nccl_check(api.AllGather(d->send.data(), d->recv.data(), wper + 4, ncclUint32, d->comm, stream), "allgather");
      exchanged += (long long)(world - 1) * (wper + 4) * 4;
      mark(3);
      merge_gathered_kernel<<<gcuda::persistent_grid(*c, (std::size_t(words) + 255) / 256, 8), 256, 0, stream>>>(
          d->recv.data(), world, wper, d->frontier_bits.data(), d->visited_bits.data(), d->counts_dev.data(), false);
      mark(4);
      cudaMemcpyAsync(d->counts_host, d->counts_dev.data(), 2 * std::size_t(world) * sizeof(long long),
                      cudaMemcpyDeviceToHost, stream);
      mark(5);
      error::throw_if_exception(cudaStreamSynchronize(stream), "dist bfs level");  // the one host sync of the level
    }
    if (peer && *d->timed_out) {
      const unsigned who = *d->timed_out - 1;
      *d->timed_out = 0;
      d->poisoned = true;
      throw error::exception_t("ess_dist_bfs: peer " + std::to_string(who) + " did not deliver its level data within " +
                               std::to_string(peer_timeout_ns() / 1000000ull) +
                               " ms (ess_tune dist_peer_timeout_ms); the handle is unusable from here on");
    }
    prev_n_f = n_f;
    n_f = 0;
    m_f = 0;
    for (int p = 0; p < world; ++p) {
      n_f += d->counts_host[2 * p];
      m_f += d->counts_host[2 * p + 1];
    }
    my_count = d->counts_host[2 * rank];
    m_u -= m_f;
  }
  cudaEventRecord(t1, stream);
  cudaEventSynchronize(t1);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, t0, t1);
  if (trace) {
    double sum[6] = {0}, gaps = 0;
    int cnt[6] = {0};
    for (std::size_t i = 1; i < marks.size(); ++i) {
      float t = 0.f;
      cudaEventElapsedTime(&t, marks[i - 1].second, marks[i].second);
      if (marks[i].first >= 0)
        sum[marks[i].first] += t, cnt[marks[i].first]++;
      else
        gaps += t;  // host turn-around between the sync of one level and the first launch of the next
    }
    if (rank == 0) {
      std::fprintf(stderr, "[dist_trace] %d levels %.3f ms:", level, ms);
      for (int k = 0; k < 6; ++k) std::fprintf(stderr, " %s=%.0fus/%d", phase_names[k], sum[k] * 1e3, cnt[k]);
      std::fprintf(stderr, " level-gaps=%.0fus\n", gaps * 1e3);
    }
    for (auto& m : marks) cudaEventDestroy(m.second);
  }
  cudaEventDestroy(t0);
  cudaEventDestroy(t1);
  d->levels = level;
  d->pull_levels = pulls;
  d->bytes_exchanged = exchanged;
  ess::fill_info(info, ms, level, pulls, level - pulls);
  if (info) info->reserved[0] = exchanged;
  return 0;
  ESS_CATCH
}

/// Start state of one partitioned SSSP: every rank knows dist(source) = 0; the owner seeds its active list.
static __global__ void sssp_seed_kernel(long long source, long long row_begin, unsigned n_local, float* replica,
                                        float* dist_local, int* active_list) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  replica[source] = 0.f;
  const long long local = source - row_begin;
  if (local >= 0 && local < (long long)n_local) {
    dist_local[local] = 0.f;
    active_list[0] = int(local);
  }
}

/// First peer-memory SSSP on this handle: allocate replica + dirty words, exchange IPC handles, map the peers.
/// Collective (every rank calls it at the same point); all ranks agree on the outcome.
static void setup_sssp_window(ess_dist_t d) {
  d->sssp_peer_tried = true;
  auto* c = d->ctx->single();
  auto stream = c->stream();
  const int world = d->world, rank = d->rank;
  const std::size_t n = std::size_t(d->n_global), chunks = (n + 1023) / 1024;
  cudaIpcMemHandle_t mine;
  std::memset(&mine, 0, sizeof(mine));
  bool ok = cudaMalloc(&d->replica_window, (n + chunks) * sizeof(float)) == cudaSuccess &&
            cudaIpcGetMemHandle(&mine, d->replica_window) == cudaSuccess;
  memory::device_array_t<unsigned char> handles(std::size_t(world + 1) * sizeof(mine));
  std::vector<cudaIpcMemHandle_t> all(world);
  unsigned char* my_slot = handles.data() + std::size_t(world) * sizeof(mine);
  cudaMemcpyAsync(my_slot, &mine, sizeof(mine), cudaMemcpyHostToDevice, stream);
  nccl_check(nccl().AllGather(my_slot, handles.data(), sizeof(mine), ncclUint8, d->comm, stream), "allgather ipc handles");
  cudaMemcpyAsync(all.data(), handles.data(), std::size_t(world) * sizeof(mine), cudaMemcpyDeviceToHost, stream);
  c->synchronize();
  for (int p = 0; p < world && ok; ++p) {
    void* mapped = d->replica_window;
    if (p != rank) {
      mapped = nullptr;
      ok = cudaIpcOpenMemHandle(&mapped, all[p], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
      if (!ok) mapped = nullptr;  // the destructor closes every non-null peer mapping: never our own window
    }
    d->replicas.value[p] = static_cast<const float*>(mapped);
    d->replicas.dirty[p] = ok ? reinterpret_cast<const unsigned*>(static_cast<const float*>(mapped) + n) : nullptr;
  }
  cudaGetLastError();
  d->counts_host[0] = ok ? 1 : 0;
  cudaMemcpyAsync(d->counts_dev.data(), d->counts_host, sizeof(long long), cudaMemcpyHostToDevice, stream);
  nccl_check(nccl().AllReduce(d->counts_dev.data(), d->counts_dev.data(), 1, ncclInt64, ncclMin, d->comm, stream),
             "allreduce sssp window");
  cudaMemcpyAsync(d->counts_host, d->counts_dev.data(), sizeof(long long), cudaMemcpyDeviceToHost, stream);
  c->synchronize();
  d->sssp_peer_ready = d->counts_host[0] == 1;
}

int ess_dist_sssp(ess_dist_t d, int64_t source, ess_run_info* info) {
  ESS_TRY
  if (!d) return ess::fail("ess_dist_sssp: null handle");
  if (d->poisoned) return ess::fail("ess_dist_sssp: an earlier peer exchange on this handle timed out; destroy and recreate it");
  if (source < 0 || source >= d->n_global) return ess::fail("ess_dist_sssp: source out of range");
  auto* c = d->ctx->single();
  auto stream = c->stream();
  auto& api = nccl();
  ess_graph_t g = d->graph;
  const int world = d->world, rank = d->rank;
  const std::size_t per = std::size_t(d->per), n = std::size_t(d->n_global);
  // exchange: fused peer-memory reduce+collect when the windows could be mapped, else ncclReduceScatter(min)
  const bool want_peer = d->peer_ready && ess::dist_peer_exchange() != 0 && world > 1 && per % 1024 == 0;
  if (want_peer && !d->sssp_peer_tried) setup_sssp_window(d);
  const bool peer = want_peer && d->sssp_peer_ready;
  if (!peer) d->replica.resize(n);
  d->dist_local.resize(per);
  float* replica = peer ? d->replica_window : d->replica.data();
  unsigned* dirty = peer ? reinterpret_cast<unsigned*>(d->replica_window + n) : nullptr;
  const std::size_t dirty_words = (n + 1023) / 1024;
  float* owned = replica + std::size_t(rank) * per;  // the reduce_scatter lands here (in place)
  float* dist_local = d->dist_local.data();
  int* active = d->fresh_list.data();
  long long* counts = d->counts_dev.data();  // [0..1] this rank, [2..3] all ranks
  cudaEvent_t t0, t1;
  cudaEventCreate(&t0);
  cudaEventCreate(&t1);
  cudaEventRecord(t0, stream);
  const float inf = gunrock::numeric_limits<float>::max();
  b200::kernels::fill_kernel<<<gcuda::persistent_grid(*c, (n + 255) / 256, 8), 256, 0, stream>>>(replica, n, inf);
  b200::kernels::fill_kernel<<<gcuda::persistent_grid(*c, (per + 255) / 256, 8), 256, 0, stream>>>(dist_local, per, inf);
  sssp_seed_kernel<<<1, 32, 0, stream>>>(source, d->row_begin, unsigned(per), replica, dist_local, active);
  long long my_count = (source >= d->row_begin && source < d->row_begin + d->per) ? 1 : 0;
  long long total = 1, relaxed = 0, exchanged = 0;
  int rounds = 0;
  if (peer) cudaMemsetAsync(counts + 4, 0, sizeof(long long), stream);  // bytes this rank pulls over NVLink
  while (total > 0) {
    ++rounds;
    if (peer) {
      const unsigned epoch = ++d->epoch;
      cudaMemsetAsync(dirty, 0, dirty_words * sizeof(unsigned), stream);  // peers finished reading: all_reduce below
      ESS_WITH_GRAPH(g, G, { partition_relax(d->ctx, G, active, my_count, dist_local, replica, dirty); })
      peer_signal_kernel<<<1, 32, 0, stream>>>(d->peers, world, rank, d->flag_off[0], epoch);
      peer_wait_kernel<<<1, 32, 0, stream>>>(d->window + d->flag_off[0], world, epoch, d->timed_out, peer_timeout_ns());
      cudaMemsetAsync(counts, 0, 2 * sizeof(long long), stream);
      const unsigned grid = gcuda::persistent_grid(*c, per / 1024, 8);
      auto* cnt = reinterpret_cast<b200::counter_t*>(counts);
      if (g->offset_bits == 64)
        sssp_peer_reduce_collect_kernel<int64_t><<<grid, 256, 0, stream>>>(
            g->g64.get_row_offsets(), unsigned(per), d->row_begin, d->replicas, world, rank, replica, dist_local, active, cnt);
      else
        sssp_peer_reduce_collect_kernel<int32_t><<<grid, 256, 0, stream>>>(
            g->g32.get_row_offsets(), unsigned(per), d->row_begin, d->replicas, world, rank, replica, dist_local, active, cnt);
      c->profiler().launches_total += 3;
    } else {
      ESS_WITH_GRAPH(g, G, { partition_relax(d->ctx, G, active, my_count, dist_local, replica); })
      nccl_check(api.ReduceScatter(replica, owned, per, ncclFloat, ncclMin, d->comm, stream), "reduce_scatter");
      exchanged += (long long)(world - 1) * (long long)per * 4;
      cudaMemsetAsync(counts, 0, 2 * sizeof(long long), stream);
      ESS_WITH_GRAPH(g, G, { partition_collect(d->ctx, G, owned, dist_local, active, reinterpret_cast<int64_t*>(counts)); })
    }
    nccl_check(api.AllReduce(counts, counts + 2, 2, ncclInt64, ncclSum, d->comm, stream), "allreduce counts");
    cudaMemcpyAsync(d->counts_host, counts, 4 * sizeof(long long), cudaMemcpyDeviceToHost, stream);
    error::throw_if_exception(cudaStreamSynchronize(stream), "dist sssp round");  // the one host sync of the round
    if (peer && *d->timed_out) {
      const unsigned who = *d->timed_out - 1;
      *d->timed_out = 0;
      d->poisoned = true;
      throw error::exception_t("ess_dist_sssp: peer " + std::to_string(who) + " did not finish its relaxation round within " +
                               std::to_string(peer_timeout_ns() / 1000000ull) +
                               " ms (ess_tune dist_peer_timeout_ms); the handle is unusable from here on");
    }
    my_count = d->counts_host[0];
    total = d->counts_host[2];
    relaxed += d->counts_host[3];
  }
  if (peer) {
    cudaMemcpyAsync(d->counts_host, counts + 4, sizeof(long long), cudaMemcpyDeviceToHost, stream);
    cudaStreamSynchronize(stream);
    exchanged = d->counts_host[0];
  }
  cudaEventRecord(t1, stream);
  cudaEventSynchronize(t1);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, t0, t1);
  cudaEventDestroy(t0);
  cudaEventDestroy(t1);
  ess::fill_info(info, ms, rounds);
  if (info) {
    info->reserved[0] = exchanged;
    info->reserved[1] = relaxed;
    info->reserved[2] = peer ? 1 : 0;
  }
  return 0;
  ESS_CATCH
}

int ess_dist_copy_dist(ess_dist_t d, float* d_out) {
  ESS_TRY
  if (!d || !d_out) return ess::fail("ess_dist_copy_dist: null argument");
  if (d->dist_local.size() != std::size_t(d->per)) return ess::fail("ess_dist_copy_dist: no SSSP has run");
  error::throw_if_exception(cudaMemcpyAsync(d_out, d->dist_local.data(), std::size_t(d->per) * sizeof(float),
                                            cudaMemcpyDeviceToDevice, d->ctx->single()->stream()),
                            "ess_dist_copy_dist");
  return 0;
  ESS_CATCH
}

int ess_dist_exchange_kind(ess_dist_t d, int* kind) {
  if (!d || !kind) return ess::fail("ess_dist_exchange_kind: null argument");
  *kind = d->peer_ready && ess::dist_peer_exchange() != 0 ? 1 : 0;
  return 0;
}

int ess_dist_copy_depth(ess_dist_t d, int32_t* d_out) {
  ESS_TRY
  if (!d || !d_out) return ess::fail("ess_dist_copy_depth: null argument");
  error::throw_if_exception(cudaMemcpyAsync(d_out, d->depth_local.data(), std::size_t(d->per) * sizeof(int32_t),
                                            cudaMemcpyDeviceToDevice, d->ctx->single()->stream()),
                            "ess_dist_copy_depth");
  return 0;
  ESS_CATCH
}

int ess_dist_depth_local(ess_dist_t d, int32_t** d_depth_local, int64_t* count) {
  if (!d) return ess::fail("ess_dist_depth_local: null handle");
  if (d_depth_local) *d_depth_local = d->depth_local.data();
  if (count) *count = d->per;
  return 0;
}

}  // extern "C"
