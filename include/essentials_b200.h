/*
 * essentials_b200.h — C ABI of the B200-native frontier operators.
 *
 * The reference (jdwapman/essentials, Gunrock 2.x) has no FFI: its boundary is a C++17 header-template API
 * (SURVEY.md §8b) that this repository mirrors under include/gunrock/. This header is the plain-C surface a
 * non-C++ host (ctypes, cgo, JNI ...) binds instead; every entry point names the reference interface it
 * stands for (paths relative to the reference tree). All pointers named d_* are DEVICE pointers owned by
 * the caller; nothing here allocates or frees caller memory; no C++ exception crosses the boundary.
 *
 * Return value: 0 on success, otherwise a cudaError_t-compatible code (cudaErrorUnknown = 999 for logical
 * errors); ess_last_error() returns the message of the calling thread's last failure.
 *
 * Types are the ones the reference's drivers use (examples/algorithms/bfs/bfs.cu:16-18):
 * vertex_t = int32, weight_t = float, edge_t = int32 or int64 chosen per graph by `offset_bits`.
 */
#ifndef ESSENTIALS_B200_H
#define ESSENTIALS_B200_H

#include <stdint.h>

#if defined(__GNUC__)
#define ESS_API __attribute__((visibility("default")))
#else
#define ESS_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* operators::load_balance_t (include/gunrock/framework/operators/configs.hxx:31-39), same values. */
enum ess_load_balance {
  ESS_LB_THREAD_MAPPED = 0,
  ESS_LB_WARP_MAPPED = 1, /* not supported, as in the reference */
  ESS_LB_BLOCK_MAPPED = 2,
  ESS_LB_BUCKETING = 3,
  ESS_LB_MERGE_PATH = 4,
  ESS_LB_MERGE_PATH_V2 = 5, /* alias of merge_path */
  ESS_LB_WORK_STEALING = 6  /* not supported, as in the reference */
};
/* operators::advance_direction_t (configs.hxx:48-52). */
enum ess_direction { ESS_DIR_FORWARD = 0, ESS_DIR_BACKWARD = 1, ESS_DIR_OPTIMIZED = 2 };
/* operators::filter_algorithm_t (configs.hxx:54-59). */
enum ess_filter { ESS_FILTER_REMOVE = 0, ESS_FILTER_PREDICATED = 1, ESS_FILTER_COMPACT = 2, ESS_FILTER_BYPASS = 3 };

typedef struct ess_context_s* ess_context_t; /* gcuda::multi_context_t, include/gunrock/cuda/context.hxx:136-206 */
typedef struct ess_graph_s* ess_graph_t;     /* graph::graph_t view, include/gunrock/graph/graph.hxx:52-317 */

/* What enact() and the enactor counters report for one run. */
typedef struct ess_run_info {
  float enact_ms;     /* value returned by gunrock::<alg>::run(): cudaEvent ms around the BSP loop
                         (include/gunrock/framework/enactor.hxx:246-253) */
  int32_t iterations; /* enactor_t::iteration at convergence */
  int32_t pull_steps; /* direction-optimised BFS: levels run bottom-up */
  int32_t push_steps; /* direction-optimised BFS: levels run top-down */
  int64_t reserved[8]; /* ess_bfs/OPTIMIZED work accounting: [0] vertices probed bottom-up, [1] in-edges read
                          bottom-up (early exit counted), [2] vertices and [3] out-edges expanded top-down,
                          [4] bottom-up hint misses (adjacency walked), [5] vertices adopted bottom-up,
                          [6] vertices claimed top-down; other entry points document their own use */
} ess_run_info;

ESS_API const char* ess_last_error(void);
ESS_API int ess_version(void);

/* gcuda::multi_context_t(device[, stream]) (context.hxx:143-181): one device. own_stream != 0 creates a new
 * non-blocking stream owned by the context, as the reference's standard_context_t does (context.hxx:82);
 * otherwise all work is enqueued on `stream` (a cudaStream_t; NULL = the legacy default stream), so it is
 * ordered with the caller's other work on that stream. */
ESS_API int ess_context_create(int device, void* stream, int own_stream, ess_context_t* out);
ESS_API int ess_context_destroy(ess_context_t ctx);
ESS_API int ess_context_synchronize(ess_context_t ctx);

/* Opt-in kernel timing with CUDA events on the context's stream (bench / roofline only; the reference's
 * counterpart is nvbench's CUPTI collection, benchmarks/bfs_bench.cu:61-65). Classes: 0 pull step, 1 push
 * expansion, 2 work preparation (scan/binning), 3 dense-state kernels (sparse<->dense, visited), 4 filters.
 * ess_profile_enable resets the accumulators; ess_profile_read resolves pending events and copies
 * accumulated milliseconds and launch counts (arrays of n_classes <= 8 entries). */
ESS_API int ess_tune(const char* knob, int value); /* development knobs, e.g. "pull_hints" (see pull.cuh) */
ESS_API int ess_profile_enable(ess_context_t ctx, int enable);
ESS_API int ess_profile_read(ess_context_t ctx, double* ms_by_class, int64_t* launches_by_class, int n_classes);

/* graph::build::from_csr<device, csr[|csc]> (include/gunrock/graph/build.hxx:21-36).
 * d_row_offsets: (n+1) x int32 or int64 (offset_bits = 32|64); d_column_indices: m x int32;
 * d_values: m x float or NULL (weight 1). CSC (in-edges), needed for backward / optimized / pull:
 *   symmetric = 1             -> the CSC view aliases the CSR arrays (undirected graph);
 *   symmetric = 2             -> same, but the arrays are a ROW RANGE of a partitioned graph (n rows, global
 *                                column ids): bottom-up hints are not built here (ess_graph_build_pull_hints);
 *   d_column_offsets != NULL  -> caller-provided transpose (same widths);
 *   otherwise                 -> no CSC view; calls that need it fail with an error. */
ESS_API int ess_graph_create(int64_t n, int64_t m, int offset_bits, const void* d_row_offsets,
                     const int32_t* d_column_indices, const float* d_values, int symmetric,
                     const void* d_column_offsets, const int32_t* d_row_indices, const float* d_csc_values,
                     ess_graph_t* out);
/* The same graph from HOST arrays — what the reference's drivers do around from_csr: load a host csr_t, assign it to
 * device vectors (format conversion + thrust copies, examples/algorithms/bfs/bfs.cu:44-66), build the views. The handle
 * owns the device copies. The transfer is pipelined on a private copy stream: offsets first, then the column indices
 * in 256 MB chunks, and the bottom-up hints of the vertices whose lists have arrived are built on the context's stream
 * while later chunks are still crossing PCIe (pinned host memory overlaps; pageable memory works, unoverlapped).
 * symmetric = 1: the CSC view aliases the copies and hints are built; 0: CSR only. Returns with the graph complete. */
ESS_API int ess_graph_create_from_host(ess_context_t ctx, int64_t n, int64_t m, int offset_bits,
                                       const void* h_row_offsets, const int32_t* h_column_indices,
                                       const float* h_values, int symmetric, ess_graph_t* out);
ESS_API int ess_graph_destroy(ess_graph_t g);
/* (Re)builds the bottom-up hints of graph::build::pull_hints (include/gunrock/graph/build.hxx; no reference
 * counterpart): per vertex, its highest-degree in-neighbour. d_degree_of_id: degree of every id that may appear
 * as an in-neighbour (required for symmetric = 2 partitions; NULL = read degrees from the graph's own offsets).
 * ess_graph_create calls it automatically for symmetric = 1 and for caller-provided CSC arrays. */
ESS_API int ess_graph_build_pull_hints(ess_graph_t g, const int32_t* d_degree_of_id);

/* CSR -> CSC by counting sort on the device (the transpose the reference performs destructively inside
 * graph/detail/build.hxx:103-110). Output buffers are caller-allocated: (n+1) offsets, m indices, m values
 * (d_values / d_out_values may both be NULL). Order inside a column is unspecified. */
ESS_API int ess_transpose_csr(int64_t n, int64_t m, int offset_bits, const void* d_row_offsets,
                      const int32_t* d_column_indices, const float* d_values, void* d_out_offsets,
                      int32_t* d_out_indices, float* d_out_values);

/* gunrock::bfs::run(G, source, distances, predecessors, context) — include/gunrock/algorithms/bfs.hxx:151-176.
 * d_depth: n x int32, INT32_MAX = unreachable. lb: ess_load_balance; direction: FORWARD (reference
 * behaviour) or OPTIMIZED (push/pull switching; needs a CSC view). alpha/beta <= 0 keep the defaults. */
ESS_API int ess_bfs(ess_context_t ctx, ess_graph_t g, int32_t source, int32_t* d_depth, int lb, int direction,
            float alpha, float beta, ess_run_info* info);

/* gunrock::bfs::run_tree: ess_bfs plus the BFS tree. d_depth, the arguments and info are exactly as for ess_bfs.
 * d_pred: n x int32, 4-byte aligned, required, must not alias d_depth. On return:
 *   d_pred[source] == source;
 *   d_pred[v] == -1 if and only if d_depth[v] == INT32_MAX (v unreached);
 *   otherwise 0 <= d_pred[v] < n, the CSR holds an edge d_pred[v] -> v, and d_depth[d_pred[v]] == d_depth[v] - 1.
 * Which of several valid parents is chosen depends on scheduling and is not deterministic. Every entry is written, so
 * what d_pred held before the call does not matter. */
ESS_API int ess_bfs_tree(ess_context_t ctx, ess_graph_t g, int32_t source, int32_t* d_depth, int32_t* d_pred, int lb,
                         int direction, float alpha, float beta, ess_run_info* info);

/* gunrock::sssp::run — include/gunrock/algorithms/sssp.hxx:155-185. d_dist: n x float, FLT_MAX = unreachable. */
ESS_API int ess_sssp(ess_context_t ctx, ess_graph_t g, int32_t source, float* d_dist, int lb, ess_run_info* info);

/* Same distances as ess_sssp through operators::advance::execute_near_far (include/gunrock/framework/operators/
 * advance/near_far.cuh): near/far priority ordering — the method the reference's load_balance_t::bucketing
 * enumerator cites (configs.hxx:35) but leaves empty (advance/bucketing.hxx:31-36) — inside one persistent
 * kernel. delta: bucket width (<= 0: 64 x mean edge weight / mean degree). info->iterations = near levels; reserved[0] levels,
 * [1] far-pile splits, [2] relaxations. */
ESS_API int ess_sssp_near_far(ess_context_t ctx, ess_graph_t g, int32_t source, float* d_dist, float delta,
                              ess_run_info* info);

/* Same distances through gunrock::sssp::run_delta (include/gunrock/algorithms/sssp.hxx): a dense active set chosen
 * per round by one streaming pass (distance dropped since last expansion AND below a threshold that advances by
 * `delta`), expanded with the merge-path advance. For low-diameter graphs with big frontiers (Kronecker/RMAT),
 * where it halves the relaxations of plain label-correcting; delta <= 0 picks mean edge weight / 2.
 * info->iterations = expanding rounds; reserved = {rounds, threshold advances, vertices expanded, passes}. */
ESS_API int ess_sssp_delta(ess_context_t ctx, ess_graph_t g, int32_t source, float* d_dist, float delta,
                           ess_run_info* info);

/* gunrock::sssp::build_tree: the shortest-path tree of distances an SSSP run returned. d_dist: n x float, read only,
 * the result of ess_sssp (any lb), ess_sssp_near_far or ess_sssp_delta from `source` on this graph. d_pred: n x int32,
 * 4-byte aligned, required, must not overlap d_dist; every entry is written. With fl(a + w) the float add SSSP uses
 * and w the CSR weight (1 without values), an edge u -> v is tight when d[u] < FLT_MAX and d[v] == fl(d[u] + w),
 * strict when also d[u] < d[v], flat when d[u] == d[v] and u != v. On return:
 *   d_pred[source] == source;
 *   d_pred[v] == -1 if and only if d_dist[v] == FLT_MAX (v unreached);
 *   a reached v with a strict tight in-edge: the smallest tail of its strict tight in-edges;
 *   any other reached v: with the vertices above as anchors and L(v) the flat hops from the nearest anchor, the
 *     smallest u with a flat edge u -> v and L(u) == L(v) - 1.
 * The tree is a pure function of the graph, d_dist and source (no cycles; byte-identical for the three SSSP entry
 * points, which return bit-identical distances). Only CSR out-edges are read: no CSC view is needed.
 * The call fails, naming the violation and its count, when d_dist is not the SSSP fixed point for `source`: an entry
 * that is NaN, negative or +inf, d_dist[source] != 0, an edge with fl(d[u] + w) < d[v] and u reached, or a reached
 * vertex without a tight path from the source. d_pred is then unspecified. info->enact_ms = the pass (CUDA events),
 * iterations = flat rounds, reserved[0] = vertices parented over a flat edge. */
ESS_API int ess_sssp_tree(ess_context_t ctx, ess_graph_t g, int32_t source, const float* d_dist, int32_t* d_pred,
                          ess_run_info* info);

/* gunrock::bc::run: betweenness centrality by Brandes' algorithm over the depths of the direction-optimised BFS
 * (include/gunrock/algorithms/bc.hxx; needs a CSC view). The graph is taken unweighted: a path is a sequence of CSR
 * edges, so parallel edges are distinct paths, and self-loops are never on a shortest path. With σ_s(v) the number of
 * shortest s -> v paths and δ_s(v) = Σ_{v->w, d(w) = d(v)+1} σ_s(v)/σ_s(w) · (1 + δ_s(w)), on return
 *   d_bc[v] = float(scale · Σ_{s ∈ sources, s != v} δ_s(v))   for every v (n x float, every entry written).
 * h_sources: HOST array of n_sources vertex ids, summed in list order (a source listed twice counts twice); NULL with
 * n_sources == 0 means every vertex in id order, which is exact BC. scale 1 gives the raw sum, 0.5 the undirected
 * convention (each unordered pair once; also the reference's single-source output), 1/((n-1)(n-2)) a normalisation.
 * σ, δ and the sum are double; the result is a pure function of (graph, sources, scale), byte-identical between runs
 * and for 32- or 64-bit offsets, host-built and misaligned graphs. Refused before any launch: a null ctx, g or d_bc,
 * n_sources < 0, n_sources == 0 with non-NULL h_sources, a source out of range, a non-finite scale, a graph without
 * a CSC view. info->enact_ms = device time of the whole call, iterations = number of sources, reserved[0] Σ levels,
 * [1] Σ reached vertices, [2] Σ edges gathered by both passes. */
ESS_API int ess_bc(ess_context_t ctx, ess_graph_t g, const int32_t* h_sources, int64_t n_sources, float scale,
                   float* d_bc, ess_run_info* info);

/* gunrock::pr::run — include/gunrock/algorithms/pr.hxx:183-216 (alpha 0.85, tol 1e-6 in examples/algorithms/pr/pr.cu:55-56).
 * pull != 0 gathers over the CSC view instead of scattering with atomics; it fails when only one of the CSR and
 * CSC views carries edge weights. */
ESS_API int ess_pagerank(ess_context_t ctx, ess_graph_t g, float alpha, float tol, int max_iterations, float* d_p, int lb,
                 int pull, ess_run_info* info);

/* gunrock::ppr::run — include/gunrock/algorithms/ppr.hxx:150-179. d_p: n x float. */
ESS_API int ess_ppr(ess_context_t ctx, ess_graph_t g, int32_t seed, float alpha, float epsilon, float* d_p, int lb,
            ess_run_info* info);

/* gunrock::kcore::run — include/gunrock/algorithms/kcore.hxx:202-222. d_k_cores: n x int32. */
ESS_API int ess_kcore(ess_context_t ctx, ess_graph_t g, int32_t* d_k_cores, int lb, ess_run_info* info);

/* gunrock::color::run — include/gunrock/algorithms/color.hxx:155-180. d_colors: n x int32. */
ESS_API int ess_color(ess_context_t ctx, ess_graph_t g, int32_t* d_colors, ess_run_info* info);

/* generate::random::uniform_distribution — include/gunrock/algorithms/generate/random.hxx:20-33. */
ESS_API int ess_randoms(ess_context_t ctx, float* d_out, int64_t n, float begin, float end);

/* ---- operator-level entry points (used by the parity tests; fixed test operators) ---------------------
 * operators::advance::execute<lb, direction, vertices, vertices>(G, op, in, out, segments, ctx) —
 * include/gunrock/framework/operators/advance/advance.hxx:91-129 — with the operator
 *     op(src, nbr, e, w) := { atomicAdd(&d_edge_calls[e], 1); return (src + nbr + e) % modulus != 0; }
 * d_out receives the kept neighbours (capacity out_capacity elements; 0 lets the library size it and only
 * report the count), *out_count their number. d_edge_calls (m x int32, caller-zeroed) may be NULL. */
ESS_API int ess_advance_probe(ess_context_t ctx, ess_graph_t g, int lb, int direction, const int32_t* d_frontier,
                      int64_t frontier_size, int32_t* d_out, int64_t out_capacity, int64_t* out_count,
                      int32_t* d_edge_calls, int32_t modulus);

/* The same fixed operator through operators::advance::execute_unique — fused advance + uniquify, the step the
 * reference leaves commented out after its advances (sssp.hxx:146-150, bfs.hxx:128-131): the operator still runs
 * once per edge (d_edge_calls), but every kept neighbour appears once in d_out. The probe runs the call twice on
 * the same bitmap (the second pass proves the map was left clear), so d_edge_calls ends at 2 per edge. */
ESS_API int ess_advance_unique_probe(ess_context_t ctx, ess_graph_t g, int lb, const int32_t* d_frontier,
                                     int64_t frontier_size, int32_t* d_out, int64_t out_capacity, int64_t* out_count,
                                     int32_t* d_edge_calls, int32_t modulus);

/* operators::filter::execute<alg>(G, op, in, out, ctx) — include/gunrock/framework/operators/filter/filter.hxx:59-86 —
 * with op(v) := { atomicAdd(&d_calls[v], 1); return v % modulus != 0; }. d_out needs `size` elements
 * (may equal d_in for BYPASS). */
ESS_API int ess_filter_probe(ess_context_t ctx, ess_graph_t g, int alg, const int32_t* d_in, int64_t size, int32_t* d_out,
                     int64_t* out_count, int32_t* d_calls, int32_t modulus);

/* operators::uniquify::execute<unique>(in, out, ctx) — include/gunrock/framework/operators/uniquify/uniquify.hxx:15-72
 * (sort + unique in the reference; here a sparse->dense->sparse round trip): d_out receives the ascending,
 * duplicate-free valid ids of d_in (d_out needs min(size, n) elements). */
ESS_API int ess_uniquify_probe(ess_context_t ctx, ess_graph_t g, const int32_t* d_in, int64_t size, int32_t* d_out,
                               int64_t* out_count);

/* math::atomic::{add,min,max,exch} (include/gunrock/util/math.hxx:77-129; float min/max:
 * include/gunrock/cuda/atomic_functions.hxx:36-123). d_old[i] = atomic::<op>(d_cell, d_values[i]) — the wrappers
 * return the value the cell held BEFORE the update, which user lambdas compare against (bfs.hxx:96-99,
 * sssp.hxx:121-127). op: 0 add, 1 min, 2 max, 3 exch; is_float selects float or int32 cells; serial != 0 applies the
 * updates in index order from one thread (deterministic), otherwise one thread per value. */
ESS_API int ess_atomic_probe(ess_context_t ctx, int op, int is_float, void* d_cell, const void* d_values, int64_t n,
                             void* d_old, int serial);

/* frontier sparse -> dense (bitmap, 1 bit per vertex; d_words: ceil(universe/32)+1 x uint32) and back
 * (ascending within 1024-vertex groups). Stand for the conversions SURVEY.md K14 R3/R4 lists; the
 * reference's boolmap_frontier_t (frontier/experimental/boolmap_frontier.hxx:25-202) has none. */
ESS_API int ess_frontier_to_bitmap(ess_context_t ctx, const int32_t* d_list, int64_t size, int64_t universe,
                           uint32_t* d_words, int64_t* popcount);
ESS_API int ess_bitmap_to_frontier(ess_context_t ctx, const uint32_t* d_words, int64_t universe, int32_t* d_list,
                           int64_t* out_count);

/* As ess_bitmap_to_frontier but only enqueues the kernel (no length is returned: the caller already knows the
 * population count). */
ESS_API int ess_bits_to_list_async(ess_context_t ctx, const uint32_t* d_words, int64_t universe, int32_t* d_list);

/* ---- multi-GPU (one process per GPU; 1-D vertex partition; exchange done by the host with NCCL) --------
 * The reference has no counterpart (operators throw on context.size() != 1, advance/advance.hxx:125-128).
 * `g` holds the rows [row_begin, row_begin + n_local) this rank owns, with GLOBAL column ids (symmetric
 * graph); bitmaps cover all global vertices; both calls only ENQUEUE work on the context's stream — the caller
 * synchronises once per level (the all_gather of the next frontier carries the counters).
 *
 * ess_bfs_partition_step, one BFS level on the owned rows:
 *   pull = 0: balanced merge-path advance over d_frontier_list (frontier_count LOCAL row ids); every neighbour
 *             not in d_visited_bits is OR-ed into d_candidate_bits (global length, zeroed here) — the host then
 *             exchanges candidate slices (all_to_all) and the owner absorbs them.
 *   pull = 1: not served here — use ess_bfs_partition_pull.
 * ess_bfs_absorb, owner side: candidate word w = OR over n_slices of d_candidates[p*slice_stride_words + w];
 *   fresh = candidate & ~visited; depth[fresh] = level; visited |= fresh; d_next_slice[w] = fresh (owned words
 *   only); fresh LOCAL ids are appended to d_fresh_list; d_counts[0] += |fresh|, d_counts[1] += sum of their
 *   degrees (two device int64 the caller zeroes). */
ESS_API int ess_bfs_partition_step(ess_context_t ctx, ess_graph_t g, int64_t row_begin, int64_t n_global, int pull,
                                   const uint32_t* d_frontier_bits, const uint32_t* d_visited_bits,
                                   uint32_t* d_candidate_bits, const int32_t* d_frontier_list,
                                   int64_t frontier_count);
 /* ess_bfs_partition_pull, one bottom-up level on the owned rows with the single-GPU pull kernel: every owned
 * vertex outside d_visited_bits that has an in-neighbour in d_frontier_bits gets depth = level, joins visited
 * and d_next_slice (owned words); d_counts[0] += |fresh|. d_counts[1] is not changed: the kernel reads no row
 * bounds of the vertices it adopts, so the sum of their degrees is not known. */
ESS_API int ess_bfs_partition_pull(ess_context_t ctx, ess_graph_t g, int64_t row_begin, int32_t level,
                                   const uint32_t* d_frontier_bits, uint32_t* d_visited_bits,
                                   uint32_t* d_next_slice, int32_t* d_depth_local, int64_t* d_counts);
/* After the all_gather of a level: d_gathered holds `world` rows of (slice_words next-frontier words | 2 x int64
 * counters). Unpacks them into the replicated frontier bitmap, ORs it into the visited bitmap and copies the
 * counters to d_counts_out (2*world int64). Enqueue only. */
ESS_API int ess_bfs_merge_gathered(ess_context_t ctx, const uint32_t* d_gathered, int32_t world, int64_t slice_words,
                                   uint32_t* d_frontier_bits, uint32_t* d_visited_bits, int64_t* d_counts_out);
ESS_API int ess_bfs_absorb(ess_context_t ctx, ess_graph_t g, int64_t row_begin, int32_t level,
                           const uint32_t* d_candidates, int32_t n_slices, int64_t slice_stride_words,
                           uint32_t* d_visited_bits, uint32_t* d_next_slice, int32_t* d_depth_local,
                           int32_t* d_fresh_list, int64_t* d_counts);

/* ---- native multi-GPU BFS driver: the level loop above in C++ with NCCL called directly ----------------
 * One process per GPU. `unique_id`: 128 bytes from ess_nccl_unique_id on rank 0, distributed by the host
 * (e.g. torch.distributed broadcast). `g`: this rank's partition (symmetric = 2, hints built). NCCL is
 * resolved at run time from the libnccl already loaded in the process. ess_dist_bfs runs one whole BFS from
 * the GLOBAL vertex id `source`: info->enact_ms is the device time of the run, iterations/pull_steps the
 * levels, reserved[0] the bytes received per rank. Depths of the owned rows: ess_dist_depth_local. */
typedef struct ess_dist_s* ess_dist_t;
ESS_API int ess_nccl_unique_id(void* out_128_bytes);
ESS_API int ess_dist_create(ess_context_t ctx, ess_graph_t g, int rank, int world, int64_t n_global,
                            const void* unique_id, ess_dist_t* out);
ESS_API int ess_dist_destroy(ess_dist_t d);
ESS_API int ess_dist_bfs(ess_dist_t d, int64_t source, float alpha, float beta, ess_run_info* info);
ESS_API int ess_dist_depth_local(ess_dist_t d, int32_t** d_depth_local, int64_t* count);
/* How ess_dist_bfs moves its bitmaps between ranks: 1 = the library's own peer-memory kernels (every rank maps
 * the others' exchange window with cudaIpcOpenMemHandle at ess_dist_create; a sender stores its slices straight
 * into the receivers' windows over NVLink and raises an epoch flag, the receiver's stream waits on the flags),
 * 0 = NCCL send/recv + all_gather (mapping failed, or ess_tune("dist_peer_exchange", 0)).
 * A rank whose stream waited longer than ess_tune("dist_peer_timeout_ms") (default 4000, wall clock) for a peer's
 * level data returns an error and marks the handle unusable: later ess_dist_bfs / ess_dist_sssp calls on it fail
 * immediately; destroy the handle on every rank and create a new one. */
ESS_API int ess_dist_exchange_kind(ess_dist_t d, int* kind);
ESS_API int ess_dist_copy_depth(ess_dist_t d, int32_t* d_out); /* owned depth slice -> caller buffer, on the stream */

/* ---- multi-GPU SSSP on the same partition (weights in the graph's values; NULL values = weight 1) --------
 * Same fixed point as gunrock::sssp::run (include/gunrock/algorithms/sssp.hxx:110-136: relax with atomic min,
 * keep what improved). Every rank holds a full-length replica of tentative distances: owned entries are exact
 * after each exchange, the rest are this rank's best candidates so far. One relaxation round =
 *   ess_sssp_partition_relax   replica[nbr] = min(replica[nbr], dist_local[src] + w) over the out-edges of the
 *                              active rows (LOCAL ids); enqueue only
 *   reduce_scatter(min)        of the replica: each owner receives the best candidate of its rows (caller's job:
 *                              ncclReduceScatter in place, or torch.distributed)
 *   ess_sssp_partition_collect rows with reduced[v] < dist_local[v] adopt it and are appended to d_active_list;
 *                              d_counts[0] += rows, d_counts[1] += their out-degrees (two int64 the caller zeroes).
 * ess_dist_sssp runs the whole loop natively. When the peers' windows are mapped (ess_dist_exchange_kind == 1 and
 * n_global/world a multiple of 1024) exchange and filter are ONE kernel over peer memory: relax also raises a dirty
 * word per 1024-entry chunk it lowered, and each owner fetches only the dirty chunks of its rows from the peers'
 * replicas (float4 loads over NVLink), takes the minimum and collects what improved; otherwise
 * ncclReduceScatter(min) + ess_sssp_partition_collect. info->iterations = rounds, reserved[0] = bytes received by
 * this rank, reserved[1] = edges relaxed (all ranks), reserved[2] = 1 if the peer-memory path ran. Distances of the
 * owned rows: ess_dist_copy_dist (FLT_MAX = unreachable). */
ESS_API int ess_sssp_partition_relax(ess_context_t ctx, ess_graph_t g, const int32_t* d_active_list,
                                     int64_t active_count, const float* d_dist_local, float* d_replica);
ESS_API int ess_sssp_partition_collect(ess_context_t ctx, ess_graph_t g, const float* d_reduced, float* d_dist_local,
                                       int32_t* d_active_list, int64_t* d_counts);
ESS_API int ess_dist_sssp(ess_dist_t d, int64_t source, ess_run_info* info);

/* The operator-API form of the partitioned run: gunrock::bfs::run / gunrock::sssp::run
 * (include/gunrock/algorithms/bfs.hxx:151-176, sssp.hxx:155-185) on this rank's rows with a gcuda::multi_context_t
 * that carries the partition descriptor — the SAME enactor contract as on one GPU (prepare_frontier ->
 * while(!is_converged) loop(), include/gunrock/framework/enactor.hxx:243-254), loop() = advance::execute<lb>
 * followed by operators::exchange::execute, which routes each level's frontier to the owners over NCCL
 * (the reference throws on more than one context, framework/operators/advance/advance.hxx:125-128).
 * d_depth_global / d_dist_global: caller-owned arrays of n_global entries; on return the OWNED slice
 * [rank*n/P, (rank+1)*n/P) holds the result (other entries are pruning bounds). Collective: every rank calls it. */
ESS_API int ess_dist_bfs_enactor(ess_dist_t dist, int64_t source, int lb, int32_t* d_depth_global, ess_run_info* info);
ESS_API int ess_dist_sssp_enactor(ess_dist_t dist, int64_t source, int lb, float* d_dist_global, ess_run_info* info);
ESS_API int ess_dist_copy_dist(ess_dist_t d, float* d_out);

#ifdef __cplusplus
}
#endif
#endif /* ESSENTIALS_B200_H */
