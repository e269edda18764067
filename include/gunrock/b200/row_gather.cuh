/**
 * @file row_gather.cuh
 * @brief Degree-binned row gather: every listed row sums a per-edge term over its edge list and hands the sum to a
 * per-row finish. PageRank pull (pr.hxx) and both passes of betweenness centrality (bc.hxx) run on it.
 *
 * Rows are binned by degree: [0, short_degree) one thread per row, [short_degree, hub_degree) one warp per row, the
 * rest one CTA (256 threads) per row; each bin is one launch. The order of every sum depends on the row's degree alone:
 * one thread walks the list in order; a warp's lanes stride it by 32 and warp_sum reduces them; a CTA's threads stride
 * it by 256, warp_sum reduces each warp and thread 0 adds the 8 warp totals in warp order. Callers that promise
 * byte-identical results (bc.hxx) rely on this order.
 */
#pragma once

#include <gunrock/b200/warp.cuh>
#include <gunrock/cuda/launch.hxx>

namespace gunrock {
namespace b200 {

constexpr int short_degree = 8;   // below: one thread per row
constexpr int hub_degree = 4096;  // from here: one CTA per row

/// Launch mode of a row of `degree` edges: 0 one thread, 1 one warp, 2 one CTA.
__host__ __device__ __forceinline__ int degree_bin(long long degree) {
  return degree < short_degree ? 0 : degree < hub_degree ? 1 : 2;
}

/// Up to three runs of row ids walked as one list of size[0] + size[1] + size[2] rows; unused runs have size 0.
template <typename vertex_t>
struct row_runs_t {
  const vertex_t* begin[3];
  counter_t size[3];
  counter_t count() const { return size[0] + size[1] + size[2]; }
  __device__ __forceinline__ vertex_t operator[](counter_t i) const {
    if (i < size[0]) return __ldg(begin[0] + i);
    i -= size[0];
    if (i < size[1]) return __ldg(begin[1] + i);
    return __ldg(begin[2] + (i - size[1]));
  }
};

namespace kernels {
/// Rows of bin `mode` (file comment): the threads on row v call sum(first, end, step) -> double over their strided
/// shares of [offsets[v], offsets[v + 1]), the shares are reduced in the fixed tree, and one thread calls
/// finish(v, total). `finish` is each thread's own copy: start() before its first row, flush() after its last (by the
/// whole warp). n_rows == rows.count(), passed in so that the compiler keeps the CTA loop of mode 2 uniform.
template <int mode, typename vertex_t, typename edge_t, typename sum_t, typename finish_t>
__global__ void __launch_bounds__(256)
    row_gather_kernel(const edge_t* __restrict__ offsets, row_runs_t<vertex_t> rows, counter_t n_rows, sum_t sum,
                      finish_t finish) {
  constexpr unsigned width = mode == 0 ? 1 : mode == 1 ? 32 : 256;  // threads per row
  __shared__ double block_acc[256 / 32];
  finish.start();
  const unsigned rank = threadIdx.x % width;
  // mode 2 takes the CTA index as is: the same value, but one the compiler sees is uniform across the CTA
  const counter_t first = mode == 2 ? blockIdx.x : (counter_t(blockIdx.x) * blockDim.x + threadIdx.x) / width;
  const counter_t stride = mode == 2 ? gridDim.x : counter_t(gridDim.x) * blockDim.x / width;
  for (counter_t i = first; i < n_rows; i += stride) {
    const vertex_t v = rows[i];
    double acc = sum(edge_t(offsets[v] + rank), offsets[v + 1], edge_t(width));
    if constexpr (mode > 0) acc = warp_sum(acc);
    if constexpr (mode == 2) {
      if (lane_id() == 0) block_acc[warp_id()] = acc;
      __syncthreads();
      if (rank == 0) {
        acc = 0;
        for (int k = 0; k < 256 / 32; ++k) acc = __dadd_rn(acc, block_acc[k]);
      }
      __syncthreads();
    }
    if (rank == 0) finish(v, acc);
  }
  finish.flush();
}
}  // namespace kernels

/// One launch of kernels::row_gather_kernel per non-empty list: rows[0] one thread per row, rows[1] one warp per row,
/// rows[2] one CTA per row.
template <typename vertex_t, typename edge_t, typename sum_t, typename finish_t>
void row_gather(gcuda::standard_context_t& ctx, const edge_t* offsets, const row_runs_t<vertex_t> (&rows)[3], sum_t sum,
                finish_t finish) {
  auto stream = ctx.stream();
  for (int mode = 0; mode < 3; ++mode) {
    const counter_t n_rows = rows[mode].count();
    if (!n_rows) continue;
    const counter_t per_cta = mode == 0 ? 256 : mode == 1 ? 8 : 1;  // rows one CTA works on at a time
    const unsigned grid = gcuda::persistent_grid(ctx, (n_rows + per_cta - 1) / per_cta, 8);
    if (mode == 0)
      kernels::row_gather_kernel<0><<<grid, 256, 0, stream>>>(offsets, rows[0], n_rows, sum, finish);
    else if (mode == 1)
      kernels::row_gather_kernel<1><<<grid, 256, 0, stream>>>(offsets, rows[1], n_rows, sum, finish);
    else
      kernels::row_gather_kernel<2><<<grid, 256, 0, stream>>>(offsets, rows[2], n_rows, sum, finish);
    ctx.profiler().launches_total += 1;
  }
}

}  // namespace b200
}  // namespace gunrock
