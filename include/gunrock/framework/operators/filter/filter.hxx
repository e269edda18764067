/**
 * @file filter.hxx
 * @brief operators::filter::execute — keep the frontier elements for which op(v) is true.
 *
 * Signatures as the reference (include/gunrock/framework/operators/filter/filter.hxx:59-67 explicit,
 * :128-152 enactor form, which ALWAYS swaps buffers unless told not to). Contract shared by all four
 * algorithms, as in the reference wrappers (predicated.hxx:24-26, compact.hxx:23-27, bypass.hxx:29-34,
 * remove.hxx:23-25): invalid (-1) elements never reach op; op may have side effects and runs exactly once
 * per valid element.
 *
 *   predicated : stable compaction in ONE pass — load (128-bit), evaluate op, CTA scan, decoupled
 *                look-back for the tile offset, scatter. (reference: thrust::copy_if)
 *   remove     : same result as predicated — the reference negates the predicate twice
 *                (remove_copy_if(!op), remove.hxx:23-34) — same kernel.
 *   compact    : two passes like mgpu::transform_compact (compact.hxx:20-36): upsweep evaluates op once,
 *                stores a keep-bit per element and counts; the host sizes the output exactly; downsweep
 *                scatters. Stable.
 *   bypass     : no compaction: out[i] = keep ? in[i] : -1, in place allowed (bypass.hxx:19-22,48-55).
 */
#pragma once

#include <gunrock/cuda/cuda.hxx>
#include <gunrock/error.hxx>
#include <gunrock/b200/lookback.cuh>
#include <gunrock/framework/operators/configs.hxx>
#include <gunrock/util/type_limits.hxx>

namespace gunrock {
namespace operators {
namespace filter {

namespace kernels {

using b200::counter_t;
using gcuda::scratch_t;
constexpr int cta_threads = 256;
constexpr int items = 4;
constexpr int per_tile = cta_threads * items;

/// 16-byte alignment of a 128-bit access. Filter inputs and outputs are caller buffers, which may be tensor views
/// at any element offset.
template <typename type_t>
__device__ __forceinline__ bool vector_aligned(const type_t* p) {
  return (reinterpret_cast<std::uintptr_t>(p) & 15u) == 0;
}

template <typename type_t>
__device__ __forceinline__ void load_items(const type_t* __restrict__ in, std::size_t first, std::size_t count,
                                           type_t (&v)[items]) {
  if (sizeof(type_t) == 4 && first + items <= count && vector_aligned(in)) {
    const int4 q = *reinterpret_cast<const int4*>(in + first);
    v[0] = type_t(q.x), v[1] = type_t(q.y), v[2] = type_t(q.z), v[3] = type_t(q.w);
  } else {
#pragma unroll
    for (int k = 0; k < items; ++k) v[k] = first + k < count ? in[first + k] : gunrock::numeric_limits<type_t>::invalid();
  }
}

/// Single-pass stable select (predicated / remove).
template <typename type_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads)
    select_kernel(const type_t* __restrict__ in, std::size_t count, type_t* __restrict__ out, operator_t op,
                  b200::tile_word_t* state, counter_t* counters) {
  __shared__ unsigned scan_u[cta_threads / 32 + 1];
  __shared__ unsigned long long prefix;
  __shared__ int s_tile;
  const int n_tiles = int((count + per_tile - 1) / per_tile);
  for (;;) {
    if (threadIdx.x == 0) s_tile = int(atomicAdd(counters + scratch_t::ticket, counter_t(1)));
    __syncthreads();
    const int tile = s_tile;
    if (tile >= n_tiles) break;
    const std::size_t first = std::size_t(tile) * per_tile + std::size_t(threadIdx.x) * items;
    type_t v[items];
    load_items(in, first, count, v);
    unsigned keep = 0;
#pragma unroll
    for (int k = 0; k < items; ++k)
      if (gunrock::util::limits::is_valid(v[k]) && op(v[k])) keep |= 1u << k;
    unsigned tile_kept;
    const unsigned before = b200::cta_exclusive_sum<cta_threads, unsigned>(__popc(keep), tile_kept, scan_u);
    if (threadIdx.x < 32) {
      const unsigned long long p = b200::lookback_exclusive(state, tile, tile_kept);
      if (threadIdx.x == 0) prefix = p;
    }
    __syncthreads();
    std::size_t at = std::size_t(prefix) + before;
#pragma unroll
    for (int k = 0; k < items; ++k)
      if (keep & (1u << k)) out[at++] = v[k];
    if (tile == n_tiles - 1 && threadIdx.x == 0) counters[scratch_t::out_count] = prefix + tile_kept;
    __syncthreads();
  }
}

/// compact, upsweep: evaluate op once per element, record 4 keep-bits per thread, per-tile counts.
template <typename type_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads)
    compact_upsweep_kernel(const type_t* __restrict__ in, std::size_t count, operator_t op,
                           unsigned char* __restrict__ keep_bits, unsigned* __restrict__ tile_counts,
                           counter_t* counters) {
  __shared__ unsigned scan_u[cta_threads / 32 + 1];
  const int n_tiles = int((count + per_tile - 1) / per_tile);
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const std::size_t first = std::size_t(tile) * per_tile + std::size_t(threadIdx.x) * items;
    type_t v[items];
    load_items(in, first, count, v);
    unsigned keep = 0;
#pragma unroll
    for (int k = 0; k < items; ++k)
      if (gunrock::util::limits::is_valid(v[k]) && op(v[k])) keep |= 1u << k;
    keep_bits[std::size_t(tile) * cta_threads + threadIdx.x] = (unsigned char)keep;
    unsigned tile_kept;
    b200::cta_exclusive_sum<cta_threads, unsigned>(__popc(keep), tile_kept, scan_u);
    if (threadIdx.x == 0) {
      tile_counts[tile] = tile_kept;
      atomicAdd(counters + scratch_t::out_count, counter_t(tile_kept));
    }
    __syncthreads();
  }
}

/// compact, middle: exclusive scan of the per-tile counts by one CTA (n_tiles is small: count/1024).
static __global__ void __launch_bounds__(1024) compact_scan_tiles_kernel(unsigned* tile_counts, unsigned long long* tile_offsets,
                                                                  int n_tiles) {
  __shared__ unsigned long long scan_e[1024 / 32 + 1];
  __shared__ unsigned long long carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < n_tiles; base += 1024) {
    const int i = base + threadIdx.x;
    unsigned long long x = i < n_tiles ? tile_counts[i] : 0ull, total;
    const unsigned long long before = b200::cta_exclusive_sum<1024, unsigned long long>(x, total, scan_e);
    if (i < n_tiles) tile_offsets[i] = carry + before;
    __syncthreads();
    if (threadIdx.x == 0) carry += total;
    __syncthreads();
  }
}

/// compact, downsweep: scatter the kept elements to their final, stable positions.
template <typename type_t>
__global__ void __launch_bounds__(cta_threads)
    compact_downsweep_kernel(const type_t* __restrict__ in, std::size_t count, type_t* __restrict__ out,
                             const unsigned char* __restrict__ keep_bits,
                             const unsigned long long* __restrict__ tile_offsets) {
  __shared__ unsigned scan_u[cta_threads / 32 + 1];
  const int n_tiles = int((count + per_tile - 1) / per_tile);
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const std::size_t first = std::size_t(tile) * per_tile + std::size_t(threadIdx.x) * items;
    const unsigned keep = keep_bits[std::size_t(tile) * cta_threads + threadIdx.x];
    unsigned tile_kept;
    const unsigned before = b200::cta_exclusive_sum<cta_threads, unsigned>(__popc(keep), tile_kept, scan_u);
    if (keep) {
      type_t v[items];
      load_items(in, first, count, v);
      std::size_t at = std::size_t(tile_offsets[tile]) + before;
#pragma unroll
      for (int k = 0; k < items; ++k)
        if (keep & (1u << k)) out[at++] = v[k];
    }
    __syncthreads();
  }
}

/// bypass: streaming map, 128-bit in / 128-bit out, in-place safe (each thread reads before it writes).
template <typename type_t, typename operator_t>
__global__ void __launch_bounds__(cta_threads)
    bypass_kernel(const type_t* in, std::size_t count, type_t* out, operator_t op) {
  const std::size_t stride = std::size_t(gridDim.x) * cta_threads * items;
  for (std::size_t first = (std::size_t(blockIdx.x) * cta_threads + threadIdx.x) * items; first < count;
       first += stride) {
    type_t v[items];
    load_items(in, first, count, v);
#pragma unroll
    for (int k = 0; k < items; ++k)
      if (gunrock::util::limits::is_valid(v[k]) && !op(v[k])) v[k] = gunrock::numeric_limits<type_t>::invalid();
    if (sizeof(type_t) == 4 && first + items <= count && vector_aligned(out)) {
      *reinterpret_cast<int4*>(out + first) = make_int4(int(v[0]), int(v[1]), int(v[2]), int(v[3]));
    } else {
#pragma unroll
      for (int k = 0; k < items; ++k)
        if (first + k < count) out[first + k] = v[k];
    }
  }
}

}  // namespace kernels

namespace detail {
using gcuda::scratch_t;

template <typename frontier_t>
void ensure(frontier_t* f, std::size_t elements) {
  if (f->get_capacity() < elements) f->reserve(elements);
}

template <typename graph_t, typename operator_t, typename frontier_t>
void select(graph_t&, operator_t op, frontier_t* input, frontier_t* output, gcuda::standard_context_t& ctx) {
  using type_t = typename frontier_t::type_t;
  const std::size_t count = input->get_number_of_elements();
  if (!count) {
    output->set_number_of_elements(0);
    return;
  }
  error::throw_if_exception(input->data() == output->data(), "filter: compacting filters cannot run in place");
  ensure(output, count);
  auto& scratch = ctx.scratch();
  auto stream = ctx.stream();
  const std::size_t n_tiles = (count + kernels::per_tile - 1) / kernels::per_tile;
  auto* state = reinterpret_cast<b200::tile_word_t*>(scratch.temp(n_tiles * sizeof(b200::tile_word_t)));
  scratch.zero(stream);
  cudaMemsetAsync(state, 0, n_tiles * sizeof(b200::tile_word_t), stream);
  ctx.profiler().begin(gcuda::profiler_t::filter_op, stream);
  kernels::select_kernel<type_t><<<gcuda::persistent_grid(ctx, n_tiles, 6), 256, 0, stream>>>(
      input->data(), count, output->data(), op, state, scratch.d);
  ctx.profiler().end(stream);
  error::check_last("filter select");
  scratch.fetch(stream);
  output->set_number_of_elements(std::size_t(scratch.h[scratch_t::out_count]));
}

template <typename graph_t, typename operator_t, typename frontier_t>
void compact(graph_t&, operator_t op, frontier_t* input, frontier_t* output, gcuda::standard_context_t& ctx) {
  using type_t = typename frontier_t::type_t;
  const std::size_t count = input->get_number_of_elements();
  if (!count) {
    output->set_number_of_elements(0);
    return;
  }
  error::throw_if_exception(input->data() == output->data(), "filter: compacting filters cannot run in place");
  auto& scratch = ctx.scratch();
  auto stream = ctx.stream();
  const std::size_t n_tiles = (count + kernels::per_tile - 1) / kernels::per_tile;
  gcuda::arena_layout_t layout;
  const std::size_t at_bits = layout.add(n_tiles * kernels::cta_threads);
  const std::size_t at_counts = layout.add(n_tiles * sizeof(unsigned));
  const std::size_t at_offsets = layout.add(n_tiles * sizeof(unsigned long long));
  unsigned char* base = scratch.temp(layout.bytes);
  auto* tile_counts = reinterpret_cast<unsigned*>(base + at_counts);
  auto* tile_offsets = reinterpret_cast<unsigned long long*>(base + at_offsets);
  scratch.zero(stream);
  const unsigned grid = gcuda::persistent_grid(ctx, n_tiles, 6);
  ctx.profiler().begin(gcuda::profiler_t::filter_op, stream);
  kernels::compact_upsweep_kernel<type_t><<<grid, 256, 0, stream>>>(input->data(), count, op, base + at_bits,
                                                                    tile_counts, scratch.d);
  kernels::compact_scan_tiles_kernel<<<1, 1024, 0, stream>>>(tile_counts, tile_offsets, int(n_tiles));
  ctx.profiler().end(stream, 2);
  error::check_last("filter compact upsweep");
  scratch.fetch(stream);  // exact size known here: allocate exactly, then scatter
  const std::size_t kept = std::size_t(scratch.h[scratch_t::out_count]);
  ensure(output, kept);
  output->set_number_of_elements(kept);
  if (kept) {
    ctx.profiler().begin(gcuda::profiler_t::filter_op, stream);
    kernels::compact_downsweep_kernel<type_t><<<grid, 256, 0, stream>>>(input->data(), count, output->data(),
                                                                        base + at_bits, tile_offsets);
    ctx.profiler().end(stream);
    error::check_last("filter compact downsweep");
    ctx.synchronize();
  }
}

template <typename graph_t, typename operator_t, typename frontier_t>
void bypass(graph_t&, operator_t op, frontier_t* input, frontier_t* output, gcuda::standard_context_t& ctx) {
  using type_t = typename frontier_t::type_t;
  const std::size_t count = input->get_number_of_elements();
  if (output->data() != input->data()) ensure(output, count);
  output->set_number_of_elements(count);
  if (!count) return;
  const std::size_t ctas = (count + kernels::per_tile - 1) / kernels::per_tile;
  ctx.profiler().begin(gcuda::profiler_t::filter_op, ctx.stream());
  kernels::bypass_kernel<type_t><<<gcuda::persistent_grid(ctx, ctas, 8), 256, 0, ctx.stream()>>>(
      input->data(), count, output->data(), op);
  ctx.profiler().end(ctx.stream());
  error::check_last("filter bypass");
  ctx.synchronize();
}
}  // namespace detail

/// Explicit-buffers form (reference filter.hxx:59-86).
template <filter_algorithm_t alg_type, typename graph_t, typename operator_t, typename frontier_t>
void execute(graph_t& G, operator_t op, frontier_t* input, frontier_t* output, gcuda::multi_context_t& context) {
  error::throw_if_exception(context.size() != 1, "`context.size() != 1` not supported");
  auto* ctx = context.get_context(0);
  if constexpr (alg_type == filter_algorithm_t::compact)
    detail::compact(G, op, input, output, *ctx);
  else if constexpr (alg_type == filter_algorithm_t::predicated || alg_type == filter_algorithm_t::remove)
    detail::select(G, op, input, output, *ctx);
  else if constexpr (alg_type == filter_algorithm_t::bypass)
    detail::bypass(G, op, input, output, *ctx);
  else
    error::throw_if_exception(cudaErrorUnknown, "Filter type not supported.");
}

/// Enactor form (reference filter.hxx:128-152).
template <filter_algorithm_t alg_type, typename graph_t, typename enactor_type, typename operator_t>
void execute(graph_t& G, enactor_type* E, operator_t op, gcuda::multi_context_t& context, bool swap_buffers = true) {
  execute<alg_type>(G, op, E->get_input_frontier(), E->get_output_frontier(), context);
  if (swap_buffers) E->swap_frontier_buffers();
}

}  // namespace filter
}  // namespace operators
}  // namespace gunrock
