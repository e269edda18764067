/**
 * @file frontier.hxx
 * @brief Frontier storage: the sparse vector view (list of ids, invalid = -1 holes allowed) and the dense
 * bit-packed view (1 bit per vertex), plus the sparse<->dense conversions.
 *
 * Sparse view keeps the reference's interface (include/gunrock/framework/frontier/frontier.hxx:37-148,
 * vector_frontier.hxx:29-256): push_back, fill, sequence, resize, reserve(size*factor), get/set_element_at,
 * data/begin/end, is_empty, get/set_number_of_elements, get_capacity, print; host copies share storage,
 * device copies carry the raw pointer (vector_frontier.hxx:65-74) so a frontier captured by value in a
 * device lambda sees the live buffer. Storage is a plain cudaMalloc'd buffer (no thrust::device_vector).
 *
 * Dense view: the reference's boolmap_frontier_t (frontier/experimental/boolmap_frontier.hxx:25-202) keeps
 * one 4-byte flag per vertex and re-reduces the whole array on every size query; it is not wired into
 * frontier_t (frontier.hxx:22,56-57). Here `bitmap` and `boolmap` name the same bit-packed class
 * (32 vertices per word, so a scale-26 frontier is 8 MiB and lives in L2): get_element_at(i) -> i or invalid,
 * set_element_at(v) sets bit v atomically, the population count is computed by a __popc kernel only when
 * the map was written since the last query.
 */
#pragma once

#include <cstdio>
#include <memory>
#include <type_traits>
#include <vector>

#include <gunrock/cuda/cuda.hxx>
#include <gunrock/framework/frontier/configs.hxx>
#include <gunrock/util/type_limits.hxx>
#include <gunrock/util/load_store.hxx>
#include <gunrock/b200/warp.cuh>

namespace gunrock {
namespace frontier {
using namespace memory;

/// CTAs of a grid-stride streaming kernel over `items` elements: SMs of the current device x 8, at most.
inline unsigned stream_ctas(std::size_t items) {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 1;
  }
  const std::size_t cap = std::size_t(sms) * 8, c = (items + 255) / 256;
  return unsigned(c < cap ? (c ? c : 1) : cap);
}

namespace kernels {

template <typename type_t>
__global__ void __launch_bounds__(256) fill_kernel(type_t* out, std::size_t count, type_t value) {
  for (std::size_t i = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count;
       i += std::size_t(gridDim.x) * blockDim.x)
    out[i] = value;
}

/// out[i] = first + i, four elements per thread through one 128-bit store when aligned.
template <typename type_t>
__global__ void __launch_bounds__(256) iota_kernel(type_t* out, std::size_t count, type_t first) {
  const std::size_t stride = std::size_t(gridDim.x) * blockDim.x;
  if constexpr (sizeof(type_t) == 4) {
    const std::size_t quads = count / 4;
    int4* out4 = reinterpret_cast<int4*>(out);  // only a frontier's own cudaMalloc'd base: 256-byte aligned
    for (std::size_t q = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; q < quads; q += stride) {
      int b = int(first) + int(q * 4);
      out4[q] = make_int4(b, b + 1, b + 2, b + 3);
    }
    for (std::size_t i = quads * 4 + std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += stride)
      out[i] = first + type_t(i);
  } else {
    for (std::size_t i = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += stride)
      out[i] = first + type_t(i);
  }
}

/// Sparse -> dense: set bit v for every valid v in the list.
template <typename type_t>
__global__ void __launch_bounds__(256)
    scatter_bits_kernel(const type_t* __restrict__ list, std::size_t count, unsigned* __restrict__ words) {
  for (std::size_t i = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count;
       i += std::size_t(gridDim.x) * blockDim.x) {
    type_t v = list[i];
    if (util::limits::is_valid(v)) atomicOr(&words[std::size_t(v) >> 5], 1u << (unsigned(v) & 31u));
  }
}

/// Population count of a word array into *total (warp shuffle reduce, one atomic per warp).
static __global__ void __launch_bounds__(256)
    popcount_kernel(const unsigned* __restrict__ words, std::size_t n_words, b200::counter_t* total) {
  unsigned long long mine = 0;
  for (std::size_t w = std::size_t(blockIdx.x) * blockDim.x + threadIdx.x; w < n_words;
       w += std::size_t(gridDim.x) * blockDim.x)
    mine += __popc(words[w]);
  mine = b200::warp_sum(mine);
  if (b200::lane_id() == 0 && mine) atomicAdd(total, mine);
}

/**
 * @brief Dense -> sparse: ordered list of set bits. One warp per 32 words (1024 vertices): lanes popcount
 * their word, a shuffle scan gives each lane its offset, one atomic per warp claims the range; output is
 * ascending within a warp's range (ranges themselves land in claim order).
 */
template <typename type_t>
__global__ void __launch_bounds__(256) gather_bits_kernel(const unsigned* __restrict__ words, std::size_t n_words,
                                                         type_t* __restrict__ list, b200::counter_t* count) {
  const unsigned lane = b200::lane_id();
  const std::size_t warps = (std::size_t(gridDim.x) * blockDim.x) >> 5;
  for (std::size_t base = ((std::size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5) * 32; base < n_words;
       base += warps * 32) {
    std::size_t w = base + lane;
    unsigned bits = w < n_words ? words[w] : 0u;
    unsigned mine = __popc(bits);
    unsigned incl = b200::warp_inclusive_sum(mine);
    unsigned total = __shfl_sync(b200::full_mask, incl, 31);
    if (total == 0) continue;
    b200::counter_t at = 0;
    if (lane == 0) at = atomicAdd(count, b200::counter_t(total));
    at = __shfl_sync(b200::full_mask, at, 0) + (incl - mine);
    while (bits) {
      unsigned b = __ffs(bits) - 1;
      bits &= bits - 1;
      list[at++] = type_t(w * 32 + b);
    }
  }
}

}  // namespace kernels

/// Shared, growable device storage behind a frontier (what the reference keeps in a
/// shared_ptr<device_vector>, vector_frontier.hxx:252). Growth keeps the first `live` elements.
template <typename type_t>
struct frontier_storage_t {
  type_t* ptr = nullptr;
  std::size_t cap = 0;
  frontier_storage_t() = default;
  frontier_storage_t(const frontier_storage_t&) = delete;
  frontier_storage_t& operator=(const frontier_storage_t&) = delete;
  ~frontier_storage_t() { memory::free(ptr); }
  void grow(std::size_t n, std::size_t live) {
    if (n <= cap) return;
    type_t* fresh = memory::allocate<type_t>(n * sizeof(type_t));
    if (ptr) {
      if (live)
        error::throw_if_exception(cudaMemcpy(fresh, ptr, live * sizeof(type_t), cudaMemcpyDeviceToDevice),
                                  "frontier grow");
      memory::free(ptr);
    }
    ptr = fresh;
    cap = n;
  }
};

template <typename vertex_t, typename edge_t, frontier_kind_t _kind>
class vector_frontier_t {
 public:
  using type_t = std::conditional_t<_kind == frontier_kind_t::vertex_frontier, vertex_t, edge_t>;

  vector_frontier_t() : raw_ptr(nullptr), num_elements(0), resizing_factor(1.0f) {
    p_storage = std::make_shared<frontier_storage_t<type_t>>();
  }
  vector_frontier_t(std::size_t size, float frontier_resizing_factor = 1.0f)
      : raw_ptr(nullptr), num_elements(size), resizing_factor(frontier_resizing_factor) {
    p_storage = std::make_shared<frontier_storage_t<type_t>>();
    p_storage->grow(size, 0);
    raw_ptr = p_storage->ptr;
  }
  ~vector_frontier_t() {}

  __host__ __device__ vector_frontier_t(const vector_frontier_t& rhs) {
#ifdef __CUDA_ARCH__
    raw_ptr = rhs.raw_ptr;
#else
    p_storage = rhs.p_storage;
    raw_ptr = rhs.p_storage ? rhs.p_storage->ptr : nullptr;
#endif
    num_elements = rhs.num_elements;
    resizing_factor = rhs.resizing_factor;
  }
  vector_frontier_t& operator=(const vector_frontier_t& rhs) {
    p_storage = rhs.p_storage;
    raw_ptr = rhs.p_storage ? rhs.p_storage->ptr : nullptr;
    num_elements = rhs.num_elements;
    resizing_factor = rhs.resizing_factor;
    return *this;
  }

  __host__ __device__ __forceinline__ std::size_t get_number_of_elements(gcuda::stream_t = 0) const {
    return num_elements;
  }
  std::size_t get_capacity() const { return p_storage->cap; }
  float get_resizing_factor() const { return resizing_factor; }
  void set_resizing_factor(float factor) { resizing_factor = factor; }
  void set_number_of_elements(std::size_t const& elements) { num_elements = elements; }

  __device__ __forceinline__ type_t get_element_at(std::size_t const& idx) const noexcept {
    return thread::load(raw_ptr + idx);
  }
  __device__ __forceinline__ void set_element_at(type_t const& element, std::size_t const& idx) const noexcept {
    thread::store(raw_ptr + idx, element);
  }

  __host__ __device__ __forceinline__ type_t* get() const { return raw_ptr; }
  type_t* data() { return sync_ptr(); }
  type_t* begin() { return sync_ptr(); }
  type_t* end() { return sync_ptr() + num_elements; }
  bool is_empty() const { return num_elements == 0; }

  void push_back(type_t const& value) {
    if (num_elements + 1 > get_capacity()) reserve_exact((num_elements + 1) * 2 + 62);
    error::throw_if_exception(
        cudaMemcpy(sync_ptr() + num_elements, &value, sizeof(type_t), cudaMemcpyHostToDevice), "frontier push_back");
    ++num_elements;
  }

  void fill(type_t const value, gcuda::stream_t stream = 0) {
    if (!num_elements) return;
    kernels::fill_kernel<<<launch_ctas(num_elements), 256, 0, stream>>>(sync_ptr(), num_elements, value);
  }

  /// Frontier = {first, first+1, ...}: `size` elements (grows the buffer when needed).
  void sequence(type_t const initial_value, std::size_t const& size, gcuda::stream_t stream = 0) {
    if (get_capacity() < size) reserve(size);
    num_elements = size;
    if (size) kernels::iota_kernel<<<launch_ctas((size + 3) / 4), 256, 0, stream>>>(sync_ptr(), size, initial_value);
  }

  /// Grow the buffer to `size` slots; slots beyond the current length are set to `default_value`.
  void resize(std::size_t const& size, type_t const default_value = gunrock::numeric_limits<type_t>::invalid()) {
    reserve_exact(size);
    if (size > num_elements)
      kernels::fill_kernel<<<launch_ctas(size - num_elements), 256>>>(sync_ptr() + num_elements, size - num_elements,
                                                                       default_value);
  }

  /// Capacity of at least size * resizing_factor (same rule as the reference); contents are kept.
  void reserve(std::size_t const& size) { reserve_exact(std::size_t(double(size) * double(resizing_factor))); }

  void print() {
    std::vector<type_t> h(num_elements);
    if (num_elements) cudaMemcpy(h.data(), sync_ptr(), num_elements * sizeof(type_t), cudaMemcpyDeviceToHost);
    std::printf("Frontier = ");
    for (auto x : h) std::printf("%lld ", (long long)x);
    std::printf("\n");
  }

 protected:
  static unsigned launch_ctas(std::size_t items) { return stream_ctas(items); }
  void reserve_exact(std::size_t n) {
    p_storage->grow(n, num_elements < p_storage->cap ? num_elements : p_storage->cap);
    raw_ptr = p_storage->ptr;
  }
  type_t* sync_ptr() {
    raw_ptr = p_storage->ptr;
    return raw_ptr;
  }

 private:
  std::shared_ptr<frontier_storage_t<type_t>> p_storage;
  type_t* raw_ptr;
  std::size_t num_elements;
  float resizing_factor;
};

/**
 * @brief Dense, bit-packed frontier over the id range [0, universe). Word w holds ids 32w..32w+31.
 */
template <typename vertex_t, typename edge_t, frontier_kind_t _kind>
class bitmap_frontier_t {
 public:
  using type_t = std::conditional_t<_kind == frontier_kind_t::vertex_frontier, vertex_t, edge_t>;
  using word_t = unsigned;

  bitmap_frontier_t() : raw_ptr(nullptr), universe(0), cached_count(0), dirty(false) {
    p_storage = std::make_shared<frontier_storage_t<word_t>>();
  }
  explicit bitmap_frontier_t(std::size_t size, float = 1.0f) : bitmap_frontier_t() { resize(size); }
  ~bitmap_frontier_t() {}

  __host__ __device__ bitmap_frontier_t(const bitmap_frontier_t& rhs) {
#ifdef __CUDA_ARCH__
    raw_ptr = rhs.raw_ptr;
#else
    p_storage = rhs.p_storage;
    raw_ptr = rhs.p_storage ? rhs.p_storage->ptr : nullptr;
#endif
    universe = rhs.universe;
    cached_count = rhs.cached_count;
    dirty = rhs.dirty;
  }

  /// Number of words backing the map.
  __host__ __device__ __forceinline__ std::size_t words() const { return (universe + 31) / 32; }
  __host__ __device__ __forceinline__ std::size_t get_universe() const { return universe; }
  std::size_t get_capacity() const { return p_storage->cap * 32; }

  /// Resize the id universe; new bits are cleared (old bits kept).
  void resize(std::size_t size, gcuda::stream_t stream = 0) {
    std::size_t old_words = words();
    universe = size;
    p_storage->grow(words() + 4, old_words);  // +1 padding word, +2..3 the size-query counter (8-byte aligned)
    raw_ptr = p_storage->ptr;
    if (words() + 1 > old_words)
      cudaMemsetAsync(raw_ptr + old_words, 0, (words() + 1 - old_words) * sizeof(word_t), stream);
  }
  void reserve(std::size_t size) {
    if (size > universe) resize(size);
  }

  /// fill(0) clears, fill(1) sets every id (the reference's guard `value!=0 || value!=1` always throws,
  /// boolmap_frontier.hxx:147-149; the intent is implemented here).
  void fill(int value, gcuda::stream_t stream = 0) {
    error::throw_if_exception(value != 0 && value != 1, "bitmap frontier: fill value must be 0 or 1");
    if (!universe) return;
    cudaMemsetAsync(raw_ptr, value ? 0xff : 0, words() * sizeof(word_t), stream);
    if (value && (universe & 31)) {  // keep the padding bits of the last word clear
      word_t last = (1u << (universe & 31)) - 1u;
      cudaMemcpyAsync(raw_ptr + words() - 1, &last, sizeof(word_t), cudaMemcpyHostToDevice, stream);
      cudaStreamSynchronize(stream);
    }
    cached_count = value ? universe : 0;
    dirty = false;
  }

  __device__ __forceinline__ type_t get_element_at(std::size_t const& idx) const noexcept {
    return ((raw_ptr[idx >> 5] >> (idx & 31)) & 1u) ? type_t(idx) : gunrock::numeric_limits<type_t>::invalid();
  }
  /// Activates `element`; `idx` is ignored (same signature as the vector view).
  __device__ __forceinline__ void set_element_at(type_t const& element, std::size_t const& = 0) const noexcept {
    atomicOr(raw_ptr + (std::size_t(element) >> 5), 1u << (unsigned(element) & 31u));
  }
  __device__ __forceinline__ bool contains(type_t const& element) const noexcept {
    return (raw_ptr[std::size_t(element) >> 5] >> (unsigned(element) & 31u)) & 1u;
  }

  /// Number of active ids; runs a popcount kernel only if the map changed since the last query.
  std::size_t get_number_of_elements(gcuda::stream_t stream = 0) {
    if (dirty) {
      // the counter lives in the spare word pair behind the map (storage is words() + 3): no allocation per query
      auto* d_total = reinterpret_cast<b200::counter_t*>(raw_ptr + ((words() + 2) & ~std::size_t(1)));
      cudaMemsetAsync(d_total, 0, sizeof(b200::counter_t), stream);
      kernels::popcount_kernel<<<stream_ctas(words()), 256, 0, stream>>>(raw_ptr, words(), d_total);
      b200::counter_t h = 0;
      cudaMemcpyAsync(&h, d_total, sizeof(h), cudaMemcpyDeviceToHost, stream);
      cudaStreamSynchronize(stream);
      cached_count = std::size_t(h);
      dirty = false;
    }
    return cached_count;
  }
  void set_number_of_elements(std::size_t const& count) {
    cached_count = count;
    dirty = false;
  }
  /// Tell the map that device code wrote bits (next size query recounts).
  void mark_dirty() { dirty = true; }
  bool is_empty(gcuda::stream_t stream = 0) { return get_number_of_elements(stream) == 0; }

  __host__ __device__ __forceinline__ word_t* get() const { return raw_ptr; }
  word_t* data() {
    raw_ptr = p_storage->ptr;
    return raw_ptr;
  }
  void print() { std::printf("Bitmap frontier: %zu of %zu active\n", get_number_of_elements(), universe); }

 private:
  std::shared_ptr<frontier_storage_t<word_t>> p_storage;
  word_t* raw_ptr;
  std::size_t universe;
  std::size_t cached_count;
  bool dirty;
};

namespace detail {
template <typename vertex_t, typename edge_t, frontier_kind_t kind, frontier_view_t view>
using underlying_t = std::conditional_t<view == frontier_view_t::vector, vector_frontier_t<vertex_t, edge_t, kind>,
                                        bitmap_frontier_t<vertex_t, edge_t, kind>>;
}

template <typename vertex_t, typename edge_t, frontier_kind_t _kind = frontier_kind_t::vertex_frontier,
          frontier_view_t _view = frontier_view_t::vector>
class frontier_t : public detail::underlying_t<vertex_t, edge_t, _kind, _view> {
 public:
  using vertex_type = vertex_t;
  using edge_type = edge_t;
  using type_t = std::conditional_t<_kind == frontier_kind_t::vertex_frontier, vertex_t, edge_t>;
  using offset_t = std::conditional_t<_kind == frontier_kind_t::vertex_frontier, edge_t, vertex_t>;
  using frontier_type = frontier_t<vertex_t, edge_t, _kind, _view>;
  using underlying_view_t = detail::underlying_t<vertex_t, edge_t, _kind, _view>;

  frontier_t() : underlying_view_t() {}
  frontier_t(std::size_t size, float frontier_resizing_factor = 1.0f)
      : underlying_view_t(size, frontier_resizing_factor) {}
  ~frontier_t() {}
  __host__ __device__ frontier_t(const frontier_t& rhs) : underlying_view_t(rhs) {}
  frontier_t& operator=(const frontier_t& rhs) = default;

  __host__ __device__ __forceinline__ constexpr frontier_kind_t get_kind() const { return _kind; }
  __host__ __device__ __forceinline__ constexpr frontier_view_t get_view() const { return _view; }
};

/// Sparse -> dense. `dense` is cleared first unless `accumulate`. Returns nothing; count is cached lazily.
template <typename V, typename E, frontier_kind_t K, frontier_view_t DV>
void convert(frontier_t<V, E, K, frontier_view_t::vector>& sparse, frontier_t<V, E, K, DV>& dense,
             gcuda::stream_t stream = 0, bool accumulate = false) {
  static_assert(DV != frontier_view_t::vector, "target must be a bitmap/boolmap frontier");
  if (!accumulate) cudaMemsetAsync(dense.data(), 0, dense.words() * sizeof(unsigned), stream);
  std::size_t count = sparse.get_number_of_elements();
  if (count) {
    std::size_t ctas = (count + 255) / 256;
    (void)ctas;
    kernels::scatter_bits_kernel<<<stream_ctas(count), 256, 0, stream>>>(sparse.data(), count, dense.data());
  }
  dense.mark_dirty();
}

/// Dense -> sparse (compaction of set bits). Synchronises the stream to learn the length.
template <typename V, typename E, frontier_kind_t K, frontier_view_t DV>
void convert(frontier_t<V, E, K, DV>& dense, frontier_t<V, E, K, frontier_view_t::vector>& sparse,
             gcuda::standard_context_t& context) {
  static_assert(DV != frontier_view_t::vector, "source must be a bitmap/boolmap frontier");
  auto& scratch = context.scratch();
  auto stream = context.stream();
  std::size_t upper = dense.get_number_of_elements(stream);
  if (sparse.get_capacity() < upper) sparse.reserve(upper);
  scratch.zero(stream);
  if (upper)
    kernels::gather_bits_kernel<<<gcuda::persistent_grid(context, (dense.words() + 255) / 256, 4), 256, 0, stream>>>(
        dense.data(), dense.words(), sparse.data(), scratch.d + gcuda::scratch_t::out_count);
  scratch.fetch(stream);
  sparse.set_number_of_elements(std::size_t(scratch.h[gcuda::scratch_t::out_count]));
}

}  // namespace frontier
}  // namespace gunrock
