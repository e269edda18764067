/**
 * @file context.hxx
 * @brief gcuda::standard_context_t (one device: stream, event, timer, properties, operator scratch) and
 * gcuda::multi_context_t (the vector of per-device contexts every operator takes).
 *
 * API kept from the reference (include/gunrock/cuda/context.hxx:54-206): the four multi_context_t
 * constructors, get_context(i), size(), enable_peer_access(), public `contexts`/`devices`;
 * standard_context_t::{stream, synchronize, event, timer, props, ptx_version, ordinal, execution_policy}.
 * Dropped: mgpu() (moderngpu is not used). Added for the B200 operators: scratch() — persistent
 * per-context device counters + pinned host mirror + a growable temp arena, so no operator call ever
 * allocates (the reference cudaMallocs inside every block_mapped advance, block_mapped.hxx:200) — and an
 * optional distributed descriptor (rank / world size) used by the 1-D partitioned multi-GPU enactors.
 */
#pragma once

#include <cstdint>
#include <functional>
#include <memory>
#include <unordered_map>
#include <vector>
#include <cuda_runtime_api.h>
#include <thrust/execution_policy.h>
#include <thrust/system/cuda/execution_policy.h>

#include <gunrock/error.hxx>
#include <gunrock/memory.hxx>
#include <gunrock/util/timer.hxx>

namespace gunrock {
namespace gcuda {

using device_id_t = int;
using stream_t = cudaStream_t;
using event_t = cudaEvent_t;
using device_properties_t = cudaDeviceProp;

struct compute_capability_t {
  int major, minor;
  constexpr int as_combined_number() const { return major * 10 + minor; }
};
constexpr compute_capability_t make_compute_capability(int combined) {
  return compute_capability_t{combined / 10, combined % 10};
}

/**
 * @brief Operator workspace living next to a stream. Slots of the counter block (device + pinned host
 * mirror) are named here so kernels and host code agree.
 */
struct scratch_t {
  enum slot : int {
    out_count = 0,    // elements appended to the output frontier
    work_total = 1,   // sum of degrees of the input frontier (edges to expand)
    overflow = 2,     // required capacity when an output buffer was too small (0 = fine)
    items = 3,        // non-empty work items after preparation
    ticket = 4,       // dynamic tile ticket for single-pass scans
    big_count = 5,    // deferred high-degree items
    aux0 = 6,
    aux1 = 7,
    aux2 = 8,
    aux3 = 9,
    quads = 10,       // 16-byte quads of column indices to expand (quad engine work domain)
    n_slots = 16
  };

  unsigned long long* d = nullptr;  // device counters
  unsigned long long* h = nullptr;  // pinned host mirror
  memory::device_array_t<unsigned char> arena;
  // cache: (graph build serial, offsets of the view) -> max degree of that view
  std::uint64_t max_degree_graph = 0;
  const void* max_degree_offsets = nullptr;
  long long max_degree_val = -1;

  scratch_t() = default;
  scratch_t(const scratch_t&) = delete;
  scratch_t& operator=(const scratch_t&) = delete;
  ~scratch_t() {
    if (d) cudaFree(d);
    if (h) cudaFreeHost(h);
  }
  void init() {
    if (d) return;
    error::throw_if_exception(cudaMalloc(&d, n_slots * sizeof(unsigned long long)), "scratch counters");
    // mapped pinned mirror: the publish kernel writes it directly, the host polls it (no DMA, no stream sync)
    error::throw_if_exception(cudaHostAlloc(&h, (n_slots + 1) * sizeof(unsigned long long), cudaHostAllocMapped),
                              "scratch mirror");
    error::throw_if_exception(cudaMemset(d, 0, n_slots * sizeof(unsigned long long)), "scratch memset");
    for (int i = 0; i <= n_slots; ++i) h[i] = 0;
    clean = true;
  }
  /// Temp arena of at least `bytes` (256-byte aligned sub-allocation is the caller's business).
  unsigned char* temp(std::size_t bytes) {
    if (arena.capacity() < bytes)
      arena.reserve(bytes + bytes / 2 + 4096, /*keep=*/false);
    return arena.data();
  }
  /// Counters are zero after every fetch(); this only has to act when a caller skipped its fetch().
  void zero(stream_t s) {
    if (!clean) cudaMemsetAsync(d, 0, n_slots * sizeof(unsigned long long), s);
    clean = false;
  }
  /// Publishes the counter block to the host mirror, re-zeroes it on the device and waits for it:
  /// the ONE host<->device round trip of an operator call. See publish_counters_kernel below.
  inline void fetch(stream_t s);

  bool clean = false;
  /// When set, an advance without an output frontier returns without its host round trip (its caller
  /// synchronises later, e.g. through a collective): used by the multi-GPU level kernels.
  bool async_when_no_output = false;
  unsigned long long sequence = 0;  // value the host waits for in h[n_slots]
};

/// Copies the counters to mapped host memory, zeroes them for the next operator, then raises the sequence
/// flag the host spins on. One warp. Replaces cudaMemcpyAsync(D2H) + cudaStreamSynchronize: the host sees the
/// result a PCIe write after the last kernel finished instead of after a DMA + driver wake-up.
static __global__ void publish_counters_kernel(unsigned long long* d, volatile unsigned long long* h,
                                               unsigned long long sequence) {
  const int i = threadIdx.x;
  if (i < scratch_t::n_slots) {
    h[i] = d[i];
    d[i] = 0;
  }
  __threadfence_system();
  __syncwarp();
  if (i == 0) h[scratch_t::n_slots] = sequence;
}

inline void scratch_t::fetch(stream_t s) {
  ++sequence;
  publish_counters_kernel<<<1, 32, 0, s>>>(d, h, sequence);
  volatile unsigned long long* flag = h + n_slots;
  for (unsigned spins = 0; *flag != sequence; ++spins) {
    if ((spins & 0x3ff) == 0x3ff) {  // every ~1k polls make sure the stream is still healthy
      cudaError_t st = cudaStreamQuery(s);
      if (st != cudaSuccess && st != cudaErrorNotReady) error::throw_if_exception(st, "operator stream");
      if (st == cudaSuccess && *flag != sequence) {  // stream drained: the flag write must be visible now
        error::throw_if_exception(cudaStreamSynchronize(s), "operator stream sync");
        if (*flag != sequence) error::throw_if_exception(cudaErrorUnknown, "counter publish lost");
      }
    }
  }
  clean = true;
}

/**
 * @brief Opt-in per-kernel-class timing with CUDA events on the launching stream (bench/roofline use).
 * Disabled by default: begin()/end() are then a single predictable branch. Events are recorded
 * asynchronously and only resolved in collect(), so an instrumented run does not add synchronisations.
 */
struct profiler_t {
  enum kernel_class : int {
    pull_step = 0,     // bottom-up level (pull.cuh)
    push_expand = 1,   // thread/block/merge-path/bucket expansion kernels
    work_prepare = 2,  // degree scan / binning / Σdeg
    dense_state = 3,   // sparse<->dense conversion, visited init, frontier degree sum
    filter_op = 4,     // filter kernels
    n_classes = 8
  };
  struct span_t {
    int cls;
    cudaEvent_t a, b;
  };
  bool enabled = false;
  std::vector<span_t> spans;
  std::size_t used = 0;
  double ms[n_classes] = {0};
  long long launches[n_classes] = {0};
  long long launches_total = 0;  ///< kernels launched by the operators on this context (always counted)

  ~profiler_t() {
    for (auto& sp : spans) {
      cudaEventDestroy(sp.a);
      cudaEventDestroy(sp.b);
    }
  }
  void begin(int cls, cudaStream_t stream) {
    if (!enabled) return;
    if (used == spans.size()) {
      span_t sp{cls, nullptr, nullptr};
      cudaEventCreate(&sp.a);
      cudaEventCreate(&sp.b);
      spans.push_back(sp);
    }
    spans[used].cls = cls;
    cudaEventRecord(spans[used].a, stream);
  }
  void end(cudaStream_t stream, int kernels = 1) {
    launches_total += kernels;
    if (!enabled) return;
    cudaEventRecord(spans[used].b, stream);
    ++used;
  }
  /// Resolve all recorded spans into ms[] / launches[] (synchronises on the last event).
  void collect() {
    for (std::size_t i = 0; i < used; ++i) {
      float t = 0.f;
      cudaEventSynchronize(spans[i].b);
      cudaEventElapsedTime(&t, spans[i].a, spans[i].b);
      ms[spans[i].cls] += double(t);
      launches[spans[i].cls] += 1;
    }
    used = 0;
  }
  void reset() {
    collect();
    for (int i = 0; i < n_classes; ++i) ms[i] = 0, launches[i] = 0;
  }
};

/// Bump allocator over scratch_t::temp(): lay out all temporaries of one operator call, then carve.
struct arena_layout_t {
  std::size_t bytes = 0;
  std::size_t add(std::size_t n) {
    std::size_t at = bytes;
    bytes += (n + 255) & ~std::size_t(255);
    return at;
  }
};

class standard_context_t {
 public:
  explicit standard_context_t(device_id_t device = 0) : _ordinal(device), _owns_stream(true) {
    cudaSetDevice(_ordinal);
    error::throw_if_exception(cudaStreamCreateWithFlags(&_stream, cudaStreamNonBlocking), "stream create");
    init();
  }
  standard_context_t(cudaStream_t stream, device_id_t device = 0)
      : _ordinal(device), _stream(stream), _owns_stream(false) {
    cudaSetDevice(_ordinal);
    init();
  }
  standard_context_t(const standard_context_t&) = delete;
  standard_context_t& operator=(const standard_context_t&) = delete;
  ~standard_context_t() {
    memory::device_pool_t::instance().unregister_stream(_stream);
    cudaEventDestroy(_event);
    if (_owns_stream) cudaStreamDestroy(_stream);
  }

  const device_properties_t& props() const { return _props; }
  void print_properties();
  compute_capability_t ptx_version() const { return make_compute_capability(_props.major * 10 + _props.minor); }
  stream_t stream() { return _stream; }
  event_t event() { return _event; }
  util::timer_t& timer() { return _timer; }
  device_id_t ordinal() const { return _ordinal; }
  int sm_count() const { return _props.multiProcessorCount; }

  void synchronize() {
    error::throw_if_exception(_stream ? cudaStreamSynchronize(_stream) : cudaDeviceSynchronize(),
                              "context synchronize");
  }

  /// Thrust policy on this stream; kept because algorithm code outside the operators calls Thrust with it.
  auto execution_policy() { return thrust::cuda::par_nosync.on(_stream); }

  scratch_t& scratch() {
    _scratch.init();
    return _scratch;
  }
  /// CTAs of `threads` threads of `kernel` that fit on one SM (occupancy API, cached per kernel).
  template <typename kernel_t>
  int resident_ctas(kernel_t kernel, int threads) {
    const void* key = reinterpret_cast<const void*>(kernel);
    auto it = _occupancy.find(key);
    if (it != _occupancy.end()) return it->second;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1) {
      cudaGetLastError();
      per_sm = 1;
    }
    _occupancy.emplace(key, per_sm);
    return per_sm;
  }
  profiler_t& profiler() { return _profiler; }

 private:
  void init() {
    memory::device_pool_t::instance().register_stream(_stream);  // the pool's release() respects work queued here
    error::throw_if_exception(cudaEventCreateWithFlags(&_event, cudaEventDisableTiming), "event create");
    error::throw_if_exception(cudaGetDeviceProperties(&_props, _ordinal), "device properties");
    _timer.set_stream(_stream);
  }

  device_properties_t _props{};
  device_id_t _ordinal;
  stream_t _stream{};
  bool _owns_stream;
  event_t _event{};
  util::timer_t _timer;
  scratch_t _scratch;
  profiler_t _profiler;
  std::unordered_map<const void*, int> _occupancy;
};

inline void standard_context_t::print_properties() {
  std::printf("device %d: %s, sm_%d%d, %d SMs, %.1f GB, L2 %.0f MB\n", _ordinal, _props.name, _props.major,
              _props.minor, _props.multiProcessorCount, _props.totalGlobalMem / 1e9, _props.l2CacheSize / 1e6);
}

/**
 * @brief Partition descriptor of a one-process-per-GPU run (1-D vertex partition: rank r owns the global vertices
 * [r * per, (r + 1) * per)). The three collectives are stream-ordered operations on device buffers and are bound
 * by the host application (essentials_b200's C ABI binds NCCL over NVLink; a single-rank binding is trivial), so
 * this header tree has no link-time dependency on a communication library. Consumed by operators::exchange and
 * by enactor_t::enact() / is_converged().
 */
struct partition_t {
  int rank = 0, world = 1;
  long long n_global = 0, per = 0;
  /// recv[p * bytes .. (p+1) * bytes) = the `bytes` bytes rank p passed as `send`.
  std::function<void(const void* send, void* recv, std::size_t bytes, cudaStream_t)> all_gather;
  /// send + send_offset[p] .. : send_bytes[p] bytes for rank p; recv + recv_offset[p] ..: recv_bytes[p] bytes from p.
  std::function<void(const void* send, const std::size_t* send_bytes, const std::size_t* send_offset, void* recv,
                     const std::size_t* recv_bytes, const std::size_t* recv_offset, cudaStream_t)>
      all_to_all_v;
  /// In-place sum over all ranks of `count` int64 values.
  std::function<void(long long* values, std::size_t count, cudaStream_t)> all_reduce_sum;
};

class multi_context_t {
 public:
  std::vector<standard_context_t*> contexts;
  std::vector<device_id_t> devices;
  static constexpr std::size_t MAX_NUMBER_OF_GPUS = 1024;

  /// 1-D partition descriptor for one-process-per-GPU runs (rank owns a contiguous vertex range); null = the
  /// context's device holds the whole graph. rank / world_size mirror it.
  int rank = 0;
  int world_size = 1;
  std::shared_ptr<partition_t> partition;
  void set_partition(std::shared_ptr<partition_t> p) {
    partition = std::move(p);
    rank = partition ? partition->rank : 0;
    world_size = partition ? partition->world : 1;
  }

  template <typename device_list_t, typename = decltype(std::declval<device_list_t>().begin())>
  explicit multi_context_t(const device_list_t& _devices) : devices(_devices.begin(), _devices.end()) {
    for (auto dev : devices) contexts.push_back(new standard_context_t(dev));
  }
  template <typename device_list_t, typename = decltype(std::declval<device_list_t>().begin())>
  multi_context_t(const device_list_t& _devices, cudaStream_t _stream) : devices(_devices.begin(), _devices.end()) {
    for (auto dev : devices) contexts.push_back(new standard_context_t(_stream, dev));
  }
  multi_context_t(device_id_t _device) : devices(1, _device) { contexts.push_back(new standard_context_t(_device)); }
  multi_context_t(device_id_t _device, cudaStream_t _stream) : devices(1, _device) {
    contexts.push_back(new standard_context_t(_stream, _device));
  }
  multi_context_t(const multi_context_t&) = delete;
  multi_context_t& operator=(const multi_context_t&) = delete;
  ~multi_context_t() {
    for (auto* c : contexts) delete c;
  }

  standard_context_t* get_context(device_id_t device) { return contexts[device]; }
  std::size_t size() const { return contexts.size(); }

  void enable_peer_access() {
    int count = int(size());
    for (int i = 0; i < count; ++i) {
      cudaSetDevice(contexts[i]->ordinal());
      for (int j = 0; j < count; ++j) {
        if (i == j) continue;
        int can = 0;
        cudaDeviceCanAccessPeer(&can, contexts[i]->ordinal(), contexts[j]->ordinal());
        if (can) {
          cudaError_t st = cudaDeviceEnablePeerAccess(contexts[j]->ordinal(), 0);
          if (st == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        }
      }
    }
    if (count) cudaSetDevice(contexts[0]->ordinal());
  }
};

}  // namespace gcuda
}  // namespace gunrock
