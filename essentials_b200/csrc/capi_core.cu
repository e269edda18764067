/**
 * @file capi_core.cu
 * @brief C ABI: errors, contexts, graph handles, transpose, random stream, frontier conversions.
 */
#include "capi_common.hxx"
#include <algorithm>
#include <memory>
#include <gunrock/algorithms/generate/random.hxx>
#include <gunrock/algorithms/sssp.hxx>

namespace ess {
std::string& last_error() {
  static thread_local std::string message;
  return message;
}
int fail(const std::exception& e) {
  last_error() = e.what();
  return 999;
}
int fail(const char* message, int code) {
  last_error() = message;
  return code;
}
}  // namespace ess

using namespace gunrock;

namespace ess {
int& dist_peer_exchange() {
  static int on = 1;
  return on;
}
int& dist_trace() {
  static int on = 0;
  return on;
}
int& dist_peer_timeout_ms() {
  static int ms = 4000;
  return ms;
}
/// ess_tune("host_chunk_edges"): column indices per H2D chunk of ess_graph_create_from_host (256 MB by default;
/// tests shrink it so that small graphs cross many chunk boundaries).
int& host_chunk_edges() {
  static int edges = 64 << 20;
  return edges;
}
}  // namespace ess

extern "C" {

const char* ess_last_error(void) { return ess::last_error().c_str(); }
int ess_version(void) { return 102; }

int ess_context_create(int device, void* stream, int own_stream, ess_context_t* out) {
  ESS_TRY
  if (!out) return ess::fail("ess_context_create: out is null");
  int count = 0;
  error::throw_if_exception(cudaGetDeviceCount(&count), "no CUDA device");
  error::throw_if_exception(device < 0 || device >= count, "ess_context_create: bad device ordinal");
  auto* h = new ess_context_s;
  if (own_stream)
    h->ctx = std::make_shared<gcuda::multi_context_t>(device);
  else
    h->ctx = std::make_shared<gcuda::multi_context_t>(device, static_cast<cudaStream_t>(stream));
  h->single()->scratch();
  *out = h;
  return 0;
  ESS_CATCH
}

int ess_context_destroy(ess_context_t ctx) {
  delete ctx;
  return 0;
}

int ess_context_synchronize(ess_context_t ctx) {
  ESS_TRY
  ctx->single()->synchronize();
  return 0;
  ESS_CATCH
}

int ess_tune(const char* knob, int value) {
  ESS_TRY
  const std::string k = knob ? knob : "";
  if (k == "advance_engine") {  // 1 = quad engine (128-bit loads, warp-autonomous rounds), 0 = round-1 scalar kernels
    gunrock::operators::advance::kernels::advance_engine() = value;
    return 0;
  }
  if (k == "pull_hints") {
    gunrock::operators::advance::kernels::pull_hints_enabled() = value;
    return 0;
  }
  if (k == "sssp_fused_unique") {
    gunrock::sssp::fused_unique() = value;
    return 0;
  }
  if (k == "dist_trace") {
    ess::dist_trace() = value;
    return 0;
  }
  if (k == "dist_peer_exchange") {
    ess::dist_peer_exchange() = value;
    return 0;
  }
  if (k == "host_chunk_edges") {
    if (value <= 0) return ess::fail("ess_tune: host_chunk_edges must be positive");
    ess::host_chunk_edges() = value;
    return 0;
  }
  if (k == "dist_peer_timeout_ms") {
    if (value <= 0) return ess::fail("ess_tune: dist_peer_timeout_ms must be positive");
    ess::dist_peer_timeout_ms() = value;
    return 0;
  }
  return ess::fail("ess_tune: unknown knob");
  ESS_CATCH
}

int ess_profile_enable(ess_context_t ctx, int enable) {
  ESS_TRY
  auto& prof = ctx->single()->profiler();
  prof.reset();
  prof.enabled = enable != 0;
  return 0;
  ESS_CATCH
}

int ess_profile_read(ess_context_t ctx, double* ms_by_class, int64_t* launches_by_class, int n_classes) {
  ESS_TRY
  auto& prof = ctx->single()->profiler();
  prof.collect();
  for (int i = 0; i < n_classes && i < gcuda::profiler_t::n_classes; ++i) {
    if (ms_by_class) ms_by_class[i] = prof.ms[i];
    if (launches_by_class) launches_by_class[i] = prof.launches[i];
  }
  // last slot: every kernel the operators launched on this context since creation (always counted)
  if (launches_by_class && n_classes >= gcuda::profiler_t::n_classes)
    launches_by_class[gcuda::profiler_t::n_classes - 1] = prof.launches_total;
  return 0;
  ESS_CATCH
}

int ess_graph_create(int64_t n, int64_t m, int offset_bits, const void* d_row_offsets,
                     const int32_t* d_column_indices, const float* d_values, int symmetric,
                     const void* d_column_offsets, const int32_t* d_row_indices, const float* d_csc_values,
                     ess_graph_t* out) {
  ESS_TRY
  if (!out || !d_row_offsets || (m > 0 && !d_column_indices)) return ess::fail("ess_graph_create: null argument");
  if (offset_bits != 32 && offset_bits != 64) return ess::fail("ess_graph_create: offset_bits must be 32 or 64");
  if (n < 0 || n > 2147483647LL) return ess::fail("ess_graph_create: vertex ids are int32");
  if (offset_bits == 32 && m > 2147483647LL) return ess::fail("ess_graph_create: m needs 64-bit offsets");
  auto* h = new ess_graph_s;
  h->offset_bits = offset_bits;
  h->n = n;
  h->m = m;
  const void* t_off = d_column_offsets;
  const int32_t* t_idx = d_row_indices;
  const float* t_val = d_csc_values;
  if (symmetric) {
    t_off = d_row_offsets;
    t_idx = d_column_indices;
    t_val = d_values;
  }
  h->has_csc = t_off != nullptr;
  auto* J = const_cast<int32_t*>(d_column_indices);
  auto* X = const_cast<float*>(d_values);
  auto* I = const_cast<int32_t*>(t_idx);
  auto* Xt = const_cast<float*>(t_val);
  if (offset_bits == 64)
    h->g64 = graph::build::from_csr_and_csc<int32_t, int64_t, float>(
        int32_t(n), int64_t(m), (int64_t*)d_row_offsets, J, X, (int64_t*)t_off, I, Xt);
  else
    h->g32 = graph::build::from_csr_and_csc<int32_t, int32_t, float>(
        int32_t(n), int32_t(m), (int32_t*)d_row_offsets, J, X, (int32_t*)t_off, I, Xt);
  if (h->has_csc && symmetric != 2 && n > 0 && m > 0) {
    int rc = ess_graph_build_pull_hints(h, nullptr);  // acceleration structure of bottom-up advance, once per graph
    if (rc) {
      delete h;
      return rc;
    }
  }
  *out = h;
  return 0;
  ESS_CATCH
}

}  // extern "C"

namespace {
/// A private copy stream and the events that order the context's stream behind its copies.
struct copy_lane_t {
  cudaStream_t stream = nullptr;
  std::vector<cudaEvent_t> events;
  copy_lane_t() { error::throw_if_exception(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking), "copy stream"); }
  ~copy_lane_t() {
    for (auto e : events) cudaEventDestroy(e);
    if (stream) cudaStreamDestroy(stream);
  }
  /// Everything enqueued on `follower` after this call waits for the copies enqueued so far.
  void publish_to(cudaStream_t follower) {
    cudaEvent_t e = nullptr;
    error::throw_if_exception(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "copy event");
    events.push_back(e);
    error::throw_if_exception(cudaEventRecord(e, stream), "copy event record");
    error::throw_if_exception(cudaStreamWaitEvent(follower, e, 0), "copy event wait");
  }
};

/// ess_graph_create_from_host for one offset width. The offsets go first (degrees and the isolated-vertex bitmap need
/// nothing else), then the column indices in chunks of `chunk_edges`; after each chunk the context's stream builds the
/// bottom-up hints of the vertices whose lists have fully arrived, so at scale-26 the ~30 ms hint build runs under the
/// ~155 ms PCIe copy instead of after it.
template <typename edge_t>
void create_from_host(ess_context_t ctx, ess_graph_s* h, const void* h_row_offsets, const int32_t* h_column_indices,
                      const float* h_values, bool symmetric) {
  auto* c = ctx->single();
  cudaStream_t work = c->stream();
  const std::size_t n = std::size_t(h->n), m = std::size_t(h->m);
  const edge_t* ho = static_cast<const edge_t*>(h_row_offsets);
  error::throw_if_exception(ho[0] != edge_t(0) || std::size_t(ho[n]) != m,
                            "ess_graph_create_from_host: row_offsets[0] must be 0 and row_offsets[n] must be m");
  h->own_offsets.resize((n + 1) * sizeof(edge_t));
  h->own_indices.resize(m);
  if (h_values) h->own_values.resize(m);
  edge_t* d_off = reinterpret_cast<edge_t*>(h->own_offsets.data());
  int32_t* d_idx = h->own_indices.data();
  float* d_val = h_values ? h->own_values.data() : nullptr;

  copy_lane_t lane;
  error::throw_if_exception(cudaMemcpyAsync(d_off, ho, (n + 1) * sizeof(edge_t), cudaMemcpyHostToDevice, lane.stream),
                            "ess_graph_create_from_host: offsets copy");
  lane.publish_to(work);
  const bool hints = symmetric && n > 0 && m > 0;
  memory::device_array_t<int32_t> degree;
  edge_t* hint_edge = nullptr;
  if (hints) {
    h->hint_head.resize(n);
    h->hint_isolated.resize((n + 31) / 32 + 1);
    if constexpr (sizeof(edge_t) == 8) {
      h->hint_edge64.resize(n);
      hint_edge = h->hint_edge64.data();
    } else {
      h->hint_edge32.resize(n);
      hint_edge = h->hint_edge32.data();
    }
    degree.resize(n);
    graph::build::detail::degrees_kernel<<<2048, 256, 0, work>>>(int32_t(n), d_off, degree.data());
    graph::build::detail::isolated_bitmap_kernel<<<2048, 256, 0, work>>>(int32_t(n), d_off, h->hint_isolated.data());
  }
  const std::size_t chunk_edges = std::size_t(ess::host_chunk_edges());  // 256 MB of column indices per copy
  std::size_t built = 0;                                  // vertices whose hints are enqueued
  for (std::size_t e0 = 0; e0 < m; e0 += chunk_edges) {
    const std::size_t e1 = std::min(m, e0 + chunk_edges);
    error::throw_if_exception(cudaMemcpyAsync(d_idx + e0, h_column_indices + e0, (e1 - e0) * sizeof(int32_t),
                                              cudaMemcpyHostToDevice, lane.stream),
                              "ess_graph_create_from_host: indices copy");
    if (!hints) continue;
    lane.publish_to(work);
    // vertices [built, arrived) end at or before e1: the last offset that is <= e1 bounds them (host-side search)
    const std::size_t arrived = std::size_t(std::upper_bound(ho, ho + n + 1, edge_t(e1)) - ho) - 1;
    graph::build::pull_hints_range(int32_t(built), int32_t(arrived), d_off, d_idx, degree.data(), h->hint_head.data(),
                                   hint_edge, work);
    built = std::max(built, arrived);
  }
  if (d_val)
    error::throw_if_exception(cudaMemcpyAsync(d_val, h_values, m * sizeof(float), cudaMemcpyHostToDevice, lane.stream),
                              "ess_graph_create_from_host: values copy");
  error::throw_if_exception(cudaStreamSynchronize(lane.stream), "ess_graph_create_from_host: copy");
  error::throw_if_exception(cudaStreamSynchronize(work), "ess_graph_create_from_host: hint build");
  error::check_last("ess_graph_create_from_host");

  auto G = graph::build::from_csr_and_csc<int32_t, edge_t, float>(int32_t(n), edge_t(m), d_off, d_idx, d_val,
                                                                  symmetric ? d_off : nullptr,
                                                                  symmetric ? d_idx : nullptr,
                                                                  symmetric ? d_val : nullptr);
  if (hints) {
    graph::graph_csc_t<int32_t, edge_t, float>& csc = G;
    csc.set_pull_hints(h->hint_head.data(), hint_edge, h->hint_isolated.data());
  }
  if constexpr (sizeof(edge_t) == 8)
    h->g64 = G;
  else
    h->g32 = G;
}
}  // namespace

extern "C" {

int ess_graph_create_from_host(ess_context_t ctx, int64_t n, int64_t m, int offset_bits, const void* h_row_offsets,
                               const int32_t* h_column_indices, const float* h_values, int symmetric,
                               ess_graph_t* out) {
  ESS_TRY
  if (!ctx || !out || !h_row_offsets || (m > 0 && !h_column_indices))
    return ess::fail("ess_graph_create_from_host: null argument");
  if (offset_bits != 32 && offset_bits != 64)
    return ess::fail("ess_graph_create_from_host: offset_bits must be 32 or 64");
  if (n < 0 || n > 2147483647LL) return ess::fail("ess_graph_create_from_host: vertex ids are int32");
  if (m < 0 || (offset_bits == 32 && m > 2147483647LL))
    return ess::fail("ess_graph_create_from_host: m needs 64-bit offsets");
  std::unique_ptr<ess_graph_s> h(new ess_graph_s);
  h->offset_bits = offset_bits;
  h->n = n;
  h->m = m;
  h->has_csc = symmetric != 0;
  if (offset_bits == 64)
    create_from_host<int64_t>(ctx, h.get(), h_row_offsets, h_column_indices, h_values, symmetric != 0);
  else
    create_from_host<int32_t>(ctx, h.get(), h_row_offsets, h_column_indices, h_values, symmetric != 0);
  *out = h.release();
  return 0;
  ESS_CATCH
}

int ess_graph_build_pull_hints(ess_graph_t h, const int32_t* d_degree_of_id) {
  ESS_TRY
  if (!h || !h->has_csc) return ess::fail("ess_graph_build_pull_hints: graph has no CSC view");
  if (h->n <= 0 || h->m <= 0) return 0;
  // The hint kernels run on the legacy default stream, which does NOT wait for non-blocking streams (torch's, or a
  // context's own): the caller's CSR arrays may still be being written (H2D copy, generator kernels) on one of
  // those. Graph creation is set-up code, so wait for the whole device before reading them.
  error::throw_if_exception(cudaDeviceSynchronize(), "ess_graph_build_pull_hints: pending work failed");
  h->hint_head.resize(std::size_t(h->n));
  h->hint_isolated.resize((std::size_t(h->n) + 31) / 32 + 1);
  if (h->offset_bits == 64) {
    h->hint_edge64.resize(std::size_t(h->n));
    graph::build::pull_hints(h->g64, h->hint_head.data(), h->hint_edge64.data(), 0, d_degree_of_id,
                             h->hint_isolated.data());
  } else {
    h->hint_edge32.resize(std::size_t(h->n));
    graph::build::pull_hints(h->g32, h->hint_head.data(), h->hint_edge32.data(), 0, d_degree_of_id,
                             h->hint_isolated.data());
  }
  return 0;
  ESS_CATCH
}

int ess_graph_destroy(ess_graph_t g) {
  delete g;
  return 0;
}

int ess_transpose_csr(int64_t n, int64_t m, int offset_bits, const void* d_row_offsets,
                      const int32_t* d_column_indices, const float* d_values, void* d_out_offsets,
                      int32_t* d_out_indices, float* d_out_values) {
  ESS_TRY
  // set-up code on the legacy default stream: wait for producers of the input arrays on non-blocking streams
  error::throw_if_exception(cudaDeviceSynchronize(), "ess_transpose_csr: pending work failed");
  if (offset_bits == 64)
    graph::build::detail::transpose_on_device<int32_t, int64_t, float>(
        int32_t(n), int64_t(m), (const int64_t*)d_row_offsets, d_column_indices, d_values, d_out_indices,
        (int64_t*)d_out_offsets, d_out_values);
  else
    graph::build::detail::transpose_on_device<int32_t, int32_t, float>(
        int32_t(n), int32_t(m), (const int32_t*)d_row_offsets, d_column_indices, d_values, d_out_indices,
        (int32_t*)d_out_offsets, d_out_values);
  return 0;
  ESS_CATCH
}

int ess_randoms(ess_context_t ctx, float* d_out, int64_t n, float begin, float end) {
  ESS_TRY
  generate::random::uniform_distribution(d_out, std::size_t(n), begin, end, ctx->single()->stream());
  error::check_last("ess_randoms");
  ctx->single()->synchronize();
  return 0;
  ESS_CATCH
}

int ess_frontier_to_bitmap(ess_context_t ctx, const int32_t* d_list, int64_t size, int64_t universe,
                           uint32_t* d_words, int64_t* popcount) {
  ESS_TRY
  auto* c = ctx->single();
  auto stream = c->stream();
  auto& scratch = c->scratch();
  const std::size_t words = (std::size_t(universe) + 31) / 32;
  cudaMemsetAsync(d_words, 0, words * sizeof(uint32_t), stream);
  if (size)
    frontier::kernels::scatter_bits_kernel<<<gcuda::persistent_grid(*c, (std::size_t(size) + 255) / 256, 8), 256, 0,
                                             stream>>>(d_list, std::size_t(size), d_words);
  scratch.zero(stream);
  frontier::kernels::popcount_kernel<<<gcuda::persistent_grid(*c, (words + 255) / 256, 8), 256, 0, stream>>>(
      d_words, words, scratch.d + gcuda::scratch_t::out_count);
  error::check_last("ess_frontier_to_bitmap");
  scratch.fetch(stream);
  if (popcount) *popcount = int64_t(scratch.h[gcuda::scratch_t::out_count]);
  return 0;
  ESS_CATCH
}

int ess_bitmap_to_frontier(ess_context_t ctx, const uint32_t* d_words, int64_t universe, int32_t* d_list,
                           int64_t* out_count) {
  ESS_TRY
  auto* c = ctx->single();
  auto stream = c->stream();
  auto& scratch = c->scratch();
  const std::size_t words = (std::size_t(universe) + 31) / 32;
  scratch.zero(stream);
  frontier::kernels::gather_bits_kernel<<<gcuda::persistent_grid(*c, (words + 255) / 256, 8), 256, 0, stream>>>(
      d_words, words, d_list, scratch.d + gcuda::scratch_t::out_count);
  error::check_last("ess_bitmap_to_frontier");
  scratch.fetch(stream);
  if (out_count) *out_count = int64_t(scratch.h[gcuda::scratch_t::out_count]);
  return 0;
  ESS_CATCH
}

int ess_bits_to_list_async(ess_context_t ctx, const uint32_t* d_words, int64_t universe, int32_t* d_list) {
  ESS_TRY
  auto* c = ctx->single();
  auto stream = c->stream();
  auto& scratch = c->scratch();
  const std::size_t words = (std::size_t(universe) + 31) / 32;
  scratch.zero(stream);  // the slot counter is left dirty on purpose: the next operator's zero() clears it
  frontier::kernels::gather_bits_kernel<<<gcuda::persistent_grid(*c, (words + 255) / 256, 8), 256, 0, stream>>>(
      d_words, words, d_list, scratch.d + gcuda::scratch_t::out_count);
  error::check_last("ess_bits_to_list_async");
  return 0;
  ESS_CATCH
}

}  // extern "C"
