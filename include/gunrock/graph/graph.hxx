/**
 * @file graph.hxx
 * @brief Non-owning graph views with device-callable accessors, and graph::build::from_csr.
 *
 * Contract kept from the reference (include/gunrock/graph/graph.hxx:52-317, csr.hxx:31-234, csc.hxx:19-142,
 * coo.hxx, properties.hxx:19-44, build.hxx:21-52): graph_t<space, V, E, W, views...> inherits one class per
 * representation; every accessor is templated on the view and defaults to the first real one; the object
 * is a POD of pointers + sizes passed BY VALUE into kernels and captured by value in user lambdas;
 * arrays are caller-owned. view_t flag values are unchanged.
 *
 * Differences, all additive: (1) CSR and CSC may be built together — required by direction-optimised
 * advance; the reference throws (graph/detail/build.hxx:85-89) and its CSC build sorts the CSR arrays in
 * place, destroying them (:103-110). Here the transpose is written into the caller's I/Aj buffers by a
 * counting sort and the CSR stays intact. (2) get_source_vertex on CSR is a plain binary search over the
 * offsets (no thrust::lower_bound with a device lambda). (3) a null weight pointer means "all ones".
 */
#pragma once

#include <atomic>
#include <cstdint>
#include <tuple>
#include <type_traits>

#include <gunrock/error.hxx>
#include <gunrock/memory.hxx>
#include <gunrock/util/load_store.hxx>
#include <gunrock/util/math.hxx>

namespace gunrock {
namespace graph {

using namespace memory;

struct graph_properties_t {
  bool directed{false};
  bool weighted{true};
  bool symmetric{false};  ///< B200 addition: CSC view aliases the CSR arrays (undirected graph).
  /// B200 addition, 1-D partitioned runs: the graph holds the rows of the global vertices
  /// [row_offset, row_offset + number_of_vertices); column ids stay global. Frontiers hold LOCAL row ids,
  /// operators are called with the GLOBAL source id (local + row_offset), so label arrays are indexed globally.
  long long row_offset{0};
  long long global_vertices{0};  ///< vertices of the whole graph (0 = this graph is the whole graph)
  graph_properties_t() = default;
};

enum view_t : uint32_t { csr = 1 << 1, csc = 1 << 2, coo = 1 << 3, invalid = 1 << 0 };

constexpr inline view_t operator|(view_t a, view_t b) { return view_t(uint32_t(a) | uint32_t(b)); }
constexpr inline view_t set(view_t a, view_t b) { return view_t(uint32_t(a) | uint32_t(b)); }
constexpr inline view_t unset(view_t a, view_t b) { return view_t(uint32_t(a) & ~uint32_t(b)); }
constexpr inline bool has(view_t a, view_t b) { return (uint32_t(a) & uint32_t(b)) == uint32_t(b); }
constexpr inline view_t toggle(view_t a, view_t b) { return view_t(uint32_t(a) ^ uint32_t(b)); }

template <typename vertex_t>
struct vertex_pair_t {
  vertex_t source;
  vertex_t destination;
};

struct empty_graph_t {};
struct empty_csr_t {};
struct empty_csc_t {};
struct empty_coo_t {};

namespace detail {
/// Process-wide counter behind graph_t::get_build_serial(); never returns 0.
inline std::uint64_t next_build_serial() {
  static std::atomic<std::uint64_t> serial{0};
  return serial.fetch_add(1, std::memory_order_relaxed) + 1;
}

/// Largest row r with offsets[r] <= e, skipping empty rows: the row that owns edge e.
template <typename vertex_t, typename edge_t>
__host__ __device__ __forceinline__ vertex_t owner_of_edge(const edge_t* offsets, vertex_t rows, edge_t e) {
  vertex_t lo = 0, hi = rows;  // offsets[lo] <= e < offsets[hi]
  while (hi - lo > 1) {
    vertex_t mid = lo + (hi - lo) / 2;
    if (offsets[mid] <= e)
      lo = mid;
    else
      hi = mid;
  }
  return lo;
}

/// Compressed-sparse adjacency shared by the CSR view (rows -> out-neighbours) and the CSC view
/// (columns -> in-neighbours). `major` is the compressed dimension.
template <typename vertex_t, typename edge_t, typename weight_t>
struct compressed_t {
  vertex_t number_of_vertices = 0;
  edge_t number_of_edges = 0;
  edge_t* offsets = nullptr;
  vertex_t* indices = nullptr;
  weight_t* values = nullptr;

  __host__ __device__ __forceinline__ edge_t start(vertex_t const& v) const { return thread::load(&offsets[v]); }
  __host__ __device__ __forceinline__ edge_t degree(vertex_t const& v) const {
    return thread::load(&offsets[v + 1]) - thread::load(&offsets[v]);
  }
  __host__ __device__ __forceinline__ vertex_t minor_of(edge_t const& e) const { return thread::load(&indices[e]); }
  __host__ __device__ __forceinline__ vertex_t major_of(edge_t const& e) const {
    return owner_of_edge(offsets, number_of_vertices, e);
  }
  __host__ __device__ __forceinline__ weight_t weight(edge_t const& e) const {
    return values ? thread::load(&values[e]) : weight_t(1);
  }
  __host__ __device__ __forceinline__ edge_t find(vertex_t const& major, vertex_t const& minor) const {
    edge_t lo = start(major), hi = start(major + 1);
    while (lo < hi) {  // adjacency lists are sorted by the builders
      edge_t mid = lo + (hi - lo) / 2;
      vertex_t x = indices[mid];
      if (x == minor) return mid;
      if (x < minor)
        lo = mid + 1;
      else
        hi = mid;
    }
    return edge_t(-1);
  }
};
}  // namespace detail

template <typename vertex_t, typename edge_t, typename weight_t>
class graph_csr_t {
  using store_t = detail::compressed_t<vertex_t, edge_t, weight_t>;

 public:
  using vertex_type = vertex_t;
  using edge_type = edge_t;
  using weight_type = weight_t;
  using vertex_pair_type = vertex_pair_t<vertex_t>;

  __host__ __device__ graph_csr_t() {}

  __host__ __device__ __forceinline__ edge_t get_number_of_neighbors(vertex_t const& v) const { return s.degree(v); }
  __host__ __device__ __forceinline__ vertex_t get_source_vertex(edge_t const& e) const { return s.major_of(e); }
  __host__ __device__ __forceinline__ vertex_t get_destination_vertex(edge_t const& e) const { return s.minor_of(e); }
  __host__ __device__ __forceinline__ edge_t get_starting_edge(vertex_t const& v) const { return s.start(v); }
  __host__ __device__ __forceinline__ vertex_pair_type get_source_and_destination_vertices(edge_t const& e) const {
    return {s.major_of(e), s.minor_of(e)};
  }
  __host__ __device__ __forceinline__ edge_t get_edge(vertex_t const& src, vertex_t const& dst) const {
    return s.find(src, dst);
  }
  __host__ __device__ __forceinline__ weight_t get_edge_weight(edge_t const& e) const { return s.weight(e); }

  /// Sorted-list intersection |N(a) ∩ N(b)|, calling on_intersection(w) per common neighbour
  /// (reference graph/csr.hxx:110-167, used by triangle counting).
  template <typename operator_type>
  __host__ __device__ __forceinline__ vertex_t get_intersection_count(vertex_t const& a, vertex_t const& b,
                                                                      operator_type on_intersection) const {
    edge_t i = s.start(a), ie = s.start(a + 1), j = s.start(b), je = s.start(b + 1);
    vertex_t hits = 0;
    while (i < ie && j < je) {
      vertex_t x = s.indices[i], y = s.indices[j];
      if (x == y) {
        on_intersection(x);
        ++hits, ++i, ++j;
      } else if (x < y)
        ++i;
      else
        ++j;
    }
    return hits;
  }

  __host__ __device__ __forceinline__ auto get_row_offsets() const { return s.offsets; }
  __host__ __device__ __forceinline__ auto get_column_indices() const { return s.indices; }
  __host__ __device__ __forceinline__ auto get_nonzero_values() const { return s.values; }
  __host__ __device__ __forceinline__ auto get_number_of_rows() const { return s.number_of_vertices; }
  __host__ __device__ __forceinline__ auto get_number_of_columns() const { return s.number_of_vertices; }
  __host__ __device__ __forceinline__ auto get_number_of_nonzeros() const { return s.number_of_edges; }
  __host__ __device__ __forceinline__ auto get_number_of_vertices() const { return s.number_of_vertices; }
  __host__ __device__ __forceinline__ auto get_number_of_edges() const { return s.number_of_edges; }

 protected:
  __host__ __device__ void set(vertex_t const& n, edge_t const& m, edge_t* row_offsets, vertex_t* column_indices,
                               weight_t* values) {
    s.number_of_vertices = n;
    s.number_of_edges = m;
    s.offsets = row_offsets;
    s.indices = column_indices;
    s.values = values;
  }

 private:
  store_t s;
};

template <typename vertex_t, typename edge_t, typename weight_t>
class graph_csc_t {
  using store_t = detail::compressed_t<vertex_t, edge_t, weight_t>;

 public:
  using vertex_type = vertex_t;
  using edge_type = edge_t;
  using weight_type = weight_t;
  using vertex_pair_type = vertex_pair_t<vertex_t>;

  __host__ __device__ graph_csc_t() {}

  // In the CSC view a vertex's "neighbours" are its IN-neighbours (reference graph/csc.hxx:43-95).
  __host__ __device__ __forceinline__ edge_t get_number_of_neighbors(vertex_t const& v) const { return s.degree(v); }
  __host__ __device__ __forceinline__ vertex_t get_source_vertex(edge_t const& e) const { return s.minor_of(e); }
  __host__ __device__ __forceinline__ vertex_t get_destination_vertex(edge_t const& e) const { return s.major_of(e); }
  __host__ __device__ __forceinline__ edge_t get_starting_edge(vertex_t const& v) const { return s.start(v); }
  __host__ __device__ __forceinline__ vertex_pair_type get_source_and_destination_vertices(edge_t const& e) const {
    return {s.minor_of(e), s.major_of(e)};
  }
  __host__ __device__ __forceinline__ edge_t get_edge(vertex_t const& src, vertex_t const& dst) const {
    return s.find(dst, src);
  }
  __host__ __device__ __forceinline__ weight_t get_edge_weight(edge_t const& e) const { return s.weight(e); }

  __host__ __device__ __forceinline__ auto get_column_offsets() const { return s.offsets; }
  __host__ __device__ __forceinline__ auto get_row_indices() const { return s.indices; }
  /// Bottom-up hints (B200 addition): caller-owned arrays filled by graph::build::pull_hints.
  __host__ __device__ void set_pull_hints(const vertex_t* head, const edge_t* head_edge,
                                          const unsigned* isolated = nullptr) {
    hint_head = head;
    hint_edge = head_edge;
    hint_isolated = isolated;
  }
  __host__ __device__ __forceinline__ const unsigned* get_pull_hint_isolated() const { return hint_isolated; }
  __host__ __device__ __forceinline__ const vertex_t* get_pull_hint_heads() const { return hint_head; }
  __host__ __device__ __forceinline__ const edge_t* get_pull_hint_edges() const { return hint_edge; }
  __host__ __device__ __forceinline__ auto get_nonzero_values() const { return s.values; }
  __host__ __device__ __forceinline__ auto get_number_of_rows() const { return s.number_of_vertices; }
  __host__ __device__ __forceinline__ auto get_number_of_columns() const { return s.number_of_vertices; }
  __host__ __device__ __forceinline__ auto get_number_of_nonzeros() const { return s.number_of_edges; }
  __host__ __device__ __forceinline__ auto get_number_of_vertices() const { return s.number_of_vertices; }
  __host__ __device__ __forceinline__ auto get_number_of_edges() const { return s.number_of_edges; }

 protected:
  __host__ __device__ void set(vertex_t const& n, edge_t const& m, edge_t* column_offsets, vertex_t* row_indices,
                               weight_t* values) {
    s.number_of_vertices = n;
    s.number_of_edges = m;
    s.offsets = column_offsets;
    s.indices = row_indices;
    s.values = values;
  }

 private:
  store_t s;
  const vertex_t* hint_head = nullptr;
  const edge_t* hint_edge = nullptr;
  const unsigned* hint_isolated = nullptr;
};

template <typename vertex_t, typename edge_t, typename weight_t>
class graph_coo_t {
 public:
  using vertex_type = vertex_t;
  using edge_type = edge_t;
  using weight_type = weight_t;
  using vertex_pair_type = vertex_pair_t<vertex_t>;

  __host__ __device__ graph_coo_t() {}

  // Coordinate lists are sorted by row when built from CSR, so row queries are binary searches.
  __host__ __device__ __forceinline__ edge_t get_starting_edge(vertex_t const& v) const {
    edge_t lo = 0, hi = number_of_edges;
    while (lo < hi) {
      edge_t mid = lo + (hi - lo) / 2;
      if (row_indices[mid] < v)
        lo = mid + 1;
      else
        hi = mid;
    }
    return lo;
  }
  __host__ __device__ __forceinline__ edge_t get_number_of_neighbors(vertex_t const& v) const {
    return get_starting_edge(v + 1) - get_starting_edge(v);
  }
  __host__ __device__ __forceinline__ vertex_t get_source_vertex(edge_t const& e) const {
    return thread::load(&row_indices[e]);
  }
  __host__ __device__ __forceinline__ vertex_t get_destination_vertex(edge_t const& e) const {
    return thread::load(&column_indices[e]);
  }
  __host__ __device__ __forceinline__ vertex_pair_type get_source_and_destination_vertices(edge_t const& e) const {
    return {get_source_vertex(e), get_destination_vertex(e)};
  }
  __host__ __device__ __forceinline__ edge_t get_edge(vertex_t const& src, vertex_t const& dst) const {
    for (edge_t e = get_starting_edge(src); e < number_of_edges && row_indices[e] == src; ++e)
      if (column_indices[e] == dst) return e;
    return edge_t(-1);
  }
  __host__ __device__ __forceinline__ weight_t get_edge_weight(edge_t const& e) const {
    return values ? thread::load(&values[e]) : weight_t(1);
  }
  __host__ __device__ __forceinline__ auto get_row_indices() const { return row_indices; }
  __host__ __device__ __forceinline__ auto get_column_indices() const { return column_indices; }
  __host__ __device__ __forceinline__ auto get_nonzero_values() const { return values; }
  __host__ __device__ __forceinline__ auto get_number_of_vertices() const { return number_of_vertices; }
  __host__ __device__ __forceinline__ auto get_number_of_edges() const { return number_of_edges; }

 protected:
  __host__ __device__ void set(vertex_t const& n, edge_t const& m, vertex_t* I, vertex_t* J, weight_t* X) {
    number_of_vertices = n;
    number_of_edges = m;
    row_indices = I;
    column_indices = J;
    values = X;
  }

 private:
  vertex_t number_of_vertices = 0;
  edge_t number_of_edges = 0;
  vertex_t* row_indices = nullptr;
  vertex_t* column_indices = nullptr;
  weight_t* values = nullptr;
};

namespace detail {
template <typename... T>
struct first_real_view;
template <typename T, typename... Rest>
struct first_real_view<T, Rest...> {
  static constexpr bool is_empty = std::is_same<T, empty_graph_t>::value || std::is_same<T, empty_csr_t>::value ||
                                   std::is_same<T, empty_csc_t>::value || std::is_same<T, empty_coo_t>::value;
  using type = std::conditional_t<is_empty, typename first_real_view<Rest...>::type, T>;
};
template <>
struct first_real_view<> {
  using type = empty_graph_t;
};
template <typename... T>
constexpr std::size_t count_real_views() {
  return ((std::is_same<T, empty_graph_t>::value || std::is_same<T, empty_csr_t>::value ||
                   std::is_same<T, empty_csc_t>::value || std::is_same<T, empty_coo_t>::value
               ? 0
               : 1) +
          ... + 0);
}
}  // namespace detail

template <memory_space_t space, typename vertex_t, typename edge_t, typename weight_t, class... graph_view_t>
class graph_t : public graph_view_t... {
  using default_view_t = typename detail::first_real_view<graph_view_t...>::type;

 public:
  using vertex_type = vertex_t;
  using edge_type = edge_t;
  using weight_type = weight_t;
  using vertex_pair_type = vertex_pair_t<vertex_t>;
  using vertex_pointer_t = vertex_t*;
  using edge_pointer_t = edge_t*;
  using weight_pointer_t = weight_t*;
  using graph_type = graph_t<space, vertex_t, edge_t, weight_t, graph_view_t...>;
  using graph_csr_view_t = graph_csr_t<vertex_t, edge_t, weight_t>;
  using graph_csc_view_t = graph_csc_t<vertex_t, edge_t, weight_t>;
  using graph_coo_view_t = graph_coo_t<vertex_t, edge_t, weight_t>;

  __host__ __device__ graph_t() : graph_view_t()... {}

  template <class input_view_t = default_view_t>
  __host__ __device__ __forceinline__ const vertex_t get_number_of_vertices() const {
    return input_view_t::get_number_of_vertices();
  }
  template <class input_view_t = default_view_t>
  __host__ __device__ __forceinline__ const edge_t get_number_of_edges() const {
    return input_view_t::get_number_of_edges();
  }
  bool is_directed() const { return properties.directed; }
  graph_properties_t& get_properties() { return properties; }
  const graph_properties_t& get_properties() const { return properties; }

  __host__ __device__ __forceinline__ std::size_t number_of_graph_representations() const {
    return detail::count_real_views<graph_view_t...>();
  }
  template <typename input_view_t>
  static constexpr bool contains_representation() {
    return std::disjunction_v<std::is_same<input_view_t, graph_view_t>...>;
  }
  __host__ __device__ __forceinline__ constexpr memory_space_t memory_space() const { return space; }

  template <class input_view_t = default_view_t, typename... args_t>
  __host__ __device__ void set(vertex_t const& n, edge_t const& m, args_t... args) {
    input_view_t::set(n, m, args...);
#ifndef __CUDA_ARCH__
    build_serial = detail::next_build_serial();
#endif
  }

  /// Identity of the arrays this graph was last set() over, unique within the process (0: set on the device, or
  /// never). Copies of a graph share it. Host caches of per-graph facts key on it rather than on array addresses,
  /// which allocators hand out again once a graph's arrays are freed.
  std::uint64_t get_build_serial() const { return build_serial; }

  template <typename input_view_t = default_view_t>
  __host__ __device__ __forceinline__ edge_t get_number_of_neighbors(vertex_t const& v) const {
    return input_view_t::get_number_of_neighbors(v);
  }
  template <typename input_view_t = default_view_t>
  __host__ __device__ __forceinline__ vertex_t get_source_vertex(edge_t const& e) const {
    return input_view_t::get_source_vertex(e);
  }
  template <typename input_view_t = default_view_t>
  __host__ __device__ __forceinline__ vertex_t get_destination_vertex(edge_t const& e) const {
    return input_view_t::get_destination_vertex(e);
  }
  template <typename input_view_t = default_view_t>
  __host__ __device__ __forceinline__ edge_t get_starting_edge(vertex_t const& v) const {
    return input_view_t::get_starting_edge(v);
  }
  template <typename input_view_t = default_view_t>
  __host__ __device__ __forceinline__ vertex_pair_type get_source_and_destination_vertices(edge_t const& e) const {
    return input_view_t::get_source_and_destination_vertices(e);
  }
  template <typename input_view_t = default_view_t>
  __host__ __device__ __forceinline__ edge_t get_edge(vertex_t const& src, vertex_t const& dst) const {
    return input_view_t::get_edge(src, dst);
  }
  template <typename input_view_t = default_view_t>
  __host__ __device__ __forceinline__ weight_t get_edge_weight(edge_t const& e) const {
    return input_view_t::get_edge_weight(e);
  }

 private:
  graph_properties_t properties;
  std::uint64_t build_serial = 0;
};

/// Raw adjacency triple handed to the advance kernels (offsets, indices, values) for one view.
template <typename vertex_t, typename edge_t, typename weight_t>
struct adjacency_t {
  const edge_t* offsets;
  const vertex_t* indices;
  const weight_t* values;  // may be null: weight 1
  vertex_t n;
  edge_t m;
  // Optional bottom-up hints (CSC only, see graph::build::pull_hints): for every vertex its in-neighbour of
  // largest degree and the id of that in-edge; null when the graph was built without them.
  const vertex_t* head = nullptr;
  const edge_t* head_edge = nullptr;
  const unsigned* isolated = nullptr;  ///< bitmap of vertices without in-edges (padding bits set), or null
  /// 1-D partition: global id of local row 0 (graph_properties_t::row_offset). Push kernels hand the operator
  /// `local row + source_offset` as the source vertex.
  vertex_t source_offset = 0;
};

/// The arrays an advance walks: CSR (rows -> out-neighbours) for forward, CSC (columns -> in-neighbours)
/// for backward. Asking for a view the graph was not built with is a compile-time error.
template <bool want_csc, typename graph_type>
auto adjacency_of(const graph_type& G) {
  using V = typename graph_type::vertex_type;
  using E = typename graph_type::edge_type;
  using W = typename graph_type::weight_type;
  if constexpr (want_csc) {
    using csc_v = typename graph_type::graph_csc_view_t;
    static_assert(graph_type::template contains_representation<csc_v>(),
                  "backward / direction-optimised advance needs a graph built with view_t::csc");
    const csc_v& c = G;
    return adjacency_t<V, E, W>{c.get_column_offsets(), c.get_row_indices(),     c.get_nonzero_values(),
                                c.get_number_of_vertices(), c.get_number_of_edges(), c.get_pull_hint_heads(),
                                c.get_pull_hint_edges(),    c.get_pull_hint_isolated()};
  } else {
    using csr_v = typename graph_type::graph_csr_view_t;
    static_assert(graph_type::template contains_representation<csr_v>(),
                  "forward advance needs a graph built with view_t::csr");
    const csr_v& c = G;
    adjacency_t<V, E, W> a{c.get_row_offsets(), c.get_column_indices(), c.get_nonzero_values(),
                           c.get_number_of_vertices(), c.get_number_of_edges()};
    a.source_offset = V(G.get_properties().row_offset);
    return a;
  }
}

template <typename graph_type>
__host__ __device__ double get_average_degree(graph_type const& G) {
  return double(G.get_number_of_edges()) / double(G.get_number_of_vertices());
}

}  // namespace graph
}  // namespace gunrock

#include <gunrock/graph/build.hxx>
