/** @file capi_bc.cu  C ABI: ess_bc (gunrock::bc::run, Brandes over the direction-optimised BFS; the reference's
 * single-source include/gunrock/algorithms/bc.hxx is the special case of one source and scale 0.5). */
#include <cmath>
#include "capi_dispatch.hxx"
#include <gunrock/algorithms/bc.hxx>

using namespace gunrock;

extern "C" int ess_bc(ess_context_t ctx, ess_graph_t g, const int32_t* h_sources, int64_t n_sources, float scale,
                      float* d_bc, ess_run_info* info) {
  ESS_TRY
  if (!ctx || !g || !d_bc) return ess::fail("ess_bc: null argument");
  if (n_sources < 0) return ess::fail("ess_bc: n_sources must not be negative");
  if (n_sources == 0 && h_sources) return ess::fail("ess_bc: n_sources == 0 needs h_sources == NULL (every vertex)");
  if (n_sources > 0 && !h_sources) return ess::fail("ess_bc: null argument");
  for (int64_t i = 0; i < n_sources; ++i)
    if (h_sources[i] < 0 || h_sources[i] >= g->n) return ess::fail("ess_bc: source out of range");
  if (!std::isfinite(scale)) return ess::fail("ess_bc: scale must be finite");
  if (!g->has_csc)
    return ess::fail("CSR and CSC sparse-matrix representations required for direction-optimized advance.");
  ESS_WITH_GRAPH(g, G, {
    long long stats[3] = {0, 0, 0};
    const std::size_t count = std::size_t(n_sources);
    float ms = bc::run(G, h_sources, count, double(scale), d_bc, ctx->ctx, stats);
    ess::fill_info(info, ms, int(n_sources ? n_sources : g->n));
    if (info)
      for (int i = 0; i < 3; ++i) info->reserved[i] = stats[i];
    return 0;
  })
  ESS_CATCH
}
