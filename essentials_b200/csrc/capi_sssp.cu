/** @file capi_sssp.cu  C ABI: ess_sssp (gunrock::sssp::run, reference include/gunrock/algorithms/sssp.hxx:155-185),
 * its near-far and delta forms, and ess_sssp_tree (gunrock::sssp::build_tree on the distances any of them returned). */
#include "capi_dispatch.hxx"
#include <gunrock/algorithms/sssp.hxx>
#include <gunrock/algorithms/sssp_tree.hxx>

using namespace gunrock;

extern "C" int ess_sssp_near_far(ess_context_t ctx, ess_graph_t g, int32_t source, float* d_dist, float delta,
                                 ess_run_info* info) {
  ESS_TRY
  if (!ctx || !g || !d_dist) return ess::fail("ess_sssp_near_far: null argument");
  if (source < 0 || source >= g->n) return ess::fail("ess_sssp_near_far: source out of range");
  ESS_WITH_GRAPH(g, G, {
    int iters = 0;
    int32_t src = source;
    long long stats[3] = {0, 0, 0};
    float ms = sssp::run<operators::load_balance_t::block_mapped, true>(G, src, d_dist, (int32_t*)nullptr, ctx->ctx,
                                                                         &iters, delta, stats);
    ess::fill_info(info, ms, iters);
    if (info)
      for (int i = 0; i < 3; ++i) info->reserved[i] = stats[i];
    return 0;
  })
  ESS_CATCH
}

extern "C" int ess_sssp(ess_context_t ctx, ess_graph_t g, int32_t source, float* d_dist, int lb, ess_run_info* info) {
  ESS_TRY
  if (!ctx || !g || !d_dist) return ess::fail("ess_sssp: null argument");
  if (source < 0 || source >= g->n) return ess::fail("ess_sssp: source out of range");
  return ess::with_load_balance(lb, [&](auto lbc) -> int {
    constexpr auto LB = decltype(lbc)::value;
    ESS_WITH_GRAPH(g, G, {
      int iters = 0;
      int32_t src = source;
      float ms = sssp::run<LB>(G, src, d_dist, (int32_t*)nullptr, ctx->ctx, &iters);
      ess::fill_info(info, ms, iters);
      return 0;
    })
  });
  ESS_CATCH
}

extern "C" int ess_sssp_delta(ess_context_t ctx, ess_graph_t g, int32_t source, float* d_dist, float delta,
                              ess_run_info* info) {
  ESS_TRY
  if (!ctx || !g || !d_dist) return ess::fail("ess_sssp_delta: null argument");
  if (source < 0 || source >= g->n) return ess::fail("ess_sssp_delta: source out of range");
  ESS_WITH_GRAPH(g, G, {
    int iters = 0;
    long long stats[4] = {0, 0, 0, 0};
    float ms = sssp::run_delta(G, source, d_dist, ctx->ctx, delta, &iters, stats);
    ess::fill_info(info, ms, iters);
    if (info)
      for (int i = 0; i < 4; ++i) info->reserved[i] = stats[i];
    return 0;
  })
  ESS_CATCH
}

extern "C" int ess_sssp_tree(ess_context_t ctx, ess_graph_t g, int32_t source, const float* d_dist, int32_t* d_pred,
                             ess_run_info* info) {
  ESS_TRY
  if (!ctx || !g || !d_dist || !d_pred) return ess::fail("ess_sssp_tree: null argument");
  if (source < 0 || source >= g->n) return ess::fail("ess_sssp_tree: source out of range");
  const auto dist_at = reinterpret_cast<std::uintptr_t>(d_dist), pred_at = reinterpret_cast<std::uintptr_t>(d_pred);
  const std::uintptr_t span = std::uintptr_t(g->n) * 4;
  if (dist_at < pred_at + span && pred_at < dist_at + span) return ess::fail("ess_sssp_tree: d_pred overlaps d_dist");
  ESS_WITH_GRAPH(g, G, {
    int rounds = 0;
    long long stats[1] = {0};
    float ms = sssp::build_tree(G, source, d_dist, d_pred, ctx->ctx, &rounds, stats);
    ess::fill_info(info, ms, rounds);
    if (info) info->reserved[0] = stats[0];
    return 0;
  })
  ESS_CATCH
}
