/** @file capi_bfs.cu  C ABI: ess_bfs (gunrock::bfs::run, reference include/gunrock/algorithms/bfs.hxx:151-176) and
 * ess_bfs_tree (gunrock::bfs::run_tree: the same run plus the parent array). */
#include <string>
#include "capi_dispatch.hxx"
#include <gunrock/algorithms/bfs.hxx>

using namespace gunrock;

namespace {
template <bool tree, operators::load_balance_t lb, operators::advance_direction_t dir, typename graph_t>
int run_bfs(ess_context_t ctx, graph_t& G, int32_t source, int32_t* d_depth, int32_t* d_pred, float alpha, float beta,
            ess_run_info* info) {
  enactor_properties_t props;
  if (alpha > 0) props.direction_alpha = alpha;
  if (beta > 0) props.direction_beta = beta;
  int pulls = 0, iters = 0;
  int32_t src = source;
  long long stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  float ms;
  if constexpr (tree)
    ms = bfs::run_tree<lb, dir>(G, src, d_depth, d_pred, ctx->ctx, props, &pulls, &iters, stats);
  else
    ms = bfs::run<lb, dir>(G, src, d_depth, (int32_t*)nullptr, ctx->ctx, props, &pulls, &iters, stats);
  ess::fill_info(info, ms, iters, pulls, iters - pulls);
  if (info)
    for (int i = 0; i < 8; ++i) info->reserved[i] = stats[i];
  return 0;
}

/// The checks and dispatch both entry points share; `what` names the entry point in error messages.
template <bool tree>
int dispatch_bfs(const char* what, ess_context_t ctx, ess_graph_t g, int32_t source, int32_t* d_depth, int32_t* d_pred,
                 int lb, int direction, float alpha, float beta, ess_run_info* info) {
  if (source < 0 || source >= g->n) return ess::fail((std::string(what) + ": source out of range").c_str());
  if (direction == ESS_DIR_OPTIMIZED && !g->has_csc)
    return ess::fail("CSR and CSC sparse-matrix representations required for direction-optimized advance.");
  if (direction != ESS_DIR_FORWARD && direction != ESS_DIR_OPTIMIZED)
    return ess::fail((std::string(what) + ": direction must be FORWARD or OPTIMIZED").c_str());
  return ess::with_load_balance(lb, [&](auto lbc) -> int {
    constexpr auto LB = decltype(lbc)::value;
    ESS_WITH_GRAPH(g, G, {
      if (direction == ESS_DIR_OPTIMIZED)
        return run_bfs<tree, LB, operators::advance_direction_t::optimized>(ctx, G, source, d_depth, d_pred, alpha,
                                                                            beta, info);
      return run_bfs<tree, LB, operators::advance_direction_t::forward>(ctx, G, source, d_depth, d_pred, alpha, beta,
                                                                        info);
    })
  });
}
}  // namespace

extern "C" int ess_bfs(ess_context_t ctx, ess_graph_t g, int32_t source, int32_t* d_depth, int lb, int direction,
                       float alpha, float beta, ess_run_info* info) {
  ESS_TRY
  if (!ctx || !g || !d_depth) return ess::fail("ess_bfs: null argument");
  return dispatch_bfs<false>("ess_bfs", ctx, g, source, d_depth, nullptr, lb, direction, alpha, beta, info);
  ESS_CATCH
}

extern "C" int ess_bfs_tree(ess_context_t ctx, ess_graph_t g, int32_t source, int32_t* d_depth, int32_t* d_pred,
                            int lb, int direction, float alpha, float beta, ess_run_info* info) {
  ESS_TRY
  if (!ctx || !g || !d_depth || !d_pred) return ess::fail("ess_bfs_tree: null argument");
  if (d_pred == d_depth) return ess::fail("ess_bfs_tree: d_pred must not alias d_depth");
  return dispatch_bfs<true>("ess_bfs_tree", ctx, g, source, d_depth, d_pred, lb, direction, alpha, beta, info);
  ESS_CATCH
}
