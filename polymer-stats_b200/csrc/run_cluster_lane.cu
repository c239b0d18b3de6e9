// run_cluster_lane.cu — launches of the composite-trial lane/warp kernels (cluster_kernels.cuh): k_run_lane_cluster, k_run_warp_cluster.
#include "handle.h"

int launch_run_cluster_lane(pmc_handle* h, const RunPlan& p, const RunArgs& a) {
  if (p.family == RunFamily::warp_cluster) {
    const unsigned grid = (unsigned)((h->nchains + 3) / 4);   // a warp per chain
    return with<0, 1>(p.ising, [&](auto IS) {
      return with<0, 1>(p.comp, [&](auto CP) {
        return p.stage ? launch(h, k_run_warp_cluster<bool(IS), kWarpClusterMinb, bool(CP), true>, grid, p.threads, p.smem, a)
                       : launch(h, k_run_warp_cluster<bool(IS), kWarpClusterMinb, bool(CP), false>, grid, p.threads, 0, a);
      });
    });
  }
  const unsigned nb = (unsigned)((h->nchains + p.threads - 1) / p.threads);
  return with<0, 1>(p.ising, [&](auto IS) {
    if (p.comp) return launch(h, k_run_lane_cluster<64, kLaneClusterMinb, bool(IS), true>, nb, p.threads, 0, a);
    return with<kLaneClusterMinb, kLaneClusterManyMinb>(p.minb, [&](auto MB) {
      return launch(h, k_run_lane_cluster<64, MB, bool(IS), false>, nb, p.threads, 0, a);
    });
  });
}
