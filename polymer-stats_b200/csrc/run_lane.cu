// run_lane.cu — launches of the O(1)-ΔU run kernels of mcmc_eap_chain.jl (lane_kernels.cuh): k_run_lane, k_run_warp.
#include "handle.h"

int launch_run_lane(pmc_handle* h, const RunPlan& p, const RunArgs& a) {
  if (p.family == RunFamily::warp) {
    const unsigned grid = (unsigned)((h->nchains + p.cpb - 1) / p.cpb);
    return with<0, 1>(p.ising, [&](auto IS) {
      return with<0, 1>(p.comp, [&](auto CP) {
        return p.cpb == 1 ? launch(h, k_run_warp<IS, warp_minb(1), bool(CP), 1>, grid, p.threads, 0, a)
                          : launch(h, k_run_warp<IS, warp_minb(4), bool(CP), 4>, grid, p.threads, 0, a);
      });
    });
  }
  const unsigned grid = (unsigned)((h->nchains + p.threads - 1) / p.threads);
  return p.comp ? launch(h, k_run_lane<64, lane_minb(true), true>, grid, p.threads, 0, a)
                : launch(h, k_run_lane<64, lane_minb(false), false>, grid, p.threads, 0, a);
}
