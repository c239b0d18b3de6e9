// run_cluster_cta.cu — launches of the composite-trial CTA kernels (cluster_kernels.cuh): k_run_cta_cluster,
// k_run_cta_cluster_spec, k_delta_segment_cta.
#include "handle.h"

int launch_run_cluster_cta(pmc_handle* h, const RunPlan& p, const RunArgs& a) {
  const unsigned nb = (unsigned)h->nchains;
  return with<0, 1>(p.cut, [&](auto CUT) {
    if (p.family == RunFamily::cta_cluster_spec)
      return with<8, 4, 2>(p.teams, [&](auto G) {
        return launch(h, k_run_cta_cluster_spec<G, cluster_spec_minb(G), bool(CUT)>, nb, p.threads, p.smem, a);
      });
    auto go = [&](auto T, auto MB) { return launch(h, k_run_cta_cluster<T, MB, bool(CUT)>, nb, T, p.smem, a); };
    switch (p.threads) {
      case 32:
        return with<kTeamMinb[0], kTeamMinb[1], kTeamMinb[2]>(p.minb, [&](auto MB) {
          return go(std::integral_constant<int, 32>(), MB);
        });
      case 64: return go(std::integral_constant<int, 64>(), std::integral_constant<int, kCluster64Minb>());
      case 128:
        return with<kCluster128Minb[0], kCluster128Minb[1], kCluster128Minb[2]>(p.minb, [&](auto MB) {
          return go(std::integral_constant<int, 128>(), MB);
        });
      case 256: return go(std::integral_constant<int, 256>(), std::integral_constant<int, kCluster256Minb>());
    }
    return pmc_fail(PMC_ERR_INVALID, "no kernel instantiated for this launch shape");
  });
}

int launch_delta_segment_cta(pmc_handle* h, const SegDeltaArgs& a) {
  const int tt = pick_cluster_threads(h->n);
  const size_t smem = cluster_delta_smem_bytes(h->n, tt);
  return with<0, 1>(h->energy_type == PMC_ENERGY_CUTOFF, [&](auto CUT) {
    return with<32, 64, 128, 256>(tt, [&](auto T) { return launch(h, k_delta_segment_cta<T, bool(CUT)>, 1, T, smem, a); });
  });
}
