// run_cta.cu — launches of the single-monomer-trial CTA-per-chain run kernels (cta_kernels.cuh): k_run_cta_win,
// k_run_cta_win_spec.
#include "handle.h"

int launch_run_cta(pmc_handle* h, const RunPlan& p, const RunArgs& a) {
  const unsigned nb = (unsigned)h->nchains;
  if (p.family == RunFamily::cta_win_spec)
    return with<8, 4, 2>(p.teams, [&](auto G) {
      return launch(h, k_run_cta_win_spec<G, spec_minb(G)>, nb, p.threads, p.smem, a);
    });
  return with<64, 128, 256, 512>(p.threads, [&](auto T) {
    return p.f32 ? launch(h, k_run_cta_win<T, win_minb(T), kRunUnroll, 1>, nb, T, p.smem, a)
                 : launch(h, k_run_cta_win<T, win_minb(T), kRunUnroll, 0>, nb, T, p.smem, a);
  });
}
