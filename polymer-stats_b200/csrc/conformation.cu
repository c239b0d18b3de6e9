// conformation.cu — launch helper of the conformation-sampling kernel (conformation.cuh).
#include "handle.h"
#include "conformation.cuh"

// One sample of every chain into h->conf, at the block size of the CTA energy kernels (the same positions, bit for bit).
int launch_conformation(pmc_handle* h) {
  pmc::ConfArgs a{};
  a.mono = h->mono; a.par = h->par; a.sums = h->conf;
  a.cols = 8 + 3 * (long long)h->n + h->conf_bins;
  a.n = h->n; a.bins = h->conf_bins;
  return with<32, 64, 128, 256, 512>(plan_run(h).cta_threads, [&](auto T) {
    return launch(h, pmc::k_conformation<decltype(T)::value>, (unsigned)h->nchains, T,
                  pmc::conformation_smem_bytes(h->n), a);
  });
}
