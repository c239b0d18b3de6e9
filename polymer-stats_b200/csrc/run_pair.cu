// run_pair.cu — launch of k_run_cta_pair (pair_kernels.cuh): long interacting chains, two SMs per chain.
#include "handle.h"
#include "pair_kernels.cuh"

namespace {
int fail(int code, const std::string& msg) { return pmc_fail(code, msg); }
}  // namespace

// When do two SMs per chain pay?  (profiles/r02b_tune_pair_small.txt, one B200)
//   * the staged copy leaves room for only one CTA per SM (n ≳ 2000): always — a launch of ≤ 148 chains is one wave and ends
//     with its slowest chain; pairs + the work-ordered queue take C5 from 0.62 to 0.71 of the DFMA peak at 50 trials;
//   * n > 768: at every ensemble size (n = 1024: 0.70–0.72 against 0.55–0.70), most for few chains;
//   * 384 < n ≤ 768: only when the chains fill between 0.55 and 0.9 of the resident CTA slots, where whole chains per SM
//     quantise badly (512 chains of n = 512 on 592 slots: 68 SMs carry four chains, 80 carry three: +15 % with pairs);
//     elsewhere the windowed one-CTA kernel is ahead (its proposals are off the critical path);
//   * shorter chains: never (the cluster barrier per trial is no longer small against the trial).
// The ensemble size is the hint's (pmc_set_ensemble_hint), so a shard decides like the whole sweep.
// Chains whose windowed one-CTA kernel does not fit shared memory (n ≳ 3900) always take pairs.  Otherwise PMC_RUN_PAIR=0
// switches pairs off and PMC_RUN_PAIR=2 forces them for any chain length (tests and experiments).
bool use_pair_kernel(const pmc_handle* h) {
  if (h->energy_type != PMC_ENERGY_INTERACTING || h->cluster_mode) return false;
  if (h->cta_threads != 128 && h->cta_threads != 256 && h->cta_threads != 512) return false;
  if (cta_smem_bytes_win(h->n) > (size_t)kSmemMax) return true;
  const int mode = env_int("PMC_RUN_PAIR", 1);
  if (mode == 0) return false;
  if (mode == 2) return true;
  if (cta_smem_bytes(h->n) > (size_t)kSmemMax / 2) return true;
  if (h->n > 768) return true;
  if (h->n > 384) {
    const int per_sm = h->cta_threads == 128 ? 4 : h->cta_threads == 256 ? 2 : 1;
    const double fill = (double)packing_chains(h) / ((double)h->sm_count * per_sm);
    return fill >= 0.55 && fill < 0.9;
  }
  return false;
}

template <int T, int MINB>
static int launch_pair_t(pmc_handle* h, const RunArgs& a, const PairQueue& q) {
  const size_t smem = cta_smem_bytes(h->n);
  int rc = set_smem(k_run_cta_pair<T, MINB, 2>, smem);
  if (rc) return rc;
  cudaLaunchConfig_t cfg{};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(T, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = h->stream;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // persistent: as many clusters as the device keeps resident (≤ one per chain); each runs chain after chain
  cfg.gridDim = dim3(2, 1, 1);
  int resident = 0;
  PMC_CU(cudaOccupancyMaxActiveClusters(&resident, k_run_cta_pair<T, MINB, 2>, &cfg));
  if (resident < 1) return fail(PMC_ERR_UNSUPPORTED, "no CTA pair fits on this device");
  const int clusters = (int)std::min<int64_t>(h->nchains, resident);
  cfg.gridDim = dim3(2 * clusters, 1, 1);
  PMC_CU(cudaLaunchKernelEx(&cfg, k_run_cta_pair<T, MINB, 2>, a, q));
  ++h->launches;
  return PMC_OK;
}

// Resident CTAs per SM the launch bound asks for: what the shared memory admits (a bound it cannot honour only takes
// registers away), at most 4 × 128, 2 × 256 or 1 × 512 threads.  PMC_PAIR_MINB overrides (experiments).
static int pair_minb(const pmc_handle* h) {
  const int fit = (int)((size_t)kSmemMax / (cta_smem_bytes(h->n) + 1024));
  const int cap = h->cta_threads == 128 ? 4 : h->cta_threads == 256 ? 2 : 1;
  int mb = std::max(1, std::min(fit, cap));
  const int o = env_int("PMC_PAIR_MINB", 0);
  if (o >= 1 && o <= cap) mb = o;
  return mb;
}

int launch_run_pair(pmc_handle* h, const RunArgs& a) {
  const int mb = pair_minb(h);
  switch (h->cta_threads * 10 + mb) {
    case 1284: PMC_PICK("k_run_cta_pair<128,4,2>"); break;
    case 1283: PMC_PICK("k_run_cta_pair<128,3,2>"); break;
    case 1282: PMC_PICK("k_run_cta_pair<128,2,2>"); break;
    case 1281: PMC_PICK("k_run_cta_pair<128,1,2>"); break;
    case 2562: PMC_PICK("k_run_cta_pair<256,2,2>"); break;
    case 2561: PMC_PICK("k_run_cta_pair<256,1,2>"); break;
    default: PMC_PICK("k_run_cta_pair<512,1,2>"); break;
  }
  const int nch = (int)h->nchains;
  if (!h->pair_work) {
    PMC_CU(pool_alloc(&h->pair_work, (size_t)nch * sizeof(unsigned long long)));
    PMC_CU(pool_alloc(&h->pair_order, (size_t)nch * sizeof(int)));
    PMC_CU(pool_alloc(&h->pair_next, sizeof(int)));
  }
  PairQueue q{};
  q.next = h->pair_next;
  if (nch <= 16384 && env_int("PMC_PAIR_ORDER", 1)) {   // heaviest predicted work first; beyond that the queue alone balances
    const int tb = 128, nb = (nch + tb - 1) / tb;
    k_predict_work<<<nb, tb, 0, h->stream>>>(h->dyn, nch, h->n, a.nsteps, h->seed, h->chain_id_base, h->pair_work);
    k_order_by_work<<<nb, tb, 0, h->stream>>>(h->pair_work, nch, h->pair_order, h->pair_next);
    h->launches += 2;
    PMC_CU(cudaGetLastError());
    q.order = h->pair_order;
  } else {
    PMC_CU(cudaMemsetAsync(h->pair_next, 0, sizeof(int), h->stream));
    q.order = nullptr;
  }
  int rc;
  switch (h->cta_threads * 10 + mb) {
    case 1284: rc = launch_pair_t<128, 4>(h, a, q); break;
    case 1283: rc = launch_pair_t<128, 3>(h, a, q); break;
    case 1282: rc = launch_pair_t<128, 2>(h, a, q); break;
    case 1281: rc = launch_pair_t<128, 1>(h, a, q); break;
    case 2562: rc = launch_pair_t<256, 2>(h, a, q); break;
    case 2561: rc = launch_pair_t<256, 1>(h, a, q); break;
    default: rc = launch_pair_t<512, 1>(h, a, q); break;
  }
  if (rc) return rc;
  PMC_CU(cudaGetLastError());
  return PMC_OK;
}
