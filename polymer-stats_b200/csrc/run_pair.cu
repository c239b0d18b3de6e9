// run_pair.cu — launch of k_run_cta_pair (pair_kernels.cuh): long interacting chains, two SMs per chain.
#include "handle.h"
#include "pair_kernels.cuh"

namespace {
int fail(int code, const std::string& msg) { return pmc_fail(code, msg); }
}  // namespace

template <int T, int MINB>
static int launch_pair_t(pmc_handle* h, size_t smem, const RunArgs& a, const PairQueue& q) {
  int rc = set_smem(k_run_cta_pair<T, MINB, kRunUnroll>, smem);
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
  PMC_CU(cudaOccupancyMaxActiveClusters(&resident, k_run_cta_pair<T, MINB, kRunUnroll>, &cfg));
  if (resident < 1) return fail(PMC_ERR_UNSUPPORTED, "no CTA pair fits on this device");
  const int clusters = (int)std::min<int64_t>(h->nchains, resident);
  cfg.gridDim = dim3(2 * clusters, 1, 1);
  PMC_CU(cudaLaunchKernelEx(&cfg, k_run_cta_pair<T, MINB, kRunUnroll>, a, q));
  ++h->launches;
  PMC_CU(cudaGetLastError());
  return PMC_OK;
}

int launch_run_pair(pmc_handle* h, const RunPlan& p, const RunArgs& a) {
  const int nch = (int)h->nchains;
  if (!h->pair_work) {
    PMC_CU(pool_alloc(&h->pair_work, (size_t)nch * sizeof(unsigned long long)));
    PMC_CU(pool_alloc(&h->pair_order, (size_t)nch * sizeof(int)));
    PMC_CU(pool_alloc(&h->pair_next, sizeof(int)));
  }
  PairQueue q{};
  q.next = h->pair_next;
  if (p.pair_order) {   // heaviest predicted work first
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
  // launch bounds 1 … win_minb(T): what the shared memory admits, or PMC_PAIR_MINB
  return with<128, 256, 512>(p.threads, [&](auto T) {
    return with_range<1, win_minb(T)>(p.minb, [&](auto MB) { return launch_pair_t<T, MB>(h, p.smem, a, q); });
  });
}
