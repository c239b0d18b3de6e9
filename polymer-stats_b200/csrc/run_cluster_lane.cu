// run_cluster_lane.cu — launches of the composite-trial lane/warp kernels (cluster_kernels.cuh): k_run_lane_cluster, k_run_warp_cluster.
#include "handle.h"

namespace {
int fail(int code, const std::string& msg) { return pmc_fail(code, msg); }
}  // namespace

// Composite-trial kernels of the non-interacting and Ising energies: chain per warp or chain per lane.
int launch_run_cluster_lane(pmc_handle* h, const RunArgs& a) {
  {
    constexpr int TB = 64;
    const unsigned nb = (unsigned)((h->nchains + TB - 1) / TB);
    const bool ising = h->energy_type == PMC_ENERGY_ISING;
    // few chains: one chain per warp with 32-trial windows; many chains: one per lane
    const int mode = env_int("PMC_LANE_CLUSTER_MODE", 0);  // 1 = lane, 2 = warp, 0 = by chain count
    if (mode == 2 || (mode == 0 && packing_chains(h) < h->warp_cluster_below)) {
      const unsigned nbw = (unsigned)((h->nchains + 3) / 4);
      const bool stage = h->n <= kWarpClusterStageMax;
      // Trials per window: an accepted trial invalidates the later trials of the window that read its segment and
      // every invalidation costs a serial re-evaluation pass, but the per-window work (draws, prefix sums,
      // averagers) is amortised over the window: 32 wins from n = 25 to 400 (profiles/r01f_tune_warp_cluster.txt).
      RunArgs aw = a;
      aw.window = 32;
      {
        const int w = env_int("PMC_WARP_CLUSTER_WIN", 0);  // experiments only
        if (w >= 1 && w <= 32) aw.window = w;
      }
      const size_t smem = stage ? (size_t)4 * h->n * sizeof(MonoRec) : 0;
#define PMC_WC(IS, CP)                                                                         \
  {                                                                                            \
    PMC_PICK("k_run_warp_cluster<" #IS ",2," #CP ">");                                         \
    if (stage) {                                                                               \
      int rc = set_smem(k_run_warp_cluster<IS, 2, CP, true>, smem);                            \
      if (rc) return rc;                                                                       \
      k_run_warp_cluster<IS, 2, CP, true><<<nbw, 128, smem, h->stream>>>(aw);                  \
    } else {                                                                                   \
      k_run_warp_cluster<IS, 2, CP, false><<<nbw, 128, 0, h->stream>>>(aw);                   \
    }                                                                                          \
  }
      if (h->compensated) { if (ising) PMC_WC(true, true) else PMC_WC(false, true) }
      else { if (ising) PMC_WC(true, false) else PMC_WC(false, false) }
#undef PMC_WC
    } else if (h->compensated) {
      PMC_PICK("k_run_lane_cluster<64,4,comp>");
      if (ising) k_run_lane_cluster<TB, 4, true, true><<<nb, TB, 0, h->stream>>>(a);
      else k_run_lane_cluster<TB, 4, false, true><<<nb, TB, 0, h->stream>>>(a);
    } else {
#define PMC_LC(TT, MB)                                                                                         \
  {                                                                                                            \
    PMC_PICK("k_run_lane_cluster<" #TT "," #MB ">");                                                           \
    const unsigned nbb = (unsigned)((h->nchains + TT - 1) / TT);                                               \
    if (ising) k_run_lane_cluster<TT, MB, true, false><<<nbb, TT, 0, h->stream>>>(a);                          \
    else k_run_lane_cluster<TT, MB, false, false><<<nbb, TT, 0, h->stream>>>(a);                               \
  }
      if (packing_chains(h) >= 32768) PMC_LC(64, 8)  // many chains: occupancy beats the spills of the 128-register build
      else PMC_LC(64, 4)
#undef PMC_LC
    }
  }
  ++h->launches;
  PMC_CU(cudaGetLastError());
  return PMC_OK;
}
