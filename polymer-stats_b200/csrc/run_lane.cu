// run_lane.cu — launches of the O(1)-ΔU run kernels of mcmc_eap_chain.jl (lane_kernels.cuh): k_run_lane, k_run_warp.
#include "handle.h"

namespace {
int fail(int code, const std::string& msg) { return pmc_fail(code, msg); }
}  // namespace

// O(1)-ΔU chains (non-interacting, Ising) of mcmc_eap_chain.jl: chain per warp or chain per lane.
int launch_run_lane(pmc_handle* h, const RunArgs& a) {
    // few chains: one chain per warp with 32-trial windows fills the machine; many chains: one per lane
    const int mode = env_int("PMC_LANE_MODE", 0);  // 1 = lane, 2 = warp, 0 = by chain count
    const long long below = h->warp_mode_below > 0 ? h->warp_mode_below : (h->energy_type == PMC_ENERGY_ISING ? 65536 : 120000);
    const bool use_warp = mode == 2 || (mode == 0 && packing_chains(h) < below);
    const bool comp = h->compensated != 0;
    if (use_warp) {
      const unsigned nb = (unsigned)((h->nchains + 3) / 4);
      const bool ising = h->energy_type == PMC_ENERGY_ISING;
      // at most one wave of warps (16 per SM): one chain per CTA, so that the block scheduler spreads the warps evenly
      const bool one_wave = packing_chains(h) <= (long long)h->sm_count * 16 && env_int("PMC_WARP_CPB", 1) == 1;
#define PMC_W(IS, MB, CP)                                                           \
  {                                                                                 \
    if (one_wave) {                                                                 \
      PMC_PICK("k_run_warp<" #IS ",16," #CP ",1>");                                  \
      k_run_warp<IS, 16, CP, 1><<<(unsigned)h->nchains, 32, 0, h->stream>>>(a);     \
    } else {                                                                        \
      PMC_PICK("k_run_warp<" #IS "," #MB "," #CP ">");                               \
      k_run_warp<IS, MB, CP><<<nb, 128, 0, h->stream>>>(a);                         \
    }                                                                               \
  }
      if (ising) { if (comp) PMC_W(1, 4, true) else PMC_W(1, 4, false) }
      else { if (comp) PMC_W(0, 4, true) else PMC_W(0, 4, false) }
#undef PMC_W
    } else {
      constexpr int TB = 64;
      const unsigned nb = (unsigned)((h->nchains + TB - 1) / TB);
#define PMC_L(MB, CP)                                    \
  {                                                      \
    PMC_PICK("k_run_lane<64," #MB "," #CP ">");            \
    k_run_lane<TB, MB, CP><<<nb, TB, 0, h->stream>>>(a);  \
  }
      if (comp) PMC_L(4, true) else PMC_L(6, false)
#undef PMC_L
    }
    ++h->launches;
    PMC_CU(cudaGetLastError());
  return PMC_OK;
}

