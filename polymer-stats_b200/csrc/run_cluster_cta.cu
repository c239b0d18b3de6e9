// run_cluster_cta.cu — launches of the composite-trial CTA kernels (cluster_kernels.cuh): k_run_cta_cluster, k_delta_segment_cta.
#include "handle.h"

namespace {
int fail(int code, const std::string& msg) { return pmc_fail(code, msg); }
}  // namespace

// Composite-trial kernels of the all-pairs and cut-off energies, one CTA (or warp) per chain.
int launch_run_cluster_cta(pmc_handle* h, const RunArgs& a) {
  {
    const int nblocks = (int)h->nchains;
    const bool cut = h->energy_type == PMC_ENERGY_CUTOFF;
#define PMC_CL(TT, MB)                                                                    \
  {                                                                                       \
    const size_t smem = cluster_smem_bytes(h->n, TT);                                     \
    if (smem > (size_t)kSmemMax) return fail(PMC_ERR_UNSUPPORTED, "chain too long for this block size"); \
    PMC_PICK(cut ? "k_run_cta_cluster<" #TT "," #MB ",cut>" : "k_run_cta_cluster<" #TT "," #MB ">");  \
    if (cut) {                                                                            \
      int rc = set_smem(k_run_cta_cluster<TT, MB, true>, smem);                           \
      if (rc) return rc;                                                                  \
      k_run_cta_cluster<TT, MB, true><<<nblocks, TT, smem, h->stream>>>(a);               \
    } else {                                                                              \
      int rc = set_smem(k_run_cta_cluster<TT, MB, false>, smem);                          \
      if (rc) return rc;                                                                  \
      k_run_cta_cluster<TT, MB, false><<<nblocks, TT, smem, h->stream>>>(a);              \
    }                                                                                     \
  }
    // Small ensembles of short chains (one-warp teams, n ≤ 160): the extra warps choose_shape grants per chain evaluate
    // DIFFERENT trials at the same time (k_run_cta_cluster_spec) instead of sharing one; PMC_CLUSTER_SPEC=0: the shared-trial
    // kernels below (experiments)
    if (pick_cluster_threads(h->n) == 32 && h->cta_threads > 32 && env_int("PMC_CLUSTER_SPEC", 1)) {
      const int groups = h->cta_threads / 32;
      const size_t smem = cluster_spec_smem_bytes(h->n, groups);
      if (smem <= (size_t)kSmemMax) {
#define PMC_SP(GG, MB)                                                                               \
  {                                                                                                  \
    PMC_PICK(cut ? "k_run_cta_cluster_spec<" #GG "," #MB ",cut>" : "k_run_cta_cluster_spec<" #GG "," #MB ">"); \
    if (cut) {                                                                                       \
      int rc = set_smem(k_run_cta_cluster_spec<GG, MB, true>, smem);                                 \
      if (rc) return rc;                                                                             \
      k_run_cta_cluster_spec<GG, MB, true><<<nblocks, 32 * GG, smem, h->stream>>>(a);                \
    } else {                                                                                         \
      int rc = set_smem(k_run_cta_cluster_spec<GG, MB, false>, smem);                                \
      if (rc) return rc;                                                                             \
      k_run_cta_cluster_spec<GG, MB, false><<<nblocks, 32 * GG, smem, h->stream>>>(a);               \
    }                                                                                                \
    ++h->launches;                                                                                   \
    PMC_CU(cudaGetLastError());                                                                      \
    return PMC_OK;                                                                                   \
  }
        if (groups == 2) PMC_SP(2, 5)
        if (groups == 4) PMC_SP(4, 3)
        if (groups == 8) PMC_SP(8, 1)
#undef PMC_SP
      }
    }
    switch (h->cta_threads > 256 ? 256 : h->cta_threads) {
      case 32:  // very short chains fit 16 per SM in shared memory: worth the 128-register build (+9 % at n=25)
        // registers beat occupancy for the one-warp teams (profiles/r02b_tune_k1.txt): 10 chains per SM at 204 registers are
        // +6 % over 12 at 170 for n = 64 … 100, 8 per SM +11 % at n = 150; only very short chains gain from 16 per SM
        if (h->n <= 40) PMC_CL(32, 16) else if (h->n <= 110) PMC_CL(32, 10) else PMC_CL(32, 8)
        break;
      case 64: PMC_CL(64, 5) break;
      case 128: {
        const int fit = cluster_fit128(h->n);
        if (fit >= 4) PMC_CL(128, 4) else if (fit == 3) PMC_CL(128, 3) else PMC_CL(128, 2)
        break;
      }
      case 256: PMC_CL(256, 1) break;
      default: return fail(PMC_ERR_INVALID, "bad cta_threads");
    }
#undef PMC_CL
  }
  ++h->launches;
  PMC_CU(cudaGetLastError());
  return PMC_OK;
}

int launch_delta_segment_cta(pmc_handle* h, const SegDeltaArgs& a) {
  {
    const int tt = pick_cluster_threads(h->n);
    const size_t smem = cluster_delta_smem_bytes(h->n, tt);
    if (smem > (size_t)kSmemMax) return fail(PMC_ERR_UNSUPPORTED, "chain too long for the composite-trial kernel");
    const bool cut = h->energy_type == PMC_ENERGY_CUTOFF;
#define PMC_DS(TT)                                                                        \
  {                                                                                       \
    if (cut) {                                                                            \
      int rc = set_smem(k_delta_segment_cta<TT, true>, smem);                             \
      if (rc) return rc;                                                                  \
      k_delta_segment_cta<TT, true><<<1, TT, smem, h->stream>>>(a);                       \
    } else {                                                                              \
      int rc = set_smem(k_delta_segment_cta<TT, false>, smem);                            \
      if (rc) return rc;                                                                  \
      k_delta_segment_cta<TT, false><<<1, TT, smem, h->stream>>>(a);                      \
    }                                                                                     \
  }
    if (tt == 32) PMC_DS(32) else if (tt == 64) PMC_DS(64) else if (tt == 128) PMC_DS(128) else PMC_DS(256)
#undef PMC_DS
  }
  ++h->launches;
  PMC_CU(cudaGetLastError());
  return PMC_OK;
}
