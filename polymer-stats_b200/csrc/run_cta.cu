// run_cta.cu — launches of the single-monomer-trial CTA-per-chain run kernels (cta_kernels.cuh): k_run_cta_win,
// k_run_cta_win_spec; chains whose windowed kernel does not fit one CTA go to k_run_cta_pair (run_pair.cu).
#include "handle.h"

namespace {
int fail(int code, const std::string& msg) { return pmc_fail(code, msg); }
}  // namespace

// FP32 rectangle (pmc_set_pair_precision): served by the windowed one-CTA kernel; every other launch stays FP64.
bool use_f32_rect(const pmc_handle* h) {
  if (h->pair_precision != 1 || h->energy_type != PMC_ENERGY_INTERACTING || h->cluster_mode) return false;
  if (use_pair_kernel(h)) return false;
  if (h->cta_threads != 64 && h->cta_threads != 128 && h->cta_threads != 256 && h->cta_threads != 512) return false;
  return cta_smem_bytes_win_f32(h->n) <= (size_t)kSmemMax;
}

int launch_run_cta(pmc_handle* h, const RunArgs& a) {
  const int nb = (int)h->nchains;
  if (h->spec_teams > 0 && h->pair_precision == 0 && env_int("PMC_RUN_PAIR", 1) != 2) {
    const size_t smem = cta_smem_bytes_spec(h->n, h->spec_teams);
#define PMC_LAUNCH_SPEC(GG, MB)                                                  \
  {                                                                              \
    PMC_PICK("k_run_cta_win_spec<" #GG "," #MB ">");                             \
    int rc = set_smem(k_run_cta_win_spec<GG, MB>, smem);                         \
    if (rc) return rc;                                                           \
    k_run_cta_win_spec<GG, MB><<<nb, 32 * GG, smem, h->stream>>>(a);             \
    ++h->launches;                                                               \
    PMC_CU(cudaGetLastError());                                                  \
    return PMC_OK;                                                               \
  }
    if (h->spec_teams == 8) PMC_LAUNCH_SPEC(8, 1)
    if (h->spec_teams == 4) PMC_LAUNCH_SPEC(4, 3)
    if (h->spec_teams == 2) PMC_LAUNCH_SPEC(2, 6)
#undef PMC_LAUNCH_SPEC
  }
  if (use_pair_kernel(h)) return launch_run_pair(h, a);
  // windowed kernel (32 proposals built at once by warp 0), FP64 or FP32 rectangle
  const bool f32 = use_f32_rect(h);
  const size_t smem = f32 ? cta_smem_bytes_win_f32(h->n) : cta_smem_bytes_win(h->n);
  if (smem > (size_t)kSmemMax) return fail(PMC_ERR_UNSUPPORTED, "chain too long for the one-CTA run kernel");
#define PMC_LAUNCH_WIN(TT, MB, PREC, NAME)                                  \
  {                                                                         \
    PMC_PICK(NAME);                                                         \
    int rc = set_smem(k_run_cta_win<TT, MB, 2, PREC>, smem);                \
    if (rc) return rc;                                                      \
    k_run_cta_win<TT, MB, 2, PREC><<<nb, TT, smem, h->stream>>>(a);         \
    break;                                                                  \
  }
#define PMC_LAUNCH_WIN2(TT, MB)                                                      \
  case TT:                                                                           \
    if (f32) PMC_LAUNCH_WIN(TT, MB, 1, "k_run_cta_win<" #TT "," #MB ",2,fp32>")     \
    else PMC_LAUNCH_WIN(TT, MB, 0, "k_run_cta_win<" #TT "," #MB ",2>")
  switch (h->cta_threads) {
    PMC_LAUNCH_WIN2(64, 8)
    PMC_LAUNCH_WIN2(128, 4)
    PMC_LAUNCH_WIN2(256, 2)
    PMC_LAUNCH_WIN2(512, 1)
    default: return fail(PMC_ERR_INVALID, "bad cta_threads");
  }
#undef PMC_LAUNCH_WIN2
#undef PMC_LAUNCH_WIN
  ++h->launches;
  PMC_CU(cudaGetLastError());
  return PMC_OK;
}
