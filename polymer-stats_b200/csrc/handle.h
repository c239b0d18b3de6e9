// handle.h — what the translation units of libpolymc_b200.so share: the handle behind the C ABI, error
// plumbing, and the launchers each kernel family's TU exports (one TU per family so that `make -j`
// compiles them in parallel).
#pragma once

#include "../../include/polymc.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <algorithm>
#include <chrono>
#include <mutex>
#include <type_traits>
#include <unordered_map>
#include <utility>
#include <vector>

#include "cluster_kernels.cuh"
#include "plan.h"

using namespace pmc;

namespace pmc {
struct ExPair;        // exchange.cuh
struct ExchangeArgs;
}  // namespace pmc

// sets the calling thread's pmc_last_error() text and returns `code`
int pmc_fail(int code, const std::string& msg);

#define PMC_CU(expr)                                                                              \
  do {                                                                                            \
    cudaError_t e__ = (expr);                                                                     \
    if (e__ != cudaSuccess) {                                                                     \
      cudaGetLastError();                                                                         \
      return pmc_fail((e__ == cudaErrorNoDevice || e__ == cudaErrorInsufficientDriver) ? PMC_ERR_NO_DEVICE \
                      : (e__ == cudaErrorMemoryAllocation)                              ? PMC_ERR_NOMEM \
                                                                                        : PMC_ERR_CUDA, \
                      std::string(#expr) + ": " + cudaGetErrorString(e__));                       \
    }                                                                                             \
  } while (0)

constexpr int kSmemMax = 232448;  // 227 KB opt-in limit per CTA on sm_100

inline int env_int(const char* name, int dflt) {
  const char* v = std::getenv(name);
  return (v && *v) ? std::atoi(v) : dflt;
}

struct pmc_handle {
  int device = 0;
  int64_t nchains = 0;
  int n = 0;
  int energy_type = 0;
  uint64_t seed = 0;
  uint32_t chain_id_base = 0;
  int init = 0;
  cudaStream_t stream = nullptr;
  MonoRec* mono = nullptr;
  MonoRec* cand = nullptr;
  ChainParams* par = nullptr;
  ChainDyn* dyn = nullptr;
  double* traj = nullptr;
  double* roll = nullptr;
  size_t traj_cap = 0, roll_cap = 0;
  double* scratch = nullptr;  // 2·nchains·n doubles (state staging) — also small outputs
  size_t scratch_cap = 0;
  int* flags = nullptr;       // nchains ints
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  float last_ms = 0.f;
  int64_t launches = 0;
  int sm_count = 148;
  int64_t shape_chains = 0;   // ensemble size the launch shape is chosen for (0 = nchains), pmc_set_ensemble_hint
  int compensated = 0;        // Neumaier-compensated accumulators in the lane/warp kernels (CTA kernels: always)
  int pair_precision = 0;     // 0: FP64 everywhere; 1: the rectangle of single-monomer trials in FP32 where a kernel exists (cta_f32.cuh)
  std::vector<ChainDyn> host_dyn;
  bool dyn_fresh = false, dynx_fresh = false;   // the host copies equal the device's (no launch since they were fetched)
  // clustering driver (mcmc_clustering_eap_chain.jl)
  int cluster_mode = 0;       // 1: the composite-trial kernels of cluster_kernels.cuh run this handle
  ChainDynX* dynx = nullptr;
  double* state = nullptr;    // [chains][rows][2n] state rows of the last pmc_run_ex
  size_t state_cap = 0;
  double* x0buf = nullptr;
  std::vector<pmc_case> cases;
  int replicas = 1;
  double kT_scale = 1.0;
  std::vector<ChainDynX> host_dynx;
  int planar = 0;             // 2-D tree
  // two SMs per chain (pair_kernels.cuh): predicted work, work-ordered queue
  unsigned long long* pair_work = nullptr;
  int* pair_order = nullptr;
  int* pair_next = nullptr;
  // replica exchange (exchange.cuh), set by pmc_set_ladders
  std::vector<int32_t> ladder;          // the rungs as given, ladders separated by -1; empty: no ladders
  pmc::ExPair* ex_pairs = nullptr;      // candidate pairs, those of even rounds first
  int64_t ex_count[2] = {0, 0};         // pairs of even / odd rounds
  unsigned long long* ex_stats = nullptr;   // [ncases][2] attempts, accepts with the next rung
  long long* ex_walker = nullptr;       // [chains] walker label of each slot
  int* ex_wstate = nullptr;             // [chains] round-trip state by walker
  long long* ex_trips = nullptr;        // [chains] round trips by walker
  int64_t ex_round = 0;                 // exchange rounds since pmc_set_ladders
  double* tt_out[3] = {nullptr, nullptr, nullptr};   // traj, roll, state rows of a whole pmc_run_tempering*
  size_t tt_cap[3] = {0, 0, 0};
  // conformation sampling (conformation.cuh), set by pmc_set_conformation; conf == nullptr: disabled
  double* conf = nullptr;               // [chains][8 + 3n + conf_bins] running sums
  int conf_bins = 0;
};

// Device memory of the handles comes from a per-device cache of freed blocks: a study creates and destroys one handle
// per bucket per call (polymc.sweep), and cudaMalloc / cudaFree (which synchronises the device) dominated such calls.
// pmc_release_cached_memory() returns everything to the driver.
cudaError_t pmc_pool_alloc(void** ptr, size_t bytes);   // on the current device
void pmc_pool_free(void* ptr);                          // back to the cache of the device it came from
template <typename P>
cudaError_t pool_alloc(P** ptr, size_t bytes) { return pmc_pool_alloc(reinterpret_cast<void**>(ptr), bytes); }

template <typename K>
int set_smem(K kernel, size_t bytes) {
  PMC_CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return PMC_OK;
}

// One launch on the handle's stream: the dynamic shared memory limit (when the kernel takes any), the launch, the count.
template <typename K, typename... Args>
int launch(pmc_handle* h, K kernel, unsigned grid, int block, size_t smem, const Args&... args) {
  if (smem > (size_t)kSmemMax) return pmc_fail(PMC_ERR_UNSUPPORTED, "chain too long for this kernel's shared memory");
  if (smem) {
    int rc = set_smem(kernel, smem);
    if (rc) return rc;
  }
  kernel<<<grid, block, smem, h->stream>>>(args...);
  ++h->launches;
  PMC_CU(cudaGetLastError());
  return PMC_OK;
}

// f(std::integral_constant<int, V>()) for the V of the list that equals v: maps a planned value onto an instantiation.
template <int... V, class F>
int with(int v, F&& f) {
  int rc = PMC_OK;
  const bool hit = ((v == V && ((rc = f(std::integral_constant<int, V>())), true)) || ...);
  return hit ? rc : pmc_fail(PMC_ERR_INVALID, "no kernel instantiated for this launch shape");
}
template <int LO, class F, int... I>
int with_offset(int v, F&& f, std::integer_sequence<int, I...>) { return with<(LO + I)...>(v, f); }
template <int LO, int HI, class F>   // v in LO … HI
int with_range(int v, F&& f) { return with_offset<LO>(v, f, std::make_integer_sequence<int, HI - LO + 1>()); }

// Block size of the composite-trial CTA kernels (and of their helper kernel k_delta_segment_cta).
// Short chains are latency bound (one serial proposal/cluster/decision chain per trial), so one warp per
// chain and many chains per SM; measured crossovers in profiles/r01e_tune_cluster.txt.  Chains whose shared-memory
// footprint (18 n doubles) leaves room for a single CTA per SM get 256 threads instead of 128: at n = 800 … 1000 one
// 128-thread CTA per SM is four warps on the whole SM (+74 % with 256 threads, profiles/r02b_tune_k35.txt).
inline int pick_cluster_threads(int n) {
  if (n <= 160) return 32;
  if (n <= 256) return 64;
  return 2 * (pmc::cluster_smem_bytes(n, 128) + 1024) > (size_t)kSmemMax ? 256 : 128;
}
// ---- launchers of the run kernels, one translation unit per kernel family: each maps a plan onto instantiations ----
int launch_run_cta(pmc_handle* h, const RunPlan& p, const pmc::RunArgs& a);           // run_cta.cu: cta_win, cta_win_spec
int launch_run_pair(pmc_handle* h, const RunPlan& p, const pmc::RunArgs& a);          // run_pair.cu: cta_pair
int launch_run_lane(pmc_handle* h, const RunPlan& p, const pmc::RunArgs& a);          // run_lane.cu: lane, warp
int launch_run_cluster_cta(pmc_handle* h, const RunPlan& p, const pmc::RunArgs& a);   // run_cluster_cta.cu
int launch_delta_segment_cta(pmc_handle* h, const pmc::SegDeltaArgs& a);              // run_cluster_cta.cu
int launch_run_cluster_lane(pmc_handle* h, const RunPlan& p, const pmc::RunArgs& a);  // run_cluster_lane.cu
int launch_exchange(pmc_handle* h, const pmc::ExchangeArgs& a, int64_t npairs);   // exchange.cu
int launch_place_rows(pmc_handle* h, double* dst, const double* src, int64_t rows, int64_t rows_total, int64_t row0,
                      int cols);                                             // exchange.cu
int launch_conformation(pmc_handle* h);                                      // conformation.cu
