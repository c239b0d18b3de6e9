// handle.h — what the translation units of libpolymc_b200.so share: the handle behind the C ABI, error
// plumbing, and the launch helpers each kernel family's TU exports (one TU per family so that `make -j`
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
#include <unordered_map>
#include <vector>

#include "cluster_kernels.cuh"

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

// Every launch helper records the kernel it picks; with dry_run set it stops there (pmc_kernel_name).
#define PMC_PICK(name_literal)        \
  do {                                \
    h->kernel_name = name_literal;    \
    if (h->dry_run) return PMC_OK;    \
  } while (0)

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
  int cta_threads = 256;      // block size of the CTA-per-chain kernels
  int sm_count = 148;
  int64_t shape_chains = 0;   // ensemble size the launch shape is chosen for (0 = nchains), pmc_set_ensemble_hint
  // O(1)-ΔU chains of the plain driver: one chain per warp below this many chains, else one per lane.  Measured
  // crossover (profiles/r02c_tune_lane_vs_warp.txt): non-interacting 14.8 vs 12.6 G updates/s at 65 536 chains and 14.5 vs
  // 17.5 at 262 144; Ising level at 65 536.  Set from the energy type in launch_run_lane.
  long long warp_mode_below = 0;
  long long warp_cluster_below = 11000;  // composite trials: chain per warp below this many chains, else per lane
  int compensated = 0;        // Neumaier-compensated accumulators in the lane/warp kernels (CTA kernels: always)
  int spec_teams = 0;         // > 0: small ensemble of short interacting chains — one-warp teams on different trials (k_run_cta_win_spec)
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
  const char* kernel_name = "";  // the MCMC kernel the last (dry or real) launch decision picked, pmc_kernel_name
  int dry_run = 0;               // launch helpers only record their decision
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

// Ensemble size the chain-per-lane / chain-per-warp packing is chosen for: like the block size it follows the
// hint, so a shard of a sweep runs the kernel the whole ensemble would (the packings sum the per-trial averager
// contributions in different orders; same kernel ⇒ results bit-identical however the sweep is sharded).
inline int64_t packing_chains(const pmc_handle* h) { return h->shape_chains > 0 ? h->shape_chains : h->nchains; }

// Block size of the composite-trial CTA kernels.
// Short chains are latency bound (one serial proposal/cluster/decision chain per trial), so one warp per
// chain and many chains per SM; measured crossovers in profiles/r01e_tune_cluster.txt.  Chains whose shared-memory
// footprint (18 n doubles) leaves room for a single CTA per SM get 256 threads instead of 128: at n = 800 … 1000 one
// 128-thread CTA per SM is four warps on the whole SM (+74 % with 256 threads, profiles/r02b_tune_k35.txt).
inline int pick_cluster_threads(int n) {
  if (n <= 160) return 32;
  if (n <= 256) return 64;
  return 2 * (pmc::cluster_smem_bytes(n, 128) + 1024) > (size_t)kSmemMax ? 256 : 128;
}
// CTAs of the 128-thread composite-trial kernel that fit one SM's shared memory (2 … 4): the launch bound follows it,
// because a bound the shared memory cannot honour only takes registers away (n = 400: 3 per SM at 168 registers are
// +8 % over a bound of 4 at 128; n = 640: 2 per SM +20 %).
inline int cluster_fit128(int n) {
  const int fit = (int)((size_t)kSmemMax / (pmc::cluster_smem_bytes(n, 128) + 1024));
  return fit >= 4 ? 4 : fit >= 3 ? 3 : 2;
}

// ---- launch helpers, one translation unit per kernel family -------------------------------------------------
int launch_run_cta(pmc_handle* h, const pmc::RunArgs& a);                    // run_cta.cu
bool use_f32_rect(const pmc_handle* h);
int launch_run_pair(pmc_handle* h, const pmc::RunArgs& a);                   // run_pair.cu
bool use_pair_kernel(const pmc_handle* h);                                   // run_pair.cu
int launch_run_lane(pmc_handle* h, const pmc::RunArgs& a);                   // run_lane.cu
int launch_run_cluster_cta(pmc_handle* h, const pmc::RunArgs& a);            // run_cluster_cta.cu
int launch_delta_segment_cta(pmc_handle* h, const pmc::SegDeltaArgs& a);     // run_cluster_cta.cu
int launch_run_cluster_lane(pmc_handle* h, const pmc::RunArgs& a);           // run_cluster_lane.cu
int launch_exchange(pmc_handle* h, const pmc::ExchangeArgs& a, int64_t npairs);   // exchange.cu
int launch_place_rows(pmc_handle* h, double* dst, const double* src, int64_t rows, int64_t rows_total, int64_t row0,
                      int cols);                                             // exchange.cu
