// plan.h — which run kernel a handle launches, with which shape: the RunPlan that plan_run (plan.cu) computes, and the
// launch bounds of the run kernels.  The launchers (run_*.cu) map a plan onto template instantiations and decide nothing;
// pmc_kernel_name formats the same plan.
#pragma once

#include <cstddef>
#include <string>

struct pmc_handle;

enum class RunFamily {
  cta_win,           // k_run_cta_win<T, MINB, UNROLL, PREC>: interacting chain per CTA, proposal windows
  cta_win_spec,      // k_run_cta_win_spec<G, MINB>: small ensembles of short chains, one-warp teams on different trials
  cta_pair,          // k_run_cta_pair<T, MINB, UNROLL>: long interacting chains, two SMs per chain
  lane,              // k_run_lane<T, MINB, COMP>: O(1)-ΔU chain per lane
  warp,              // k_run_warp<ISING, MINB, COMP, CPB>: O(1)-ΔU chain per warp
  cta_cluster,       // k_run_cta_cluster<T, MINB, CUT>: composite trials, chain per CTA
  cta_cluster_spec,  // k_run_cta_cluster_spec<G, MINB, CUT>: composite trials, one-warp teams on different trials
  lane_cluster,      // k_run_lane_cluster<T, MINB, ISING, COMP>
  warp_cluster,      // k_run_warp_cluster<ISING, MINB, COMP, STAGE>
};

struct RunPlan {
  RunFamily family = RunFamily::cta_win;
  int threads = 0;          // block size of the run kernel
  int minb = 0;             // its launch bound: resident CTAs per SM
  int teams = 0;            // spec kernels: one-warp teams per CTA
  int cpb = 0;              // k_run_warp: chains per CTA
  bool f32 = false;         // FP32 rectangle (PREC = 1)
  bool cut = false;         // cut-off pair sum
  bool ising = false;
  bool comp = false;        // Neumaier-compensated accumulators of the lane/warp kernels
  bool stage = false;       // k_run_warp_cluster: records staged in shared memory
  bool pair_order = false;  // k_run_cta_pair: chains taken heaviest predicted work first
  size_t smem = 0;          // dynamic shared memory of the run kernel
  int cta_threads = 0;      // block size of the CTA helper kernels (energy, ΔU, re-initialisation)
};

// Everything the next run of `h` launches, from its driver, energy type, n, ensemble size, precision and the
// environment as it is now.  Pure: no launch, no state.
RunPlan plan_run(const pmc_handle* h);
// The instantiation a plan launches, e.g. "k_run_cta_win<128,4,2>" (pmc_kernel_name).
std::string kernel_name(const RunPlan& p);

// ---- launch bounds of the run kernels ---------------------------------------------------------------------------
// The planner tests residency with these and the launchers pass them as template arguments, so the two cannot drift.
constexpr int kRunUnroll = 2;   // UNROLL of k_run_cta_win and k_run_cta_pair

// k_run_cta_win: 16 warps per SM at every block size.  The same number of CTAs per SM bounds k_run_cta_pair (less where
// the shared memory admits fewer, pair_minb) and gives the CTA slots the pair kernel's fill rule counts.
constexpr int win_minb(int threads) { return 512 / threads; }
// k_run_cta_win_spec and k_run_cta_cluster_spec by teams per CTA (8, 4, 2)
constexpr int spec_minb(int teams) { return teams == 8 ? 1 : teams == 4 ? 3 : 6; }
constexpr int cluster_spec_minb(int teams) { return teams == 8 ? 1 : teams == 4 ? 3 : 5; }
// k_run_cta_cluster with one-warp teams, by chain length: n ≤ 40, n ≤ 110, longer.  Registers beat occupancy here
// (profiles/r02b_tune_k1.txt): 10 chains per SM at 204 registers are +6 % over 12 at 170 for n = 64 … 100, 8 per SM
// +11 % at n = 150; only very short chains gain from 16 per SM (+9 % at n = 25).
constexpr int kTeamMinb[3] = {16, 10, 8};
// k_run_cta_cluster with 64, 128 (as many CTAs as the shared memory holds, cluster_fit128) and 256 threads
constexpr int kCluster64Minb = 5, kCluster128Minb[3] = {4, 3, 2}, kCluster256Minb = 1;
// k_run_warp: 16 warps per SM, whether one chain (one warp) or four per CTA
constexpr int warp_minb(int cpb) { return 16 / cpb; }
// k_run_lane (64 threads): the 128-register build where the compensated accumulators need it
constexpr int lane_minb(bool comp) { return comp ? 4 : 6; }
// k_run_lane_cluster (64 threads): many chains trade the 128-register build's spills for occupancy
constexpr int kLaneClusterMinb = 4, kLaneClusterManyMinb = 8;
constexpr int kWarpClusterMinb = 2;   // k_run_warp_cluster, 128 threads
