// plan.cu — the launch planner: which run kernel a handle uses, with which block size, launch bound and shared memory.
//
// Environment overrides (read here and nowhere else, at every plan, that is at every run and every query):
//   PMC_RUN_PAIR=0|2           CTA pairs off / forced for any chain length (tests, tools/soak.py)
//   PMC_LANE_MODE=1|2          O(1)-ΔU chains: chain per lane / per warp (tests, tools/soak.py)
//   PMC_LANE_CLUSTER_MODE=1|2  the same for composite trials (tests, tools/soak.py)
//   PMC_RUN_SPEC=0             no k_run_cta_win_spec (tools/tune_spec_plain.py)
//   PMC_CLUSTER_SPEC=0         no k_run_cta_cluster_spec (tools/tune_spec.py)
//   PMC_PAIR_MINB=m            launch bound of k_run_cta_pair (tools/tune_pair_minb.py)
//   PMC_PAIR_ORDER=0           CTA pairs without the work-ordered queue (tools/c5_tail.py)
#include "handle.h"

namespace {

constexpr size_t kSmemPerSm = 233472;   // 228 KB of shared memory per SM on sm_100

// Ensemble size the shape is chosen for: the hint (pmc_set_ensemble_hint) when there is one, so a shard of a sweep runs the
// kernel the whole ensemble would (the packings sum the per-trial averager contributions in different orders; same kernel
// ⇒ results bit-identical however the sweep is sharded).
int64_t shape_chains(const pmc_handle* h) { return h->shape_chains > 0 ? h->shape_chains : h->nchains; }

// Block size of the interacting one-CTA kernels: enough threads to cover the mean rectangle (n²/6 pairs) without leaving
// most lanes idle on short chains.
int pick_cta_threads(int n) { return n <= 128 ? 64 : n <= 1024 ? 128 : n <= 1536 ? 256 : 512; }

// CTAs of the 128-thread composite-trial kernel that fit one SM's shared memory (2 … 4): the launch bound follows it,
// because a bound the shared memory cannot honour only takes registers away (n = 400: 3 per SM at 168 registers are
// +8 % over a bound of 4 at 128; n = 640: 2 per SM +20 %).
int cluster_fit128(int n) {
  const int fit = (int)((size_t)kSmemMax / (pmc::cluster_smem_bytes(n, 128) + 1024));
  for (int mb : kCluster128Minb)
    if (fit >= mb) return mb;
  return kCluster128Minb[2];
}

int cluster_minb(int threads, int n) {
  if (threads == 32) return kTeamMinb[n <= 40 ? 0 : n <= 110 ? 1 : 2];
  return threads == 64 ? kCluster64Minb : threads == 128 ? cluster_fit128(n) : kCluster256Minb;
}

// Block size for the ensemble at hand.  `base` is the shape that wins on a full machine (many chains per SM).
// A small ensemble leaves SMs idle — 148 chains of n=100 are one warp per SM — so each chain gets 2× or 4× the
// threads until the warps resident per SM reach what the base shape has when the machine is full
// (profiles/r01f_tune_small_ensembles.txt: +50–80 % at one chain per SM, nothing lost on large ensembles).
int scaled_threads(int base, int minb, size_t smem, int tmax, int64_t chains, int sms, int max_scale = 4) {
  const int fit = (int)std::max<size_t>(1, kSmemPerSm / (smem + 1024));     // CTAs per SM that fit in shared memory
  const int resident_max = std::min(minb, fit);
  const double sat = (double)resident_max * (base / 32);                     // warps per SM, full machine
  const double res = std::min((double)chains / sms, (double)resident_max) * (base / 32);
  int scale = 1;
  while (scale < max_scale && base * scale * 2 <= tmax && res * scale * 2 <= sat) scale *= 2;
  return base * scale;
}

// Block size of the CTA helper kernels of every handle but the composite-trial CTA ones, and of k_run_cta_win / pair.
int cta_block(const pmc_handle* h, int64_t chains) {
  const int base = pick_cta_threads(h->n);
  return scaled_threads(base, win_minb(base), pmc::cta_smem_bytes_win(h->n), 512, chains, h->sm_count);
}

// The most one-warp teams (8, 4, 2; the first `tries` of them) whose CTAs are all resident at once: a second wave costs
// more than the teams gain (profiles/r02d_tune_spec.txt: 500 chains on 444 slots of four teams lose to two teams).
// 0: none.
template <class Smem, class Minb, class Fits>
int spec_teams(int64_t chains, int sms, int tries, Smem smem, Minb minb, Fits fits) {
  const int teams[3] = {8, 4, 2};
  for (int k = 0; k < tries; ++k) {
    const int fit = (int)std::min<size_t>((size_t)minb(teams[k]), kSmemPerSm / (smem(teams[k]) + 1024));
    if (fit >= 1 && chains <= (int64_t)sms * fit && fits(teams[k])) return teams[k];
  }
  return 0;
}

// Composite trials with a pair sum (all-pairs, cut-off): one CTA per chain.  Short chains are latency bound (one serial
// proposal/cluster/decision chain per trial), so one warp per chain and many chains per SM; measured crossovers in
// profiles/r01e_tune_cluster.txt.  Small ensembles of one-warp-team chains (n ≤ 160) give the extra warps DIFFERENT trials
// of the same chain (k_run_cta_cluster_spec) instead of sharing one.
void plan_cluster_cta(const pmc_handle* h, int64_t chains, RunPlan& p) {
  const int n = h->n, base = pick_cluster_threads(n);
  auto delta_fits = [&](int t) { return pmc::cluster_delta_smem_bytes(n, t) <= (size_t)kSmemMax; };
  if (base == 32 && env_int("PMC_CLUSTER_SPEC", 1) != 0) {
    p.teams = spec_teams(chains, h->sm_count, 3, [&](int g) { return pmc::cluster_spec_smem_bytes(n, g); },
                         cluster_spec_minb, [&](int g) { return delta_fits(32 * g); });
    p.cta_threads = p.teams ? 32 * p.teams : 32;
  } else {
    p.cta_threads = scaled_threads(base, cluster_minb(base, n), pmc::cluster_smem_bytes(n, base), 256, chains, h->sm_count);
    while (p.cta_threads > base && !delta_fits(p.cta_threads)) p.cta_threads /= 2;
  }
  p.cut = h->energy_type == PMC_ENERGY_CUTOFF;
  p.threads = p.cta_threads;
  if (p.teams) {
    p.family = RunFamily::cta_cluster_spec;
    p.minb = cluster_spec_minb(p.teams);
    p.smem = pmc::cluster_spec_smem_bytes(n, p.teams);
  } else {
    p.family = RunFamily::cta_cluster;
    p.minb = cluster_minb(p.threads, n);
    p.smem = pmc::cluster_smem_bytes(n, p.threads);
  }
}

// When do two SMs per chain pay?  (profiles/r02b_tune_pair_small.txt, one B200)
//   * the staged copy leaves room for only one CTA per SM (n ≳ 2000): always — a launch of ≤ 148 chains is one wave and ends
//     with its slowest chain; pairs + the work-ordered queue take C5 from 0.62 to 0.71 of the DFMA peak at 50 trials;
//   * n > 768: at every ensemble size (n = 1024: 0.70–0.72 against 0.55–0.70), most for few chains;
//   * 384 < n ≤ 768: only when the chains fill between 0.55 and 0.9 of the resident CTA slots, where whole chains per SM
//     quantise badly (512 chains of n = 512 on 592 slots: 68 SMs carry four chains, 80 carry three: +15 % with pairs);
//     elsewhere the windowed one-CTA kernel is ahead (its proposals are off the critical path);
//   * shorter chains: never (the cluster barrier per trial is no longer small against the trial).
// Chains whose windowed one-CTA kernel does not fit shared memory (n ≳ 3900) always take pairs.  Otherwise PMC_RUN_PAIR=0
// switches pairs off and PMC_RUN_PAIR=2 forces them for any chain length.
bool use_pair_kernel(int n, int threads, int64_t chains, int sms, int mode) {
  if (threads != 128 && threads != 256 && threads != 512) return false;
  if (pmc::cta_smem_bytes_win(n) > (size_t)kSmemMax) return true;
  if (mode == 0) return false;
  if (mode == 2) return true;
  if (pmc::cta_smem_bytes(n) > (size_t)kSmemMax / 2) return true;
  if (n > 768) return true;
  if (n > 384) {
    const double fill = (double)chains / ((double)sms * win_minb(threads));
    return fill >= 0.55 && fill < 0.9;
  }
  return false;
}

// Single-monomer trials of interacting chains: one CTA per chain (k_run_cta_win, or k_run_cta_win_spec for small
// ensembles of short chains), two SMs per chain for long chains (k_run_cta_pair).
void plan_cta(const pmc_handle* h, int64_t chains, RunPlan& p) {
  const int n = h->n;
  p.threads = p.cta_threads;
  const int pair_mode = env_int("PMC_RUN_PAIR", 1);
  // Small ensembles of short chains: one-warp teams on DIFFERENT trials of the window instead of more warps on one trial.
  // Unlike the composite trial, the single-monomer trial has almost no serial head and shares well among warps, so this
  // pays only where a warp is enough for a trial (profiles/r02e_tune_spec_plain.txt): n ≤ 64 with the largest number of
  // teams whose CTAs are all resident at once (+10–70 %), and n ≤ 110 when every chain can have a whole SM (eight teams,
  // +17–29 %); above that the one-trial kernels win.  FP64 only.
  if (n <= 110 && h->pair_precision == PMC_PAIR_FP64 && pair_mode != 2 && env_int("PMC_RUN_SPEC", 1) != 0) {
    p.teams = spec_teams(chains, h->sm_count, n <= 64 ? 3 : 1, [&](int g) { return pmc::cta_smem_bytes_spec(n, g); },
                         spec_minb, [](int) { return true; });
    if (p.teams) {
      p.family = RunFamily::cta_win_spec;
      p.threads = 32 * p.teams;
      p.minb = spec_minb(p.teams);
      p.smem = pmc::cta_smem_bytes_spec(n, p.teams);
      return;
    }
  }
  if (use_pair_kernel(n, p.threads, chains, h->sm_count, pair_mode)) {
    p.family = RunFamily::cta_pair;
    p.smem = pmc::cta_smem_bytes(n);
    // what the shared memory admits (a bound it cannot honour only takes registers away), at most win_minb
    const int fit = (int)((size_t)kSmemMax / (p.smem + 1024)), cap = win_minb(p.threads);
    p.minb = std::max(1, std::min(fit, cap));
    const int o = env_int("PMC_PAIR_MINB", 0);
    if (o >= 1 && o <= cap) p.minb = o;
    // heaviest predicted work first; beyond 16 384 chains the queue alone balances
    p.pair_order = h->nchains <= 16384 && env_int("PMC_PAIR_ORDER", 1) != 0;
    return;
  }
  // windowed kernel, FP64 or FP32 rectangle (pmc_set_pair_precision)
  p.family = RunFamily::cta_win;
  p.minb = win_minb(p.threads);
  p.f32 = h->pair_precision == PMC_PAIR_FP32 && pmc::cta_smem_bytes_win_f32(n) <= (size_t)kSmemMax;
  p.smem = p.f32 ? pmc::cta_smem_bytes_win_f32(n) : pmc::cta_smem_bytes_win(n);
}

// O(1)-ΔU chains (non-interacting, Ising): one chain per warp with 32-trial windows fills the machine for few chains, one
// per lane for many.  Measured crossover (profiles/r02c_tune_lane_vs_warp.txt): non-interacting 14.8 vs 12.6 G updates/s
// at 65 536 chains and 14.5 vs 17.5 at 262 144; Ising level at 65 536.  PMC_LANE_MODE: 1 = lane, 2 = warp.
constexpr int64_t kWarpBelowIsing = 65536, kWarpBelowNonint = 120000;
void plan_lane(const pmc_handle* h, int64_t chains, RunPlan& p) {
  const int mode = env_int("PMC_LANE_MODE", 0);
  const int64_t below = p.ising ? kWarpBelowIsing : kWarpBelowNonint;
  if (mode == 2 || (mode == 0 && chains < below)) {
    p.family = RunFamily::warp;
    // at most one wave of warps (16 per SM): one chain per CTA, so that the block scheduler spreads the warps evenly
    p.cpb = chains <= (int64_t)h->sm_count * 16 ? 1 : 4;
    p.threads = 32 * p.cpb;
    p.minb = warp_minb(p.cpb);
  } else {
    p.family = RunFamily::lane;
    p.threads = 64;
    p.minb = lane_minb(p.comp);
  }
}

// Composite trials of the non-interacting and Ising energies: chain per warp below this many chains, else per lane.
// PMC_LANE_CLUSTER_MODE: 1 = lane, 2 = warp.
constexpr int64_t kWarpClusterBelow = 11000, kLaneClusterMany = 32768;
void plan_lane_cluster(const pmc_handle* h, int64_t chains, RunPlan& p) {
  const int mode = env_int("PMC_LANE_CLUSTER_MODE", 0);
  if (mode == 2 || (mode == 0 && chains < kWarpClusterBelow)) {
    p.family = RunFamily::warp_cluster;
    p.threads = 128;
    p.minb = kWarpClusterMinb;
    p.stage = h->n <= kWarpClusterStageMax;
    p.smem = p.stage ? (size_t)4 * h->n * sizeof(MonoRec) : 0;
  } else {
    p.family = RunFamily::lane_cluster;
    p.threads = 64;
    // many chains: occupancy beats the spills of the 128-register build
    p.minb = !p.comp && chains >= kLaneClusterMany ? kLaneClusterManyMinb : kLaneClusterMinb;
  }
}

}  // namespace

RunPlan plan_run(const pmc_handle* h) {
  RunPlan p;
  const int64_t chains = shape_chains(h);
  p.cta_threads = cta_block(h, chains);
  p.ising = h->energy_type == PMC_ENERGY_ISING;
  p.comp = h->compensated != 0;
  const bool pair_sum = h->energy_type == PMC_ENERGY_INTERACTING || h->energy_type == PMC_ENERGY_CUTOFF;
  if (h->cluster_mode && pair_sum) plan_cluster_cta(h, chains, p);
  else if (h->cluster_mode) plan_lane_cluster(h, chains, p);
  else if (h->energy_type == PMC_ENERGY_INTERACTING) plan_cta(h, chains, p);
  else plan_lane(h, chains, p);
  return p;
}

std::string kernel_name(const RunPlan& p) {
  char b[96];
  const char* comp = p.comp ? "true" : "false";
  switch (p.family) {
    case RunFamily::cta_win:
      std::snprintf(b, sizeof b, "k_run_cta_win<%d,%d,%d%s>", p.threads, p.minb, kRunUnroll, p.f32 ? ",fp32" : ""); break;
    case RunFamily::cta_win_spec: std::snprintf(b, sizeof b, "k_run_cta_win_spec<%d,%d>", p.teams, p.minb); break;
    case RunFamily::cta_pair: std::snprintf(b, sizeof b, "k_run_cta_pair<%d,%d,%d>", p.threads, p.minb, kRunUnroll); break;
    case RunFamily::lane: std::snprintf(b, sizeof b, "k_run_lane<%d,%d,%s>", p.threads, p.minb, comp); break;
    case RunFamily::warp:
      std::snprintf(b, sizeof b, p.cpb == 1 ? "k_run_warp<%d,%d,%s,1>" : "k_run_warp<%d,%d,%s>", (int)p.ising, p.minb, comp);
      break;
    case RunFamily::cta_cluster:
      std::snprintf(b, sizeof b, "k_run_cta_cluster<%d,%d%s>", p.threads, p.minb, p.cut ? ",cut" : ""); break;
    case RunFamily::cta_cluster_spec:
      std::snprintf(b, sizeof b, "k_run_cta_cluster_spec<%d,%d%s>", p.teams, p.minb, p.cut ? ",cut" : ""); break;
    case RunFamily::lane_cluster:
      std::snprintf(b, sizeof b, "k_run_lane_cluster<%d,%d%s>", p.threads, p.minb, p.comp ? ",comp" : ""); break;
    case RunFamily::warp_cluster:   // the name has no staging flag
      std::snprintf(b, sizeof b, "k_run_warp_cluster<%s,%d,%s>", p.ising ? "true" : "false", p.minb, comp); break;
  }
  return b;
}
