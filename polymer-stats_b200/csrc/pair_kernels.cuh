// pair_kernels.cuh — long interacting chains: TWO SMs per chain (a 2-CTA thread-block cluster), chains taken from a
// work-ordered queue.
//
// At n ≈ 4096 the staged chain (x, μ, E: 7n doubles = 229 KB) fills one SM's shared memory, so the CTA-per-chain kernel
// runs one chain per SM, and with ≤ 148 chains per GPU (config C5 on 8 GPUs) the launch is ONE wave: it ends with its
// slowest chain, whose work Σ_trials idx·(n−1−idx) spreads by ±6 % (1σ) over 50 trials — the FP64 pipe was 82 % busy
// while resident but 68 % of elapsed (profiles/r01f_ncu_full_k_run_cta_C5_n4096.txt).  Here
//   * both CTAs of a cluster hold the SAME chain in their shared memory and each evaluates half of the flattened
//     changed-pair set (row {idx}×rest + rectangle heads×tails); the two partial sums are exchanged through
//     distributed shared memory (one remote store + one cluster barrier per trial) and added in a fixed order, so both
//     CTAs take the same accept/reject decision and apply it to their own copy — no other traffic between them;
//   * a cluster runs chain after chain from a global queue ordered by PREDICTED work, heaviest first (LPT): the
//     monomer index of every trial is a counter-based draw that does not depend on the chain's state
//     (mcmc_eap_chain.jl:277 `idx = rand(1:n)`), so Σ idx·(n−1−idx) of a launch is known before it starts.
// The Markov chain, its Philox stream and the order of the pair-sum reduction inside a CTA are those of k_run_cta_win; only
// the split of the pair set over 2·T threads differs (results agree with the one-CTA kernels to rounding, decisions are
// the same: tests/test_gpu_round2.py::test_c5_run_kernel_trajectory_n4096).
#pragma once

#include <cooperative_groups.h>

#include "cta_kernels.cuh"

namespace pmc {

namespace cg = cooperative_groups;

// The 2·NW warps of a CTA pair that share the pair work of one chain; every CTA has its own copy of the chain.
template <int NW>
struct PairTeam {
  static constexpr int kWarps = 2 * NW;
  static constexpr int kThreads = 2 * NW * 32;
  static constexpr int kLocalThreads = NW * 32;
  __device__ __forceinline__ static int rank() { return (int)cg::this_cluster().block_rank(); }
  __device__ __forceinline__ static int tid() { return rank() * NW * 32 + (int)threadIdx.x; }
  __device__ __forceinline__ static int ltid() { return (int)threadIdx.x; }
  __device__ __forceinline__ static int warp() { return rank() * NW + (int)(threadIdx.x >> 5); }
  __device__ __forceinline__ static int lane() { return (int)(threadIdx.x & 31); }
  __device__ __forceinline__ static void sync() { __syncthreads(); }
};

struct PairQueue {
  const int* order;   // chain ids, heaviest predicted work first (null: 0, 1, 2, …)
  int* next;          // queue head
};

// Predicted pair work of one launch per chain: Σ over its trials of (n−1) + idx·(n−1−idx).
__global__ void k_predict_work(const ChainDyn* __restrict__ dyn, int nchains, int n, long long nsteps, uint64_t seed,
                               uint32_t chain_id_base, unsigned long long* __restrict__ work) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nchains) return;
  const long long step0 = dyn[c].step;
  const uint32_t init = (uint32_t)dyn[c].init;
  unsigned long long w = 0;
  for (long long s = 1; s <= nsteps; ++s) {
    const uint4 a = philox_at(seed, chain_id_base + (uint32_t)c, init, SUB_STEP_A, (uint64_t)(step0 + s));
    const uint64_t v = ((uint64_t)a.y << 32) | a.x;
    const unsigned long long idx = __umul64hi(v, (uint64_t)n);
    w += (unsigned long long)(n - 1) + idx * (unsigned long long)(n - 1 - (long long)idx);
  }
  work[c] = w;
}

// order[] = chain ids by decreasing work: rank of chain c = #{d : w_d > w_c or (w_d == w_c and d < c)} — O(chains²)
// comparisons, a few hundred chains at the lengths this kernel is for.
__global__ void k_order_by_work(const unsigned long long* __restrict__ work, int nchains, int* __restrict__ order,
                                int* __restrict__ next) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c == 0) *next = 0;
  if (c >= nchains) return;
  const unsigned long long w = work[c];
  int r = 0;
  for (int d = 0; d < nchains; ++d) {
    const unsigned long long wd = work[d];
    r += (wd > w) || (wd == w && d < c);
  }
  order[r] = c;
}

// The hot loop of mcmc_eap_chain.jl:276-350 for interacting chains, one chain per CTA PAIR.
template <int T, int MINB, int UNROLL = 2>
__global__ void __launch_bounds__(T, MINB) k_run_cta_pair(const RunArgs a, const PairQueue q) {
  using TEAM = PairTeam<T / 32>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const CtaView S = carve(smem_raw, a.n);
  // exchange slots in the unused tail of `part` (block_sum uses T/32 entries, load_chain 3·T/32 ≤ 48 of 96):
  // xch[parity][rank] partial pair sums, xnext = the chain id handed out by rank 0
  double* xch = S.part + 64;
  int* xnext = reinterpret_cast<int*>(S.part + 72);
  double* xch_peer = cluster.map_shared_rank(xch, rank ^ 1);
  int* xnext_peer = cluster.map_shared_rank(xnext, rank ^ 1);
  const int tid = threadIdx.x;
  const int n = a.n;
  cluster.sync();   // both CTAs have started before either touches the other's shared memory

  for (;;) {
    // ---- next chain of the queue (both CTAs must agree) ---------------------------------------------------------
    if (rank == 0 && tid == 0) {
      const int k = atomicAdd(q.next, 1);
      const int c = k < a.nchains ? (q.order ? q.order[k] : k) : -1;
      *xnext = c;
      *xnext_peer = c;
    }
    cluster.sync();
    const int c = *xnext;
    if (c < 0) break;
    MonoRec* mono = a.mono + (size_t)c * n;
    if (tid == 0) {
      *S.par = a.par[c];
      *S.dyn = a.dyn[c];
    }
    __syncthreads();
    const ChainParams& P = *S.par;
    load_chain<T>(mono, P, n, S);
    const uint32_t chain_id = a.chain_id_base + (uint32_t)c;
    const double b = P.b, inv_kT = P.inv_kT;
    const long long step0 = S.dyn->step;
    long long row = 0;
    if (tid == 0) make_proposal(a, P, *S.dyn, mono, chain_id, (uint32_t)S.dyn->init, step0 + 1, S.prop[1]);

    for (long long s = 1; s <= a.nsteps; ++s) {
      const long long step = step0 + s;
      __syncthreads();  // (A) proposal of this trial and state updates of the previous one are visible
      const Proposal* pr = &S.prop[s & 1];
      const int idx = pr->idx;
      const bool skip = pr->skip;
      const double dnx = pr->dnx, dny = pr->dny, dnz = pr->dnz;
      double dsum = 0.0;
      bool accept = false;
      // both CTAs see the same proposal (same record, same draws), so both skip or none does
      double* slot = xch + 2 * (int)(s & 1);
      if (!skip) {
        const double part = delta_pairs_partial<TEAM, UNROLL>(S, n, 1, b, idx, pr->mx, pr->my, pr->mz, dnx, dny, dnz);
        const double mine = block_sum<T>(part, S.part, /*trailing_sync=*/false);
        if (tid == 0) {
          slot[rank] = mine;
          xch_peer[2 * (int)(s & 1) + rank] = mine;
        }
      }
      // One cluster barrier per trial, skipped trials included: it publishes the peer's half (release/acquire at cluster
      // scope) and, two trials later, guarantees the peer has read a slot before it is written again.
      cluster.sync();
      if (!skip) accept = decide(pr->single, slot[0] + slot[1], inv_kT, pr->eps, dsum);
      if (accept) shift_tail(S, idx + 1, n, b * dnx, b * dny, b * dnz, tid, T);   // apply move! to this CTA's copy
      if (tid == 0) {
        // both CTAs store the same record: each later reads back what its own SM wrote
        if (accept) move_pivot(S, mono, *pr, idx, b, dnx, dny, dnz);
        after_decision(P, *S.dyn, *pr, accept, dsum, step);
      }
      const bool isrow = a.stepout > 0 && (step % a.stepout) == 0;
      if (isrow && tid < 32 && rank == 0) emit_row(a, *S.dyn, c, row, step, S.rowbuf, tid);
      if (isrow) ++row;
      if (tid == 0 && s < a.nsteps)
        make_proposal(a, P, *S.dyn, mono, chain_id, (uint32_t)S.dyn->init, step + 1, S.prop[(s + 1) & 1]);
    }
    __syncthreads();
    if (tid == 0 && rank == 0) a.dyn[c] = *S.dyn;
    cluster.sync();   // nobody overwrites the exchange slots or the staged chain while the peer still reads them
  }
}

}  // namespace pmc
