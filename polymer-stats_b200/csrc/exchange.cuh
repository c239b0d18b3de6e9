// exchange.cuh — replica exchange (parallel tempering) between the rungs of a kT / force ladder (DESIGN.md §12).
//
// A ladder is an ordered list of cases of one handle; replica r of rung k pairs with replica r of rung k+1.  An
// exchange round swaps configurations between the two slots of a pair with the Metropolis rule that keeps every
// rung's distribution π_s(x) ∝ exp(−U_s(x)/kT_s)·Ω(x) exact.  It runs between two launches of the run kernels,
// which it does not touch: a slot keeps its parameters, accumulators, step sizes, counters and random stream.
#pragma once

#include "chain_math.cuh"

namespace pmc {

enum : uint32_t { SUB_EXCHANGE = 7 };

// One candidate pair: slot a is the lower rung.  flags bit 0: a is the bottom rung of its ladder; bit 1: b is the top.
struct ExPair {
  int a, b, stat, flags;
};

// Δ of the swap of slots a and b (accept iff Δ ≥ 0 or ε < exp(Δ)):
//   Δ = β_a [U_a(x_a) − U_a(x_b)] + β_b [U_b(x_b) − U_b(x_a)],  β = 1/kT,
//   U_a(x_b) = U_b(x_b) + r_b·(F_b − F_a)  (written to *Uab, the energy slot a keeps after an accepted swap),
//   U_b(x_a) = U_a(x_a) + r_a·(F_a − F_b)  (*Uba).
// The order of the FP64 operations is fixed here, without contraction into FMA, so that a restatement on the CPU
// (tests/tempering_ref.py) computes the same bits from the same inputs.
__host__ __device__ inline double exchange_delta(double kTa, double kTb, double Ua, double Ub, const double ra[3],
                                                 const double rb[3], double Fxa, double Fza, double Fxb, double Fzb,
                                                 double* Uab, double* Uba) {
#ifdef __CUDA_ARCH__
#define PMC_ADD __dadd_rn
#define PMC_SUB __dsub_rn
#define PMC_MUL __dmul_rn
#define PMC_DIV __ddiv_rn
#else
#define PMC_ADD(x, y) ((x) + (y))
#define PMC_SUB(x, y) ((x) - (y))
#define PMC_MUL(x, y) ((x) * (y))
#define PMC_DIV(x, y) ((x) / (y))
#endif
  const double dFx = PMC_SUB(Fxb, Fxa), dFz = PMC_SUB(Fzb, Fza);
  const double wb = PMC_ADD(PMC_MUL(rb[0], dFx), PMC_MUL(rb[2], dFz));   // r_b·(F_b − F_a)
  const double wa = PMC_ADD(PMC_MUL(ra[0], dFx), PMC_MUL(ra[2], dFz));   // r_a·(F_b − F_a)
  *Uab = PMC_ADD(Ub, wb);
  *Uba = PMC_SUB(Ua, wa);
  const double ba = PMC_DIV(1.0, kTa), bb = PMC_DIV(1.0, kTb);
  return PMC_ADD(PMC_MUL(ba, PMC_SUB(Ua, *Uab)), PMC_MUL(bb, PMC_SUB(Ub, *Uba)));
#undef PMC_ADD
#undef PMC_SUB
#undef PMC_MUL
#undef PMC_DIV
}

// ε of the attempt of round `round` on the pair whose lower slot is global chain `chain_id` at stream tag `init`.
__device__ __forceinline__ double draw_exchange_eps(uint64_t seed, uint32_t chain_id, uint32_t init, long long round) {
  const uint4 w = philox_at<false>(seed, chain_id, init, SUB_EXCHANGE, (uint64_t)round);
  return u53(w.x, w.y);
}

struct ExchangeArgs {
  MonoRec* mono;
  const ChainParams* par;
  ChainDyn* dyn;
  ChainDynX* dynx;
  const ExPair* pairs;          // the pairs of this round's parity
  unsigned long long* stats;    // [ncases][2] attempts, accepts with the next rung
  long long* walker;            // [chains] global id of the initial configuration a slot holds
  int* wstate;                  // [chains] by walker: 0 bottom not yet visited, 1 heading up, 2 top visited, heading down
  long long* trips;             // [chains] by walker: completed bottom → top → bottom trips
  int* accepted;                // [chains] 1 at the lower slot of an accepted pair (zeroed by the host)
  uint64_t seed;
  uint32_t chain_id_base;
  int n;
  long long round;
};

// A walker arrives at slot `slot` (bottom / top of its ladder per the pair flags).
__device__ __forceinline__ void walker_arrives(const ExchangeArgs& a, long long walker, bool bottom, bool top) {
  const long long w = walker - (long long)a.chain_id_base;
  if (bottom) {
    if (a.wstate[w] == 2) a.trips[w] += 1;
    a.wstate[w] = 1;
  } else if (top && a.wstate[w] == 1) {
    a.wstate[w] = 2;
  }
}

// One CTA per candidate pair.  Thread 0 decides; on acceptance the CTA swaps the two chains' records with 16-byte
// accesses and thread 0 swaps the scalars that travel with the configuration.
template <int T>
__global__ void __launch_bounds__(T) k_exchange(const ExchangeArgs a) {
  __shared__ int take;
  const ExPair pr = a.pairs[blockIdx.x];
  if (threadIdx.x == 0) {
    const ChainDyn& Da = a.dyn[pr.a];
    const ChainDyn& Db = a.dyn[pr.b];
    const ChainParams& Pa = a.par[pr.a];
    const ChainParams& Pb = a.par[pr.b];
    double Uab, Uba;
    const double delta = exchange_delta(Pa.kT, Pb.kT, Da.U, Db.U, Da.r, Db.r, Pa.Fx, Pa.Fz, Pb.Fx, Pb.Fz, &Uab, &Uba);
    int acc = delta >= 0.0;
    if (!acc) acc = draw_exchange_eps(a.seed, a.chain_id_base + (uint32_t)pr.a, (uint32_t)Da.init, a.round) < exp(delta);
    atomicAdd(&a.stats[2 * pr.stat], 1ull);
    if (acc) {
      atomicAdd(&a.stats[2 * pr.stat + 1], 1ull);
      a.accepted[pr.a] = 1;
      ChainDyn& A = a.dyn[pr.a];
      ChainDyn& B = a.dyn[pr.b];
      const double Om = A.Omega, su = A.su;
      A.Omega = B.Omega; B.Omega = Om;
      A.su = B.su; B.su = su;
      for (int k = 0; k < 3; ++k) {
        const double r = A.r[k], p = A.p[k];
        A.r[k] = B.r[k]; B.r[k] = r;
        A.p[k] = B.p[k]; B.p[k] = p;
      }
      A.U = Uab;
      B.U = Uba;
      ChainDynX& X = a.dynx[pr.a];
      ChainDynX& Y = a.dynx[pr.b];
      const double sp = X.spsi, c2 = X.scos2;
      X.spsi = Y.spsi; Y.spsi = sp;
      X.scos2 = Y.scos2; Y.scos2 = c2;
      X.carry = 0.0;   // the acceptor is re-bound to the configuration the slot now holds
      Y.carry = 0.0;
      const long long wa = a.walker[pr.a], wb = a.walker[pr.b];
      a.walker[pr.a] = wb;
      a.walker[pr.b] = wa;
      walker_arrives(a, wb, pr.flags & 1, false);
      walker_arrives(a, wa, false, pr.flags & 2);
    }
    take = acc;
  }
  __syncthreads();
  if (!take) return;
  static_assert(sizeof(MonoRec) % sizeof(int4) == 0, "MonoRec must be a whole number of 16-byte words");
  constexpr int W = sizeof(MonoRec) / sizeof(int4);
  int4* xa = reinterpret_cast<int4*>(a.mono + (size_t)pr.a * a.n);
  int4* xb = reinterpret_cast<int4*>(a.mono + (size_t)pr.b * a.n);
  for (int i = threadIdx.x; i < W * a.n; i += T) {
    const int4 va = xa[i], vb = xb[i];
    xa[i] = vb;
    xb[i] = va;
  }
}

}  // namespace pmc
