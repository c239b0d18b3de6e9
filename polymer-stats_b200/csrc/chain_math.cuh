// chain_math.cuh — device-side chain physics shared by every kernel of libpolymc_b200.
//
// Restates, for one monomer / one pair at a time, the arithmetic of
//   inc/eap_chain.jl:40-58 (n̂, ψ, u, ubend), :176-187 and :200-207 (pair terms), :230-257 (move!),
//   :263-333 (refl_n!, cluster_flip!), inc/dipole_response.jl:7-29, inc/acceptance.jl:29-37,
//   mcmc_eap_chain.jl:277-280
// in the changed-pair ΔU form of SURVEY.md §8a.  All arithmetic is FP64.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace pmc {

constexpr double kPi = 3.14159265358979323846;
constexpr double kInv4Pi = 0.07957747154594767;  // 1/(4π), hoisted out of the pair term

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. SC'11).  Stream definition (DESIGN.md "RNG streams"):
//   key = (seed_lo, seed_hi), counter = (pos_lo, pos_hi, chain_id, (init << 8) | sub)
// ---------------------------------------------------------------------------------------------
enum : uint32_t { SUB_STEP_A = 0, SUB_STEP_B = 1, SUB_INIT = 2, SUB_REINIT = 3, SUB_CLUSTER_UP = 4,
                  SUB_CLUSTER_DOWN = 5, SUB_CLUSTER_GATE = 6 };

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// Shared (not inlined) copies of the long library routines.  The chain-per-lane and chain-per-warp composite-trial
// kernels are serial, latency-bound code whose top stall is instruction fetch (profiles/r01f_*): a trial calls
// acos up to 8 times, sincos 4, log 3, Philox 5+, and one inlined copy per call site (≈100–200 SASS instructions
// each) makes the loop body several times the 32 KB instruction cache.  With SH = true every call site jumps to
// the same copy (K4 +31 %, K2 +11 % from acos alone).  The CTA kernels, where these calls are rare next to the
// pair loops, keep the inlined versions (SH = false, the default everywhere).
static __device__ __noinline__ uint4 philox_shared(uint4 c, uint2 k) { return philox4x32_10(c, k); }
static __device__ __noinline__ void sincos_shared(double x, double* s, double* c) { sincos(x, s, c); }
static __device__ __noinline__ double log_shared(double x) { return log(x); }
static __device__ __noinline__ double exp_shared(double x) { return exp(x); }
static __device__ __noinline__ double acos_shared(double x) { return acos(x); }

// Call sites without an explicit choice use the inlined versions.
constexpr bool kSharedLib = false;

template <bool SH>
struct Lib {
  __device__ __forceinline__ static uint4 philox(uint4 c, uint2 k) { return SH ? philox_shared(c, k) : philox4x32_10(c, k); }
  __device__ __forceinline__ static void sincos_(double x, double* s, double* c) {
    if (SH) sincos_shared(x, s, c);
    else sincos(x, s, c);
  }
  __device__ __forceinline__ static double log_(double x) { return SH ? log_shared(x) : log(x); }
  __device__ __forceinline__ static double exp_(double x) { return SH ? exp_shared(x) : exp(x); }
  __device__ __forceinline__ static double acos_(double x) { return SH ? acos_shared(x) : acos(x); }
};

template <bool SH = kSharedLib>
__device__ __forceinline__ uint4 philox_at(uint64_t seed, uint32_t chain_id, uint32_t init, uint32_t sub,
                                           uint64_t pos) {
  return Lib<SH>::philox(make_uint4((uint32_t)pos, (uint32_t)(pos >> 32), chain_id, (init << 8) | sub),
                         make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}

__device__ __forceinline__ double u53(uint32_t lo, uint32_t hi) {
  const uint64_t v = ((uint64_t)hi << 32) | lo;
  return (double)(v >> 11) * 0x1.0p-53;
}

// cluster_flip! draws an unbounded number of uniforms per trial (eap_chain.jl:273,291,307): uniform #k
// of the upward / downward growth is word pair (k&1) of the Philox block at position
// step + ((k>>1) << 40) of stream SUB_CLUSTER_UP / _DOWN (steps stay below 2^40).
template <bool SH = kSharedLib>
__device__ __forceinline__ uint4 cluster_block(uint64_t seed, uint32_t chain_id, uint32_t init, long long step,
                                               uint32_t sub, int k) {
  return philox_at<SH>(seed, chain_id, init, sub, (uint64_t)step + (((uint64_t)k >> 1) << 40));
}

template <bool SH = kSharedLib>
__device__ __forceinline__ double draw_cluster(uint64_t seed, uint32_t chain_id, uint32_t init, long long step,
                                               uint32_t sub, int k) {
  const uint4 w = cluster_block<SH>(seed, chain_id, init, step, sub, k);
  return (k & 1) ? u53(w.z, w.w) : u53(w.x, w.y);
}

template <bool SH = kSharedLib>
__device__ __forceinline__ double draw_cluster_gate(uint64_t seed, uint32_t chain_id, uint32_t init,
                                                    long long step) {
  const uint4 w = philox_at<SH>(seed, chain_id, init, SUB_CLUSTER_GATE, (uint64_t)step);
  return u53(w.x, w.y);
}

// ---------------------------------------------------------------------------------------------
// Per-monomer record in HBM.  (phi, theta) is the independent state (EAPChain.ϕs/θs,
// eap_chain.jl:22,25); n̂ and sinθ are the caches a proposal needs (n̂s, sθs, :27,:28).
// ---------------------------------------------------------------------------------------------
struct __align__(16) MonoRec {
  double phi, theta;
  double nx, ny;
  double nz, sth;
};

// Per-chain constants (one case of the sweep).
struct ChainParams {
  double alpha, beta, m;  // μ = (alpha·n̂z + m)·n̂ + beta·ẑ : dielectric alpha=(K1-K2)E0, beta=K2·E0; polar m=mu
  double E0, kT, inv_kT, Fz, Fx, b;
  double adj_lb, adj_ub, adj_scale;
  double cF;              // 0.2 + 0.8 exp(-(Fx²+Fz²)/kT), average.jl:121-122
  double gauge0;          // log_gauge without Ω0: -(K1+2K2)E0² n/(3kT)  or  -mu·E0·n/(3kT) (average.jl:109-118)
  double phi_step0, theta_step0;
  long long steps_per_adjust;
  int do_flips, umbrella, force_init, pad;
  // clustering driver (mcmc_clustering_eap_chain.jl): bending energy, cut-off pair sum, cluster flips
  double kappa, psi0;     // --bend-mod, --bend-angle (eap_chain.jl:54-58)
  double crad2;           // (cutoff-radius · mlen)², eap_chain.jl:102,172
  double cluster_prob;    // cluster_flip! returns early iff rand() <= cluster_prob (eap_chain.jl:273)
  int clustering, alpha_carry, cutoff_full;
  int planar;             // 2-D tree (2D/inc/eap_chain.jl): state is ϕ only, n̂ = (cosϕ, 0, sinϕ), no solid angle
};

constexpr int kNumAcc = 17;  // 16 sums (rolling.csv order) + normaliser

// Per-chain mutable scalars.
struct ChainDyn {
  double U, Omega, su;    // running energy, Σ log sinθ, Σ u_i
  double r[3], p[3];      // end-to-end vector, net dipole
  double phi_step, theta_step;
  double log_gauge;       // AntiDipoleWeightFunction.log_gauge (fixed at construction)
  double drift_max;       // max |U_running - U_recomputed| seen at re-synchronisation
  double acc[kNumAcc], comp[kNumAcc];  // Neumaier-compensated sums
  long long nacc, natt, nacc_total, steps_total, step;
  int init, valid;
};

// Extra per-chain scalars of the clustering driver (kept apart from ChainDyn so that the tuned kernels
// of mcmc_eap_chain.jl are untouched).
struct ChainDynX {
  double spsi, scos2;           // running Σψ_i and Σcos²θ_i (mcmc_clustering_eap_chain.jl:243-244)
  double carry;                 // logπ_prev − logπ(chain) = log α of the last accepted trial (acceptance.jl:30-33)
  double acc[2], comp[2];       // Σ of the two extra averagers (Neumaier-compensated)
  double ncluster, cluster_sum, cluster_max;  // trials with a cluster flip, Σ cluster sizes, largest cluster
};

// ---------------------------------------------------------------------------------------------
// Small math helpers
// ---------------------------------------------------------------------------------------------
// 1/sqrt(x) to ≈1 ulp: MUFU.RSQ64H seed + one cubically convergent correction
//   y ← y (1 + e/2 + 3e²/8), e = 1 - x y²   (seed error ≲2^-20 ⇒ result error ≲2^-60).
__device__ __forceinline__ double rsqrt_cubic(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double e = fma(-x, y * y, 1.0);
  const double t = fma(e, 0.375, 0.5);
  return fma(y * e, t, y);
}

#ifndef PMC_RSQRT_VARIANT
#define PMC_RSQRT_VARIANT 0
#endif
#if PMC_RSQRT_VARIANT != 0
// Measured negative result (tools/rect_bench.cu, profiles/r01f_rect_bench_rsqrt_variants.txt), not in the product
// build: 3 instead of 5 FP64-pipe instructions per 1/sqrt by refining the seed on the FP32 pipe (MUFU.RSQ of the
// rounded x + one FP32 Newton step, error ≲2^-23) and one quadratic FP64 step y ← y + (y/2)e (≲3e-14 relative).
// The FP64 pipe takes an issue slot every other cycle and the rectangle loop already fills most of the others,
// so the ≈16 extra FP32/integer/XU instructions per 1/sqrt cost more than the 2 DFMA they save.
// Variant 1: F2F width conversions; 2: conversions on the integer pipe; 3: 2 without the range check.
__device__ __forceinline__ double rsqrt_mixed(double x) {
#if PMC_RSQRT_VARIANT == 1
  const float xf = (float)x;
#else
  const int hi = __double2hiint(x), lo = __double2loint(x);
#if PMC_RSQRT_VARIANT == 2
  if ((unsigned)(hi - 0x38100000) >= 0x0fe00000u) return rsqrt_cubic(x);  // outside the FP32 normal range
#endif
  const float xf = __int_as_float(__funnelshift_l(lo, hi - 0x38000000, 3));  // truncated, not rounded
#endif
  float yf;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(yf) : "f"(xf));
  const float ef = fmaf(-(xf * yf), yf, 1.0f);
  yf = fmaf(0.5f * yf, ef, yf);
#if PMC_RSQRT_VARIANT == 1
  if (!(fabsf(ef) <= 1e-3f)) return rsqrt_cubic(x);
  const double y = (double)yf;
  const int yhi = __double2hiint(y), ylo = __double2loint(y);
#else
  const int yb = __float_as_int(yf);
  const int yhi = (yb >> 3) + 0x38000000, ylo = yb << 29;
  const double y = __hiloint2double(yhi, ylo);
#endif
  const double h = __hiloint2double(yhi - 0x00100000, ylo);  // y/2
  const double e = fma(-x, y * y, 1.0);
  return fma(h, e, y);
}
__device__ __forceinline__ double rsqrt_fast(double x) { return rsqrt_mixed(x); }
#else
__device__ __forceinline__ double rsqrt_fast(double x) { return rsqrt_cubic(x); }
#endif

// 4π × one dipole-dipole pair term (eap_chain.jl:200-207): μa·μb/r³ − 3(μa·r)(μb·r)/r⁵.
__device__ __forceinline__ double pair_g(double ax, double ay, double az, double bx, double by, double bz,
                                         double rx, double ry, double rz) {
  const double r2 = fma(rz, rz, fma(ry, ry, rx * rx));
  const double mm = fma(az, bz, fma(ay, by, ax * bx));
  const double a = fma(az, rz, fma(ay, ry, ax * rx));
  const double b = fma(bz, rz, fma(by, ry, bx * rx));
  const double y = rsqrt_fast(r2);
  const double y2 = y * y;
  const double t = fma(-3.0 * a * b, y2, mm);
  return t * (y2 * y);
}

// One term of UCutoff (eap_chain.jl:176-187): zero when r² > crad².
__device__ __forceinline__ double pair_g_cut(double ax, double ay, double az, double bx, double by, double bz,
                                             double rx, double ry, double rz, double crad2) {
  const double r2 = fma(rz, rz, fma(ry, ry, rx * rx));
  const double g = pair_g(ax, ay, az, bx, by, bz, rx, ry, rz);
  return (r2 > crad2) ? 0.0 : g;
}

// ψ (eap_chain.jl:45-47): acos(min(1, max(-1, n̂_a·n̂_b)))
template <bool SH = kSharedLib>
__device__ __forceinline__ double psi_of(double ax, double ay, double az, double bx, double by, double bz) {
  const double d = fma(az, bz, fma(ay, by, ax * bx));
  return Lib<SH>::acos_(fmin(1.0, fmax(-1.0, d)));
}

// ubend (eap_chain.jl:54-58)
__device__ __forceinline__ double ubend_of(const ChainParams& P, double psi) {
  const double t = psi - P.psi0;
  return 0.5 * P.kappa * t * t;
}

// pflip_linear of a bond (eap_chain.jl:267,290): (1 + n̂_a·n̂_b)/2
__device__ __forceinline__ double link_prob(double ax, double ay, double az, double bx, double by, double bz) {
  return (1.0 + (ax * bx + ay * by + az * bz)) / 2.0;
}

// refl_n! (eap_chain.jl:263-265) = move!(chain, i, 0, π − 2θ_i): θ ← clamp(θ + (π − 2θ)).
__device__ __forceinline__ double reflect_theta(double theta) {
  return fmin(kPi, fmax(0.0, theta + (kPi - 2.0 * theta)));
}

__device__ __forceinline__ void mu_of(const ChainParams& P, double nx, double ny, double nz, double& mx,
                                      double& my, double& mz) {
  const double f = P.alpha * nz + P.m;
  mx = f * nx;
  my = f * ny;
  mz = f * nz + P.beta;
}

// Neumaier compensated add: (s, c) += v.
__device__ __forceinline__ void comp_add(double& s, double& c, double v) {
  const double t = s + v;
  c += (fabs(s) >= fabs(v)) ? ((s - t) + v) : ((v - t) + s);
  s = t;
}

// ---------------------------------------------------------------------------------------------
// One trial move of monomer idx (steps 1-4 of SURVEY Appendix A).
// ---------------------------------------------------------------------------------------------
struct Proposal {
  double nx, ny, nz;      // n̂'
  double mx, my, mz;      // μ'
  double dnx, dny, dnz;   // Δn̂
  double dmx, dmy, dmz;   // Δμ
  double phi, theta, sth; // new angles and sinθ'
  double du, drF, dOmega; // Δu_idx, −b(FxΔn̂x+FzΔn̂z), log(sinθ'/sinθ)
  double single;          // −(du+drF)/kT + dΩ [+ Δw]: everything but the pair sum
  double eps;
  int idx;
  int skip;               // sinθ' == 0 ⇒ logπ' = −Inf ⇒ certain rejection (eap_chain.jl:236-238)
  int clamped;
  int pad;
};

// Raw random draws of one trial: idx, dϕ, [Bool], dθ, ϵ (mcmc_eap_chain.jl:277-280,287).
struct Draws {
  double u_phi, u_theta, eps;
  int idx, flipbit;
};

template <bool SH = kSharedLib>
__device__ __forceinline__ Draws draw_step(uint64_t seed, uint32_t chain_id, uint32_t init, long long step,
                                           int n) {
  const uint4 a = philox_at<SH>(seed, chain_id, init, SUB_STEP_A, (uint64_t)step);
  const uint4 b = philox_at<SH>(seed, chain_id, init, SUB_STEP_B, (uint64_t)step);
  Draws d;
  const uint64_t v = ((uint64_t)a.y << 32) | a.x;
  d.idx = (int)__umul64hi(v, (uint64_t)n);
  d.u_phi = u53(a.z, a.w);
  d.flipbit = (int)(a.z & 1u);
  d.u_theta = u53(b.x, b.y);
  d.eps = u53(b.z, b.w);
  return d;
}

// move! up to the energy (eap_chain.jl:232-251) for given increments.
template <bool SH = kSharedLib>
__device__ __forceinline__ void build_proposal(const ChainParams& P, const MonoRec& rec, int idx, double dphi,
                                               double dtheta, double eps, Proposal& q) {
  q.idx = idx;
  q.eps = eps;
  q.phi = rec.phi + dphi;  // never wrapped (:232)
  const double traw = rec.theta + dtheta;
  q.theta = fmin(kPi, fmax(0.0, traw));  // clamped, not reflected (:236)
  q.clamped = (q.theta != traw);
  double sph, cph, sth, cth;
  Lib<SH>::sincos_(q.phi, &sph, &cph);
  Lib<SH>::sincos_(q.theta, &sth, &cth);
  q.sth = sth;
  q.nx = cph * sth;
  q.ny = sph * sth;
  q.nz = cth;
  mu_of(P, q.nx, q.ny, q.nz, q.mx, q.my, q.mz);
  double omx, omy, omz;
  mu_of(P, rec.nx, rec.ny, rec.nz, omx, omy, omz);
  q.dnx = q.nx - rec.nx;
  q.dny = q.ny - rec.ny;
  q.dnz = q.nz - rec.nz;
  q.dmx = q.mx - omx;
  q.dmy = q.my - omy;
  q.dmz = q.mz - omz;
  q.dOmega = Lib<SH>::log_(sth / rec.sth);             // :238
  q.du = -0.5 * P.E0 * q.mz - (-0.5 * P.E0 * omz);     // u = −½E0μz, :53
  q.drF = -P.b * (q.dnx * P.Fx + q.dnz * P.Fz);        // −Δr·F, energy.jl:8
  const double dw = P.umbrella ? q.du * P.inv_kT * P.cF : 0.0;  // average.jl:120-124
  q.single = -(q.du + q.drF) * P.inv_kT + q.dOmega + dw;
  q.skip = (sth == 0.0);
}

// move! of the planar chain (2D/inc/eap_chain.jl:171-187): ϕ += dϕ, n̂ = (cosϕ, sinϕ) in the x–z plane
// (the field is along the second axis, 2D/inc/dipole_response.jl:7-10), no θ and no solid-angle term.
// In the record: n̂y = 0, sinθ ≡ 1 (so every log(sinθ'/sinθ) is exactly 0), θ ≡ 0.
template <bool SH = kSharedLib>
__device__ __forceinline__ void build_proposal_planar(const ChainParams& P, const MonoRec& rec, int idx, double dphi,
                                                      double eps, Proposal& q) {
  q.idx = idx;
  q.eps = eps;
  q.phi = rec.phi + dphi;
  q.theta = 0.0;
  q.clamped = 0;
  double sph, cph;
  Lib<SH>::sincos_(q.phi, &sph, &cph);
  q.sth = 1.0;
  q.nx = cph; q.ny = 0.0; q.nz = sph;
  mu_of(P, q.nx, q.ny, q.nz, q.mx, q.my, q.mz);
  double omx, omy, omz;
  mu_of(P, rec.nx, rec.ny, rec.nz, omx, omy, omz);
  q.dnx = q.nx - rec.nx; q.dny = 0.0; q.dnz = q.nz - rec.nz;
  q.dmx = q.mx - omx; q.dmy = q.my - omy; q.dmz = q.mz - omz;
  q.dOmega = 0.0;
  q.du = -0.5 * P.E0 * q.mz - (-0.5 * P.E0 * omz);   // u = −½E0μ[2], 2D/inc/eap_chain.jl:64
  q.drF = -P.b * (q.dnx * P.Fx + q.dnz * P.Fz);      // −Δr·[Fx;Fz], 2D/inc/energy.jl:8
  const double dw = P.umbrella ? q.du * P.inv_kT * P.cF : 0.0;
  q.single = -(q.du + q.drF) * P.inv_kT + dw;
  q.skip = 0;
}

// Proposal increments from raw draws: rand(Uniform(-s,s)) = -s + 2s·u (mcmc_eap_chain.jl:278-280).
__device__ __forceinline__ void increments(const ChainParams& P, const Draws& d, double theta_old,
                                           double phi_step, double theta_step, double& dphi, double& dtheta) {
  dphi = -phi_step + (2.0 * phi_step) * d.u_phi;
  dtheta = ((P.do_flips && d.flipbit) ? kPi - 2.0 * theta_old : 0.0) + (-theta_step + (2.0 * theta_step) * d.u_theta);
}

// Metropolis on Δlogπ (acceptance.jl:32): NaN and −Inf both reject.
template <bool SH = kSharedLib>
__device__ __forceinline__ bool metropolis(double dlogpi, double eps) {
  return (dlogpi >= 0.0) || (eps < Lib<SH>::exp_(dlogpi));
}

// Step-size adaptation, mcmc_eap_chain.jl:301-322 (counters reset only when a change fires).
__device__ __forceinline__ void adapt_apply(const ChainParams& P, double& phi_step, double& theta_step,
                                            long long& nacc, long long& natt) {
  const double ratio = (double)nacc / (double)natt;
  if (ratio > P.adj_ub && phi_step != kPi && theta_step != kPi / 2) {
    nacc = 0;
    natt = 0;
    phi_step = fmin(kPi, phi_step * P.adj_scale);
    theta_step = fmin(kPi / 2, theta_step * P.adj_scale);
  } else if (ratio < P.adj_lb) {
    nacc = 0;
    natt = 0;
    phi_step /= P.adj_scale;
    theta_step /= P.adj_scale;
  }
}

__device__ __forceinline__ void adapt_steps(const ChainParams& P, long long step, double& phi_step,
                                            double& theta_step, long long& nacc, long long& natt) {
  if (P.adj_scale != 1.0 && P.steps_per_adjust > 0 && step % P.steps_per_adjust == 0)
    adapt_apply(P, phi_step, theta_step, nacc, natt);
}

// `step % period == 0` for consecutive steps without the 64-bit division: trials left until the next multiple.
struct Countdown {
  long long left, period;
  __device__ __forceinline__ void start(long long step0, long long per) {  // the first step seen is step0 + 1
    period = per;
    left = per > 0 ? per - (step0 % per) : -1;
  }
  __device__ __forceinline__ bool tick() {
    if (period <= 0) return false;
    if (--left != 0) return false;
    left = period;
    return true;
  }
};

// record! of the 8 averagers (average.jl:40-48; umbrella :63-73) on the current state.  STRIDE: distance between
// consecutive accumulators (1: a thread's own array; 32: one lane's column of a [17][32] shared-memory tile).
template <bool COMP = true, int STRIDE = 1>
__device__ __forceinline__ void record_averages(const ChainParams& P, double* acc, double* comp,
                                                const double* r, const double* p, double U, double su,
                                                double log_gauge) {
  double wgt = 1.0;
  if (P.umbrella) wgt = 1.0 / Lib<kSharedLib>::exp_(su * P.inv_kT * P.cF - log_gauge);
  const double v[kNumAcc] = {r[0], r[1], r[2], r[0] * r[0], r[1] * r[1], r[2] * r[2],
                             r[0] * r[0] + r[1] * r[1] + r[2] * r[2],
                             p[0], p[1], p[2], p[0] * p[0], p[1] * p[1], p[2] * p[2],
                             p[0] * p[0] + p[1] * p[1] + p[2] * p[2],
                             U, U * U, 1.0};
#pragma unroll
  for (int k = 0; k < kNumAcc; ++k) {
    if (COMP) comp_add(acc[k * STRIDE], comp[k * STRIDE], v[k] * wgt);
    else acc[k * STRIDE] += v[k] * wgt;  // plain Float64 sums, as the reference's default --numeric-type (average.jl:40-48)
  }
}

}  // namespace pmc
