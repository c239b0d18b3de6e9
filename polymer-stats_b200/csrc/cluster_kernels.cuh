// cluster_kernels.cuh — the trial of the clustering driver (mcmc_clustering_eap_chain.jl:267-279):
//   move!(trial, idx, dϕ, dθ)  →  α = cluster_flip!(trial, idx)  →  acceptor(trial, ϵ; α)
// with bending energy (--bend-mod/--bend-angle, eap_chain.jl:54-58), the cut-off pair sum (UCutoff,
// eap_chain.jl:165-192) and the two extra averagers ⟨Σcos²θ⟩, ⟨Σψ/(n−1)⟩ (:243-244).
//
// The reference deep-copies the chain, calls move! and then refl_n! (= move!(i, 0, π−2θ_i)) for every
// monomer of the cluster, each with a full O(n²) energy recompute (eap_chain.jl:311-315).  Here the whole
// composite trial is ONE segment update: monomers lo..hi get new directions and dipoles, the tail j>hi is
// translated rigidly by D = bΣΔn̂, so the changed pair terms are segment×everything plus the rectangle
// heads(i<lo)×tails(j>hi) (same rectangle code as the single-monomer kernels), the changed bond angles
// are lo−1..hi.  A trial without a cluster is the segment lo = hi = idx.
//
// Two packings, as for mcmc_eap_chain.jl: one CTA per chain (all-pairs and cut-off energies), one chain
// per lane (non-interacting and Ising energies).
#pragma once

#include "lane_kernels.cuh"

namespace pmc {

// Sums reduced over the CTA for one composite trial.
enum { R_PAIR = 0, R_BEND, R_PSI, R_USELF, R_OMEGA, R_COS2, R_PX, R_PY, R_PZ, kNumRed };

struct ClusterCtl {
  int idx, lo, hi, reflect;
  double up, lp;      // link probabilities at the two ends of the cluster before the flip (eap_chain.jl:276-305)
  double Dx, Dy, Dz;  // tail translation bΣΔn̂ of a segment built by warp 0
  unsigned dirty;     // proposals of the current window invalidated by an accepted trial
  unsigned pad;
};

// What the composite trial needs of the single-monomer move (a Proposal without the single-monomer energy terms,
// which the segment sums recompute), plus the gate decision of cluster_flip!: one entry of the proposal window.
struct ClProposal {
  double nx, ny, nz, sth;  // n̂', sinθ'
  double phi, theta;       // new angles
  double dOmega, eps;
  int idx, reflect;
};

struct ClView {
  double *nhx, *nhy, *nhz;  // n̂_i of the current state (eap_chain.jl:27)
  double *nnx, *nny, *nnz;  // n̂'_i of the trial, valid on the segment
  double *xnx, *xny, *xnz;  // x'_i of the trial, valid on the segment
  double *psi, *psn;        // bond angles ψ_i of the current state (eap_chain.jl:29) and of the trial (bonds lo−1..hi)
  double* red;              // [kNumRed][warps] warp partials
  ClProposal* win;          // [kWin]
  ClusterCtl* ctl;
  ChainDynX* dx;
};

// Bytes of the composite-trial arrays that follow the CtaView part.
__host__ __device__ inline size_t cluster_extra_bytes(int n, int threads) {
  size_t b = (size_t)11 * n * sizeof(double) + (size_t)kNumRed * (threads / 32) * sizeof(double);
  b += kWin * sizeof(ClProposal) + sizeof(ClusterCtl) + sizeof(ChainDynX);
  return (b + 15) & ~(size_t)15;
}
// run kernel (compact CtaView) / parity-seam kernel (full CtaView with its Proposal slots)
__host__ __device__ inline size_t cluster_smem_bytes(int n, int threads) {
  return cta_smem_bytes_compact(n, threads) + cluster_extra_bytes(n, threads);
}
__host__ __device__ inline size_t cluster_delta_smem_bytes(int n, int threads) {
  return cta_smem_bytes(n) + cluster_extra_bytes(n, threads);
}

__device__ __forceinline__ ClView carve_cluster(unsigned char* base, int n, int threads) {
  ClView X;
  double* d = reinterpret_cast<double*>(base);
  X.nhx = d; X.nhy = d + n; X.nhz = d + 2 * n;
  X.nnx = d + 3 * n; X.nny = d + 4 * n; X.nnz = d + 5 * n;
  X.xnx = d + 6 * n; X.xny = d + 7 * n; X.xnz = d + 8 * n;
  X.psi = d + 9 * n; X.psn = d + 10 * n;
  X.red = d + 11 * n;
  X.win = reinterpret_cast<ClProposal*>(X.red + kNumRed * (threads / 32));
  X.ctl = reinterpret_cast<ClusterCtl*>(X.win + kWin);
  X.dx = reinterpret_cast<ChainDynX*>(X.ctl + 1);
  return X;
}

// n̂ and the bond angles ψ of the staged chain.  Ends with a barrier.
template <int T>
__device__ __forceinline__ void load_nhat(const MonoRec* __restrict__ mono, int n, const ClView& X) {
  for (int i = team_tid<T>(); i < n; i += T) {
    const MonoRec r = mono[i];
    X.nhx[i] = r.nx; X.nhy[i] = r.ny; X.nhz[i] = r.nz;
  }
  team_sync<T>();
  for (int i = team_tid<T>(); i + 1 < n; i += T)
    X.psi[i] = psi_of(X.nhx[i], X.nhy[i], X.nhz[i], X.nhx[i + 1], X.nhy[i + 1], X.nhz[i + 1]);
  team_sync<T>();
}

// n̂ of monomer i on the chain that carries the single-monomer move (cluster_flip! runs on the trial
// chain AFTER move!, mcmc_clustering_eap_chain.jl:272-273).
template <class PQ>
__device__ __forceinline__ void nhat_trial(const ClView& X, const PQ& q, int i, double& x, double& y, double& z) {
  if (i == q.idx) { x = q.nx; y = q.ny; z = q.nz; }
  else { x = X.nhx[i]; y = X.nhy[i]; z = X.nhz[i]; }
}

// Draw and build the single-monomer part of trial `step` (mcmc_clustering_eap_chain.jl:267-270; the 2-D driver
// draws no dθ, 2D/mcmc_clustering_eap_chain.jl:238-241).
__device__ __forceinline__ void make_proposal_cl(const RunArgs& a, const ChainParams& P, const ChainDyn& D,
                                                 const MonoRec* mono, uint32_t chain_id, long long step, Proposal& q) {
  const Draws d = draw_step(a.seed, chain_id, (uint32_t)D.init, step, a.n);
  const MonoRec rec = mono[d.idx];
  double dphi, dtheta;
  increments(P, d, rec.theta, D.phi_step, D.theta_step, dphi, dtheta);
  if (P.planar) build_proposal_planar(P, rec, d.idx, dphi, d.eps, q);
  else build_proposal(P, rec, d.idx, dphi, dtheta, d.eps, q);
}

// The gate of cluster_flip!.  3-D: `if rand() <= ϵflip; return 1.0; end` BEFORE the growth (eap_chain.jl:273):
// flips with 1 − ϵflip;  2-D: `if rand() <= ϵflip … flip` AFTER the growth (2D/inc/eap_chain.jl:233): flips with ϵflip.
template <bool SH = kSharedLib>
__device__ __forceinline__ int cluster_gate(const ChainParams& P, uint64_t seed, uint32_t chain_id, uint32_t init,
                                            long long step) {
  if (!P.clustering) return 0;
  const double gate = draw_cluster_gate<SH>(seed, chain_id, init, step);
  return P.planar ? (gate <= P.cluster_prob) : !(gate <= P.cluster_prob);
}

// One entry of the proposal window: everything of trial `step` that depends on the chain only through the record
// of its own monomer.
__device__ __forceinline__ void make_window_entry(const RunArgs& a, const ChainParams& P, const ChainDyn& D,
                                                  const MonoRec* mono, uint32_t chain_id, long long step,
                                                  ClProposal& w) {
  Proposal q;
  make_proposal_cl(a, P, D, mono, chain_id, step, q);
  w.nx = q.nx; w.ny = q.ny; w.nz = q.nz; w.sth = q.sth;
  w.phi = q.phi; w.theta = q.theta;
  w.dOmega = q.dOmega; w.eps = q.eps;
  w.idx = q.idx;
  w.reflect = cluster_gate(P, a.seed, chain_id, (uint32_t)D.init, step);
}

// cluster_flip! up to the flips (eap_chain.jl:273-309), by one warp: the growth draws are counter-based,
// so 32 bonds are tested per round and the first failing one ends the growth — same result as the
// reference's sequential loop on the same uniforms.
template <class PQ>
__device__ __forceinline__ void warp_cluster_grow(const ClView& X, const PQ& q, int reflect, const ChainParams& P, int n,
                                                  uint64_t seed, uint32_t chain_id, uint32_t init, long long step,
                                                  ClusterCtl& out) {
  constexpr unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int idx = q.idx;
  int lo = idx, hi = idx;
  double up = 0.0, lp = 0.0;
  if (reflect) {
    // upward: bond (u,u+1), eap_chain.jl:276-289
    for (int k0 = 0;; k0 += 32) {
      const int bnd = hi + lane;
      bool stop = true;
      double pr = 0.0;
      if (bnd < n - 1) {
        double ax, ay, az, bx, by, bz;
        nhat_trial(X, q, bnd, ax, ay, az);
        nhat_trial(X, q, bnd + 1, bx, by, bz);
        pr = link_prob(ax, ay, az, bx, by, bz);
        stop = !(draw_cluster(seed, chain_id, init, step, SUB_CLUSTER_UP, k0 + lane) <= pr);
      }
      const unsigned m = __ballot_sync(FULL, stop);
      if (m) {
        const int f = __ffs(m) - 1;
        up = __shfl_sync(FULL, pr, f);  // 0 when the chain end stopped the growth (:277-279)
        hi += f;
        break;
      }
      hi += 32;
    }
    // downward: bond (l−1,l), eap_chain.jl:292-305
    for (int k0 = 0;; k0 += 32) {
      const int l = lo - lane;
      bool stop = true;
      double pr = 0.0;
      if (l > 0) {
        double ax, ay, az, bx, by, bz;
        nhat_trial(X, q, l, ax, ay, az);
        nhat_trial(X, q, l - 1, bx, by, bz);
        pr = link_prob(ax, ay, az, bx, by, bz);
        stop = !(draw_cluster(seed, chain_id, init, step, SUB_CLUSTER_DOWN, k0 + lane) <= pr);
      }
      const unsigned m = __ballot_sync(FULL, stop);
      if (m) {
        const int f = __ffs(m) - 1;
        lp = __shfl_sync(FULL, pr, f);
        lo -= f;
        break;
      }
      lo -= 32;
    }
  }
  if (lane == 0) {
    out.idx = idx; out.lo = lo; out.hi = hi; out.reflect = reflect;
    out.up = up; out.lp = lp;
  }
}

// New angles of segment monomer c: move! for idx (already in the proposal), then refl_n! if the cluster
// is flipped.  Returns ϕ', θ'.
template <class PQ>
__device__ __forceinline__ void segment_angles(const MonoRec* __restrict__ mono, const PQ& q, int c,
                                               bool reflect, int planar, double& phi, double& theta,
                                               double& sth_before) {
  if (c == q.idx) {
    phi = q.phi; theta = q.theta; sth_before = q.sth;
  } else {
    const MonoRec r = mono[c];
    phi = r.phi; theta = r.theta; sth_before = r.sth;
  }
  if (reflect) {
    if (planar) phi += kPi;  // flip_n! = move!(chain, i, π), 2D/inc/eap_chain.jl:189-191
    else theta = reflect_theta(theta);
  }
}

// n̂ and sinθ from the angles: (cosϕ sinθ, sinϕ sinθ, cosθ) (eap_chain.jl:40) or the planar (cosϕ, 0, sinϕ).
template <bool SH = kSharedLib>
__device__ __forceinline__ void direction_of(int planar, double phi, double theta, double& nx, double& ny, double& nz,
                                             double& sth) {
  double sph, cph;
  Lib<SH>::sincos_(phi, &sph, &cph);
  if (planar) {
    nx = cph; ny = 0.0; nz = sph; sth = 1.0;
  } else {
    double cth;
    Lib<SH>::sincos_(theta, &sth, &cth);
    nx = cph * sth; ny = sph * sth; nz = cth;
  }
}

// refl_n! / flip_n! of one monomer by symmetry, without transcendentals: refl_n! maps θ → π−θ, i.e.
// n̂ → (n̂x, n̂y, −n̂z) with sinθ unchanged (eap_chain.jl:263-265); the planar flip_n! maps ϕ → ϕ+π, i.e. n̂ → −n̂
// (2D/inc/eap_chain.jl:189-191).  Equal to the reference's recomputed cos/sin in real arithmetic.
__device__ __forceinline__ void flip_dir(int planar, double nx, double ny, double nz, double& fx, double& fy,
                                         double& fz) {
  if (planar) { fx = -nx; fy = -ny; fz = -nz; }
  else { fx = nx; fy = ny; fz = -nz; }
}

// S.E[c] of a segment monomer whose record keeps its sinθ (flipped by symmetry).
constexpr double kKeepSinTheta = -1.0;

// New direction of segment monomer c: n̂', sinθ' and this monomer's share of the changed single-monomer sums.
template <class PQ>
__device__ __forceinline__ void segment_monomer(const CtaView& S, const ClView& X, const MonoRec* __restrict__ mono,
                                                const ChainParams& P, const PQ& q, int c, bool reflect,
                                                double* acc, double& dnx, double& dny, double& dnz) {
  double nx, ny, nz, sth;
  if (!reflect) {  // the segment is idx alone
    nx = q.nx; ny = q.ny; nz = q.nz; sth = q.sth;
    acc[R_OMEGA] += q.dOmega;
  } else if (c != q.idx && (P.planar || X.nhz[c] != -1.0)) {
    // refl_n! / flip_n! of an unmoved monomer by symmetry, no transcendental: θ → π−θ is n̂ → (n̂x, n̂y, −n̂z)
    // with sinθ and hence Ω unchanged (eap_chain.jl:263-265); the planar ϕ → ϕ+π is n̂ → −n̂.  A monomer
    // sitting at θ = π (cosθ = −1) reflects to sinθ' = 0 exactly and goes the literal way below.
    double ox = X.nhx[c], oy = X.nhy[c], oz = X.nhz[c];
    flip_dir(P.planar, ox, oy, oz, nx, ny, nz);
    sth = kKeepSinTheta;  // the record keeps its sinθ
  } else {
    double phi, theta, sb;
    segment_angles(mono, q, c, true, P.planar, phi, theta, sb);
    direction_of(P.planar, phi, theta, nx, ny, nz, sth);
    if (!P.planar) acc[R_OMEGA] += (c == q.idx ? q.dOmega : 0.0) + Lib<kSharedLib>::log_(sth / sb);  // Ω += log(sθ'/sθ), eap_chain.jl:238
  }
  X.nnx[c] = nx; X.nny[c] = ny; X.nnz[c] = nz;
  S.E[c] = sth;
  double ux, uy, uz;
  mu_of(P, nx, ny, nz, ux, uy, uz);
  const double ox = S.mx[c], oy = S.my[c], oz = S.mz[c];
  acc[R_USELF] += -0.5 * P.E0 * uz - (-0.5 * P.E0 * oz);
  acc[R_PX] += ux - ox; acc[R_PY] += uy - oy; acc[R_PZ] += uz - oz;
  const double onz = X.nhz[c];
  acc[R_COS2] += nz * nz - onz * onz;
  dnx = nx - X.nhx[c]; dny = ny - X.nhy[c]; dnz = nz - onz;
}

// Segments of at most 32 monomers (nearly all of them) are built by the warp that selected the cluster:
// one monomer per lane, positions by a warp scan (update_xs! restricted to the segment, eap_chain.jl:49-51).
// Leaves n̂', x' in X.nn / X.xn, sinθ' in S.E, D = bΣΔn̂ in ctl; the lanes keep their partial sums in acc.
template <class PQ>
__device__ __forceinline__ void warp_segment_build(const CtaView& S, const ClView& X, const MonoRec* __restrict__ mono,
                                                   const ChainParams& P, const PQ& q, int lo, int hi,
                                                   bool reflect, double* acc, ClusterCtl& ctl) {
  constexpr unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int c = lo + lane;
  double dx = 0, dy = 0, dz = 0;
  if (c <= hi) segment_monomer(S, X, mono, P, q, c, reflect, acc, dx, dy, dz);
  double ix = dx, iy = dy, iz = dz;
#pragma unroll 1
  for (int o = 1; o < 32; o <<= 1) {
    const double tx = __shfl_up_sync(FULL, ix, o);
    const double ty = __shfl_up_sync(FULL, iy, o);
    const double tz = __shfl_up_sync(FULL, iz, o);
    if (lane >= o) { ix += tx; iy += ty; iz += tz; }
  }
  if (c <= hi) {
    X.xnx[c] = S.sx[c] + P.b * ((ix - dx) + 0.5 * dx);
    X.xny[c] = S.sy[c] + P.b * ((iy - dy) + 0.5 * dy);
    X.xnz[c] = S.sz[c] + P.b * ((iz - dz) + 0.5 * dz);
  }
  if (lane == 31) { ctl.Dx = P.b * ix; ctl.Dy = P.b * iy; ctl.Dz = P.b * iz; }
}

// The same for longer segments, by the whole CTA: contiguous chunks per thread and a block scan.
// Contains two CTA barriers.
template <int T, class PQ>
__device__ __forceinline__ void cta_segment_build(const CtaView& S, const ClView& X, const MonoRec* __restrict__ mono,
                                                  const ChainParams& P, const PQ& q, int lo, int hi,
                                                  bool reflect, double* acc, double& Dx, double& Dy, double& Dz) {
  constexpr int W = T / 32;
  const int tid = team_tid<T>(), lane = tid & 31, warp = tid >> 5;
  const int m = hi - lo + 1;
  const int C = (m + T - 1) / T;
  const int c0 = min(hi + 1, lo + tid * C), c1 = min(hi + 1, c0 + C);
  double lx = 0, ly = 0, lz = 0;
  for (int c = c0; c < c1; ++c) {
    double dx, dy, dz;
    segment_monomer(S, X, mono, P, q, c, reflect, acc, dx, dy, dz);
    lx += dx; ly += dy; lz += dz;
  }
  double ix = lx, iy = ly, iz = lz;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double tx = __shfl_up_sync(0xffffffffu, ix, o);
    const double ty = __shfl_up_sync(0xffffffffu, iy, o);
    const double tz = __shfl_up_sync(0xffffffffu, iz, o);
    if (lane >= o) { ix += tx; iy += ty; iz += tz; }
  }
  if (lane == 31) { S.part[warp] = ix; S.part[W + warp] = iy; S.part[2 * W + warp] = iz; }
  team_sync<T>();
  double ox = 0, oy = 0, oz = 0, tx = 0, ty = 0, tz = 0;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const double px = S.part[w], py = S.part[W + w], pz = S.part[2 * W + w];
    if (w < warp) { ox += px; oy += py; oz += pz; }
    tx += px; ty += py; tz += pz;
  }
  double sxx = ox + (ix - lx), syy = oy + (iy - ly), szz = oz + (iz - lz);  // exclusive prefix of the chunk
  for (int c = c0; c < c1; ++c) {
    const double dx = X.nnx[c] - X.nhx[c], dy = X.nny[c] - X.nhy[c], dz = X.nnz[c] - X.nhz[c];
    X.xnx[c] = S.sx[c] + P.b * (sxx + 0.5 * dx);
    X.xny[c] = S.sy[c] + P.b * (syy + 0.5 * dy);
    X.xnz[c] = S.sz[c] + P.b * (szz + 0.5 * dz);
    sxx += dx; syy += dy; szz += dz;
  }
  Dx = P.b * tx; Dy = P.b * ty; Dz = P.b * tz;
  team_sync<T>();  // X.nn, X.xn, S.E visible
}

// The changed-term sums over bonds and pairs for a built segment, added to this thread's acc and reduced
// over the CTA: the kNumRed sums end up in every thread.  One CTA barrier.
template <int T, bool CUT, int UNROLL = 1>
__device__ __forceinline__ void segment_sums(const CtaView& S, const ClView& X, const ChainParams& P, int n,
                                             int energy_type, int lo, int hi, double Dx, double Dy, double Dz,
                                             double* acc, double* sums) {
  constexpr int W = T / 32;
  using TEAM = typename std::conditional<T == 32, WarpTeam, Team<W>>::type;
  const int tid = team_tid<T>(), lane = tid & 31, warp = tid >> 5;
  // ---- bonds lo−1..hi: ψ and bending energy (eap_chain.jl:45-47,54-58,246-251) ---------------------------
  {
    const int b0 = max(lo - 1, 0), b1 = min(hi, n - 2);
    for (int i = b0 + tid; i <= b1; i += T) {
      const bool an = i >= lo, bn = i + 1 <= hi;
      const double ax = X.nhx[i], ay = X.nhy[i], az = X.nhz[i];
      const double bx = X.nhx[i + 1], by = X.nhy[i + 1], bz = X.nhz[i + 1];
      const double psi_old = X.psi[i];
      const double psi_new = psi_of(an ? X.nnx[i] : ax, an ? X.nny[i] : ay, an ? X.nnz[i] : az,
                                    bn ? X.nnx[i + 1] : bx, bn ? X.nny[i + 1] : by, bn ? X.nnz[i + 1] : bz);
      X.psn[i] = psi_new;
      acc[R_PSI] += psi_new - psi_old;
      acc[R_BEND] += ubend_of(P, psi_new) - ubend_of(P, psi_old);
    }
  }
  // ---- pair terms: segment × everything (each pair once) and heads [0,lo) × tails (hi,n) ---------------
  if (energy_type == 1 || energy_type == 3) {
    double a = 0.0;
    const int H = lo, Tl = n - 1 - hi;
    // short chains (≤ 2 warps): eB = μ_B·D on the fly — a barrier costs more than 3 DFMA per broadcast item;
    // longer chains: the pre-pass into S.E and its barrier are amortised, and the rectangle loop is unrolled
    constexpr bool EFLY = (T <= 64);
    constexpr int UR = (T <= 64) ? 1 : 2;   // rectangle unroll
    const bool rect = H > 0 && Tl > 0;
    // lane side = the one that wastes fewer lanes; r = x_L − x_B, so r' = r − D (L = head) or r + D (L = tail)
    const long long costH = (long long)((H + 31) >> 5) * Tl;
    const long long costT = (long long)((Tl + 31) >> 5) * H;
    const bool lanes_are_heads = costH <= costT;
    const double sgn = lanes_are_heads ? 1.0 : -1.0;
    const int baseA = lanes_are_heads ? 0 : hi + 1, A = lanes_are_heads ? H : Tl;
    const int baseB = lanes_are_heads ? hi + 1 : 0, B = lanes_are_heads ? Tl : H;
    if (!EFLY && rect)
      for (int k = tid; k < B; k += T)
        S.E[baseB + k] = sgn * fma(S.mz[baseB + k], Dz, fma(S.my[baseB + k], Dy, S.mx[baseB + k] * Dx));
    for (int c = lo; c <= hi; ++c) {
      const double xi = S.sx[c], yi = S.sy[c], zi = S.sz[c];
      const double oxm = S.mx[c], oym = S.my[c], ozm = S.mz[c];
      const double xni = X.xnx[c], yni = X.xny[c], zni = X.xnz[c];
      double nmx, nmy, nmz;
      mu_of(P, X.nnx[c], X.nny[c], X.nnz[c], nmx, nmy, nmz);
      for (int j = tid; j < n; j += T) {
        if (j >= lo && j <= c) continue;
        const double jx = S.sx[j], jy = S.sy[j], jz = S.sz[j];
        const double ux = S.mx[j], uy = S.my[j], uz = S.mz[j];
        double njx = jx, njy = jy, njz = jz, vx = ux, vy = uy, vz = uz;
        if (j > hi) { njx += Dx; njy += Dy; njz += Dz; }
        else if (j >= lo) {
          njx = X.xnx[j]; njy = X.xny[j]; njz = X.xnz[j];
          mu_of(P, X.nnx[j], X.nny[j], X.nnz[j], vx, vy, vz);
        }
        if (CUT)
          a += pair_g_cut(nmx, nmy, nmz, vx, vy, vz, xni - njx, yni - njy, zni - njz, P.crad2) -
               pair_g_cut(oxm, oym, ozm, ux, uy, uz, xi - jx, yi - jy, zi - jz, P.crad2);
        else
          a += pair_g(nmx, nmy, nmz, vx, vy, vz, xni - njx, yni - njy, zni - njz) -
               pair_g(oxm, oym, ozm, ux, uy, uz, xi - jx, yi - jy, zi - jz);
      }
    }
    if (!EFLY) team_sync<T>();  // S.E visible (uniform: every thread of the CTA takes this branch)
    if (rect) a += rect_sum<TEAM, UR, CUT, EFLY>(S, baseA, A, baseB, B, sgn * Dx, sgn * Dy, sgn * Dz, P.crad2);
    acc[R_PAIR] += a;
  }
  // ---- reduce ------------------------------------------------------------------------------------------
  // butterfly over the nine sums with the five steps ROLLED: a fifth of the code of nine unrolled warp_sums — these
  // kernels are short of instruction cache, not of issue slots (profiles/r02c_hot_lines_k_run_cta_cluster_K1.txt)
#pragma unroll 1
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int k = 0; k < kNumRed; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < kNumRed; ++k) X.red[k * W + warp] = acc[k];
  }
  team_sync<T>();
#pragma unroll
  for (int k = 0; k < kNumRed; ++k) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < W; ++w) s += X.red[k * W + w];
    sums[k] = s;
  }
  sums[R_PAIR] *= kInv4Pi;
}

// α of cluster_flip! (eap_chain.jl:317-330) from the link probabilities before and after the flip.
__device__ __forceinline__ double cluster_log_alpha(const ClView& X, int n, int lo, int hi, double up, double lp) {
  const double nup = (hi < n - 1) ? link_prob(X.nnx[hi], X.nny[hi], X.nnz[hi], X.nhx[hi + 1], X.nhy[hi + 1], X.nhz[hi + 1]) : 0.0;
  const double nlp = (lo > 0) ? link_prob(X.nnx[lo], X.nny[lo], X.nnz[lo], X.nhx[lo - 1], X.nhy[lo - 1], X.nhz[lo - 1]) : 0.0;
  return Lib<kSharedLib>::log_(((1.0 - nup) * (1.0 - nlp)) / ((1.0 - up) * (1.0 - lp)));
}

// record! of the two extra averagers (mcmc_clustering_eap_chain.jl:243-244), same weight as the others.
template <bool COMP>
__device__ __forceinline__ void record_extras(const ChainParams& P, ChainDynX& DX, double su, double log_gauge,
                                              int n) {
  double wgt = 1.0;
  if (P.umbrella) wgt = 1.0 / Lib<kSharedLib>::exp_(su * P.inv_kT * P.cF - log_gauge);
  if (COMP) {
    comp_add(DX.acc[0], DX.comp[0], DX.scos2 * wgt);
    comp_add(DX.acc[1], DX.comp[1], DX.spsi / (double)(n - 1) * wgt);
  } else {  // plain Float64 sums, the reference's default --numeric-type (average.jl:40-48)
    DX.acc[0] += DX.scos2 * wgt;
    DX.acc[1] += DX.spsi / (double)(n - 1) * wgt;
  }
}

// Step adaptation, the 8 + 2 averagers: everything after the decision (mcmc_clustering_eap_chain.jl:287-311).
__device__ __forceinline__ void bookkeep_cluster(const ChainParams& P, ChainDyn& D, ChainDynX& DX, bool adapt_now, int n,
                                                 bool compensated) {
  if (adapt_now) adapt_apply(P, D.phi_step, D.theta_step, D.nacc, D.natt);
  if (compensated) {
    record_averages<true>(P, D.acc, D.comp, D.r, D.p, D.U, D.su, D.log_gauge);
    record_extras<true>(P, DX, D.su, D.log_gauge, n);
  } else {
    record_averages<false>(P, D.acc, D.comp, D.r, D.p, D.U, D.su, D.log_gauge);
    record_extras<false>(P, DX, D.su, D.log_gauge, n);
  }
}

// Decision quantities of one composite trial from the reduced sums (identical in every thread).
struct SegDecision {
  double dU, dsu, dlogpi, la;
};

__device__ __forceinline__ SegDecision segment_decision(const ChainParams& P, int energy_type, const double* sums,
                                                        double Dx, double Dz, double la, double carry) {
  SegDecision d;
  const bool bare = (energy_type == 3) && !P.cutoff_full;  // the UCutoff functor is the bare pair sum
  const double drF = -(Dx * P.Fx + Dz * P.Fz);             // −Δr·F, energy.jl:8
  d.dsu = sums[R_USELF] + sums[R_BEND];                    // Δ sum(chain.us)
  d.dU = bare ? sums[R_PAIR] : d.dsu + drF + sums[R_PAIR];
  const double dw = P.umbrella ? d.dsu * P.inv_kT * P.cF : 0.0;  // average.jl:120-124
  d.la = la;
  d.dlogpi = -d.dU * P.inv_kT + sums[R_OMEGA] + dw + la - carry;  // acceptance.jl:30-31
  return d;
}

__device__ __forceinline__ void stage_row_cluster(const ChainDyn& D, const ChainDynX& DX, long long step,
                                                  double* rowbuf /* 8 + 19 */) {
  stage_row(D, step, rowbuf);
  const double nrm = D.acc[16] + D.comp[16];
  rowbuf[25] = (DX.acc[0] + DX.comp[0]) / nrm;
  rowbuf[26] = (DX.acc[1] + DX.comp[1]) / nrm;
}

constexpr int kRowDoublesCluster = 28;

// The team, thread tid: output row `row` after trial `step`, with the two extra averagers and, if a.state, the angles of
// every monomer.  Starts with a team barrier (the records of the trial are visible).
template <int T>
__device__ __forceinline__ void emit_row_cluster(const RunArgs& a, const ChainDyn& D, const ChainDynX& DX,
                                                 const MonoRec* mono, int c, long long row, long long step,
                                                 double* rowbuf, int tid) {
  team_sync<T>();
  if (row < a.rows) {
    if (tid == 0) stage_row_cluster(D, DX, step, rowbuf);
    if (a.state) {
      double* st = a.state + ((size_t)c * a.rows + row) * 2 * (size_t)a.n;
      for (int m = tid; m < a.n; m += T) {
        const MonoRec r = mono[m];
        st[2 * m] = r.phi; st[2 * m + 1] = r.theta;
      }
    }
    team_sync<T>();
    if (tid < 8) a.traj[((size_t)c * a.rows + row) * 8 + tid] = rowbuf[tid];
    if (tid < a.roll_cols) a.roll[((size_t)c * a.rows + row) * a.roll_cols + tid] = rowbuf[8 + tid];
  }
}

// The trial chain becomes the chain (mcmc_clustering_eap_chain.jl:274-275), threads tid, tid + T, …: monomers lo … hi
// take the records, n̂, x and μ of the trial from the arrays of the team that evaluated it (St.E = sinθ', Xt), the tail
// j > hi moves by D, and the bond angles lo−1 … hi follow.
template <int T>
__device__ __forceinline__ void commit_segment(const CtaView& S, const ClView& X, const CtaView& St, const ClView& Xt,
                                               MonoRec* mono, const ChainParams& P, const ClProposal& q, int n, int lo,
                                               int hi, bool reflect, double Dx, double Dy, double Dz, int tid) {
  for (int m = lo + tid; m <= hi; m += T) {
    double phi, theta, sb;
    segment_angles(mono, q, m, reflect, P.planar, phi, theta, sb);
    MonoRec rec;
    rec.phi = phi; rec.theta = theta;
    rec.nx = Xt.nnx[m]; rec.ny = Xt.nny[m]; rec.nz = Xt.nnz[m];
    rec.sth = (St.E[m] == kKeepSinTheta) ? sb : St.E[m];
    mono[m] = rec;
    X.nhx[m] = rec.nx; X.nhy[m] = rec.ny; X.nhz[m] = rec.nz;
    S.sx[m] = Xt.xnx[m]; S.sy[m] = Xt.xny[m]; S.sz[m] = Xt.xnz[m];
    double ux, uy, uz;
    mu_of(P, rec.nx, rec.ny, rec.nz, ux, uy, uz);
    S.mx[m] = ux; S.my[m] = uy; S.mz[m] = uz;
  }
  shift_tail(S, hi + 1, n, Dx, Dy, Dz, tid, T);
  for (int i = max(lo - 1, 0) + tid; i <= min(hi, n - 2); i += T) X.psi[i] = Xt.psn[i];
}

// Thread 0 (lane kernel: every thread): the increments of an accepted composite trial and its α carry, the trial
// counters and the cluster statistics.
__device__ __forceinline__ void commit_trial(const ChainParams& P, ChainDyn& D, ChainDynX& DX, bool accept,
                                             long long step, double dU, double dOmega, double dsu, double Dx,
                                             double Dy, double Dz, double dpx, double dpy, double dpz, double dpsi,
                                             double dcos2, double la, bool reflect, int lo, int hi) {
  if (accept) {
    D.U += dU;
    D.Omega += dOmega;
    D.su += dsu;
    D.r[0] += Dx; D.r[1] += Dy; D.r[2] += Dz;
    D.p[0] += dpx; D.p[1] += dpy; D.p[2] += dpz;
    DX.spsi += dpsi;
    DX.scos2 += dcos2;
    DX.carry = P.alpha_carry ? la : 0.0;  // logπ_prev = logπ + log α (acceptance.jl:32-33)
    D.nacc += 1;
    D.nacc_total += 1;
  }
  D.natt += 1;
  D.steps_total += 1;
  D.step = step;
  if (reflect) {
    const double sz = (double)(hi - lo + 1);
    DX.ncluster += 1.0; DX.cluster_sum += sz; DX.cluster_max = fmax(DX.cluster_max, sz);
  }
}

// The hot loop of mcmc_clustering_eap_chain.jl:267-336 for one chain per CTA (T = 32: a one-warp CTA, the team
// barriers are __syncwarp).
//
// Proposal window, as in k_run_cta_win: the serial head of a trial (3 Philox blocks, 2 sincos, log, the record
// read from HBM/L2) is taken off the per-trial critical path by building the single-monomer moves and the gate
// decisions of the next kWin trials at once, one trial per lane of warp 0.  A window entry depends on the
// chain only through the record of its own monomer: an accepted trial marks the later entries whose monomer
// lies in its segment [lo, hi] dirty and those are rebuilt when their turn comes.  Windows never cross a
// step-size adaptation boundary.  The cluster growth reads the neighbours' current directions and stays per trial.
template <int T, int MINB, bool CUT>
__global__ void __launch_bounds__(T, MINB) k_run_cta_cluster(const RunArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  static_assert(kRowDoublesCluster <= kRowDoublesCompact, "row buffer");
  const CtaView S = carve_compact(smem_raw, a.n, T);
  const ClView X = carve_cluster(smem_raw + cta_smem_bytes_compact(a.n, T), a.n, T);
  double* rowbuf = S.rowbuf;
  const int c = blockIdx.x;
  const int tid = team_tid<T>();
  const int n = a.n;
  MonoRec* mono = a.mono + (size_t)c * n;
  if (tid == 0) {
    *S.par = a.par[c];
    *S.dyn = a.dyn[c];
    *X.dx = a.dynx[c];
  }
  team_sync<T>();
  const ChainParams& P = *S.par;
  load_chain<T>(mono, P, n, S);
  load_nhat<T>(mono, n, X);
  const uint32_t chain_id = a.chain_id_base + (uint32_t)c;
  const long long step0 = S.dyn->step;
  const uint32_t init = (uint32_t)S.dyn->init;
  const bool adapt_on = P.adj_scale != 1.0 && P.steps_per_adjust > 0;
  long long row = 0;
  Countdown row_due;
  row_due.start(step0, a.stepout);

  long long s = 1;
  while (s <= a.nsteps) {
    // ---- window [s, s+wlen) ------------------------------------------------------------------------------
    long long to_boundary;
    const int wlen = window_len(a, P, adapt_on, step0, s, to_boundary);
    if (tid < 32)
      build_window(step0 + s, wlen, X.ctl->dirty, tid,
                   [&](int e, long long st) { make_window_entry(a, P, *S.dyn, mono, chain_id, st, X.win[e]); });
    team_sync<T>();  // window visible
    for (int k = 0; k < wlen; ++k) {
      const long long step = step0 + s + k;
      const ClProposal* q = &X.win[k];
      double acc[kNumRed];
#pragma unroll
      for (int r = 0; r < kNumRed; ++r) acc[r] = 0.0;
      if (tid < 32) {
        if ((X.ctl->dirty >> k) & 1u) {  // an earlier trial of this window changed this monomer: rebuild
          __syncwarp();
          if (tid == 0) make_window_entry(a, P, *S.dyn, mono, chain_id, step, X.win[k]);
          __syncwarp();
        }
        warp_cluster_grow(X, *q, q->reflect, P, n, a.seed, chain_id, init, step, *X.ctl);
        __syncwarp();
        if (X.ctl->hi - X.ctl->lo < 32)
          warp_segment_build(S, X, mono, P, *q, X.ctl->lo, X.ctl->hi, X.ctl->reflect != 0, acc, *X.ctl);
      }
      team_sync<T>();  // proposal, cluster and (short) segment are visible
      const int lo = X.ctl->lo, hi = X.ctl->hi;
      const bool reflect = X.ctl->reflect != 0;
      const double carry = X.dx->carry;
      double sums[kNumRed], Dx = X.ctl->Dx, Dy = X.ctl->Dy, Dz = X.ctl->Dz;
      if (hi - lo >= 32) cta_segment_build<T>(S, X, mono, P, *q, lo, hi, reflect, acc, Dx, Dy, Dz);
      segment_sums<T, CUT>(S, X, P, n, a.energy_type, lo, hi, Dx, Dy, Dz, acc, sums);
      const double la = reflect ? cluster_log_alpha(X, n, lo, hi, X.ctl->up, X.ctl->lp) : 0.0;
      const SegDecision dec = segment_decision(P, a.energy_type, sums, Dx, Dz, la, carry);
      const bool accept = metropolis(dec.dlogpi, q->eps);
      if (accept) {
        commit_segment<T>(S, X, S, X, mono, P, *q, n, lo, hi, reflect, Dx, Dy, Dz, tid);
        if (tid < 32) mark_stale(X.win, k, wlen, lo, hi, X.ctl->dirty, tid);
      }
      if (tid == 0) {
        commit_trial(P, *S.dyn, *X.dx, accept, step, dec.dU, sums[R_OMEGA], dec.dsu, Dx, Dy, Dz, sums[R_PX], sums[R_PY],
                     sums[R_PZ], sums[R_PSI], sums[R_COS2], dec.la, reflect, lo, hi);
        bookkeep_cluster(P, *S.dyn, *X.dx, /*adapt_now=*/k + 1 == to_boundary, n, a.compensated != 0);
      }
      if (row_due.tick()) emit_row_cluster<T>(a, *S.dyn, *X.dx, mono, c, row++, step, rowbuf, tid);
      team_sync<T>();  // state, records and the dirty mask of this trial are visible
    }
    s += wlen;
  }
  if (tid == 0) {
    a.dyn[c] = *S.dyn;
    a.dynx[c] = *X.dx;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Small ensembles: G one-warp teams per chain, each evaluating a DIFFERENT trial of the window at the same time.
//
// The reference's studies are a few hundred chains of n ≈ 100: one warp per chain leaves a B200 idle, and more warps
// on the same trial (k_run_cta_cluster<64|128>) stop paying at the serial head of a trial.  But at the parameters of
// those studies a trial is rejected far more often than not (acceptance 1–40 %), and a rejected trial leaves the chain
// as it was — so trial k+1 can be evaluated on the current chain while trial k is still open, and its evaluation stands
// unless k is accepted.  Here the G warps of a CTA evaluate trials k … k+G−1 of the proposal window against the shared,
// read-only chain, each into its own scratch arrays; then the trials are committed in order by the whole CTA: a
// rejected trial only does its bookkeeping, the first accepted one is applied and ends the batch (the speculations
// behind it saw a stale chain and are evaluated again).  Every decision is taken on exactly the state the sequential
// chain would show it: same trajectories as the one-team kernels (tests/test_gpu_cluster.py run through this kernel
// whenever the ensemble is small).
struct SpecResult {
  double sums[kNumRed];
  SegDecision dec;
  double Dx, Dy, Dz;
  int lo, hi, reflect, accept;
};

__host__ __device__ inline size_t cluster_spec_group_bytes(int n) {   // private arrays of one extra team
  size_t b = (size_t)8 * n * sizeof(double) + sizeof(ClusterCtl);
  return (b + 15) & ~(size_t)15;
}
__host__ __device__ inline size_t cluster_spec_smem_bytes(int n, int groups) {
  return cta_smem_bytes_compact(n, 32 * groups) + cluster_extra_bytes(n, 32 * groups) +
         (size_t)(groups - 1) * cluster_spec_group_bytes(n) + (((size_t)groups * sizeof(SpecResult) + 15) & ~(size_t)15);
}

template <int G, int MINB, bool CUT>
__global__ void __launch_bounds__(32 * G, MINB) k_run_cta_cluster_spec(const RunArgs a) {
  constexpr int T = 32 * G;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const CtaView S = carve_compact(smem_raw, a.n, T);
  const ClView X = carve_cluster(smem_raw + cta_smem_bytes_compact(a.n, T), a.n, T);
  unsigned char* extra = smem_raw + cta_smem_bytes_compact(a.n, T) + cluster_extra_bytes(a.n, T);
  SpecResult* res = reinterpret_cast<SpecResult*>(extra + (size_t)(G - 1) * cluster_spec_group_bytes(a.n));
  double* rowbuf = S.rowbuf;
  const int c = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, g = tid >> 5;
  const int n = a.n;
  MonoRec* mono = a.mono + (size_t)c * n;
  // team t's views: the chain (x, μ, n̂, ψ) is shared and read-only while trials are evaluated; sinθ'/E, n̂', x', ψ',
  // the reduction slots and the cluster control block are the team's own
  auto team_arrays = [&](int t, CtaView& St, ClView& Xt) {
    St = S;
    Xt = X;
    St.part = S.part + 3 * t;
    Xt.red = X.red + kNumRed * t;
    if (t > 0) {
      double* d = reinterpret_cast<double*>(extra + (size_t)(t - 1) * cluster_spec_group_bytes(n));
      St.E = d;
      Xt.nnx = d + n; Xt.nny = d + 2 * n; Xt.nnz = d + 3 * n;
      Xt.xnx = d + 4 * n; Xt.xny = d + 5 * n; Xt.xnz = d + 6 * n;
      Xt.psn = d + 7 * n;
      Xt.ctl = reinterpret_cast<ClusterCtl*>(d + 8 * n);
    }
  };
  CtaView Sg;
  ClView Xg;
  team_arrays(g, Sg, Xg);
  if (tid == 0) {
    *S.par = a.par[c];
    *S.dyn = a.dyn[c];
    *X.dx = a.dynx[c];
  }
  __syncthreads();
  const ChainParams& P = *S.par;
  load_chain<T>(mono, P, n, S);
  load_nhat<T>(mono, n, X);
  const uint32_t chain_id = a.chain_id_base + (uint32_t)c;
  const long long step0 = S.dyn->step;
  const uint32_t init = (uint32_t)S.dyn->init;
  const bool adapt_on = P.adj_scale != 1.0 && P.steps_per_adjust > 0;
  long long row = 0;
  Countdown row_due;
  row_due.start(step0, a.stepout);

  long long s = 1;
  while (s <= a.nsteps) {
    // ---- window [s, s+wlen) --------------------------------------------------------------------------------
    long long to_boundary;
    const int wlen = window_len(a, P, adapt_on, step0, s, to_boundary);
    if (tid < 32)
      build_window(step0 + s, wlen, X.ctl->dirty, tid,
                   [&](int e, long long st) { make_window_entry(a, P, *S.dyn, mono, chain_id, st, X.win[e]); });
    __syncthreads();  // window visible
    int k = 0;
    while (k < wlen) {
      const int nb = min(G, wlen - k);
      // ---- phase 1: team g evaluates trial k+g on the current chain ------------------------------------------
      if (g < nb) {
        const int kk = k + g;
        const long long step = step0 + s + kk;
        if ((X.ctl->dirty >> kk) & 1u) {  // an accepted trial of this window moved this monomer: rebuild the entry
          if (lane == 0) make_window_entry(a, P, *S.dyn, mono, chain_id, step, X.win[kk]);
          __syncwarp();
        }
        const ClProposal* q = &X.win[kk];
        double acc[kNumRed], sums[kNumRed];
#pragma unroll
        for (int r = 0; r < kNumRed; ++r) acc[r] = 0.0;
        warp_cluster_grow(Xg, *q, q->reflect, P, n, a.seed, chain_id, init, step, *Xg.ctl);
        __syncwarp();
        if (Xg.ctl->hi - Xg.ctl->lo < 32)
          warp_segment_build(Sg, Xg, mono, P, *q, Xg.ctl->lo, Xg.ctl->hi, Xg.ctl->reflect != 0, acc, *Xg.ctl);
        __syncwarp();
        const int lo = Xg.ctl->lo, hi = Xg.ctl->hi;
        const bool reflect = Xg.ctl->reflect != 0;
        double Dx = Xg.ctl->Dx, Dy = Xg.ctl->Dy, Dz = Xg.ctl->Dz;
        if (hi - lo >= 32) cta_segment_build<32>(Sg, Xg, mono, P, *q, lo, hi, reflect, acc, Dx, Dy, Dz);
        segment_sums<32, CUT>(Sg, Xg, P, n, a.energy_type, lo, hi, Dx, Dy, Dz, acc, sums);
        const double la = reflect ? cluster_log_alpha(Xg, n, lo, hi, Xg.ctl->up, Xg.ctl->lp) : 0.0;
        // the α carry changes only when a trial is accepted: valid for every trial that is committed from this batch
        const SegDecision dec = segment_decision(P, a.energy_type, sums, Dx, Dz, la, X.dx->carry);
        const bool accept = metropolis(dec.dlogpi, q->eps);
        if (lane == 0) {
          SpecResult& R = res[g];
#pragma unroll
          for (int r = 0; r < kNumRed; ++r) R.sums[r] = sums[r];
          R.dec = dec;
          R.Dx = Dx; R.Dy = Dy; R.Dz = Dz;
          R.lo = lo; R.hi = hi; R.reflect = reflect ? 1 : 0; R.accept = accept ? 1 : 0;
        }
      }
      __syncthreads();  // all evaluations of the batch are in
      // ---- phase 2: commit in order, by the whole CTA; the first accepted trial ends the batch ------------------
      int committed = 0;
      for (int b = 0; b < nb; ++b) {
        const SpecResult& R = res[b];
        const int kk = k + b;
        const long long step = step0 + s + kk;
        const ClProposal* q = &X.win[kk];
        const bool accept = R.accept != 0, reflect = R.reflect != 0;
        const int lo = R.lo, hi = R.hi;
        if (accept) {  // the trial chain of team b becomes the chain
          CtaView Sb;
          ClView Xb;
          team_arrays(b, Sb, Xb);
          commit_segment<T>(S, X, Sb, Xb, mono, P, *q, n, lo, hi, reflect, R.Dx, R.Dy, R.Dz, tid);
          if (tid < 32) mark_stale(X.win, kk, wlen, lo, hi, X.ctl->dirty, tid);
        }
        if (tid == 0) {
          commit_trial(P, *S.dyn, *X.dx, accept, step, R.dec.dU, R.sums[R_OMEGA], R.dec.dsu, R.Dx, R.Dy, R.Dz,
                       R.sums[R_PX], R.sums[R_PY], R.sums[R_PZ], R.sums[R_PSI], R.sums[R_COS2], R.dec.la, reflect, lo, hi);
          bookkeep_cluster(P, *S.dyn, *X.dx, /*adapt_now=*/kk + 1 == to_boundary, n, a.compensated != 0);
        }
        if (row_due.tick()) emit_row_cluster<T>(a, *S.dyn, *X.dx, mono, c, row++, step, rowbuf, tid);
        ++committed;
        if (accept) break;  // the speculations behind this trial saw the chain before it
      }
      k += committed;
      __syncthreads();  // state, records, running scalars and the dirty mask are visible
    }
    s += wlen;
  }
  if (tid == 0) {
    a.dyn[c] = *S.dyn;
    a.dynx[c] = *X.dx;
  }
}

// Non-mutating changed-term sums of one scripted composite trial (same device code as the run kernel).
struct SegDeltaArgs {
  const MonoRec* mono;
  const ChainParams* par;
  double* out;  // {dU, dOmega, dU_pairs, du_self, drF, dU_bend, dΣψ, dΣcos²θ, dp1, dp2, dp3, log α}
  int n, energy_type, chain, idx, lo, hi, reflect;
  double dphi, dtheta;
};

template <int T, bool CUT>
__global__ void __launch_bounds__(T) k_delta_segment_cta(const SegDeltaArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const CtaView S = carve(smem_raw, a.n);
  const ClView X = carve_cluster(smem_raw + cta_smem_bytes(a.n), a.n, T);
  const int tid = threadIdx.x, n = a.n;
  const MonoRec* mono = a.mono + (size_t)a.chain * n;
  if (tid == 0) *S.par = a.par[a.chain];
  __syncthreads();
  const ChainParams& P = *S.par;
  load_chain<T>(mono, P, n, S);
  load_nhat<T>(mono, n, X);
  if (tid == 0) {
    if (P.planar) build_proposal_planar(P, mono[a.idx], a.idx, a.dphi, 0.0, S.prop[0]);
    else build_proposal(P, mono[a.idx], a.idx, a.dphi, a.dtheta, 0.0, S.prop[0]);
  }
  __syncthreads();
  const Proposal& q = S.prop[0];
  const bool reflect = a.reflect != 0;
  const int lo = reflect ? a.lo : a.idx, hi = reflect ? a.hi : a.idx;
  __shared__ ClusterCtl dctl;
  double acc[kNumRed], sums[kNumRed], Dx, Dy, Dz;
#pragma unroll
  for (int k = 0; k < kNumRed; ++k) acc[k] = 0.0;
  if (hi - lo < 32) {  // the two build paths of the run kernel
    if (tid < 32) warp_segment_build(S, X, mono, P, q, lo, hi, reflect, acc, dctl);
    __syncthreads();
    Dx = dctl.Dx; Dy = dctl.Dy; Dz = dctl.Dz;
  } else {
    cta_segment_build<T>(S, X, mono, P, q, lo, hi, reflect, acc, Dx, Dy, Dz);
  }
  segment_sums<T, CUT>(S, X, P, n, a.energy_type, lo, hi, Dx, Dy, Dz, acc, sums);
  if (tid == 0) {
    double up = 0.0, lp = 0.0;  // link probabilities before the flip, on the chain carrying the move
    if (reflect) {
      double ax, ay, az, bx, by, bz;
      if (hi < n - 1) { nhat_trial(X, q, hi, ax, ay, az); nhat_trial(X, q, hi + 1, bx, by, bz); up = link_prob(ax, ay, az, bx, by, bz); }
      if (lo > 0) { nhat_trial(X, q, lo, ax, ay, az); nhat_trial(X, q, lo - 1, bx, by, bz); lp = link_prob(ax, ay, az, bx, by, bz); }
    }
    const double la = reflect ? cluster_log_alpha(X, n, lo, hi, up, lp) : 0.0;
    const SegDecision d = segment_decision(P, a.energy_type, sums, Dx, Dz, la, 0.0);
    a.out[0] = d.dU; a.out[1] = sums[R_OMEGA]; a.out[2] = sums[R_PAIR]; a.out[3] = sums[R_USELF];
    a.out[4] = -(Dx * P.Fx + Dz * P.Fz); a.out[5] = sums[R_BEND]; a.out[6] = sums[R_PSI]; a.out[7] = sums[R_COS2];
    a.out[8] = sums[R_PX]; a.out[9] = sums[R_PY]; a.out[10] = sums[R_PZ]; a.out[11] = la;
  }
}

// ---------------------------------------------------------------------------------------------
// One chain per lane: non-interacting and Ising energies (+ bending), O(|cluster|) per trial.
// ---------------------------------------------------------------------------------------------
struct LaneSeg {
  double dOmega, du_self, dbend, dpsi, dcos2, dpair;  // dpair: 4π × Σ(new − old) of U_Ising terms
  double dpx, dpy, dpz, sx, sy, sz;                   // Δp, ΣΔn̂
};

// Contribution of one flipped cluster monomer (not idx) with current direction (nx,ny,nz) to the sums.
__device__ __forceinline__ void lane_add_flipped(const ChainParams& P, const MonoRec& r, LaneSeg& o) {
  const double nx = r.nx, ny = r.ny, nz = r.nz;
  double fx, fy, fz;
  flip_dir(P.planar, nx, ny, nz, fx, fy, fz);
  // a monomer sitting at θ = π (the only θ in [0, π] with reflect_theta(θ) == 0) reflects to sinθ' = 0 ⇒ Ω' = −Inf ⇒
  // the trial is rejected (eap_chain.jl:236-238)
  if (!P.planar && r.theta == kPi) o.dOmega = -INFINITY;
  double ux, uy, uz, vx, vy, vz;
  mu_of(P, nx, ny, nz, ux, uy, uz);
  mu_of(P, fx, fy, fz, vx, vy, vz);
  o.du_self += -0.5 * P.E0 * vz - (-0.5 * P.E0 * uz);
  o.dpx += vx - ux; o.dpy += vy - uy; o.dpz += vz - uz;
  o.sx += fx - nx; o.sy += fy - ny; o.sz += fz - nz;
}

// ψ, bending and (Ising) pair-term change of ONE bond between monomers a and b (b = a+1).
template <bool ISING, bool SH = kSharedLib>
__device__ __forceinline__ void lane_bond_delta(const ChainParams& P, double aox, double aoy, double aoz, double anx,
                                                double any_, double anz, double box, double boy, double boz,
                                                double bnx, double bny, double bnz, LaneSeg& o) {
  const double psi_old = psi_of<SH>(aox, aoy, aoz, box, boy, boz);
  const double psi_new = psi_of<SH>(anx, any_, anz, bnx, bny, bnz);
  o.dpsi += psi_new - psi_old;
  o.dbend += ubend_of(P, psi_new) - ubend_of(P, psi_old);
  if (ISING) {  // U_Ising (eap_chain.jl:215-228): separation x_a − x_b = −(b/2)(n̂_a + n̂_b)
    const double hb = -0.5 * P.b;
    double uox, uoy, uoz, unx, uny, unz, vox, voy, voz, vnx, vny, vnz;
    mu_of(P, aox, aoy, aoz, uox, uoy, uoz);
    mu_of(P, anx, any_, anz, unx, uny, unz);
    mu_of(P, box, boy, boz, vox, voy, voz);
    mu_of(P, bnx, bny, bnz, vnx, vny, vnz);
    o.dpair += pair_g(unx, uny, unz, vnx, vny, vnz, hb * (anx + bnx), hb * (any_ + bny), hb * (anz + bnz)) -
               pair_g(uox, uoy, uoz, vox, voy, voz, hb * (aox + box), hb * (aoy + boy), hb * (aoz + boz));
  }
}

// Final record of the moved monomer idx: move! (the proposal), then refl_n!/flip_n! if its cluster is flipped.
// This one is computed literally from the angles (a θ clamped to π reflects to θ = 0 ⇒ sinθ = 0 ⇒ rejection).
template <bool SH = kSharedLib>
__device__ __forceinline__ void lane_idx_record(const ChainParams& P, const Proposal& q, bool reflect, MonoRec& nrec,
                                                double& dOmega) {
  if (!reflect) {
    nrec = record_of(q);
    dOmega = q.dOmega;
    return;
  }
  double phi = q.phi, theta = q.theta;
  if (P.planar) phi += kPi; else theta = reflect_theta(theta);
  nrec.phi = phi; nrec.theta = theta;
  direction_of<SH>(P.planar, phi, theta, nrec.nx, nrec.ny, nrec.nz, nrec.sth);
  dOmega = P.planar ? 0.0 : q.dOmega + Lib<SH>::log_(nrec.sth / q.sth);
}

// Changed-term sums of the composite trial for O(1)-per-bond energies.  Reflecting a whole cluster is an
// orthogonal map of every direction in it (and μ' = ±Rμ for both chain types), so bond angles and
// nearest-neighbour pair terms INSIDE the cluster are unchanged; what changes is: the bonds next to the moved
// monomer idx, the two bonds at the ends of the cluster, and the single-monomer sums (u, p, r) of the flipped
// monomers — no transcendental per cluster monomer.  `o` enters holding the flipped-monomer sums (c ≠ idx).
template <bool ISING, bool SH = kSharedLib>
__device__ __forceinline__ void lane_segment_finish(const MonoRec* __restrict__ mono, int n, const ChainParams& P,
                                                    const MonoRec& rec, const MonoRec& nrec, int idx, int lo, int hi,
                                                    bool reflect, LaneSeg& o, double& la, double up, double lp) {
  // the moved monomer
  {
    double ux, uy, uz, vx, vy, vz;
    mu_of(P, rec.nx, rec.ny, rec.nz, ux, uy, uz);
    mu_of(P, nrec.nx, nrec.ny, nrec.nz, vx, vy, vz);
    o.du_self += -0.5 * P.E0 * vz - (-0.5 * P.E0 * uz);
    o.dpx += vx - ux; o.dpy += vy - uy; o.dpz += vz - uz;
    o.dcos2 += nrec.nz * nrec.nz - rec.nz * rec.nz;
    o.sx += nrec.nx - rec.nx; o.sy += nrec.ny - rec.ny; o.sz += nrec.nz - rec.nz;
  }
  // bonds (idx−1,idx) and (idx,idx+1)
  if (idx > 0) {
    const MonoRec l = mono[idx - 1];
    double fx = l.nx, fy = l.ny, fz = l.nz;
    if (reflect && idx - 1 >= lo) flip_dir(P.planar, l.nx, l.ny, l.nz, fx, fy, fz);
    lane_bond_delta<ISING, SH>(P, l.nx, l.ny, l.nz, fx, fy, fz, rec.nx, rec.ny, rec.nz, nrec.nx, nrec.ny, nrec.nz, o);
  }
  if (idx + 1 < n) {
    const MonoRec r = mono[idx + 1];
    double fx = r.nx, fy = r.ny, fz = r.nz;
    if (reflect && idx + 1 <= hi) flip_dir(P.planar, r.nx, r.ny, r.nz, fx, fy, fz);
    lane_bond_delta<ISING, SH>(P, rec.nx, rec.ny, rec.nz, nrec.nx, nrec.ny, nrec.nz, r.nx, r.ny, r.nz, fx, fy, fz, o);
  }
  la = 0.0;
  if (!reflect) return;
  // the two ends of the cluster (when they are not the bonds of idx) and α (eap_chain.jl:317-330)
  double nup = 0.0, nlp = 0.0;
  if (hi < n - 1) {
    const MonoRec b = mono[hi + 1];
    double hx, hy, hz;  // new direction of monomer hi
    if (hi == idx) { hx = nrec.nx; hy = nrec.ny; hz = nrec.nz; }
    else {
      const MonoRec t = mono[hi];
      flip_dir(P.planar, t.nx, t.ny, t.nz, hx, hy, hz);
      lane_bond_delta<ISING, SH>(P, t.nx, t.ny, t.nz, hx, hy, hz, b.nx, b.ny, b.nz, b.nx, b.ny, b.nz, o);
    }
    nup = link_prob(hx, hy, hz, b.nx, b.ny, b.nz);
  }
  if (lo > 0) {
    const MonoRec b = mono[lo - 1];
    double hx, hy, hz;  // new direction of monomer lo
    if (lo == idx) { hx = nrec.nx; hy = nrec.ny; hz = nrec.nz; }
    else {
      const MonoRec t = mono[lo];
      flip_dir(P.planar, t.nx, t.ny, t.nz, hx, hy, hz);
      lane_bond_delta<ISING, SH>(P, b.nx, b.ny, b.nz, b.nx, b.ny, b.nz, t.nx, t.ny, t.nz, hx, hy, hz, o);
    }
    nlp = link_prob(hx, hy, hz, b.nx, b.ny, b.nz);
  }
  la = Lib<SH>::log_(((1.0 - nup) * (1.0 - nlp)) / ((1.0 - up) * (1.0 - lp)));
}

// Sequential cluster growth for one lane (eap_chain.jl:276-305) on the chain carrying the move; every monomer
// that joins the cluster adds its flipped-monomer sums on the way.
template <bool SH = kSharedLib>
__device__ __forceinline__ void lane_cluster_grow(const MonoRec* __restrict__ mono, const Proposal& q,
                                                  const ChainParams& P, int n, uint64_t seed, uint32_t chain_id,
                                                  uint32_t init, long long step, int& lo, int& hi, double& up,
                                                  double& lp, LaneSeg& o) {
  const int idx = q.idx;
  hi = idx;
  double ax = q.nx, ay = q.ny, az = q.nz;
  uint4 w = make_uint4(0u, 0u, 0u, 0u);  // uniforms #k and #k+1 (k even) share one Philox block (draw_cluster)
  for (int k = 0;; ++k) {
    if (hi >= n - 1) { up = 0.0; break; }
    const MonoRec b = mono[hi + 1];
    up = link_prob(ax, ay, az, b.nx, b.ny, b.nz);
    if (!(k & 1)) w = cluster_block<SH>(seed, chain_id, init, step, SUB_CLUSTER_UP, k);
    if (((k & 1) ? u53(w.z, w.w) : u53(w.x, w.y)) <= up) {
      hi += 1; ax = b.nx; ay = b.ny; az = b.nz;
      lane_add_flipped(P, b, o);
    } else break;
  }
  lo = idx;
  ax = q.nx; ay = q.ny; az = q.nz;
  for (int k = 0;; ++k) {
    if (lo <= 0) { lp = 0.0; break; }
    const MonoRec b = mono[lo - 1];
    lp = link_prob(ax, ay, az, b.nx, b.ny, b.nz);
    if (!(k & 1)) w = cluster_block<SH>(seed, chain_id, init, step, SUB_CLUSTER_DOWN, k);
    if (((k & 1) ? u53(w.z, w.w) : u53(w.x, w.y)) <= lp) {
      lo -= 1; ax = b.nx; ay = b.ny; az = b.nz;
      lane_add_flipped(P, b, o);
    } else break;
  }
}

__device__ __forceinline__ void lane_seg_zero(LaneSeg& o) {
  o.dOmega = o.du_self = o.dbend = o.dpsi = o.dcos2 = o.dpair = 0.0;
  o.dpx = o.dpy = o.dpz = o.sx = o.sy = o.sz = 0.0;
}

template <int T, int MINB, bool ISING, bool COMP>
__global__ void __launch_bounds__(T, MINB) k_run_lane_cluster(const RunArgs a) {
  const int c = blockIdx.x * T + threadIdx.x;
  if (c >= a.nchains) return;
  const int n = a.n;
  MonoRec* mono = a.mono + (size_t)c * n;
  const ChainParams P = a.par[c];
  ChainDyn D = a.dyn[c];
  ChainDynX DX = a.dynx[c];
  const uint32_t chain_id = a.chain_id_base + (uint32_t)c;
  const long long step0 = D.step;
  long long row = 0;
  for (long long s = 1; s <= a.nsteps; ++s) {
    const long long step = step0 + s;
    const Draws d = draw_step<true>(a.seed, chain_id, (uint32_t)D.init, step, n);
    const MonoRec rec = mono[d.idx];
    double dphi, dtheta;
    increments(P, d, rec.theta, D.phi_step, D.theta_step, dphi, dtheta);
    Proposal q;
    if (P.planar) build_proposal_planar<true>(P, rec, d.idx, dphi, d.eps, q);
    else build_proposal<true>(P, rec, d.idx, dphi, dtheta, d.eps, q);
    int lo = d.idx, hi = d.idx;
    double up = 0.0, lp = 0.0;
    bool reflect = false;
    if (P.clustering) {
      const bool g = draw_cluster_gate<true>(a.seed, chain_id, (uint32_t)D.init, step) <= P.cluster_prob;
      reflect = P.planar ? g : !g;  // the gate has opposite senses in the two trees (see warp_cluster_grow)
    }
    LaneSeg g;
    lane_seg_zero(g);
    if (reflect) lane_cluster_grow<true>(mono, q, P, n, a.seed, chain_id, (uint32_t)D.init, step, lo, hi, up, lp, g);
    MonoRec nrec;
    double dOm_idx;
    lane_idx_record<true>(P, q, reflect, nrec, dOm_idx);
    g.dOmega += dOm_idx;
    double la;
    lane_segment_finish<ISING, true>(mono, n, P, rec, nrec, d.idx, lo, hi, reflect, g, la, up, lp);
    const double Dx = P.b * g.sx, Dy = P.b * g.sy, Dz = P.b * g.sz;
    const double dpairs = kInv4Pi * g.dpair;
    const double dsu = g.du_self + g.dbend;
    const double dU = dsu - (Dx * P.Fx + Dz * P.Fz) + dpairs;
    const double dw = P.umbrella ? dsu * P.inv_kT * P.cF : 0.0;
    const double dlogpi = -dU * P.inv_kT + g.dOmega + dw + la - DX.carry;
    const bool accept = metropolis<true>(dlogpi, q.eps);
    if (accept) {
      if (reflect)
        for (int k = lo; k <= hi; ++k) {
          if (k == d.idx) continue;
          MonoRec r = mono[k];  // refl_n! / flip_n! of the record
          if (P.planar) { r.phi += kPi; r.nx = -r.nx; r.ny = -r.ny; r.nz = -r.nz; }
          else { r.theta = reflect_theta(r.theta); r.nz = -r.nz; }
          mono[k] = r;
        }
      mono[d.idx] = nrec;
    }
    commit_trial(P, D, DX, accept, step, dU, g.dOmega, dsu, Dx, Dy, Dz, g.dpx, g.dpy, g.dpz, g.dpsi, g.dcos2, la, reflect,
                 lo, hi);
    bookkeep<COMP>(P, D, step);
    record_extras<COMP>(P, DX, D.su, D.log_gauge, n);
    if (a.stepout > 0 && (step % a.stepout) == 0) {
      if (row < a.rows) {
        double rb[kRowDoublesCluster];
        stage_row_cluster(D, DX, step, rb);
        double* t = a.traj + ((size_t)c * a.rows + row) * 8;
        double* r = a.roll + ((size_t)c * a.rows + row) * a.roll_cols;
#pragma unroll
        for (int k = 0; k < 8; ++k) t[k] = rb[k];
        for (int k = 0; k < a.roll_cols; ++k) r[k] = rb[8 + k];
        if (a.state) {
          double* st = a.state + ((size_t)c * a.rows + row) * 2 * (size_t)n;
          for (int k = 0; k < n; ++k) { st[2 * k] = mono[k].phi; st[2 * k + 1] = mono[k].theta; }
        }
      }
      ++row;
    }
  }
  a.dyn[c] = D;
  a.dynx[c] = DX;
}

// One chain per WARP for O(1)-per-bond energies: every lane takes one TRIAL of the same chain (32 composite trials
// per window), as k_run_warp does for mcmc_eap_chain.jl.  The reference's studies are a few hundred chains (20 cases
// × 25 runs, run/Ising_2025-12-17.jl); with one chain per lane they are a handful of warps in which every lane walks
// its Markov chain alone at the latency of a dependent chain of record reads.
//
// A composite trial reads the records lo−1..hi+1 of its segment (the grown cluster and the two bonds that ended the
// growth; lo = hi = idx without a cluster) and, if accepted, writes lo..hi.  Its draws are counter-based, so every
// lane can evaluate its trial speculatively on the current chain: segment, changed-term sums, log α, and
// base = logπ' − logπ without the carried log α of the acceptor (acceptance.jl:30-33), which depends on the LAST
// ACCEPTED trial and is applied when the trial's turn comes.  The window is then resolved in order: the warp walks the
// undecided trials; a trial whose speculation is still valid is decided (carry threaded through the walk); an
// accepted trial invalidates every undecided trial whose read interval meets its write interval; the walk stops at
// the first invalid trial, the accepted trials write their (disjoint) segments, the invalid ones are re-evaluated on
// the new chain, and the walk resumes.  Every trial is decided on exactly the state the sequential loop would
// show it: the chain performs the reference's Markov chain (trajectory parity with the oracle).  Running r, p, U, Σu,
// Σψ, Σcos²θ after each trial — the averagers record every trial — are inclusive prefix sums of the accepted
// increments; each lane keeps its own accumulators, combined at output rows and at the end.  Windows never cross an
// adaptation boundary or an output row.
// STAGE: the chain's records are staged in shared memory for the launch (48 n bytes per warp; chains of up to
// kWarpClusterStageMax monomers) — the evaluations are dependent chains of record reads.
constexpr int kWarpClusterStageMax = 1024;

template <bool ISING, int MINB, bool COMP, bool STAGE>
__global__ void __launch_bounds__(128, MINB) k_run_warp_cluster(const RunArgs a) {
  constexpr unsigned FULL = 0xffffffffu;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  const int c = (int)((blockIdx.x * 128u + threadIdx.x) >> 5);
  if (c >= a.nchains) return;
  const int n = a.n;
  MonoRec* const gmono = a.mono + (size_t)c * n;
  MonoRec* mono = gmono;
  if (STAGE) {
    mono = reinterpret_cast<MonoRec*>(smem_raw) + (size_t)(threadIdx.x >> 5) * n;
    for (int k = lane; k < n; k += 32) mono[k] = gmono[k];
    __syncwarp();
  }
  const ChainParams P = a.par[c];
  ChainDyn D = a.dyn[c];      // uniform scalars (every lane holds a copy); accumulators: per lane
  ChainDynX DX = a.dynx[c];
  double acc[kNumAcc], comp[kNumAcc], xacc[2], xcomp[2];
#pragma unroll
  for (int k = 0; k < kNumAcc; ++k) {
    acc[k] = lane == 0 ? D.acc[k] : 0.0;
    comp[k] = lane == 0 ? D.comp[k] : 0.0;
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    xacc[k] = lane == 0 ? DX.acc[k] : 0.0;
    xcomp[k] = lane == 0 ? DX.comp[k] : 0.0;
  }
  const uint32_t chain_id = a.chain_id_base + (uint32_t)c;
  const uint32_t init = (uint32_t)D.init;
  const long long step0 = D.step;
  const bool adapt_on = P.adj_scale != 1.0 && P.steps_per_adjust > 0;
  long long row = 0;
  long long s = 1;
  while (s <= a.nsteps) {
    long long wl = a.nsteps - s + 1;
    if (wl > a.window) wl = a.window;
    if (adapt_on) {
      const long long tb = P.steps_per_adjust - ((step0 + s - 1) % P.steps_per_adjust);
      if (wl > tb) wl = tb;
    }
    if (a.stepout > 0) {
      const long long tr = a.stepout - ((step0 + s - 1) % a.stepout);
      if (wl > tr) wl = tr;
    }
    const int wlen = (int)wl;
    const bool active = lane < wlen;
    const long long step = step0 + s + lane;
    Draws d;
    d.idx = 0; d.flipbit = 0; d.u_phi = d.u_theta = d.eps = 0.0;
    int reflect = 0;
    if (active) {
      d = draw_step<true>(a.seed, chain_id, init, step, n);
      reflect = cluster_gate<true>(P, a.seed, chain_id, init, step);
    }
    // the speculative evaluation of this lane's trial
    int lo = d.idx, hi = d.idx;
    double base = 0.0, la = 0.0;
    double dU = 0, dOm = 0, dsu = 0, Dx = 0, Dy = 0, Dz = 0, dpx = 0, dpy = 0, dpz = 0, dpsi = 0, dcos2 = 0;
    MonoRec nrec;
    nrec.phi = nrec.theta = nrec.nx = nrec.ny = nrec.nz = nrec.sth = 0.0;
    bool pending = active, valid = false, accepted = false, written = false, acc0 = false;
    double carry = DX.carry;
    unsigned pmask;
    while ((pmask = __ballot_sync(FULL, pending)) != 0u) {
      if (pending && !valid) {
        const MonoRec rec = mono[d.idx];
        double dphi, dtheta;
        increments(P, d, rec.theta, D.phi_step, D.theta_step, dphi, dtheta);
        Proposal q;
        if (P.planar) build_proposal_planar<true>(P, rec, d.idx, dphi, d.eps, q);
        else build_proposal<true>(P, rec, d.idx, dphi, dtheta, d.eps, q);
        lo = hi = d.idx;
        double up = 0.0, lp = 0.0;
        LaneSeg g;
        lane_seg_zero(g);
        if (reflect) lane_cluster_grow<true>(mono, q, P, n, a.seed, chain_id, init, step, lo, hi, up, lp, g);
        double dOm_idx;
        lane_idx_record<true>(P, q, reflect != 0, nrec, dOm_idx);
        g.dOmega += dOm_idx;
        lane_segment_finish<ISING, true>(mono, n, P, rec, nrec, d.idx, lo, hi, reflect != 0, g, la, up, lp);
        Dx = P.b * g.sx; Dy = P.b * g.sy; Dz = P.b * g.sz;
        const double dpairs = kInv4Pi * g.dpair;
        dsu = g.du_self + g.dbend;
        dU = dsu - (Dx * P.Fx + Dz * P.Fz) + dpairs;
        const double dw = P.umbrella ? dsu * P.inv_kT * P.cF : 0.0;
        base = -dU * P.inv_kT + g.dOmega + dw + la;  // Δlogπ of the lane kernel before `- carry`
        acc0 = metropolis<true>(base, d.eps);              // the decision when nothing is carried (the usual case)
        dOm = g.dOmega; dpx = g.dpx; dpy = g.dpy; dpz = g.dpz; dpsi = g.dpsi; dcos2 = g.dcos2;
        valid = true;
      }
      // ---- walk the undecided trials in order ---------------------------------------------------------------
      unsigned walk = pmask;
      while (walk) {
        const int j = __ffs(walk) - 1;
        walk &= walk - 1;
        const int fj = __shfl_sync(FULL, (int)valid | ((int)acc0 << 1), j);
        if (!(fj & 1)) break;  // stale: re-evaluate after the writes of this pass
        bool aj = (fj & 2) != 0;
        if (carry != 0.0)  // uniform; x − 0 = x exactly, so the precomputed decision is the same one otherwise
          aj = metropolis<true>(__shfl_sync(FULL, base, j) - carry, __shfl_sync(FULL, d.eps, j));
        if (lane == j) { accepted = aj; pending = false; }
        if (aj) {
          const double lj = __shfl_sync(FULL, la, j);
          const int wlo = __shfl_sync(FULL, lo, j), whi = __shfl_sync(FULL, hi, j);
          carry = P.alpha_carry ? lj : 0.0;  // logπ_prev = logπ + log α (acceptance.jl:32-33)
          if (pending && lo - 1 <= whi && hi + 1 >= wlo) valid = false;
        }
      }
      // ---- the trials accepted in this pass write their segments (pairwise disjoint) --------------------------
      if (accepted && !written) {
        if (reflect)
          for (int k = lo; k <= hi; ++k) {
            if (k == d.idx) continue;
            MonoRec r = mono[k];  // refl_n! / flip_n! of the record
            if (P.planar) { r.phi += kPi; r.nx = -r.nx; r.ny = -r.ny; r.nz = -r.nz; }
            else { r.theta = reflect_theta(r.theta); r.nz = -r.nz; }
            mono[k] = r;
          }
        mono[d.idx] = nrec;
        written = true;
      }
      __syncwarp();  // record writes of this pass are visible to the re-evaluations
    }
    // ---- running state after each trial: inclusive prefix sums of the accepted increments ---------------------
    if (!accepted) { dU = dOm = dsu = Dx = Dy = Dz = dpx = dpy = dpz = dpsi = dcos2 = 0.0; }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double t0 = __shfl_up_sync(FULL, Dx, o), t1 = __shfl_up_sync(FULL, Dy, o), t2 = __shfl_up_sync(FULL, Dz, o);
      const double t3 = __shfl_up_sync(FULL, dpx, o), t4 = __shfl_up_sync(FULL, dpy, o), t5 = __shfl_up_sync(FULL, dpz, o);
      const double t6 = __shfl_up_sync(FULL, dU, o), t7 = __shfl_up_sync(FULL, dsu, o), t8 = __shfl_up_sync(FULL, dOm, o);
      const double t9 = __shfl_up_sync(FULL, dpsi, o), t10 = __shfl_up_sync(FULL, dcos2, o);
      if (lane >= o) {
        Dx += t0; Dy += t1; Dz += t2; dpx += t3; dpy += t4; dpz += t5; dU += t6; dsu += t7; dOm += t8;
        dpsi += t9; dcos2 += t10;
      }
    }
    if (active) {
      const double r[3] = {D.r[0] + Dx, D.r[1] + Dy, D.r[2] + Dz};
      const double p[3] = {D.p[0] + dpx, D.p[1] + dpy, D.p[2] + dpz};
      const double su = D.su + dsu;
      record_averages<COMP>(P, acc, comp, r, p, D.U + dU, su, D.log_gauge);
      double wgt = 1.0;  // record_extras (mcmc_clustering_eap_chain.jl:243-244)
      if (P.umbrella) wgt = 1.0 / exp(su * P.inv_kT * P.cF - D.log_gauge);
      const double v0 = (DX.scos2 + dcos2) * wgt, v1 = (DX.spsi + dpsi) / (double)(n - 1) * wgt;
      if (COMP) { comp_add(xacc[0], xcomp[0], v0); comp_add(xacc[1], xcomp[1], v1); }
      else { xacc[0] += v0; xacc[1] += v1; }
    }
    const int last = wlen - 1;
    D.r[0] += __shfl_sync(FULL, Dx, last); D.r[1] += __shfl_sync(FULL, Dy, last); D.r[2] += __shfl_sync(FULL, Dz, last);
    D.p[0] += __shfl_sync(FULL, dpx, last); D.p[1] += __shfl_sync(FULL, dpy, last); D.p[2] += __shfl_sync(FULL, dpz, last);
    D.U += __shfl_sync(FULL, dU, last);
    D.su += __shfl_sync(FULL, dsu, last);
    D.Omega += __shfl_sync(FULL, dOm, last);
    DX.spsi += __shfl_sync(FULL, dpsi, last);
    DX.scos2 += __shfl_sync(FULL, dcos2, last);
    DX.carry = carry;
    const int nacc_w = __popc(__ballot_sync(FULL, accepted));
    D.nacc += nacc_w; D.nacc_total += nacc_w;
    D.natt += wlen; D.steps_total += wlen;
    {  // cluster statistics: trials with a flip, Σ sizes, largest (counted whether accepted or not)
      const bool fl = active && reflect;
      int sz = fl ? hi - lo + 1 : 0, mx = sz;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sz += __shfl_xor_sync(FULL, sz, o);
        mx = max(mx, __shfl_xor_sync(FULL, mx, o));
      }
      DX.ncluster += (double)__popc(__ballot_sync(FULL, fl));
      DX.cluster_sum += (double)sz;
      DX.cluster_max = fmax(DX.cluster_max, (double)mx);
    }
    const long long step_last = step0 + s + last;
    D.step = step_last;
    adapt_steps(P, step_last, D.phi_step, D.theta_step, D.nacc, D.natt);  // no-op unless a boundary
    if (a.stepout > 0 && (step_last % a.stepout) == 0) {
      double tot[kNumAcc], xt[2];
#pragma unroll
      for (int k = 0; k < kNumAcc; ++k) tot[k] = warp_sum(acc[k] + comp[k]);
#pragma unroll
      for (int k = 0; k < 2; ++k) xt[k] = warp_sum(xacc[k] + xcomp[k]);
      if (row < a.rows) {
        if (lane == 0) {
          double* t = a.traj + ((size_t)c * a.rows + row) * 8;
          double* rr = a.roll + ((size_t)c * a.rows + row) * a.roll_cols;
          t[0] = (double)step_last;
          t[1] = D.r[0]; t[2] = D.r[1]; t[3] = D.r[2];
          t[4] = D.p[0]; t[5] = D.p[1]; t[6] = D.p[2];
          t[7] = D.U;
          rr[0] = (double)step_last;
#pragma unroll
          for (int k = 0; k < 16; ++k) rr[1 + k] = tot[k] / tot[16];
          if (a.roll_cols > 17) { rr[17] = xt[0] / tot[16]; rr[18] = xt[1] / tot[16]; }
        }
        if (a.state) {
          double* st = a.state + ((size_t)c * a.rows + row) * 2 * (size_t)n;
          for (int k = lane; k < n; k += 32) { st[2 * k] = mono[k].phi; st[2 * k + 1] = mono[k].theta; }
        }
      }
      ++row;
    }
    s += wlen;
  }
  // combine the per-lane accumulators
#pragma unroll
  for (int k = 0; k < kNumAcc; ++k) {
    D.acc[k] = warp_sum(acc[k] + comp[k]);
    D.comp[k] = 0.0;
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    DX.acc[k] = warp_sum(xacc[k] + xcomp[k]);
    DX.comp[k] = 0.0;
  }
  if (lane == 0) {
    a.dyn[c] = D;
    a.dynx[c] = DX;
  }
  if (STAGE) {
    __syncwarp();
    for (int k = lane; k < n; k += 32) gmono[k] = mono[k];
  }
}

// Non-mutating sums of one scripted composite trial through the lane path's device code.
template <bool ISING>
__global__ void k_delta_segment_lane(const SegDeltaArgs a) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  const int n = a.n;
  const MonoRec* mono = a.mono + (size_t)a.chain * n;
  const ChainParams P = a.par[a.chain];
  const MonoRec rec = mono[a.idx];
  Proposal q;
  if (P.planar) build_proposal_planar(P, rec, a.idx, a.dphi, 0.0, q);
  else build_proposal(P, rec, a.idx, a.dphi, a.dtheta, 0.0, q);
  const bool reflect = a.reflect != 0;
  const int lo = reflect ? a.lo : a.idx, hi = reflect ? a.hi : a.idx;
  LaneSeg g;
  lane_seg_zero(g);
  double up = 0.0, lp = 0.0;
  if (reflect) {
    for (int k = lo; k <= hi; ++k) {
      if (k == a.idx) continue;
      const MonoRec r = mono[k];
      lane_add_flipped(P, r, g);
    }
    // link probabilities before the flip, on the chain carrying the move
    if (hi < n - 1) {
      const MonoRec b = mono[hi + 1];
      const MonoRec t = mono[hi];
      const bool m = hi == a.idx;
      up = link_prob(m ? q.nx : t.nx, m ? q.ny : t.ny, m ? q.nz : t.nz, b.nx, b.ny, b.nz);
    }
    if (lo > 0) {
      const MonoRec b = mono[lo - 1];
      const MonoRec t = mono[lo];
      const bool m = lo == a.idx;
      lp = link_prob(m ? q.nx : t.nx, m ? q.ny : t.ny, m ? q.nz : t.nz, b.nx, b.ny, b.nz);
    }
  }
  MonoRec nrec;
  double dOm_idx;
  lane_idx_record(P, q, reflect, nrec, dOm_idx);
  g.dOmega += dOm_idx;
  double la;
  lane_segment_finish<ISING>(mono, n, P, rec, nrec, a.idx, lo, hi, reflect, g, la, up, lp);
  const double Dx = P.b * g.sx, Dz = P.b * g.sz;
  const double dpairs = kInv4Pi * g.dpair;
  a.out[0] = g.du_self + g.dbend - (Dx * P.Fx + Dz * P.Fz) + dpairs;
  a.out[1] = g.dOmega; a.out[2] = dpairs; a.out[3] = g.du_self;
  a.out[4] = -(Dx * P.Fx + Dz * P.Fz); a.out[5] = g.dbend; a.out[6] = g.dpsi; a.out[7] = g.dcos2;
  a.out[8] = g.dpx; a.out[9] = g.dpy; a.out[10] = g.dpz; a.out[11] = la;
}

// A fresh `mcmc(nsteps, pargs, chain)` call on the current chains (mcmc_clustering_eap_chain.jl:171-265):
// new averagers, counters, step sizes and acceptor; the RNG stream tag advances.  The running scalars and
// the weight function are re-synchronised by k_energy_cta afterwards (rebind_gauge).
static __global__ void k_begin_stage(ChainDyn* dyn, ChainDynX* dynx, const ChainParams* par, int nchains, int new_init) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nchains) return;
  ChainDyn& D = dyn[c];
  ChainDynX& X = dynx[c];
  D.phi_step = par[c].phi_step0;
  D.theta_step = par[c].theta_step0;
  D.nacc = D.natt = D.nacc_total = D.steps_total = D.step = 0;
  D.init = new_init;
  D.drift_max = 0.0;
  for (int k = 0; k < kNumAcc; ++k) { D.acc[k] = 0.0; D.comp[k] = 0.0; }
  X.carry = 0.0;
  X.acc[0] = X.acc[1] = X.comp[0] = X.comp[1] = 0.0;
  X.ncluster = X.cluster_sum = X.cluster_max = 0.0;
}

// --x0/--dx0 initial chains (eap_chain.jl:63-78): ϕ = ϕ0 + U(0,dx0[1]), θ = θ0 + U(0,dx0[2]); the uniforms
// are those of the random-init stream.
static __global__ void k_fill_x0(MonoRec* mono, long long total, int n, uint64_t seed, uint32_t chain_id_base,
                          uint32_t init, const double* x0, int x0_len, double dx0_phi, double dx0_theta) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total) return;
  const long long c = g / n;
  const int k = (int)(g - c * n);
  const uint4 w = philox_at(seed, chain_id_base + (uint32_t)c, init, SUB_INIT, (uint64_t)k);
  const double p0 = x0_len == 2 ? x0[0] : x0[2 * k], t0 = x0_len == 2 ? x0[1] : x0[2 * k + 1];
  mono[g] = make_record(p0 + (0.0 + (dx0_phi - 0.0) * u53(w.x, w.y)), t0 + (0.0 + (dx0_theta - 0.0) * u53(w.z, w.w)));
}

}  // namespace pmc
