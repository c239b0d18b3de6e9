// cta_kernels.cuh — one CTA per chain: the interacting (all-pairs dipole-dipole) hot path.
//
// The chain (positions x, dipoles μ; eap_chain.jl:31,33 `μs`, `xs`) is staged in shared memory as
// SoA FP64 arrays.  A single-monomer rotation at idx translates the whole tail j>idx rigidly
// (positions are a cumulative sum of directions, eap_chain.jl:49-51), so the exact energy change
// touches the row {idx}×rest and the rectangle heads(i<idx)×tails(j>idx) — (idx)(n-1-idx)+(n-1)
// pairs (SURVEY.md §8a).  The rectangle is flattened over the CTA's warps: one side of the
// rectangle is held in registers one item per lane, the other side is read from shared memory as
// warp-wide broadcasts, and the partial sums are reduced with warp shuffles.
#pragma once

#include <type_traits>

#include "chain_math.cuh"

namespace pmc {

constexpr int kPartDoubles = 96;  // 3 × 32 warp partials (block scan of n̂ needs three)
constexpr int kRowDoubles = 26;   // 8 trajectory + 17 rolling values (+1 pad)

struct CtaView {
  double *sx, *sy, *sz;   // positions x_i (eap_chain.jl:49-51)
  double *mx, *my, *mz;   // dipoles μ_i
  double *E;              // μ_B · D_eff of the broadcast-side items of the current trial
  double *part;           // warp partial sums
  double *rowbuf;         // staging of one output row
  Proposal* prop;         // [2] ping-pong
  ChainDyn* dyn;
  ChainParams* par;
};

__host__ __device__ inline size_t cta_smem_bytes(int n) {
  size_t b = (size_t)7 * n * sizeof(double);
  b += (kPartDoubles + kRowDoubles) * sizeof(double);
  b += 2 * sizeof(Proposal) + sizeof(ChainDyn) + sizeof(ChainParams);
  return (b + 15) & ~(size_t)15;
}

__device__ __forceinline__ CtaView carve(unsigned char* base, int n) {
  CtaView S;
  double* d = reinterpret_cast<double*>(base);
  S.sx = d; S.sy = d + n; S.sz = d + 2 * n;
  S.mx = d + 3 * n; S.my = d + 4 * n; S.mz = d + 5 * n;
  S.E = d + 6 * n;
  S.part = d + 7 * n;
  S.rowbuf = S.part + kPartDoubles;
  S.prop = reinterpret_cast<Proposal*>(S.rowbuf + kRowDoubles);
  S.dyn = reinterpret_cast<ChainDyn*>(S.prop + 2);
  S.par = reinterpret_cast<ChainParams*>(S.dyn + 1);
  return S;
}

// Compact layout for the composite-trial run kernel (cluster_kernels.cuh), where shared memory per chain sets
// the number of resident chains: 3 partials per warp, a 28-double row buffer, no ping-pong proposals.
constexpr int kRowDoublesCompact = 28;

__host__ __device__ inline size_t cta_smem_bytes_compact(int n, int threads) {
  size_t b = (size_t)7 * n * sizeof(double);
  b += (size_t)(3 * (threads / 32) + kRowDoublesCompact) * sizeof(double);
  b += sizeof(ChainDyn) + sizeof(ChainParams);
  return (b + 15) & ~(size_t)15;
}

__device__ __forceinline__ CtaView carve_compact(unsigned char* base, int n, int threads) {
  CtaView S;
  double* d = reinterpret_cast<double*>(base);
  S.sx = d; S.sy = d + n; S.sz = d + 2 * n;
  S.mx = d + 3 * n; S.my = d + 4 * n; S.mz = d + 5 * n;
  S.E = d + 6 * n;
  S.part = d + 7 * n;
  S.rowbuf = S.part + 3 * (threads / 32);
  S.prop = nullptr;
  S.dyn = reinterpret_cast<ChainDyn*>(S.rowbuf + kRowDoublesCompact);
  S.par = reinterpret_cast<ChainParams*>(S.dyn + 1);
  return S;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// A team = the threads that share one chain.  T = 32: one warp (several chains may share a CTA, see
// k_run_cta_cluster), team-local thread id = lane and the team barrier is __syncwarp; T > 32: the whole CTA.
template <int T>
__device__ __forceinline__ int team_tid() { return T == 32 ? (int)(threadIdx.x & 31) : (int)threadIdx.x; }
template <int T>
__device__ __forceinline__ void team_sync() {
  if (T == 32) __syncwarp();
  else __syncthreads();
}

// Sum over the CTA, result in every thread.  `trailing_sync` protects `part` for immediate reuse.
template <int T>
__device__ __forceinline__ double block_sum(double v, double* part, bool trailing_sync = true) {
  constexpr int W = T / 32;
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int w = 0; w < W; ++w) s += part[w];
  if (trailing_sync) __syncthreads();
  return s;
}

// Stage one chain: x = b(cumsum(n̂) − n̂/2) (update_xs!, eap_chain.jl:49-51) by a block scan, and
// μ (dipole_response.jl).  Ends with a barrier.
template <int T>
__device__ void load_chain(const MonoRec* __restrict__ mono, const ChainParams& P, int n, const CtaView& S) {
  constexpr int W = T / 32;
  const int tid = team_tid<T>(), lane = tid & 31, warp = tid >> 5;
  const int C = (n + T - 1) / T;
  const int i0 = min(n, tid * C), i1 = min(n, i0 + C);
  double lx = 0, ly = 0, lz = 0;
  for (int i = i0; i < i1; ++i) {
    lx += mono[i].nx;
    ly += mono[i].ny;
    lz += mono[i].nz;
  }
  // inclusive warp scan
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
  double ox = 0, oy = 0, oz = 0;
  for (int w = 0; w < warp && w < W; ++w) { ox += S.part[w]; oy += S.part[W + w]; oz += S.part[2 * W + w]; }
  double sxx = ox + (ix - lx), syy = oy + (iy - ly), szz = oz + (iz - lz);  // exclusive prefix
  for (int i = i0; i < i1; ++i) {
    const MonoRec r = mono[i];
    sxx += r.nx; syy += r.ny; szz += r.nz;
    S.sx[i] = P.b * (sxx - 0.5 * r.nx);
    S.sy[i] = P.b * (syy - 0.5 * r.ny);
    S.sz[i] = P.b * (szz - 0.5 * r.nz);
    double ux, uy, uz;
    mu_of(P, r.nx, r.ny, r.nz, ux, uy, uz);
    S.mx[i] = ux; S.my[i] = uy; S.mz[i] = uz;
  }
  team_sync<T>();
}

// 4π × dipole-dipole energy of the staged chain: U_interaction (eap_chain.jl:196-211) or
// U_Ising (:215-228).  Result in every thread.
template <int T>
__device__ double cta_pair_energy(const CtaView& S, int n, int energy_type, double crad2 = 0.0) {
  constexpr int W = T / 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double acc = 0.0;
  if (energy_type == 3) {  // UCutoff, eap_chain.jl:171-192
    for (int i = warp; i < n - 1; i += W) {
      const double xi = S.sx[i], yi = S.sy[i], zi = S.sz[i];
      const double ax = S.mx[i], ay = S.my[i], az = S.mz[i];
      for (int j = i + 1 + lane; j < n; j += 32)
        acc += pair_g_cut(ax, ay, az, S.mx[j], S.my[j], S.mz[j], xi - S.sx[j], yi - S.sy[j], zi - S.sz[j], crad2);
    }
  } else if (energy_type == 1) {
    for (int i = warp; i < n - 1; i += W) {
      const double xi = S.sx[i], yi = S.sy[i], zi = S.sz[i];
      const double ax = S.mx[i], ay = S.my[i], az = S.mz[i];
      for (int j = i + 1 + lane; j < n; j += 32)
        acc += pair_g(ax, ay, az, S.mx[j], S.my[j], S.mz[j], xi - S.sx[j], yi - S.sy[j], zi - S.sz[j]);
    }
  } else if (energy_type == 2) {
    for (int i = tid; i < n - 1; i += T)
      acc += pair_g(S.mx[i], S.my[i], S.mz[i], S.mx[i + 1], S.my[i + 1], S.mz[i + 1],
                    S.sx[i] - S.sx[i + 1], S.sy[i] - S.sy[i + 1], S.sz[i] - S.sz[i + 1]);
  }
  return block_sum<T>(acc, S.part);
}

// The rectangle heads×tails, 39 FP64 instructions per pair (old and new energy of one pair):
//   lane item L in registers (x_L, μ_L, −3μ_L, cL = −3μ_L·D, wL = −2p_L), broadcast item B from shared
//   memory (x_B, μ_B, eB = μ_B·D, vB = |D|² + 2p_B);  r = x_L − x_B,  r' = r − D;
//   μ_L·r' = μ_L·r − μ_L·D and μ_B·r' = μ_B·r − eB save two dot products;
//   |r'|² = r² − 2r·D + |D|² = (r² + wL) + vB with r·D = p_L − p_B, p_k = (x_k − x_idx)·D the projection on
//   the move measured from the rotated monomer: 2 DADD instead of forming r' (3 DADD + 1 DMUL + 2 DFMA).
//   Measured from the pivot, the rounding error of |r'|² is of order eps·|x_k − x_idx|·|D|, the order r
//   itself already carries;
//   g = y³(μ_L·μ_B + (−3μ_L·r)(μ_B·r) y²),  y = 1/|r|.
// Shared-memory loads are not free next to the FP64 pipe (≈1.7 issue cycles per LDS.64 against 2 per
// DFMA, tools/fp64_mix.cu), so each lane keeps NL=2 lane items and every broadcast item loaded from
// shared memory serves two pairs; an odd last group of 32 lane items runs with NL=1.
// A team = the warps that share the pair work of one chain: here the whole CTA.
template <int NW>
struct Team {
  static constexpr int kWarps = NW;
  static constexpr int kThreads = NW * 32;
  static constexpr int kLocalThreads = NW * 32;   // threads that share ONE copy of the staged chain (see PairTeam)
  __device__ __forceinline__ static int tid() { return (int)threadIdx.x; }
  __device__ __forceinline__ static int ltid() { return tid(); }
  __device__ __forceinline__ static int warp() { return (int)(threadIdx.x >> 5); }
  __device__ __forceinline__ static int lane() { return (int)(threadIdx.x & 31); }
  __device__ __forceinline__ static void sync() { __syncthreads(); }
};

// One warp as the team (chains of ≤ 160 monomers in the composite-trial kernel).
struct WarpTeam {
  static constexpr int kWarps = 1;
  static constexpr int kThreads = 32;
  static constexpr int kLocalThreads = 32;
  __device__ __forceinline__ static int tid() { return (int)(threadIdx.x & 31); }
  __device__ __forceinline__ static int ltid() { return tid(); }
  __device__ __forceinline__ static int warp() { return 0; }
  __device__ __forceinline__ static int lane() { return (int)(threadIdx.x & 31); }
  __device__ __forceinline__ static void sync() { __syncwarp(); }
};

struct LaneItem {
  double x, y, z;     // position
  double ax, ay, az;  // μ
  double tx, ty, tz;  // −3μ
  double c;           // −3μ·D
  double w;           // −2(x − x_idx)·D (Q2 form only, see rect_lane_w)
};

__device__ __forceinline__ LaneItem load_lane_item(const CtaView& S, int L, double Dx, double Dy, double Dz) {
  LaneItem it;
  it.x = S.sx[L]; it.y = S.sy[L]; it.z = S.sz[L];
  it.ax = S.mx[L]; it.ay = S.my[L]; it.az = S.mz[L];
  it.tx = -3.0 * it.ax; it.ty = -3.0 * it.ay; it.tz = -3.0 * it.az;
  it.c = fma(it.tz, Dz, fma(it.ty, Dy, it.tx * Dx));
  it.w = 0.0;
  return it;
}

// Projection of x on the move, measured from the pivot (px, py, pz) = x_idx: p = (x − x_idx)·D.
__device__ __forceinline__ double rect_proj(double x, double y, double z, double px, double py, double pz, double Dx,
                                            double Dy, double Dz) {
  return fma(z - pz, Dz, fma(y - py, Dy, (x - px) * Dx));
}

// wL = −2p_L of a lane item.
__device__ __forceinline__ void rect_lane_w(LaneItem& it, double px, double py, double pz, double Dx, double Dy,
                                            double Dz) {
  it.w = -2.0 * rect_proj(it.x, it.y, it.z, px, py, pz, Dx, Dy, Dz);
}

// Broadcast-side values of one trial, written by the pre-pass before rect_sum.  Q2 form: {eB, vB} of broadcast
// item k (counted from the start of the broadcast side) interleaved at S.E[2k], S.E[2k+1] and read with one 16-byte
// load, so the broadcast side must have at most n/2 items (S.E holds n doubles).  Otherwise eB at S.E[baseB + k].
template <bool Q2>
__device__ __forceinline__ void rect_prepass_item(const CtaView& S, int baseB, int k, double px, double py, double pz,
                                                  double Dx, double Dy, double Dz) {
  const int j = baseB + k;
  const double e = fma(S.mz[j], Dz, fma(S.my[j], Dy, S.mx[j] * Dx));
  if constexpr (Q2) {
    const double dd = fma(Dz, Dz, fma(Dy, Dy, Dx * Dx));
    reinterpret_cast<double2*>(S.E)[k] =
        make_double2(e, fma(2.0, rect_proj(S.sx[j], S.sy[j], S.sz[j], px, py, pz, Dx, Dy, Dz), dd));
  }
  else
    S.E[j] = e;
}

// new − old of one pair: lane item `it` against broadcast item (bx,by,bz; ux,uy,uz; e; p2 = vB, Q2 form only).
// CUT: UCutoff (eap_chain.jl:176-187) — a term is zero when its own r² exceeds crad².
template <bool CUT = false, bool Q2 = false>
__device__ __forceinline__ double rect_pair(const LaneItem& it, double bx, double by, double bz, double ux,
                                            double uy, double uz, double e, double p2, double Dx, double Dy, double Dz,
                                            double acc, double crad2 = 0.0) {
  const double rx = it.x - bx, ry = it.y - by, rz = it.z - bz;
  const double mm = fma(it.az, uz, fma(it.ay, uy, it.ax * ux));
  const double r2 = fma(rz, rz, fma(ry, ry, rx * rx));
  const double a3 = fma(it.tz, rz, fma(it.ty, ry, it.tx * rx));
  const double bb = fma(uz, rz, fma(uy, ry, ux * rx));
  double q2;
  if constexpr (Q2) {
    q2 = (r2 + it.w) + p2;
  } else {
    const double qx = rx - Dx, qy = ry - Dy, qz = rz - Dz;
    q2 = fma(qz, qz, fma(qy, qy, qx * qx));
  }
  const double a3n = a3 - it.c;
  const double bn = bb - e;
  const double y = rsqrt_fast(r2);
  const double yn = rsqrt_fast(q2);
  const double y2 = y * y, yn2 = yn * yn;
  const double t = fma(a3 * bb, y2, mm);
  const double tn = fma(a3n * bn, yn2, mm);
  if constexpr (CUT) {
    const double gn = tn * (yn2 * yn), go = t * (y2 * y);
    return acc + ((q2 > crad2 ? 0.0 : gn) - (r2 > crad2 ? 0.0 : go));
  } else {
    acc = fma(tn, yn2 * yn, acc);
    return fma(-t, y2 * y, acc);
  }
}

// EFLY: eB = μ_B·D is computed in the loop (3 DFMA per broadcast item) instead of being read from S.E —
// saves the pre-pass and its barrier where barriers cost more than FP64 issue slots (short chains).
// Q2: |r'|² from the projections (rect_prepass_item<true> has filled S.E); `pivot` = idx, the rotated monomer.
// The pivot is read from shared memory with each lane item: its index costs one register in the loop, its position six.
template <class TEAM, int UNROLL = 2, bool CUT = false, bool EFLY = false, bool Q2 = false>
__device__ __forceinline__ double rect_sum(const CtaView& S, int baseA, int A, int baseB, int B, double Dx,
                                           double Dy, double Dz, double crad2 = 0.0, int pivot = 0) {
  static_assert(!(Q2 && EFLY), "the Q2 form reads 2p_B from the pre-pass");
  constexpr int W = TEAM::kWarps;
  const int lane = TEAM::lane(), warp = TEAM::warp();
  const int G = (A + 31) >> 5;
  const double* __restrict__ bxp = S.sx + baseB;
  const double* __restrict__ byp = S.sy + baseB;
  const double* __restrict__ bzp = S.sz + baseB;
  const double* __restrict__ mxp = S.mx + baseB;
  const double* __restrict__ myp = S.my + baseB;
  const double* __restrict__ mzp = S.mz + baseB;
  const double* __restrict__ ep = S.E + baseB;
  const double2* __restrict__ e2p = reinterpret_cast<const double2*>(S.E);
  auto lane_item = [&](int L) {
    LaneItem it = load_lane_item(S, L, Dx, Dy, Dz);
    if (Q2) {
      rect_lane_w(it, S.sx[pivot], S.sy[pivot], S.sz[pivot], Dx, Dy, Dz);
      // With wL the two lane items fill the 128 registers of k_run_cta_win<128,4,2>, and ptxas would recompute
      // −3μ inside the pair loop (5 DMUL per 4 pairs) rather than spill per-trial values outside it.  Hiding how −3μ
      // was made keeps it in registers: 39 FP64 per pair in the loop (profiles/r04_rect_q2_sass.txt).
      asm("" : "+d"(it.tx), "+d"(it.ty), "+d"(it.tz));
    }
    return it;
  };
  // eB (and vB) of broadcast item k, whose μ is (ux, uy, uz)
  auto bvals = [&](int k, double ux, double uy, double uz, double& e, double& p2) {
    if constexpr (Q2) {
      const double2 v = e2p[k];
      e = v.x; p2 = v.y;
    } else {
      e = EFLY ? fma(uz, Dz, fma(uy, Dy, ux * Dx)) : ep[k];
      p2 = 0.0;
    }
  };
  double acc = 0.0;
  // phase 1: group pairs (64 lane items per warp pass), two pairs per broadcast load
  const int G2 = G >> 1;
  {
    const int U = G2 * B;
    int u = (int)(((long long)U * warp) / W);
    const int u1 = (int)(((long long)U * (warp + 1)) / W);
    if (u < u1) {
      int g = u / B;
      int k = u - g * B;
      while (u < u1) {
        const int l0 = g * 64 + lane, l1 = l0 + 32;
        const bool v0 = l0 < A, v1 = l1 < A;
        const LaneItem i0 = lane_item(baseA + min(l0, A - 1));
        const LaneItem i1 = lane_item(baseA + min(l1, A - 1));
        const int kend = min(B, k + (u1 - u));
        u += kend - k;
        double a0 = 0.0, a1 = 0.0;
#pragma unroll UNROLL
        for (; k < kend; ++k) {
          const double bx = bxp[k], by = byp[k], bz = bzp[k];
          const double ux = mxp[k], uy = myp[k], uz = mzp[k];
          double e, p2;
          bvals(k, ux, uy, uz, e, p2);
          a0 = rect_pair<CUT, Q2>(i0, bx, by, bz, ux, uy, uz, e, p2, Dx, Dy, Dz, a0, crad2);
          a1 = rect_pair<CUT, Q2>(i1, bx, by, bz, ux, uy, uz, e, p2, Dx, Dy, Dz, a1, crad2);
        }
        acc += (v0 ? a0 : 0.0) + (v1 ? a1 : 0.0);
        k = 0;
        ++g;
      }
    }
  }
  // phase 2: the odd last group of 32 lane items
  if (G & 1) {
    int k = (int)(((long long)B * warp) / W);
    const int kend = (int)(((long long)B * (warp + 1)) / W);
    if (k < kend) {
      const int li = (G - 1) * 32 + lane;
      const bool valid = li < A;
      const LaneItem it = lane_item(baseA + min(li, A - 1));
      double a0 = 0.0, a1 = 0.0;
      auto pair = [&](int kk, double a) {
        double e, p2;
        bvals(kk, mxp[kk], myp[kk], mzp[kk], e, p2);
        return rect_pair<CUT, Q2>(it, bxp[kk], byp[kk], bzp[kk], mxp[kk], myp[kk], mzp[kk], e, p2, Dx, Dy, Dz, a,
                                  crad2);
      };
      for (; k + 1 < kend; k += 2) {
        a0 = pair(k, a0);
        a1 = pair(k + 1, a1);
      }
      if (k < kend) a0 = pair(k, a0);
      acc += valid ? (a0 + a1) : 0.0;
    }
  }
  return acc;
}

// 4π × Σ over changed pairs of (new − old): this thread's share (row part + rectangle).  Contains one
// team barrier (after E).
template <class TEAM, int UNROLL = 2>
__device__ __forceinline__ double delta_pairs_partial(const CtaView& S, int n, int energy_type, double b, int idx,
                                                      double npx, double npy, double npz,   // μ'
                                                      double dnx, double dny, double dnz) { // Δn̂
  constexpr int T = TEAM::kThreads;
  const int tid = TEAM::tid();
  const double Dx = b * dnx, Dy = b * dny, Dz = b * dnz;  // tail translation
  const double hx = 0.5 * Dx, hy = 0.5 * Dy, hz = 0.5 * Dz;
  const int H = idx, Tl = n - 1 - idx;
  // lane side = the one that wastes fewer lanes
  bool rect = (energy_type == 1) && H > 0 && Tl > 0;
  bool lanes_are_heads = true;
  if (rect) {
    const long long costH = (long long)((H + 31) >> 5) * Tl;
    const long long costT = (long long)((Tl + 31) >> 5) * H;
    lanes_are_heads = costH <= costT;
    // {eB, 2p_B} of the broadcast side fill 2B of the n doubles of S.E: at most one side (H + Tl = n − 1) has more
    // than n/2 items, and it goes on the lanes
    if (2 * (lanes_are_heads ? Tl : H) > n) lanes_are_heads = !lanes_are_heads;
  }
  // D_eff: r = x_L − x_B.  L=head,B=tail: r' = r − D.  L=tail,B=head: r' = r + D.
  const double sgn = lanes_are_heads ? 1.0 : -1.0;
  const double ex = sgn * Dx, ey = sgn * Dy, ez = sgn * Dz;
  const int baseA = lanes_are_heads ? 0 : idx + 1, A = lanes_are_heads ? H : Tl;
  const int baseB = lanes_are_heads ? idx + 1 : 0, B = lanes_are_heads ? Tl : H;
  const double xi = S.sx[idx], yi = S.sy[idx], zi = S.sz[idx];  // the pivot of the Q2 projections
  if (rect)  // every copy of the staged chain needs its own E
    for (int k = TEAM::ltid(); k < B; k += TEAM::kLocalThreads)
      rect_prepass_item<true>(S, baseB, k, xi, yi, zi, ex, ey, ez);
  // row {idx}×rest: both μ_idx and the separation change.
  double acc = 0.0;
  {
    const double ox = S.mx[idx], oy = S.my[idx], oz = S.mz[idx];
    int jlo = 0, jhi = n - 1;
    if (energy_type == 2) { jlo = max(0, idx - 1); jhi = min(n - 1, idx + 1); }
    if (energy_type == 0) { jlo = 1; jhi = 0; }
    for (int j = jlo + tid; j <= jhi; j += T) {
      if (j == idx) continue;
      const double rx = xi - S.sx[j], ry = yi - S.sy[j], rz = zi - S.sz[j];
      const double s = (j < idx) ? 1.0 : -1.0;  // x'_idx − x'_j = r ± (b/2)Δn̂
      const double ux = S.mx[j], uy = S.my[j], uz = S.mz[j];
      acc += pair_g(npx, npy, npz, ux, uy, uz, fma(s, hx, rx), fma(s, hy, ry), fma(s, hz, rz)) -
             pair_g(ox, oy, oz, ux, uy, uz, rx, ry, rz);
    }
  }
  TEAM::sync();  // E visible
  if (rect) acc += rect_sum<TEAM, UNROLL, false, false, true>(S, baseA, A, baseB, B, ex, ey, ez, 0.0, idx);
  return acc;
}

// Whole-CTA version: summed over the CTA, result in every thread; no trailing barrier.
template <int T, int UNROLL = 2>
__device__ __forceinline__ double cta_delta_pairs(const CtaView& S, int n, int energy_type, double b, int idx,
                                                  double npx, double npy, double npz, double dnx, double dny,
                                                  double dnz) {
  const double acc = delta_pairs_partial<Team<T / 32>, UNROLL>(S, n, energy_type, b, idx, npx, npy, npz, dnx, dny, dnz);
  return block_sum<T>(acc, S.part, /*trailing_sync=*/false);
}

}  // namespace pmc

#define PMC_CTA_BUILDING_BLOCKS 1
#include "cta_f32.cuh"

namespace pmc {

// ---------------------------------------------------------------------------------------------
// Kernels
// ---------------------------------------------------------------------------------------------
struct RunArgs {
  MonoRec* mono;
  const ChainParams* par;
  ChainDyn* dyn;
  double* traj;  // [chains][rows][8]
  double* roll;  // [chains][rows][17]
  long long nsteps, stepout, rows;
  uint64_t seed;
  uint32_t chain_id_base;
  int n;
  int nchains;
  int energy_type;
  // clustering driver only (cluster_kernels.cuh)
  ChainDynX* dynx;
  double* state;   // [chains][rows][2n] (phi,theta interleaved) or null
  int roll_cols;   // 17, or 19 with the two extra averagers
  int compensated; // Neumaier-compensated accumulators (accum_mode 1 or umbrella weights), else plain sums
  int window;      // k_run_warp_cluster: trials per window (≤ 32)
};

// Thread 0 (window: lane k for trial step + k): draw and build the proposal of trial `step`.  `init` = D.init (the
// window passes the copy it keeps in a register, the rebuild of a stale entry reads D).
__device__ __forceinline__ void make_proposal(const RunArgs& a, const ChainParams& P, const ChainDyn& D,
                                              const MonoRec* mono, uint32_t chain_id, uint32_t init, long long step,
                                              Proposal& q) {
  const Draws d = draw_step(a.seed, chain_id, init, step, a.n);
  const MonoRec rec = mono[d.idx];
  double dphi, dtheta;
  increments(P, d, rec.theta, D.phi_step, D.theta_step, dphi, dtheta);
  build_proposal(P, rec, d.idx, dphi, dtheta, d.eps, q);
}

// State update of an accepted move and the trial counters (mcmc_eap_chain.jl:288-292).
__device__ __forceinline__ void apply_decision(const ChainParams& P, ChainDyn& D, const Proposal& q, bool accept,
                                               double dU_pairs, long long step) {
  if (accept) {
    D.U += q.du + q.drF + dU_pairs;
    D.Omega += q.dOmega;
    D.su += q.du;
    D.r[0] += P.b * q.dnx; D.r[1] += P.b * q.dny; D.r[2] += P.b * q.dnz;
    D.p[0] += q.dmx; D.p[1] += q.dmy; D.p[2] += q.dmz;
    D.nacc += 1;
    D.nacc_total += 1;
  }
  D.natt += 1;
  D.steps_total += 1;
  D.step = step;
}

// Step adaptation (:301-322) then the 8 averagers (:327-328) on the post-decision state.
template <bool COMP = true>
__device__ __forceinline__ void bookkeep(const ChainParams& P, ChainDyn& D, long long step) {
  adapt_steps(P, step, D.phi_step, D.theta_step, D.nacc, D.natt);
  record_averages<COMP>(P, D.acc, D.comp, D.r, D.p, D.U, D.su, D.log_gauge);
}

// Thread 0 (lane kernel: every thread): everything after the accept/reject decision.
template <bool COMP = true>
__device__ __forceinline__ void after_decision(const ChainParams& P, ChainDyn& D, const Proposal& q, bool accept,
                                               double dU_pairs, long long step) {
  apply_decision(P, D, q, accept, dU_pairs, step);
  bookkeep<COMP>(P, D, step);
}

__device__ __forceinline__ void stage_row(const ChainDyn& D, long long step, double* rowbuf) {
  rowbuf[0] = (double)step;  // the reference's hcat promotes step to Float64 (mcmc_eap_chain.jl:331)
  rowbuf[1] = D.r[0]; rowbuf[2] = D.r[1]; rowbuf[3] = D.r[2];
  rowbuf[4] = D.p[0]; rowbuf[5] = D.p[1]; rowbuf[6] = D.p[2];
  rowbuf[7] = D.U;
  rowbuf[8] = (double)step;
  const double nrm = D.acc[16] + D.comp[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) rowbuf[9 + k] = (D.acc[k] + D.comp[k]) / nrm;
}

// Warp 0, lane = tid: output row `row` of chain c after trial `step`, staged by lane 0.
__device__ __forceinline__ void emit_row(const RunArgs& a, const ChainDyn& D, int c, long long row, long long step,
                                         double* rowbuf, int tid) {
  if (tid == 0) stage_row(D, step, rowbuf);
  __syncwarp();
  if (row < a.rows) {
    if (tid < 8) a.traj[((size_t)c * a.rows + row) * 8 + tid] = rowbuf[tid];
    if (tid < 17) a.roll[((size_t)c * a.rows + row) * 17 + tid] = rowbuf[8 + tid];
  }
  __syncwarp();
}

// The record of monomer q.idx after the move of q.
__device__ __forceinline__ MonoRec record_of(const Proposal& q) {
  MonoRec rec;
  rec.phi = q.phi; rec.theta = q.theta;
  rec.nx = q.nx; rec.ny = q.ny; rec.nz = q.nz; rec.sth = q.sth;
  return rec;
}

// move! of an accepted trial, tail part: x_j += D for j ≥ first, by threads tid, tid + stride, …
__device__ __forceinline__ void shift_tail(const CtaView& S, int first, int n, double Dx, double Dy, double Dz, int tid,
                                           int stride) {
  for (int j = first + tid; j < n; j += stride) {
    S.sx[j] += Dx; S.sy[j] += Dy; S.sz[j] += Dz;
  }
}

// move! of an accepted single-monomer trial, by one thread: x_idx += (b/2)Δn̂, μ_idx = μ', and the record.
__device__ __forceinline__ void move_pivot(const CtaView& S, MonoRec* mono, const Proposal& q, int idx, double b,
                                           double dnx, double dny, double dnz) {
  S.sx[idx] += 0.5 * b * dnx; S.sy[idx] += 0.5 * b * dny; S.sz[idx] += 0.5 * b * dnz;
  S.mx[idx] = q.mx; S.my[idx] = q.my; S.mz[idx] = q.mz;
  mono[idx] = record_of(q);
}

// The accept/reject decision from the summed pair partials; explicit rounding so that every kernel takes
// bit-identical decisions.
__device__ __forceinline__ bool decide(double single, double tsum, double inv_kT, double eps, double& dsum) {
  dsum = __dmul_rn(kInv4Pi, tsum);
  return metropolis(__fma_rn(-dsum, inv_kT, single), eps);
}

// Proposal windows: the serial part of a trial (Philox, sincos, log, …) is taken off the per-trial critical path by
// building the proposals of the next kWin trials at once, one trial per lane of warp 0.  A proposal depends on the
// chain only through the record of its own monomer, so it stays valid unless an earlier trial of the window moves
// that monomer: accepted trials mark later proposals on the monomers they moved stale, and those are rebuilt
// (serially, rarely) when their turn comes.  A window never crosses a step-size adaptation boundary
// (mcmc_eap_chain.jl:301-322).
constexpr int kWin = 32;

// Trials of the window that starts at trial s.  to_boundary = trials until the adaptation rule runs next (0: never).
__device__ __forceinline__ int window_len(const RunArgs& a, const ChainParams& P, bool adapt_on, long long step0,
                                          long long s, long long& to_boundary) {
  long long wl = a.nsteps - s + 1;
  if (wl > kWin) wl = kWin;
  to_boundary = 0;
  if (adapt_on) {
    to_boundary = P.steps_per_adjust - ((step0 + s - 1) % P.steps_per_adjust);  // ≥ 1
    if (wl > to_boundary) wl = to_boundary;
  }
  return (int)wl;
}

// Warp 0, lane = tid: entry `tid` of the window is trial step + tid, built by make(tid, step + tid); no entry is stale.
template <class Make>
__device__ __forceinline__ void build_window(long long step, int wlen, unsigned& dirty, int tid, Make&& make) {
  if (tid < wlen) make(tid, step + tid);
  if (tid == 0) dirty = 0u;
}

// Warp 0, lane = tid: trial k of the window was accepted and moved monomers lo … hi; later entries on them are stale.
template <class Entry>
__device__ __forceinline__ void mark_stale(const Entry* win, int k, int wlen, int lo, int hi, unsigned& dirty,
                                           int tid) {
  const int widx = win[tid].idx;
  const bool stale = tid > k && tid < wlen && widx >= lo && widx <= hi;
  const unsigned m = __ballot_sync(0xffffffffu, stale);
  if (tid == 0 && m) dirty |= m;
}

__host__ __device__ inline size_t cta_smem_bytes_win(int n) {
  return (cta_smem_bytes(n) + kWin * sizeof(Proposal) + 16 + 15) & ~(size_t)15;
}
__host__ __device__ inline size_t cta_smem_bytes_win_f32(int n) { return cta_smem_bytes_win(n) + f32_smem_bytes(n); }

// The hot loop (mcmc_eap_chain.jl:276-350) for one interacting chain per CTA, with proposal windows.
// PREC = 1: the rectangle of every trial in FP32 (cta_f32.cuh; pmc_set_pair_precision), everything else as PREC = 0.
template <int T, int MINB, int UNROLL = 2, int PREC = 0>
__global__ void __launch_bounds__(T, MINB) k_run_cta_win(const RunArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const CtaView S = carve(smem_raw, a.n);
  Proposal* win = reinterpret_cast<Proposal*>(smem_raw + cta_smem_bytes(a.n));
  unsigned* dirty = reinterpret_cast<unsigned*>(win + kWin);
  const F32View F = carve_f32(smem_raw + cta_smem_bytes_win(a.n), PREC ? a.n : 0, S.E);
  const int c = blockIdx.x;
  const int tid = threadIdx.x;
  const int n = a.n;
  MonoRec* mono = a.mono + (size_t)c * n;
  if (tid == 0) {
    *S.par = a.par[c];
    *S.dyn = a.dyn[c];
  }
  __syncthreads();
  const ChainParams& P = *S.par;
  load_chain<T>(mono, P, n, S);
  if (PREC) fill_mu_f32<Team<T / 32>>(S, F, n);   // visible after the window barrier below
  const uint32_t chain_id = a.chain_id_base + (uint32_t)c;
  const double b = P.b, inv_kT = P.inv_kT;
  const long long step0 = S.dyn->step;
  const uint32_t init = (uint32_t)S.dyn->init;
  const bool adapt_on = P.adj_scale != 1.0 && P.steps_per_adjust > 0;
  long long row = 0;

  long long s = 1;
  while (s <= a.nsteps) {
    // ---- window [s, s+wlen) ----------------------------------------------------------------------
    long long to_boundary;
    const int wlen = window_len(a, P, adapt_on, step0, s, to_boundary);
    if (tid < 32)
      build_window(step0 + s, wlen, *dirty, tid,
                   [&](int e, long long st) { make_proposal(a, P, *S.dyn, mono, chain_id, init, st, win[e]); });
    __syncthreads();  // window visible
    for (int k = 0; k < wlen; ++k) {
      const long long step = step0 + s + k;
      if ((*dirty >> k) & 1u) {  // an earlier trial of this window moved the same monomer: rebuild
        if (tid == 0) make_proposal(a, P, *S.dyn, mono, chain_id, (uint32_t)S.dyn->init, step, win[k]);
        __syncthreads();
      }
      const Proposal* q = &win[k];
      const int idx = q->idx;
      const bool skip = q->skip;
      const double dnx = q->dnx, dny = q->dny, dnz = q->dnz;
      double dsum = 0.0;
      bool accept = false;
      if (!skip) {
        const double t = PREC ? cta_delta_pairs_f32<T>(S, F, n, b, idx, q->mx, q->my, q->mz, dnx, dny, dnz)
                              : cta_delta_pairs<T, UNROLL>(S, n, 1, b, idx, q->mx, q->my, q->mz, dnx, dny, dnz);
        accept = decide(q->single, t, inv_kT, q->eps, dsum);
      }
      if (accept) {
        shift_tail(S, idx + 1, n, b * dnx, b * dny, b * dnz, tid, T);
        if (tid < 32) mark_stale(win, k, wlen, idx, idx, *dirty, tid);
      }
      if (tid == 0) {
        if (accept) {
          move_pivot(S, mono, *q, idx, b, dnx, dny, dnz);
          if (PREC) F.pb[idx] = make_float4((float)q->mx, (float)q->my, (float)q->mz, 0.0f);   // w is rebuilt per trial
        }
        after_decision(P, *S.dyn, *q, accept, dsum, step);
      }
      const bool isrow = a.stepout > 0 && (step % a.stepout) == 0;
      if (isrow && tid < 32) emit_row(a, *S.dyn, c, row, step, S.rowbuf, tid);
      if (isrow) ++row;
      __syncthreads();  // state, records and dirty mask of this trial are visible
    }
    s += wlen;
  }
  if (tid == 0) a.dyn[c] = *S.dyn;
}

// Small ensembles of short chains: G one-warp teams per chain, each evaluating a DIFFERENT trial of the window at once.
//
// A few hundred chains of n ≈ 100 (what one study of the reference runs) cannot fill 148 SMs, and more warps on ONE trial
// stop paying at its serial parts.  A rejected trial leaves the chain as it was — and at the parameters of those studies
// most trials are rejected — so trials k … k+G−1 of the proposal window are evaluated at the same time against the
// shared, read-only staged chain (each team has its own E array), and then committed in order by the whole CTA: a
// rejected trial only does its bookkeeping, the first accepted one is applied and ends the batch (what was evaluated
// behind it saw a stale chain and is evaluated again).  Every decision is taken on exactly the state the sequential
// chain would show it.  The composite-trial counterpart is k_run_cta_cluster_spec (cluster_kernels.cuh).
struct SpecTrial {
  double dsum;
  int accept, pad;
};

// The E arrays of teams 1…G−1 start 16-byte aligned (rect_prepass_item reads S.E as double2).
__host__ __device__ inline int spec_e_stride(int n) { return (n + 1) & ~1; }

__host__ __device__ inline size_t cta_smem_bytes_spec(int n, int groups) {
  return cta_smem_bytes_win(n) +
         (((size_t)(groups - 1) * spec_e_stride(n) * sizeof(double) + (size_t)groups * sizeof(SpecTrial) + 15) & ~(size_t)15);
}

template <int G, int MINB>
__global__ void __launch_bounds__(32 * G, MINB) k_run_cta_win_spec(const RunArgs a) {
  constexpr int T = 32 * G;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const CtaView S = carve(smem_raw, a.n);
  Proposal* win = reinterpret_cast<Proposal*>(smem_raw + cta_smem_bytes(a.n));
  unsigned* dirty = reinterpret_cast<unsigned*>(win + kWin);
  double* extraE = reinterpret_cast<double*>(smem_raw + cta_smem_bytes_win(a.n));
  SpecTrial* res = reinterpret_cast<SpecTrial*>(extraE + (size_t)(G - 1) * spec_e_stride(a.n));
  const int c = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, g = tid >> 5;
  const int n = a.n;
  MonoRec* mono = a.mono + (size_t)c * n;
  CtaView Sg = S;                       // this team's view: its own E array, everything else shared
  if (g > 0) Sg.E = extraE + (size_t)(g - 1) * spec_e_stride(n);
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
  const uint32_t init = (uint32_t)S.dyn->init;
  const bool adapt_on = P.adj_scale != 1.0 && P.steps_per_adjust > 0;
  long long row = 0;
  Countdown row_due;
  row_due.start(step0, a.stepout);

  long long s = 1;
  while (s <= a.nsteps) {
    long long to_boundary;
    const int wlen = window_len(a, P, adapt_on, step0, s, to_boundary);
    if (tid < 32)
      build_window(step0 + s, wlen, *dirty, tid,
                   [&](int e, long long st) { make_proposal(a, P, *S.dyn, mono, chain_id, init, st, win[e]); });
    __syncthreads();  // window visible
    int k = 0;
    while (k < wlen) {
      const int nb = min(G, wlen - k);
      // ---- phase 1: team g evaluates trial k+g on the current chain ------------------------------------------
      if (g < nb) {
        const int kk = k + g;
        if ((*dirty >> kk) & 1u) {  // an accepted trial of this window moved the same monomer: rebuild the entry
          if (lane == 0) make_proposal(a, P, *S.dyn, mono, chain_id, (uint32_t)S.dyn->init, step0 + s + kk, win[kk]);
          __syncwarp();
        }
        const Proposal* q = &win[kk];
        double dsum = 0.0;
        bool accept = false;
        if (!q->skip) {
          const double part = delta_pairs_partial<WarpTeam, 1>(Sg, n, 1, b, q->idx, q->mx, q->my, q->mz, q->dnx, q->dny, q->dnz);
          accept = decide(q->single, warp_sum(part), inv_kT, q->eps, dsum);
        }
        if (lane == 0) {
          res[g].dsum = dsum;
          res[g].accept = accept ? 1 : 0;
        }
      }
      __syncthreads();  // all evaluations of the batch are in
      // ---- phase 2: commit in order; the first accepted trial ends the batch ---------------------------------
      int committed = 0;
      for (int bb = 0; bb < nb; ++bb) {
        const int kk = k + bb;
        const long long step = step0 + s + kk;
        const Proposal* q = &win[kk];
        const bool accept = res[bb].accept != 0;
        const int idx = q->idx;
        if (accept) {
          shift_tail(S, idx + 1, n, b * q->dnx, b * q->dny, b * q->dnz, tid, T);
          if (tid < 32) mark_stale(win, kk, wlen, idx, idx, *dirty, tid);
        }
        if (tid == 0) {
          if (accept) move_pivot(S, mono, *q, idx, b, q->dnx, q->dny, q->dnz);
          apply_decision(P, *S.dyn, *q, accept, res[bb].dsum, step);
          if (kk + 1 == to_boundary) adapt_apply(P, S.dyn->phi_step, S.dyn->theta_step, S.dyn->nacc, S.dyn->natt);
          record_averages<true>(P, S.dyn->acc, S.dyn->comp, S.dyn->r, S.dyn->p, S.dyn->U, S.dyn->su, S.dyn->log_gauge);
        }
        const bool isrow = row_due.tick();
        if (isrow && tid < 32) emit_row(a, *S.dyn, c, row, step, S.rowbuf, tid);
        if (isrow) ++row;
        ++committed;
        if (accept) break;  // the speculations behind this trial saw the chain before it
      }
      k += committed;
      __syncthreads();  // state, records, running scalars and the dirty mask are visible
    }
    s += wlen;
  }
  if (tid == 0) a.dyn[c] = *S.dyn;
}

// Recompute {U, Σu, U_dd, Ω, r, p} of chains from their records (EAPChain ctor tail,
// eap_chain.jl:124-133).  Optionally writes them to out4 / obs6 and/or re-synchronises dyn.
struct EnergyArgs {
  const MonoRec* mono;
  const ChainParams* par;
  ChainDyn* dyn;
  double* out4;  // [nchains][4] or null
  double* obs6;  // [nchains][6] or null
  int n, energy_type, first_chain;
  int update_dyn, rebind_gauge;
  ChainDynX* dynx;  // re-synchronised together with dyn
  double* out8;     // [nchains][8] = {U, Σu (incl. bending), U_dd, Ω, U_bend, Σψ/(n−1), Σcos²θ, 0} or null
};

// Σ over bonds of ubend (eap_chain.jl:54-58) and ψ (:45-47), Σ over monomers of cos²θ: this thread's share.
template <int T>
__device__ __forceinline__ void bond_sums_partial(const MonoRec* __restrict__ mono, const ChainParams& P, int n,
                                                  double& ub, double& sp, double& c2) {
  ub = 0.0; sp = 0.0; c2 = 0.0;
  for (int i = threadIdx.x; i < n; i += T) {
    const MonoRec a = mono[i];
    c2 += a.nz * a.nz;
    if (i + 1 < n) {
      const MonoRec b = mono[i + 1];
      const double psi = psi_of(a.nx, a.ny, a.nz, b.nx, b.ny, b.nz);
      sp += psi;
      ub += ubend_of(P, psi);
    }
  }
}

// Totals of one chain, in every thread.
struct ChainTotals {
  double U, su, udd, om, ub, sp, c2;
  double rx, ry, rz, px, py, pz;
};

// Stage the chain of records `mono` and sum its totals.
template <int T>
__device__ __forceinline__ ChainTotals chain_totals(const MonoRec* __restrict__ mono, const ChainParams& P, int n,
                                                    int energy_type, const CtaView& S) {
  const int tid = threadIdx.x;
  load_chain<T>(mono, P, n, S);
  ChainTotals t;
  double su = 0, om = 0, px = 0, py = 0, pz = 0;
  for (int i = tid; i < n; i += T) {
    su += -0.5 * P.E0 * S.mz[i];
    om += log(mono[i].sth);
    px += S.mx[i]; py += S.my[i]; pz += S.mz[i];
  }
  double ub, sp, c2;
  bond_sums_partial<T>(mono, P, n, ub, sp, c2);
  t.su = block_sum<T>(su, S.part);
  t.om = block_sum<T>(om, S.part);
  t.px = block_sum<T>(px, S.part);
  t.py = block_sum<T>(py, S.part);
  t.pz = block_sum<T>(pz, S.part);
  t.ub = block_sum<T>(ub, S.part);
  t.sp = block_sum<T>(sp, S.part);
  t.c2 = block_sum<T>(c2, S.part);
  t.su += t.ub;  // us[i] = u + ubend (eap_chain.jl:130)
  t.udd = kInv4Pi * cta_pair_energy<T>(S, n, energy_type, P.crad2);
  // end_to_end (eap_chain.jl:405): x_n + (b/2) n̂_n
  t.rx = S.sx[n - 1] + 0.5 * P.b * mono[n - 1].nx;
  t.ry = S.sy[n - 1] + 0.5 * P.b * mono[n - 1].ny;
  t.rz = S.sz[n - 1] + 0.5 * P.b * mono[n - 1].nz;
  // energy.jl:7-23; the UCutoff functor (eap_chain.jl:171-192) is the bare pair sum unless cutoff_full
  const bool bare = (energy_type == 3) && !P.cutoff_full;
  t.U = bare ? t.udd : t.su + t.udd - (t.rx * P.Fx + t.rz * P.Fz);
  return t;
}

template <int T>
__global__ void __launch_bounds__(T) k_energy_cta(const EnergyArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const CtaView S = carve(smem_raw, a.n);
  const int c = a.first_chain + blockIdx.x;
  const int tid = threadIdx.x, n = a.n;
  const MonoRec* mono = a.mono + (size_t)c * n;
  if (tid == 0) *S.par = a.par[c];
  __syncthreads();
  const ChainParams& P = *S.par;
  const ChainTotals t = chain_totals<T>(mono, P, n, a.energy_type, S);
  if (tid == 0) {
    if (a.out4) {
      double* o = a.out4 + (size_t)blockIdx.x * 4;
      o[0] = t.U; o[1] = t.su; o[2] = t.udd; o[3] = t.om;
    }
    if (a.out8) {
      double* o = a.out8 + (size_t)blockIdx.x * 8;
      o[0] = t.U; o[1] = t.su; o[2] = t.udd; o[3] = t.om;
      o[4] = t.ub; o[5] = t.sp / (double)(n - 1); o[6] = t.c2; o[7] = 0.0;
    }
    if (a.obs6) {
      double* o = a.obs6 + (size_t)blockIdx.x * 6;
      o[0] = t.rx; o[1] = t.ry; o[2] = t.rz; o[3] = t.px; o[4] = t.py; o[5] = t.pz;
    }
    if (a.update_dyn) {
      ChainDyn& D = a.dyn[c];
      if (D.valid) D.drift_max = fmax(D.drift_max, fabs(D.U - t.U));
      D.U = t.U; D.su = t.su; D.Omega = t.om;
      D.r[0] = t.rx; D.r[1] = t.ry; D.r[2] = t.rz;
      D.p[0] = t.px; D.p[1] = t.py; D.p[2] = t.pz;
      if (a.rebind_gauge || !D.valid) D.log_gauge = P.gauge0 + t.om;
      D.valid = 1;
      if (a.dynx) {
        a.dynx[c].spsi = t.sp;
        a.dynx[c].scos2 = t.c2;
      }
    }
  }
}

// Non-mutating ΔU of one scripted move on one interacting chain: what the run kernels evaluate for this move, with
// the rectangle in FP32 (cta_f32.cuh) for PREC = 1.
struct DeltaArgs {
  const MonoRec* mono;
  const ChainParams* par;
  double* out;  // {dU, dOmega, clamped, dU_pairs}
  int n, energy_type, chain, idx;
  double dphi, dtheta;
};

template <int T, int PREC = 0>
__global__ void __launch_bounds__(T) k_delta_cta(const DeltaArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const CtaView S = carve(smem_raw, a.n);
  const F32View F = carve_f32(smem_raw + ((cta_smem_bytes(a.n) + 15) & ~(size_t)15), PREC ? a.n : 0, S.E);
  const int tid = threadIdx.x, n = a.n;
  const MonoRec* mono = a.mono + (size_t)a.chain * n;
  if (tid == 0) *S.par = a.par[a.chain];
  __syncthreads();
  const ChainParams& P = *S.par;
  load_chain<T>(mono, P, n, S);
  if (PREC) fill_mu_f32<Team<T / 32>>(S, F, n);
  if (tid == 0) build_proposal(P, mono[a.idx], a.idx, a.dphi, a.dtheta, 0.0, S.prop[0]);
  __syncthreads();
  const Proposal* q = &S.prop[0];
  const double dsum =
      kInv4Pi * (PREC ? cta_delta_pairs_f32<T>(S, F, n, P.b, a.idx, q->mx, q->my, q->mz, q->dnx, q->dny, q->dnz)
                      : cta_delta_pairs<T>(S, n, a.energy_type, P.b, a.idx, q->mx, q->my, q->mz, q->dnx, q->dny, q->dnz));
  if (tid == 0) {
    a.out[0] = q->du + q->drF + dsum;
    a.out[1] = q->dOmega;
    a.out[2] = (double)q->clamped;
    a.out[3] = dsum;
  }
}

// Re-initialisation (mcmc_eap_chain.jl:352-361): candidate records are in `cand`.
struct ReinitArgs {
  MonoRec* mono;
  const MonoRec* cand;
  const ChainParams* par;
  ChainDyn* dyn;
  int* replaced;  // may be null
  uint64_t seed;
  uint32_t chain_id_base;
  int n, energy_type, new_init;
};

template <int T>
__global__ void __launch_bounds__(T) k_reinit_cta(const ReinitArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const CtaView S = carve(smem_raw, a.n);
  const int c = blockIdx.x, tid = threadIdx.x, n = a.n;
  const MonoRec* cand = a.cand + (size_t)c * n;
  MonoRec* mono = a.mono + (size_t)c * n;
  if (tid == 0) *S.par = a.par[c];
  __syncthreads();
  const ChainParams& P = *S.par;
  const ChainTotals t = chain_totals<T>(cand, P, n, a.energy_type, S);
  const ChainDyn& D0 = a.dyn[c];
  const uint4 w = philox_at(a.seed, a.chain_id_base + (uint32_t)c, (uint32_t)a.new_init, SUB_REINIT, 0);
  const double eps = u53(w.x, w.y);
  // metropolis_acc (acceptance.jl:1-3) with Π sinθ written as exp(Σ log sinθ)
  const bool take = P.force_init || (eps <= exp(-(t.U - D0.U) * P.inv_kT + (t.om - D0.Omega)));
  __syncthreads();
  if (take)
    for (int i = tid; i < n; i += T) mono[i] = cand[i];
  if (tid == 0) {
    ChainDyn& D = a.dyn[c];
    if (take) {
      D.U = t.U; D.su = t.su; D.Omega = t.om;
      D.r[0] = t.rx; D.r[1] = t.ry; D.r[2] = t.rz;
      D.p[0] = t.px; D.p[1] = t.py; D.p[2] = t.pz;
    }
    D.init = a.new_init;
    D.step = 0;
    if (a.replaced) a.replaced[c] = take ? 1 : 0;
  }
}

}  // namespace pmc
