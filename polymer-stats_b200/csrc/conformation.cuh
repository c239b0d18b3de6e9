// conformation.cuh — running sums of the shape of every chain (DESIGN.md §13): gyration tensor, bond-orientation
// correlation, per-bond orientation profile and extension histogram, one sample of the current configuration per call.
//
// Like k_exchange it runs between two launches of the run kernels and reads only the records and the chain constants.
// Row of one chain, cols = 8 + 3n + B doubles of sums over samples:
//   0: 1 · 1–6: S_xx S_yy S_zz S_xy S_xz S_yz of S = (1/n) Σ_i (x_i − x̄)(x_i − x̄)ᵀ · 7: (tr S)²
//   8 + s: C_s = Σ_{i=0}^{n−1−s} n̂_i·n̂_{i+s} · 8 + n + i: n̂z_i · 8 + 2n + i: n̂z_i² · 8 + 3n + k: histogram of
//   ζ = r_z / (n b) on [−1, 1] in B bins.
#pragma once

#include "cta_kernels.cuh"

namespace pmc {

constexpr int kConfMaxBins = 1 << 16;   // the finest extension histogram pmc_set_conformation accepts

struct ConfArgs {
  const MonoRec* mono;
  const ChainParams* par;
  double* sums;   // [chains][cols]
  long long cols;
  int n, bins;
};

// x, y, z (3n) | n̂ (3n; load_chain stages μ there first) | block-scan partials | ChainParams.  Six n doubles: at the
// longest chain pmc_create accepts (n ≈ 4100) that is ≈ 197 KB.
__host__ __device__ inline size_t conformation_smem_bytes(int n) {
  return (size_t)(6 * n + kPartDoubles) * sizeof(double) + sizeof(ChainParams);
}

// One CTA per chain.  Positions come from load_chain at the block size of the energy kernels, so x and r_z are the
// bits chain_totals computes (the histogram bin agrees with pmc_observables).  Every sum has a fixed order and every
// column has one writer: repeated calls are bit-identical.  The sample count, the profile and the histogram are one
// uncontracted addition per sample, so a CPU restatement reproduces them bit for bit.
template <int T>
__global__ void __launch_bounds__(T) k_conformation(const ConfArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n = a.n, tid = threadIdx.x;
  double* d = reinterpret_cast<double*>(smem_raw);
  CtaView S{};
  S.sx = d; S.sy = d + n; S.sz = d + 2 * n;
  S.mx = d + 3 * n; S.my = d + 4 * n; S.mz = d + 5 * n;
  S.part = d + 6 * n;
  ChainParams* Ps = reinterpret_cast<ChainParams*>(S.part + kPartDoubles);
  const MonoRec* mono = a.mono + (size_t)blockIdx.x * n;
  double* row = a.sums + (size_t)blockIdx.x * (size_t)a.cols;
  if (tid == 0) *Ps = a.par[blockIdx.x];
  __syncthreads();
  const ChainParams& P = *Ps;
  load_chain<T>(mono, P, n, S);
  double* ux = S.mx;
  double* uy = S.my;
  double* uz = S.mz;
  double lx = 0, ly = 0, lz = 0;
  for (int i = tid; i < n; i += T) {
    const MonoRec r = mono[i];
    ux[i] = r.nx; uy[i] = r.ny; uz[i] = r.nz;
    row[8 + n + i] = __dadd_rn(row[8 + n + i], r.nz);
    row[8 + 2 * n + i] = __dadd_rn(row[8 + 2 * n + i], __dmul_rn(r.nz, r.nz));
    lx += S.sx[i]; ly += S.sy[i]; lz += S.sz[i];
  }
  const double inv_n = __drcp_rn((double)n);
  const double cx = block_sum<T>(lx, S.part) * inv_n, cy = block_sum<T>(ly, S.part) * inv_n,
               cz = block_sum<T>(lz, S.part) * inv_n;
  double q[6] = {0, 0, 0, 0, 0, 0};
  for (int i = tid; i < n; i += T) {
    const double dx = S.sx[i] - cx, dy = S.sy[i] - cy, dz = S.sz[i] - cz;
    q[0] += dx * dx; q[1] += dy * dy; q[2] += dz * dz;
    q[3] += dx * dy; q[4] += dx * dz; q[5] += dy * dz;
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) q[k] = block_sum<T>(q[k], S.part) * inv_n;   // its barriers also publish n̂
  if (tid == 0) {
    row[0] = __dadd_rn(row[0], 1.0);
#pragma unroll
    for (int k = 0; k < 6; ++k) row[1 + k] += q[k];
    const double tr = q[0] + q[1] + q[2];
    row[7] += tr * tr;
    if (a.bins > 0) {
      const double rz = S.sz[n - 1] + 0.5 * P.b * mono[n - 1].nz;   // chain_totals' end-to-end z
      const double zeta = __ddiv_rn(rz, __dmul_rn((double)n, P.b));
      const double u = __dmul_rn(__dmul_rn(__dadd_rn(zeta, 1.0), (double)a.bins), 0.5);
      const int k = u < 1.0 ? 0 : u >= (double)(a.bins - 1) ? a.bins - 1 : (int)floor(u);
      row[8 + 3 * n + k] = __dadd_rn(row[8 + 3 * n + k], 1.0);
    }
  }
  // C_s: thread p takes the lags p and n − 1 − p, n + 1 dot products in all (the middle lag of an odd n once)
  for (int p = tid; p < (n + 1) / 2; p += T) {
    const int s1 = n - 1 - p;
    double c0 = 0.0;
    for (int i = 0; i + p < n; ++i) c0 += ux[i] * ux[i + p] + uy[i] * uy[i + p] + uz[i] * uz[i + p];
    row[8 + p] += c0;
    if (s1 != p) {
      double c1 = 0.0;
      for (int i = 0; i + s1 < n; ++i) c1 += ux[i] * ux[i + s1] + uy[i] * uy[i + s1] + uz[i] * uz[i + s1];
      row[8 + s1] += c1;
    }
  }
}

}  // namespace pmc
