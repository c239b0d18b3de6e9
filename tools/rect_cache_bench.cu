// Microbenchmark for VERDICT r01 "next" #5 (developer tool, not product code): would an old-pair-energy cache in HBM beat
// the rectangle loop that recomputes the old term?
//
// The product evaluates, per changed pair, the old and the new energy: 43 FP64 instructions (rect_pair, cta_kernels.cuh).
// With f_ij of the CURRENT state cached in HBM a trial reads the old term (8 B per pair) and evaluates only the new one
// (24 FP64 instructions); an accepted trial must write the new terms back, which means evaluating them a second time
// (they cannot be kept on chip: 44 000 per trial at n=512) and storing 8 B per pair.
//
// Layout tried: one n×n matrix per chain, g[j][i] (row = the larger monomer index j, contiguous in the smaller index i),
// heads always on the lanes so that a warp's loads / stores are contiguous 256 B pieces of a row; 2 MB per chain at n=512
// (8.6 GB for the 4096 chains of C2).  Kernels: the product loop (baseline), the cached loop on the reject path
// (read old, evaluate new) and on the accept path (evaluate new again, store).  Throughput of a Markov chain with
// acceptance rate AR = reject-path time + AR × accept-path time.
//
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o tools/rect_cache_bench tools/rect_cache_bench.cu
#include <cstdio>
#include <cmath>
#include <cuda_runtime.h>
#include "../polymer-stats_b200/csrc/cta_kernels.cuh"
using namespace pmc;

__device__ __forceinline__ void fill_chain(const CtaView& S, int n, int T) {
  for (int i = threadIdx.x; i < n; i += T) {
    const double t = 0.37 * i + 0.01 * blockIdx.x;
    S.sx[i] = 0.9 * i * 0.3 + sin(t); S.sy[i] = cos(1.3 * t) * 3.0; S.sz[i] = 0.5 * i * 0.2 + sin(0.7 * t);
    S.mx[i] = sin(t) * 0.3; S.my[i] = cos(t) * 0.3; S.mz[i] = 1.0 + 0.1 * sin(2 * t);
  }
  __syncthreads();
}

__device__ __forceinline__ int trial_idx(int r, int n) { return (int)((r * 2654435761u + blockIdx.x * 40503u) % (unsigned)n); }

// new term only: 4π f(μ_L, μ_B, r − D), same operation order as the new half of rect_pair
__device__ __forceinline__ double new_term(const LaneItem& it, double bx, double by, double bz, double ux, double uy,
                                           double uz, double e, double Dx, double Dy, double Dz) {
  const double qx = (it.x - bx) - Dx, qy = (it.y - by) - Dy, qz = (it.z - bz) - Dz;
  const double mm = fma(it.az, uz, fma(it.ay, uy, it.ax * ux));
  const double q2 = fma(qz, qz, fma(qy, qy, qx * qx));
  const double a3n = fma(it.tz, qz, fma(it.ty, qy, it.tx * qx));
  const double bn = fma(uz, qz, fma(uy, qy, ux * qx));
  const double yn = rsqrt_fast(q2);
  const double yn2 = yn * yn;
  const double tn = fma(a3n * bn, yn2, mm);
  return tn * (yn2 * yn);
}

// MODE 0: product loop.  MODE 1: cached, reject path (read old, evaluate new).  MODE 2: cached, accept path (evaluate
// new, store it).  PF: rows of the cache in flight per warp (software prefetch depth).
template <int T, int MINB, int MODE, int PF>
__global__ void __launch_bounds__(T, MINB) k_rect(double* out, double* __restrict__ cache, int n, int reps) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const CtaView S = carve(smem_raw, n);
  fill_chain(S, n, T);
  double* g = cache + (size_t)blockIdx.x * n * n;
  constexpr int W = T / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  using TEAM = Team<W>;
  double acc = 0.0;
  for (int r = 0; r < reps; ++r) {
    const int idx = trial_idx(r, n);
    const double Dx = 0.1 + 1e-3 * (r & 7), Dy = -0.2, Dz = 0.15;
    const int H = idx, Tl = n - 1 - idx;
    if (H <= 0 || Tl <= 0) continue;
    for (int k = threadIdx.x; k < Tl; k += T)
      S.E[idx + 1 + k] = fma(S.mz[idx + 1 + k], Dz, fma(S.my[idx + 1 + k], Dy, S.mx[idx + 1 + k] * Dx));
    __syncthreads();
    if (MODE == 0) {
      acc += rect_sum<TEAM, 2, false, false>(S, 0, H, idx + 1, Tl, Dx, Dy, Dz);
    } else {
      // heads on the lanes (64 per pass, two per lane), tails broadcast; the (pass × tail) space split over the warps
      const int G2 = (H + 63) >> 6;
      const int U = G2 * Tl;
      int u = (int)(((long long)U * warp) / W);
      const int u1 = (int)(((long long)U * (warp + 1)) / W);
      while (u < u1) {
        const int gq = u / Tl;
        int k = u - gq * Tl;
        const int l0 = gq * 64 + lane, l1 = l0 + 32;
        const bool v0 = l0 < H, v1 = l1 < H;
        const LaneItem i0 = load_lane_item(S, min(l0, H - 1), Dx, Dy, Dz);
        const LaneItem i1 = load_lane_item(S, min(l1, H - 1), Dx, Dy, Dz);
        const int kend = min(Tl, k + (u1 - u));
        u += kend - k;
        double a0 = 0.0, a1 = 0.0;
        if (MODE == 1) {
          double o0[PF], o1[PF];
#pragma unroll
          for (int p = 0; p < PF; ++p) {   // prefetch PF rows
            const int kk = min(k + p, Tl - 1);
            const double* row = g + (size_t)(idx + 1 + kk) * n;
            o0[p] = v0 ? __ldcs(row + l0) : 0.0;
            o1[p] = v1 ? __ldcs(row + l1) : 0.0;
          }
          for (; k < kend; k += PF) {
#pragma unroll
            for (int p = 0; p < PF; ++p) {
              const int kk = k + p;
              if (kk < kend) {
                const int B = idx + 1 + kk;
                const double bx = S.sx[B], by = S.sy[B], bz = S.sz[B], ux = S.mx[B], uy = S.my[B], uz = S.mz[B], e = S.E[B];
                a0 += new_term(i0, bx, by, bz, ux, uy, uz, e, Dx, Dy, Dz) - o0[p];
                a1 += new_term(i1, bx, by, bz, ux, uy, uz, e, Dx, Dy, Dz) - o1[p];
              }
              const int kn = min(kk + PF, Tl - 1);   // refill the slot
              const double* row = g + (size_t)(idx + 1 + kn) * n;
              o0[p] = v0 ? __ldcs(row + l0) : 0.0;
              o1[p] = v1 ? __ldcs(row + l1) : 0.0;
            }
          }
        } else {
          for (; k < kend; ++k) {
            const int B = idx + 1 + k;
            const double bx = S.sx[B], by = S.sy[B], bz = S.sz[B], ux = S.mx[B], uy = S.my[B], uz = S.mz[B], e = S.E[B];
            double* row = g + (size_t)B * n;
            const double f0 = new_term(i0, bx, by, bz, ux, uy, uz, e, Dx, Dy, Dz);
            const double f1 = new_term(i1, bx, by, bz, ux, uy, uz, e, Dx, Dy, Dz);
            if (v0) __stcs(row + l0, f0);
            if (v1) __stcs(row + l1, f1);
            a0 += f0; a1 += f1;
          }
        }
        acc += (v0 ? a0 : 0.0) + (v1 ? a1 : 0.0);
      }
    }
    __syncthreads();
  }
  out[blockIdx.x * T + threadIdx.x] = acc;
}

template <int MODE, int PF>
static float run(double* d, double* cache, int n, int blocks, int reps, size_t smem) {
  constexpr int T = 128, MINB = 4;
  cudaFuncSetAttribute(k_rect<T, MINB, MODE, PF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_rect<T, MINB, MODE, PF><<<blocks, T, smem>>>(d, cache, n, 4);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  float best = 1e30f;
  for (int it = 0; it < 3; ++it) {
    cudaEventRecord(e0);
    k_rect<T, MINB, MODE, PF><<<blocks, T, smem>>>(d, cache, n, reps);
    cudaEventRecord(e1); cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    best = fminf(best, ms);
  }
  return best;
}

int main() {
  const int n = 512, T = 128, blocks = 148 * 4 * 4, reps = 100;
  const size_t smem = cta_smem_bytes(n);
  double* d; cudaMalloc(&d, sizeof(double) * blocks * T);
  double* cache;
  const size_t cbytes = (size_t)blocks * n * n * sizeof(double);
  if (cudaMalloc(&cache, cbytes) != cudaSuccess) { printf("cannot allocate the %.1f GB cache\n", cbytes / 1e9); return 1; }
  cudaMemset(cache, 0, cbytes);
  double pairs = 0, lane_pairs = 0;
  for (int b = 0; b < blocks; ++b)
    for (int r = 0; r < reps; ++r) {
      const int idx = (int)((r * 2654435761u + b * 40503u) % (unsigned)n);
      pairs += (double)idx * (n - 1 - idx);
      lane_pairs += (double)((idx + 63) / 64 * 64) * (n - 1 - idx);
    }
  printf("n=%d, %d chains, %d trials each: %.3e rectangle pairs per launch; cache %.1f GB (n*n doubles per chain)\n", n, blocks, reps,
         pairs, cbytes / 1e9);
  printf("heads-on-lanes only (needed for contiguous cache rows) evaluates %.3fx the pairs of the product's lane-side choice\n",
         lane_pairs / pairs);
  const float t0 = run<0, 1>(d, cache, n, blocks, reps, smem);
  printf("product loop (old + new, 43 FP64 instr/pair):          %8.3f ms  %7.1f G pairs/s\n", t0, pairs / t0 / 1e6);
  const float t1a = run<1, 2>(d, cache, n, blocks, reps, smem);
  printf("cached, reject path, 2 rows in flight per warp:        %8.3f ms  %7.1f G pairs/s  %6.2f TB/s read\n", t1a, pairs / t1a / 1e6, pairs * 8 / t1a / 1e9);
  const float t1b = run<1, 4>(d, cache, n, blocks, reps, smem);
  printf("cached, reject path, 4 rows in flight per warp:        %8.3f ms  %7.1f G pairs/s  %6.2f TB/s read\n", t1b, pairs / t1b / 1e6, pairs * 8 / t1b / 1e9);
  const float t1c = run<1, 8>(d, cache, n, blocks, reps, smem);
  printf("cached, reject path, 8 rows in flight per warp:        %8.3f ms  %7.1f G pairs/s  %6.2f TB/s read\n", t1c, pairs / t1c / 1e6, pairs * 8 / t1c / 1e9);
  const float t2 = run<2, 1>(d, cache, n, blocks, reps, smem);
  printf("cached, accept path (evaluate new again + store):      %8.3f ms  %7.1f G pairs/s  %6.2f TB/s written\n", t2, pairs / t2 / 1e6, pairs * 8 / t2 / 1e9);
  const float t1 = fminf(t1a, fminf(t1b, t1c));
  for (double ar : {0.2, 0.3, 0.4}) {
    const double tc = t1 + ar * t2;
    printf("Markov chain at acceptance rate %.1f: cached %.3f ms vs product %.3f ms  ->  %.2fx\n", ar, tc, (double)t0, t0 / tc);
  }
  cudaError_t err = cudaDeviceSynchronize();
  if (err != cudaSuccess) { printf("CUDA error: %s\n", cudaGetErrorString(err)); return 1; }
  return 0;
}
