// Microbenchmark of the rectangle loop (rect_sum, cta_kernels.cuh) alone, and accuracy of rsqrt_fast under
// -DPMC_RSQRT_VARIANT=0|1, and of the two forms of |r'|² under -DRECT_Q2=0|1 (developer tool, not product code;
// the Q2 form keeps the broadcast side at most n/2 long: both builds time the trials whose tails are that short).
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -DPMC_RSQRT_VARIANT=1 -o tools/rect_bench_v1 tools/rect_bench.cu
#include <cstdio>
#include <cmath>
#include <cuda_runtime.h>
#include "../polymer-stats_b200/csrc/cta_kernels.cuh"
using namespace pmc;
#ifndef RECT_Q2
#define RECT_Q2 1   // 0: r' formed and squared (the form before the projections)
#endif

template <int T, int MINB>
__global__ void __launch_bounds__(T, MINB) k_rect(double* out, int n, int reps) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const CtaView S = carve(smem_raw, n);
  // a random-walk-like chain
  for (int i = threadIdx.x; i < n; i += T) {
    const double t = 0.37 * i + 0.01 * blockIdx.x;
    S.sx[i] = 0.9 * i * 0.3 + sin(t); S.sy[i] = cos(1.3 * t) * 3.0; S.sz[i] = 0.5 * i * 0.2 + sin(0.7 * t);
    S.mx[i] = sin(t) * 0.3; S.my[i] = cos(t) * 0.3; S.mz[i] = 1.0 + 0.1 * sin(2 * t);
  }
  __syncthreads();
  double acc = 0.0;
  using TEAM = Team<T / 32>;
  for (int r = 0; r < reps; ++r) {
    const int idx = (int)((r * 2654435761u + blockIdx.x * 40503u) % (unsigned)n);
    const double Dx = 0.1 + 1e-3 * (r & 7), Dy = -0.2, Dz = 0.15;
    const int H = idx, Tl = n - 1 - idx;
    if (H > 0 && Tl > 0) {
      // heads on the lanes: the tails' {eB, 2p_B} take 2·Tl doubles of S.E in the Q2 form
      if (2 * Tl > n) continue;
      const double px = S.sx[idx], py = S.sy[idx], pz = S.sz[idx];
      for (int k = threadIdx.x; k < Tl; k += T) rect_prepass_item<RECT_Q2>(S, idx + 1, k, px, py, pz, Dx, Dy, Dz);
      __syncthreads();
      acc += rect_sum<TEAM, 2, false, false, RECT_Q2>(S, 0, H, idx + 1, Tl, Dx, Dy, Dz, 0.0, idx);
      __syncthreads();
    }
  }
  out[blockIdx.x * T + threadIdx.x] = acc;
}

__global__ void k_acc(double* out, int n) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  double maxerr = 0;
  for (int i = t; i < n; i += gridDim.x * blockDim.x) {
    const double m = 1.0 + (double)(i % 1000003) / 1000003.0 * 3.0;
    const double x = ldexp(m, (i % 61) - 30);
    const double y = rsqrt_fast(x);
    const double yy = y * y, yy_lo = fma(y, y, -yy);
    const double r = fma(-x, yy, 1.0) - x * yy_lo;
    maxerr = fmax(maxerr, fabs(r) * 0.5);
  }
  out[t] = maxerr;
}

int main() {
  const int n = 512, T = 128, MINB = 4, blocks = 148 * 4 * 4, reps = 200;
  const size_t smem = cta_smem_bytes(n);
  cudaFuncSetAttribute(k_rect<T, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  double* d; cudaMalloc(&d, sizeof(double) * blocks * T);
  k_rect<T, MINB><<<blocks, T, smem>>>(d, n, 10);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  float best = 1e30f;
  for (int it = 0; it < 3; ++it) {
    cudaEventRecord(e0);
    k_rect<T, MINB><<<blocks, T, smem>>>(d, n, reps);
    cudaEventRecord(e1); cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    best = fminf(best, ms);
  }
  // pairs: Σ over blocks and reps of idx(n-1-idx), same sequence as the kernel
  double pairs = 0;
  for (int b = 0; b < blocks; ++b)
    for (int r = 0; r < reps; ++r) {
      const int idx = (int)((r * 2654435761u + b * 40503u) % (unsigned)n);
      if (2 * (n - 1 - idx) > n) continue;
      pairs += (double)idx * (n - 1 - idx);
    }
  static double h[148 * 4 * 4 * 128];
  cudaMemcpy(h, d, sizeof(double) * blocks * T, cudaMemcpyDeviceToHost);
  double cs = 0; for (int i = 0; i < blocks * T; ++i) cs += h[i];
  printf("q2 %d variant %d: rect loop %.3f ms, %.3e pairs -> %.2f G pairs/s = %.2f TFLOP/s algorithmic (68 flop/pair), checksum %.15e\n",
         RECT_Q2, PMC_RSQRT_VARIANT, best, pairs, pairs / best / 1e6, pairs * 68 / best / 1e9, cs);
  const int TT = 256 * 148;
  double* e; cudaMalloc(&e, TT * sizeof(double));
  k_acc<<<148, 256>>>(e, 200000000);
  static double he[256 * 148]; cudaMemcpy(he, e, sizeof(he), cudaMemcpyDeviceToHost);
  double m = 0; for (int i = 0; i < TT; ++i) m = fmax(m, he[i]);
  printf("variant %d: max relative error of rsqrt_fast = %.3e (%.1f ulp)\n", PMC_RSQRT_VARIANT, m, m / 1.11e-16);
  cudaError_t err = cudaDeviceSynchronize();
  if (err != cudaSuccess) { printf("CUDA error: %s\n", cudaGetErrorString(err)); return 1; }
  return 0;
}
