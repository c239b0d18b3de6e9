// exchange.cu — launch helpers of the replica-exchange kernels (exchange.cuh).
#include "handle.h"
#include "exchange.cuh"

namespace {

// Rows of one chunk of a tempering run, [chains][rows][cols], placed at row `row0` of [chains][rows_total][cols].
__global__ void k_place_rows(double* __restrict__ dst, const double* __restrict__ src, long long nchains, long long rows,
                             long long rows_total, long long row0, int cols) {
  const long long per = rows * cols;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < nchains * per;
       g += (long long)gridDim.x * blockDim.x) {
    const long long c = g / per, k = g - c * per;
    dst[(c * rows_total + row0) * cols + k] = src[g];
  }
}

}  // namespace

int launch_exchange(pmc_handle* h, const pmc::ExchangeArgs& a, int64_t npairs) {
  if (npairs <= 0) return PMC_OK;
  k_exchange<128><<<(unsigned)npairs, 128, 0, h->stream>>>(a);
  ++h->launches;
  PMC_CU(cudaGetLastError());
  return PMC_OK;
}

int launch_place_rows(pmc_handle* h, double* dst, const double* src, int64_t rows, int64_t rows_total, int64_t row0,
                      int cols) {
  if (rows <= 0) return PMC_OK;
  const long long total = (long long)h->nchains * rows * cols;
  const int tb = 256;
  const long long blocks = std::min<long long>((total + tb - 1) / tb, (long long)h->sm_count * 16);
  k_place_rows<<<(unsigned)blocks, tb, 0, h->stream>>>(dst, src, (long long)h->nchains, (long long)rows,
                                                       (long long)rows_total, (long long)row0, cols);
  ++h->launches;
  PMC_CU(cudaGetLastError());
  return PMC_OK;
}
