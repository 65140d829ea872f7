// Block reduction and the energy of one chain on CSR couplings, shared by the chromatic sweep kernel
// (sparse_gibbs.cu) and the Houdayer move on sparse couplings (sparse_houdayer.cu).  block_sum_d adds the warps' partial
// sums in warp order, so the value depends on blockDim: a kernel that must report the sweep kernel's energies bit for
// bit launches with the sweep kernel's thread count for that N (sparse_threads).
#pragma once
#include "common.cuh"

namespace {

// threads per CTA of the sparse kernels: one per four sites, whole warps, 32 .. 256
inline int sparse_threads(int N) {
  int threads = (N + 3) / 4;
  threads = (threads + 31) / 32 * 32;
  return threads < 32 ? 32 : (threads > 256 ? 256 : threads);
}

__device__ __forceinline__ double block_sum_d(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < nw; ++w) t += red[w];
  return t;
}

// E = -1/2 s^T J s - b^T s (tsu/gibbs.py:215-236) of the bits s [N] (any nonzero byte is a 1), for every thread of
// the block; bias may be nullptr.  The pointers and N are taken by reference so that a caller passing fields of its
// kernel parameters reads them where this function reads them: sparse_gibbs_kernel compiles to the same SASS as when
// it read them through its SparseParams.
__device__ double sparse_energy(const int32_t* const& rowptr, const int32_t* const& col, const double* const& val,
                                const double* const& bias, const int& N, const uint8_t* s, double* red) {
  double acc = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    if (!s[i]) continue;
    double h = 0.0;
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k)
      if (s[col[k]]) h += val[k];
    acc += -0.5 * h - (bias ? bias[i] : 0.0);
  }
  return block_sum_d(acc, red);
}

}  // namespace
