// Population-annealing steps on the chain states of any back end (tsu_population_resample, tsu_population_moments):
// rows of row_bytes bytes with a float64 energy each, resampled by the kernels the lattice uses (population.cuh).

#include "common.cuh"
#include "population.cuh"

namespace {

// the order key of each population's lowest energy into Q.min_key[p] (atomicMin: the caller sets it to ~0 first).
// Grid (x, n_pop): blockIdx.x strides over a population.
__global__ void __launch_bounds__(kPaThreads) pa_min_kernel(const double* __restrict__ energy, PopParams Q) {
  const int p = blockIdx.y;
  unsigned long long key = ~0ull;
  for (int j = blockIdx.x * kPaThreads + threadIdx.x; j < Q.rp; j += gridDim.x * kPaThreads)
    key = min(key, order_key(energy[(size_t)p * Q.rp + j]));
  __shared__ unsigned long long part[kPaThreads / 32];
  key = warp_min(key);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = key;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kPaThreads / 32; ++w) key = min(key, part[w]);
    atomicMin(Q.min_key + p, key);
  }
}

// One block per population: (sum E, sum E^2) in float64.  Thread t sums chains t, t + 256, ... in order, then the
// warps reduce by a fixed butterfly and thread 0 adds the warp totals in order: the bits depend only on the
// population's energies.
constexpr int kMomentThreads = 256;

__global__ void __launch_bounds__(kMomentThreads) pa_moments_kernel(const double* __restrict__ energy, int rp,
                                                                   double* __restrict__ moments) {
  const double* e = energy + (size_t)blockIdx.x * rp;
  double s1 = 0.0, s2 = 0.0;
  for (int j = threadIdx.x; j < rp; j += kMomentThreads) {
    const double v = e[j];
    s1 = __dadd_rn(s1, v);
    s2 = __dadd_rn(s2, __dmul_rn(v, v));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s1 = __dadd_rn(s1, __shfl_xor_sync(0xffffffffu, s1, o));
    s2 = __dadd_rn(s2, __shfl_xor_sync(0xffffffffu, s2, o));
  }
  __shared__ double part[2][kMomentThreads / 32];
  if ((threadIdx.x & 31) == 0) {
    part[0][threadIdx.x >> 5] = s1;
    part[1][threadIdx.x >> 5] = s2;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kMomentThreads / 32; ++w) {
      s1 = __dadd_rn(s1, part[0][w]);
      s2 = __dadd_rn(s2, part[1][w]);
    }
    moments[2 * (size_t)blockIdx.x] = s1;
    moments[2 * (size_t)blockIdx.x + 1] = s2;
  }
}

bool populations_ok(int n_chains, int n_populations) {
  return n_chains >= 1 && n_populations >= 1 && n_populations <= 65535 && n_chains % n_populations == 0;
}

}  // namespace

extern "C" {

int tsu_population_resample(const void* d_state, void* d_state_out, const int32_t* d_family, int32_t* d_family_out,
                            const double* d_energy, const double* d_dbeta, int n_chains, int n_populations,
                            long long row_bytes, uint64_t seed, uint32_t sweep, uint32_t chain0,
                            unsigned long long* d_weight_sum, double* d_energy_ref, void* d_work, size_t work_bytes,
                            uintptr_t stream) {
  TSU_CHECK_ARG(d_state && d_state_out && d_family && d_family_out && d_energy && d_dbeta && d_weight_sum &&
                d_energy_ref && d_work);
  TSU_CHECK_ARG(populations_ok(n_chains, n_populations) && row_bytes >= 1);
  TSU_CHECK_ARG(d_state != d_state_out && d_family != d_family_out);
  TSU_CHECK_ARG((reinterpret_cast<uintptr_t>(d_work) & 7) == 0 &&
                work_bytes >= (size_t)tsu_ising2d_population_work_bytes(n_chains, n_populations));
  const PopParams Q = pop_params(d_work, n_chains, n_populations);
  cudaStream_t st = tsu_stream(stream);
  const cudaError_t e = cudaMemsetAsync(Q.min_key, 0xff, sizeof(unsigned long long) * n_populations, st);
  if (e != cudaSuccess) return (int)e;
  long long bx = (Q.rp + kPaThreads - 1) / kPaThreads;
  const long long cap = (148LL * 8 + n_populations - 1) / n_populations;  // about 8 CTAs per SM in total
  if (bx > cap) bx = cap;
  pa_min_kernel<<<dim3((unsigned)bx, (unsigned)n_populations), kPaThreads, 0, st>>>(d_energy, Q);
  // 16-byte rows at 16-byte addresses copy as uint4, anything else byte by byte
  const bool vec = row_bytes % 16 == 0 &&
                   ((reinterpret_cast<uintptr_t>(d_state) | reinterpret_cast<uintptr_t>(d_state_out)) & 15) == 0;
  if (vec)
    return launch_pa_resample(Q, d_energy, d_dbeta, seed, sweep, chain0, d_weight_sum, d_energy_ref,
                              static_cast<const uint4*>(d_state), static_cast<uint4*>(d_state_out), d_family,
                              d_family_out, row_bytes / 16, st);
  return launch_pa_resample(Q, d_energy, d_dbeta, seed, sweep, chain0, d_weight_sum, d_energy_ref,
                            static_cast<const uint8_t*>(d_state), static_cast<uint8_t*>(d_state_out), d_family,
                            d_family_out, row_bytes, st);
}

int tsu_population_moments(const double* d_energy, int n_chains, int n_populations, double* d_moments,
                           uintptr_t stream) {
  TSU_CHECK_ARG(d_energy && d_moments && populations_ok(n_chains, n_populations));
  pa_moments_kernel<<<n_populations, kMomentThreads, 0, tsu_stream(stream)>>>(d_energy, n_chains / n_populations,
                                                                              d_moments);
  TSU_RETURN_LAUNCH_STATUS();
}

}  // extern "C"
