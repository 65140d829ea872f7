// Chromatic heat-bath Gibbs sampler for SPARSE couplings (sm_100a): chains of spins (IsingChain,
// tsu/models/ising.py:265-304), irregular graphs, MAX-CUT instances - anything whose coupling matrix is mostly
// zeros.  The reference walks the N x N matrix row by row whatever its content (gibbs.py:79-100: one np.dot of length
// N per spin); here a site visit costs its degree.
//
// Sites are grouped into colour classes (greedy colouring on the host: no two coupled sites share a colour).  A sweep
// visits the classes in order; the sites of one class do not interact, so a thread block updates them concurrently and
// the result equals a sequential sweep (gibbs.py:153-160) that visits the sites class by class - which is what the
// reference computes with update_order="random" when the permutation is that order (the parity goldens do exactly
// this).  Rule per visit, as in the reference: h_i = sum_j J_ij s_j + b_i including a self term (gibbs.py:96-99),
// p = sigmoid(h_i / T) with the +-20 clamp (gibbs.py:61-77), new bit = 1 iff u < p (gibbs.py:126).
//
// One CTA per chain; the chain's bits live in shared memory (one byte per site) for all sweeps of the call;
// CSR rows stream from L2.  The uniform of (site, chain, sweep) is the dense sampler's
// (Philox counter = (site, chain, sweep, 'DENS'), 53 bits), so the dense kernel run in the same visiting order gives
// the same bits.

#include "common.cuh"
#include "philox.cuh"
#include "sparse_energy.cuh"

namespace {

struct SparseParams {
  const int32_t* rowptr;   // [N + 1]
  const int32_t* col;      // [nnz] column indices, ascending within a row
  const double* val;       // [nnz]
  const double* bias;      // [N] or nullptr
  const int32_t* colour_ptr;    // [n_colours + 1] offsets into colour_sites
  const int32_t* colour_sites;  // [N] sites grouped by colour (the visiting order of a sweep)
  uint8_t* state;          // [n_chains][N]
  const double* T_chain;   // [n_chains] or nullptr
  const double* T_sweep;   // [total sweeps] or nullptr
  const double* uniforms;  // parity mode: [sweep][chain][N] in visiting order, or nullptr
  uint8_t* samples;        // [n_samples][n_chains][N] or nullptr
  double* energy;          // [n_chains] or nullptr
  uint8_t* best_state;     // [n_chains][N] (track_best)
  double* best_energy;     // [n_chains]
  double T;
  int n_chains, N, n_colours;
  int n_burnin, n_samples, sweeps_per_sample, track_best;
  uint32_t k0, k1, sweep0, chain0;
};

__device__ __forceinline__ double sigmoid_clamped_d(double x) {  // tsu/gibbs.py:61-77
  if (x > 20.0) return 1.0;
  if (x < -20.0) return 0.0;
  return 1.0 / (1.0 + exp(-x));
}

__global__ void __launch_bounds__(256) sparse_gibbs_kernel(SparseParams P) {
  extern __shared__ unsigned char smem_s[];
  __shared__ double red[32];
  uint8_t* s = smem_s;
  const int N = P.N, chain = blockIdx.x;
  uint8_t* gstate = P.state + (size_t)chain * N;
  for (int j = threadIdx.x; j < N; j += blockDim.x) s[j] = gstate[j] ? 1 : 0;
  __syncthreads();

  double best_e = 0.0;
  if (P.track_best) {
    best_e = sparse_energy(P.rowptr, P.col, P.val, P.bias, P.N, s, red);
    for (int j = threadIdx.x; j < N; j += blockDim.x) P.best_state[(size_t)chain * N + j] = s[j];
  }
  const int total = P.n_burnin + P.n_samples * P.sweeps_per_sample;
  int next_sample_at = P.n_burnin + P.sweeps_per_sample;
  int sample_idx = 0;
  for (int sw = 0; sw < total; ++sw) {
    const double T = P.T_chain ? P.T_chain[chain] : (P.T_sweep ? P.T_sweep[sw] : P.T);
    const double* u_sweep = P.uniforms ? P.uniforms + ((size_t)sw * P.n_chains + chain) * N : nullptr;
    for (int c = 0; c < P.n_colours; ++c) {
      const int begin = P.colour_ptr[c], end = P.colour_ptr[c + 1];
      for (int idx = begin + threadIdx.x; idx < end; idx += blockDim.x) {
        const int i = P.colour_sites[idx];
        double h = 0.0;
        for (int k = P.rowptr[i]; k < P.rowptr[i + 1]; ++k)
          if (s[P.col[k]]) h += P.val[k];   // ascending column order; includes the self term if J_ii is stored
        if (P.bias) h += P.bias[i];
        double u;
        if (u_sweep) {
          u = u_sweep[idx];
        } else {
          const tsu_u32x4 o = tsu_philox4x32_10((uint32_t)i, P.chain0 + (uint32_t)chain, P.sweep0 + (uint32_t)sw,
                                                TSU_STREAM_DENSE, P.k0, P.k1);
          const unsigned long long m = (((unsigned long long)o.x << 32) | o.y) >> 11;
          u = (double)m * (1.0 / 9007199254740992.0);
        }
        s[i] = (u < sigmoid_clamped_d(h / T)) ? 1 : 0;   // nobody else of this colour reads s[i]
      }
      __syncthreads();
    }
    if (P.track_best) {  // gibbs.py:387-391
      const double e = sparse_energy(P.rowptr, P.col, P.val, P.bias, P.N, s, red);
      if (e < best_e) {
        best_e = e;
        for (int j = threadIdx.x; j < N; j += blockDim.x) P.best_state[(size_t)chain * N + j] = s[j];
      }
      __syncthreads();
    }
    if (sw + 1 == next_sample_at) {
      if (P.samples && sample_idx < P.n_samples) {
        uint8_t* dst = P.samples + ((size_t)sample_idx * P.n_chains + chain) * N;
        for (int j = threadIdx.x; j < N; j += blockDim.x) dst[j] = s[j];
      }
      ++sample_idx;
      next_sample_at += P.sweeps_per_sample;
    }
  }
  for (int j = threadIdx.x; j < N; j += blockDim.x) gstate[j] = s[j];
  if (P.energy) {
    const double e = sparse_energy(P.rowptr, P.col, P.val, P.bias, P.N, s, red);
    if (threadIdx.x == 0) P.energy[chain] = e;
  }
  if (P.track_best && threadIdx.x == 0) P.best_energy[chain] = best_e;
}

}  // namespace

extern "C" int tsu_sparse_gibbs_run(const int32_t* d_rowptr, const int32_t* d_col, const double* d_val,
                                    const double* d_bias, const int32_t* d_colour_ptr, const int32_t* d_colour_sites,
                                    int n_colours, uint8_t* d_state, int n_chains, int N, double T,
                                    const double* d_T_chain, const double* d_T_sweep, int n_burnin, int n_samples,
                                    int sweeps_per_sample, const double* d_uniforms, uint8_t* d_samples,
                                    double* d_energy, int track_best, uint8_t* d_best_state, double* d_best_energy,
                                    uint64_t seed, uint32_t sweep0, uint32_t chain0, uintptr_t stream) {
  TSU_CHECK_ARG(d_rowptr && d_col && d_val && d_colour_ptr && d_colour_sites && d_state);
  TSU_CHECK_ARG(n_chains > 0 && N > 0 && n_colours > 0);
  TSU_CHECK_ARG(n_burnin >= 0 && n_samples >= 0 && sweeps_per_sample >= 0);
  TSU_CHECK_ARG(n_samples == 0 || sweeps_per_sample > 0);
  TSU_CHECK_ARG(d_T_chain || d_T_sweep || T > 0);
  TSU_CHECK_ARG(!track_best || (d_best_state && d_best_energy));
  const size_t smem = ((size_t)N + 15) / 16 * 16;
  if (smem > 200 * 1024) return TSU_ERR_UNSUPPORTED;  // one byte per site in shared memory
  if (smem > 40 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(sparse_gibbs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  SparseParams P;
  P.rowptr = d_rowptr;
  P.col = d_col;
  P.val = d_val;
  P.bias = d_bias;
  P.colour_ptr = d_colour_ptr;
  P.colour_sites = d_colour_sites;
  P.state = d_state;
  P.T_chain = d_T_chain;
  P.T_sweep = d_T_sweep;
  P.uniforms = d_uniforms;
  P.samples = d_samples;
  P.energy = d_energy;
  P.best_state = d_best_state;
  P.best_energy = d_best_energy;
  P.T = T;
  P.n_chains = n_chains;
  P.N = N;
  P.n_colours = n_colours;
  P.n_burnin = n_burnin;
  P.n_samples = n_samples;
  P.sweeps_per_sample = sweeps_per_sample;
  P.track_best = track_best;
  P.k0 = (uint32_t)seed;
  P.k1 = (uint32_t)(seed >> 32);
  P.sweep0 = sweep0;
  P.chain0 = chain0;
  sparse_gibbs_kernel<<<n_chains, sparse_threads(N), smem, tsu_stream(stream)>>>(P);
  TSU_RETURN_LAUNCH_STATUS();
}
