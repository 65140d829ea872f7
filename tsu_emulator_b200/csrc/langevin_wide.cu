// Overdamped-Langevin kernels for dim > 64 (sm_100a): the same sampler as langevin.cu, for states too large for the
// register kernel's one-thread-per-chain layout.
//
// The update, restart jitter, first_chain_exact, chain0, injected normals [chain][1 + n_burnin + n_steps][dim] and
// trajectory [chain][n_steps][dim] are those of tsu_langevin_run.  Two rules make these kernels the same sampler as
// the register kernels, coordinate for coordinate:
//   1. Same noise per coordinate: coordinate i takes element i % PER of Philox block b = i / PER of (chain, step)
//      (tsu_langevin::philox_normals; PER = 2 in float64, 4 in float32), so its draw does not depend on dim.
//   2. Same per-coordinate arithmetic and summation order: the gradient terms and the update are the device
//      functions of langevin_body.cuh that the register kernels call, summed in the same order (QUADRATIC_FORM over
//      ascending j, one thread per output; MIXTURE d2_k over ascending i, tot and g_i over ascending k).
// A coordinate of a dim-dimensional run that does not couple to the others therefore has the bits of a lower-dim run.
//
// Kernels (caps in langevin_wide.cuh):
//   separable_kernel  QUADRATIC, DOUBLE_WELL.  One thread per (chain, Philox block): PER coordinates in registers for
//                     the whole run, reads and writes coalesced over [chain][dim].
//   qform_kernel      QUADRATIC_FORM.  The gradient of all chains is X A^T - b, a GEMM per step.  A CTA owns TC chains
//                     (8 in float64, 16 in float32) and stages their state in shared memory; each thread owns PER
//                     consecutive rows and accumulates them for all TC chains in ascending k, streaming A^T (converted
//                     to `real` once per launch into a scratch buffer) from L2 with 16-byte coalesced loads.  No
//                     split-K and no tensor cores: rule 2 fixes the order of every sum.  The new state goes to d_x,
//                     which is reloaded into shared memory at the next step.
//   mixture_kernel    MIXTURE.  A CTA owns 256 / KP chains (KP = K rounded up to a power of two); one thread per
//                     (chain, centre) sums d2_k, then the CTA runs over (chain, Philox block) for g and the update.
//                     Centres are read through L1 / L2 from the caller's float64 parameters.

#include "common.cuh"
#include "langevin_wide.cuh"

namespace {

using tsu_langevin::BoxMuller;
using tsu_langevin::LangevinParams;

enum { ENERGY_QUADRATIC = 0, ENERGY_MIXTURE = 1, ENERGY_DOUBLE_WELL = 2, ENERGY_QUADRATIC_FORM = 3 };

constexpr int kThreads = 256;

// normals of Philox block b (coordinates b*PER ..) of (chain, step): injected rows or Philox + Box-Muller
template <typename real>
__device__ __forceinline__ void block_normals(const LangevinParams& P, unsigned long long chain_g, long long chain,
                                              int b, int step, real* t) {
  constexpr int PER = BoxMuller<real>::kPerCall;
  if (P.normals) {
    const long long rows = 1LL + P.n_burnin + P.n_steps;
    const real* src = reinterpret_cast<const real*>(P.normals) + ((size_t)chain * rows + step) * P.dim + (size_t)b * PER;
#pragma unroll
    for (int q = 0; q < PER; ++q)
      if (b * PER + q < P.dim) t[q] = src[q];
    return;
  }
  tsu_langevin::philox_normals<real>(P, chain_g, b, step, t);
}

// start of coordinates b*PER .. of a chain: x_init, plus the restart jitter for every chain but an exact first one
template <typename real>
__device__ __forceinline__ void start_block(const LangevinParams& P, unsigned long long chain_g, long long chain, int b,
                                            real* x) {
  constexpr int PER = BoxMuller<real>::kPerCall;
  const real* xi = reinterpret_cast<const real*>(P.x_init);
#pragma unroll
  for (int q = 0; q < PER; ++q)
    if (b * PER + q < P.dim) x[q] = xi ? xi[b * PER + q] : (real)0;
  if (!(chain == 0 && P.first_chain_exact) && P.jitter != 0.0) {
    real z[PER];
    block_normals<real>(P, chain_g, chain, b, 0, z);
#pragma unroll
    for (int q = 0; q < PER; ++q)
      if (b * PER + q < P.dim) x[q] = tsu_langevin::jitter_start(x[q], (real)P.jitter, z[q]);
  }
}

// ------------------------------------------------------------------------------------------------ separable
template <typename real>
__global__ void __launch_bounds__(kThreads) separable_kernel(LangevinParams P) {
  constexpr int PER = BoxMuller<real>::kPerCall;
  const int dim = P.dim;
  const int nblk = (dim + PER - 1) / PER;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= P.n_chains * nblk) return;
  const long long chain = tid / nblk;
  const int b = (int)(tid - chain * nblk);
  const int i0 = b * PER;
  const unsigned long long chain_g = P.chain0 + (unsigned long long)chain;

  // parameters as langevin_kernel stages them: (real) of the float64 value, then the same products
  const bool quad = P.energy_kind == ENERGY_QUADRATIC;
  const real c0 = (quad ? (real)2 : (real)4) * (real)P.params[0];  // 2a (QUADRATIC) or 4a (DOUBLE_WELL)
  real w[PER], mu[PER];
  const real dw_b = quad ? (real)0 : (real)P.params[1];
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    w[q] = (real)0;
    mu[q] = (real)0;
    if (quad && i0 + q < dim) {
      mu[q] = (real)P.params[1 + i0 + q];
      w[q] = (real)P.params[1 + dim + i0 + q];
    }
  }

  real x[PER], z[PER];
  start_block<real>(P, chain_g, chain, b, x);
  const real drift = (real)P.drift, noise = (real)P.noise;
  const int total = P.n_burnin + P.n_steps;
  real* traj = reinterpret_cast<real*>(P.traj);
  for (int s = 0; s < total; ++s) {
    block_normals<real>(P, chain_g, chain, b, s + 1, z);
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const real g = quad ? tsu_langevin::grad_quadratic(c0, w[q], x[q], mu[q])
                          : tsu_langevin::grad_double_well(c0, dw_b, x[q]);
      x[q] = tsu_langevin::em_update(x[q], g, z[q], drift, noise);
    }
    if (traj && s >= P.n_burnin) {
      real* dst = traj + ((size_t)chain * P.n_steps + (s - P.n_burnin)) * dim + i0;
#pragma unroll
      for (int q = 0; q < PER; ++q)
        if (i0 + q < dim) dst[q] = x[q];
    }
  }
  real* out = reinterpret_cast<real*>(P.x) + (size_t)chain * dim + i0;
#pragma unroll
  for (int q = 0; q < PER; ++q)
    if (i0 + q < dim) out[q] = x[q];
}

// ------------------------------------------------------------------------------------------------ quadratic form
template <typename real>
struct Vec;
template <>
struct Vec<double> {
  using T = double2;
};
template <>
struct Vec<float> {
  using T = float4;
};

// At[k][i] = (real)A[i][k] for i < dim, 0 for dim <= i < ld;  bt[i] = (real)b[i] (0 past dim)
template <typename real>
__global__ void qform_stage_kernel(const double* __restrict__ params, int dim, int ld, real* __restrict__ At,
                                   real* __restrict__ bt) {
  __shared__ double tile[32][33];
  const int i_base = blockIdx.x * 32, k_base = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {  // coalesced over k along a row of A
    const int i = i_base + r, k = k_base + threadIdx.x;
    tile[r][threadIdx.x] = (i < dim && k < dim) ? params[(size_t)i * dim + k] : 0.0;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {  // coalesced over i along a row of A^T
    const int k = k_base + r, i = i_base + threadIdx.x;
    if (k < dim && i < ld) At[(size_t)k * ld + i] = (real)tile[threadIdx.x][r];
  }
  if (blockIdx.y == 0 && threadIdx.y == 0) {
    const int i = i_base + threadIdx.x;
    if (i < ld) bt[i] = i < dim ? (real)params[(size_t)dim * dim + i] : (real)0;
  }
}

// TC chains per CTA; thread t owns rows r0 + t*PER .. r0 + t*PER + PER-1 of every row block r0 (kThreads*PER rows)
template <typename real, int TC>
__global__ void __launch_bounds__(kThreads) qform_kernel(LangevinParams P, const real* __restrict__ At,
                                                         const real* __restrict__ bt, int ld) {
  constexpr int PER = BoxMuller<real>::kPerCall;  // rows per thread = reals per 16-byte load
  using V = typename Vec<real>::T;
  extern __shared__ double smem_raw[];
  real* xs = reinterpret_cast<real*>(smem_raw);  // [TC][ldx]
  const int dim = P.dim;
  const int ldx = (dim + PER - 1) / PER * PER;
  const int nblk = ldx / PER;
  const long long tile0 = (long long)blockIdx.x * TC;
  const int nc = (int)min((long long)TC, P.n_chains - tile0);  // chains of this tile
  real* X = reinterpret_cast<real*>(P.x);
  real* traj = reinterpret_cast<real*>(P.traj);

  // start state -> d_x
  for (int w = threadIdx.x; w < nc * nblk; w += kThreads) {
    const int c = w / nblk, b = w - c * nblk;
    const long long chain = tile0 + c;
    real x[PER];
    start_block<real>(P, P.chain0 + (unsigned long long)chain, chain, b, x);
#pragma unroll
    for (int q = 0; q < PER; ++q)
      if (b * PER + q < dim) X[(size_t)chain * dim + b * PER + q] = x[q];
  }

  const real drift = (real)P.drift, noise = (real)P.noise;
  const int total = P.n_burnin + P.n_steps;
  const int kfull = dim / PER * PER;
  for (int s = 0; s < total; ++s) {
    __syncthreads();  // the previous step's d_x writes are visible, and nobody reads xs any more
    for (int w = threadIdx.x; w < TC * ldx; w += kThreads) {
      const int c = w / ldx, i = w - c * ldx;
      xs[w] = (c < nc && i < dim) ? X[(size_t)(tile0 + c) * dim + i] : (real)0;
    }
    __syncthreads();
    for (int r0 = 0; r0 < dim; r0 += kThreads * PER) {
      const int i0 = r0 + threadIdx.x * PER;
      if (i0 >= dim) break;  // ld >= i0 + PER: the A^T loads below stay inside a padded row
      real acc[TC][PER];
      {
        const V bv = *reinterpret_cast<const V*>(bt + i0);
        const real* bb = reinterpret_cast<const real*>(&bv);
#pragma unroll
        for (int c = 0; c < TC; ++c)
#pragma unroll
          for (int q = 0; q < PER; ++q) acc[c][q] = -bb[q];
      }
      // full k tiles of PER: one 16-byte load of x per chain, one of A^T per k
      for (int k = 0; k < kfull; k += PER) {
        real a[PER][PER];  // a[u][q] = A[i0 + q][k + u]
#pragma unroll
        for (int u = 0; u < PER; ++u) {
          const V v = __ldg(reinterpret_cast<const V*>(At + (size_t)(k + u) * ld + i0));
          const real* vv = reinterpret_cast<const real*>(&v);
#pragma unroll
          for (int q = 0; q < PER; ++q) a[u][q] = vv[q];
        }
#pragma unroll
        for (int c = 0; c < TC; ++c) {
          const V xv = *reinterpret_cast<const V*>(xs + c * ldx + k);
          const real* xx = reinterpret_cast<const real*>(&xv);
#pragma unroll
          for (int u = 0; u < PER; ++u)
#pragma unroll
            for (int q = 0; q < PER; ++q) acc[c][q] = tsu_langevin::qform_term(acc[c][q], a[u][q], xx[u]);
        }
      }
      // last partial k tile
      for (int k = kfull; k < dim; ++k) {
        const V v = __ldg(reinterpret_cast<const V*>(At + (size_t)k * ld + i0));
        const real* vv = reinterpret_cast<const real*>(&v);
#pragma unroll
        for (int c = 0; c < TC; ++c) {
          const real xk = xs[c * ldx + k];
#pragma unroll
          for (int q = 0; q < PER; ++q) acc[c][q] = tsu_langevin::qform_term(acc[c][q], vv[q], xk);
        }
      }
      // update: rows i0 .. i0 + PER - 1 are Philox block i0 / PER
#pragma unroll
      for (int c = 0; c < TC; ++c) {
        if (c >= nc) break;
        const long long chain = tile0 + c;
        real z[PER];
        block_normals<real>(P, P.chain0 + (unsigned long long)chain, chain, i0 / PER, s + 1, z);
        real* dst = traj && s >= P.n_burnin ? traj + ((size_t)chain * P.n_steps + (s - P.n_burnin)) * dim : nullptr;
#pragma unroll
        for (int q = 0; q < PER; ++q) {
          const int i = i0 + q;
          if (i < dim) {
            const real xn = tsu_langevin::em_update(xs[c * ldx + i], acc[c][q], z[q], drift, noise);
            X[(size_t)chain * dim + i] = xn;
            if (dst) dst[i] = xn;
          }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ mixture
// params = [K, p[K], c[K][dim]];  e[c][k] = p_k exp(-d2_k / 2) in shared memory
template <typename real>
__global__ void __launch_bounds__(kThreads) mixture_kernel(LangevinParams P, int K, int KP) {
  constexpr int PER = BoxMuller<real>::kPerCall;
  __shared__ real e_s[kThreads];  // [TC][KP]
  const int dim = P.dim;
  const int TC = kThreads / KP;
  const int nblk = (dim + PER - 1) / PER;
  const long long tile0 = (long long)blockIdx.x * TC;
  const int nc = (int)min((long long)TC, P.n_chains - tile0);
  const double* cen = P.params + 1 + K;
  real* X = reinterpret_cast<real*>(P.x);
  real* traj = reinterpret_cast<real*>(P.traj);

  for (int w = threadIdx.x; w < nc * nblk; w += kThreads) {
    const int c = w / nblk, b = w - c * nblk;
    const long long chain = tile0 + c;
    real x[PER];
    start_block<real>(P, P.chain0 + (unsigned long long)chain, chain, b, x);
#pragma unroll
    for (int q = 0; q < PER; ++q)
      if (b * PER + q < dim) X[(size_t)chain * dim + b * PER + q] = x[q];
  }

  const real drift = (real)P.drift, noise = (real)P.noise;
  const int total = P.n_burnin + P.n_steps;
  for (int s = 0; s < total; ++s) {
    __syncthreads();
    {  // d2_k over ascending i, one thread per (chain, centre)
      const int c = threadIdx.x / KP, k = threadIdx.x - c * KP;
      if (c < nc && k < K) {
        const real* x = X + (size_t)(tile0 + c) * dim;
        const double* ck = cen + (size_t)k * dim;
        real d2 = (real)0;
        for (int i = 0; i < dim; ++i) d2 = tsu_langevin::mixture_d2_term(d2, x[i], (real)ck[i]);
        e_s[threadIdx.x] = tsu_langevin::mixture_weight((real)P.params[1 + k], d2);
      }
    }
    __syncthreads();
    for (int w = threadIdx.x; w < nc * nblk; w += kThreads) {
      const int c = w / nblk, b = w - c * nblk;
      const long long chain = tile0 + c;
      const real* e = e_s + c * KP;
      real tot = (real)0;
      for (int k = 0; k < K; ++k) tot += e[k];
      const real inv = tsu_langevin::mixture_inv(tot);
      real z[PER];
      block_normals<real>(P, P.chain0 + (unsigned long long)chain, chain, b, s + 1, z);
      real* dst = traj && s >= P.n_burnin ? traj + ((size_t)chain * P.n_steps + (s - P.n_burnin)) * dim : nullptr;
#pragma unroll
      for (int q = 0; q < PER; ++q) {
        const int i = b * PER + q;
        if (i < dim) {
          const real xi = X[(size_t)chain * dim + i];
          real g = (real)0;
          for (int k = 0; k < K; ++k) g = tsu_langevin::mixture_grad_term(g, e[k], xi, (real)cen[(size_t)k * dim + i]);
          g *= inv;
          const real xn = tsu_langevin::em_update(xi, g, z[q], drift, noise);
          X[(size_t)chain * dim + i] = xn;
          if (dst) dst[i] = xn;
        }
      }
    }
  }
}

template <typename real>
int launch_wide(const LangevinParams& P, int mixture_k, cudaStream_t st) {
  constexpr int PER = BoxMuller<real>::kPerCall;
  if (P.energy_kind == ENERGY_QUADRATIC || P.energy_kind == ENERGY_DOUBLE_WELL) {
    const long long threads = P.n_chains * (long long)((P.dim + PER - 1) / PER);
    separable_kernel<real><<<(unsigned)((threads + kThreads - 1) / kThreads), kThreads, 0, st>>>(P);
    TSU_RETURN_LAUNCH_STATUS();
  }
  if (P.energy_kind == ENERGY_MIXTURE) {
    int KP = 1;
    while (KP < mixture_k) KP *= 2;
    const long long TC = kThreads / KP;
    mixture_kernel<real><<<(unsigned)((P.n_chains + TC - 1) / TC), kThreads, 0, st>>>(P, mixture_k, KP);
    TSU_RETURN_LAUNCH_STATUS();
  }
  // QUADRATIC_FORM
  constexpr int TC = sizeof(real) == 8 ? 8 : 16;
  const int dim = P.dim;
  const int ld = (dim + kThreads * PER - 1) / (kThreads * PER) * (kThreads * PER);  // whole row blocks, zero padded
  real* scratch = nullptr;
  cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&scratch), sizeof(real) * ((size_t)dim * ld + ld), st);
  if (e != cudaSuccess) return (int)e;
  real* At = scratch;
  real* bt = scratch + (size_t)dim * ld;
  qform_stage_kernel<real><<<dim3((unsigned)(ld / 32), (unsigned)((dim + 31) / 32)), dim3(32, 8), 0, st>>>(P.params, dim, ld,
                                                                                                          At, bt);
  e = cudaGetLastError();
  if (e == cudaSuccess) {
    const int ldx = (dim + PER - 1) / PER * PER;
    const size_t smem = sizeof(real) * (size_t)TC * ldx;
    if (smem > 48 * 1024)
      e = cudaFuncSetAttribute(qform_kernel<real, TC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) {
      qform_kernel<real, TC><<<(unsigned)((P.n_chains + TC - 1) / TC), kThreads, smem, st>>>(P, At, bt, ld);
      e = cudaGetLastError();
    }
  }
  const cudaError_t ef = cudaFreeAsync(scratch, st);
  if (e == cudaSuccess) e = ef;
  return e == cudaSuccess ? TSU_OK : (int)e;
}

}  // namespace

int tsu_langevin::langevin_wide_launch(const LangevinParams& P, int dtype, int mixture_k, uintptr_t stream) {
  return dtype == 0 ? launch_wide<float>(P, mixture_k, tsu_stream(stream))
                    : launch_wide<double>(P, mixture_k, tsu_stream(stream));
}
