// Chain loop of the fused overdamped-Langevin sampler (see langevin.cu for what it replaces), shared by the prebuilt
// kernels for the built-in energies and by the kernels NVRTC compiles for traced Python energies
// (tsu_langevin_jit_prepare): the gradient is a functor `grad(dim, x, g)`.  Keep it free of host headers.
#pragma once
#ifdef __CUDACC_RTC__
typedef unsigned int uint32_t;
typedef unsigned long long uint64_t;
typedef unsigned long size_t;
#else
#include <stdint.h>
#include <stddef.h>
#endif
#include "philox.cuh"

namespace tsu_langevin {

constexpr int kMaxDynDim = 64;

struct LangevinParams {
  void* x;
  const void* x_init;
  const void* normals;
  void* traj;
  const double* params;
  long long n_chains;
  unsigned long long chain0;
  int dim, energy_kind, n_params;
  int n_burnin, n_steps;
  int first_chain_exact;
  double jitter, drift, noise;  // drift = dt / gamma, noise = sqrt(2 T dt / gamma)
  uint32_t k0, k1;
};

__device__ __forceinline__ float lg2_fast(float x) {  // x in [2^-25, 1): no denormal handling needed
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <typename real>
struct BoxMuller;

template <>
struct BoxMuller<float> {
  static constexpr int kPerCall = 4;
  // 4 normals from one Philox block (24-bit uniforms, exactly representable in float)
  __device__ static __forceinline__ void draw(const tsu_u32x4& o, float z[4]) {
    const float u1 = ((float)(o.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(o.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u3 = ((float)(o.z >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u4 = ((float)(o.w >> 8) + 0.5f) * (1.0f / 16777216.0f);
    // fast-math forms (MUFU lg2 / rsq / sin / cos, absolute error ~2^-21): the float32 kernel is instruction bound and
    // the library logf / sincospif cost three times as many instructions as the rest of the step
    const float a1 = -1.3862943611f * lg2_fast(u1), a2 = -1.3862943611f * lg2_fast(u3);  // -2 ln u > 0 (u < 1)
    // (u rounds to 1.0f for the top uniforms: a = 0 -> r = 0, guarded against 0 * inf)
    const float r1 = a1 * rsqrtf(fmaxf(a1, 1e-30f)), r2 = a2 * rsqrtf(fmaxf(a2, 1e-30f));
    const float t1 = 6.2831853072f * u2, t2 = 6.2831853072f * u4;
    z[0] = r1 * __cosf(t1);
    z[1] = r1 * __sinf(t1);
    z[2] = r2 * __cosf(t2);
    z[3] = r2 * __sinf(t2);
  }
};

template <>
struct BoxMuller<double> {
  static constexpr int kPerCall = 2;
  // 2 normals from one Philox block (53-bit uniforms)
  __device__ static __forceinline__ void draw(const tsu_u32x4& o, double z[2]) {
    const unsigned long long a = (((unsigned long long)o.x << 32) | o.y) >> 11;
    const unsigned long long b = (((unsigned long long)o.z << 32) | o.w) >> 11;
    const double u1 = ((double)a + 0.5) * (1.0 / 9007199254740992.0);
    const double u2 = ((double)b + 0.5) * (1.0 / 9007199254740992.0);
    const double r = sqrt(-2.0 * log(u1));
    double s, c;
    sincospi(2.0 * u2, &s, &c);
    z[0] = r * c;
    z[1] = r * s;
  }
};

// The PER = BoxMuller<real>::kPerCall normals of Philox block b of (chain, step): coordinates b*PER .. b*PER+PER-1.
// The counter does not involve dim, so a coordinate draws the same normal at every dim; the 16-bit block field
// bounds dim at 65536 * PER.
template <typename real>
__device__ __forceinline__ void philox_normals(const LangevinParams& P, unsigned long long chain_g, int b, int step,
                                               real* t) {
  tsu_u32x4 o = tsu_philox4x32_10((uint32_t)chain_g, ((uint32_t)(chain_g >> 32) & 0xFFFFu) | ((uint32_t)b << 16),
                                  (uint32_t)step, TSU_STREAM_LANGEVIN, P.k0, P.k1);
  BoxMuller<real>::draw(o, t);
}

// Per-coordinate arithmetic of the built-in energies and of the Euler-Maruyama update.  The register kernels
// (langevin.cu) and the wide kernels (langevin_wide.cu) both evaluate through these, in the same summation order,
// so nvcc contracts them the same way in both and a coordinate gets the same bits at every dim.
// QUADRATIC: dE/dx_i = 2a w_i (x_i - mu_i)
template <typename real>
__device__ __forceinline__ real grad_quadratic(real two_a, real w, real x, real mu) { return two_a * w * (x - mu); }
// DOUBLE_WELL: dE/dx_i = 4a x_i (x_i^2 - b)
template <typename real>
__device__ __forceinline__ real grad_double_well(real a4, real b, real x) { return a4 * x * (x * x - b); }
// QUADRATIC_FORM: g_i = -b_i + sum_j A_ij x_j over ascending j; each term contracts to acc = fma(A_ij, x_j, acc)
template <typename real>
__device__ __forceinline__ real qform_term(real acc, real a, real x) { return acc + a * x; }
// MIXTURE: d2_k = sum_i (x_i - c_ki)^2 over ascending i; e_k = p_k exp(-d2_k / 2); tot = sum_k e_k over ascending k;
// g_i = (sum_k e_k (x_i - c_ki) over ascending k) / (tot + 1e-10)
template <typename real>
__device__ __forceinline__ real mixture_d2_term(real d2, real x, real c) {
  real d = x - c;
  return d2 + d * d;
}
template <typename real>
__device__ __forceinline__ real mixture_weight(real p, real d2) { return p * (real)exp((real)-0.5 * d2); }
template <typename real>
__device__ __forceinline__ real mixture_grad_term(real g, real e, real x, real c) { return g + e * (x - c); }
template <typename real>
__device__ __forceinline__ real mixture_inv(real tot) { return (real)1 / (tot + (real)1e-10); }
// restart jitter: x <- x_init + jitter z  (core.py:142-143)
template <typename real>
__device__ __forceinline__ real jitter_start(real x, real jitter, real z) { return x + jitter * z; }
// x <- x - g dt/gamma + sqrt(2 T dt/gamma) z  (core.py:74-80 order of operations)
template <typename real>
__device__ __forceinline__ real em_update(real x, real g, real z, real drift, real noise) {
  return x + (-g * drift) + noise * z;
}

// N(0,1) vector for (chain, step): injected rows or Philox + Box-Muller
template <typename real, int DIM>
__device__ __forceinline__ void normal_vector(const LangevinParams& P, unsigned long long chain_g, long long chain_l,
                                              int step, int dim, real* z) {
  if (P.normals) {
    const long long rows = 1LL + P.n_burnin + P.n_steps;
    const real* src = reinterpret_cast<const real*>(P.normals) + ((size_t)chain_l * rows + step) * dim;
#pragma unroll
    for (int i = 0; i < (DIM > 0 ? DIM : kMaxDynDim); ++i)
      if (i < dim) z[i] = src[i];
    return;
  }
  constexpr int PER = BoxMuller<real>::kPerCall;
  constexpr int MAXD = DIM > 0 ? DIM : kMaxDynDim;
#pragma unroll
  for (int b = 0; b < (MAXD + PER - 1) / PER; ++b) {
    if (b * PER < dim) {
      real t[PER];
      philox_normals<real>(P, chain_g, b, step, t);
#pragma unroll
      for (int q = 0; q < PER; ++q)
        if (b * PER + q < MAXD && b * PER + q < dim) z[b * PER + q] = t[q];
    }
  }
}


// one chain per thread: restart jitter, n_burnin + n_steps Euler-Maruyama steps, optional trajectory (core.py:140-159)
template <typename real, int DIM, typename Grad>
__device__ __forceinline__ void langevin_chain(const LangevinParams& P, const Grad& grad) {
  const long long chain = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (chain >= P.n_chains) return;
  const unsigned long long chain_g = P.chain0 + (unsigned long long)chain;
  const int dim = DIM > 0 ? DIM : P.dim;
  constexpr int MAXD = DIM > 0 ? DIM : kMaxDynDim;
  real x[MAXD], z[MAXD], g[MAXD];

  const real* xi = reinterpret_cast<const real*>(P.x_init);
#pragma unroll
  for (int i = 0; i < MAXD; ++i)
    if (i < dim) x[i] = xi ? xi[i] : (real)0;
  // every chain but the first of a call starts at x_init + jitter * N(0, I)  (core.py:142-143)
  if (!(chain == 0 && P.first_chain_exact) && P.jitter != 0.0) {
    normal_vector<real, DIM>(P, chain_g, chain, 0, dim, z);
#pragma unroll
    for (int i = 0; i < MAXD; ++i)
      if (i < dim) x[i] = jitter_start(x[i], (real)P.jitter, z[i]);
  }
  const real drift = (real)P.drift, noise = (real)P.noise;
  const int total = P.n_burnin + P.n_steps;
  real* traj = reinterpret_cast<real*>(P.traj);
  for (int s = 0; s < total; ++s) {
    grad(dim, x, g);
    normal_vector<real, DIM>(P, chain_g, chain, s + 1, dim, z);
#pragma unroll
    for (int i = 0; i < MAXD; ++i)
      if (i < dim) x[i] = em_update(x[i], g[i], z[i], drift, noise);
    if (traj && s >= P.n_burnin) {
      real* dst = traj + ((size_t)chain * P.n_steps + (s - P.n_burnin)) * dim;
#pragma unroll
      for (int i = 0; i < MAXD; ++i)
        if (i < dim) dst[i] = x[i];
    }
  }
  real* out = reinterpret_cast<real*>(P.x) + (size_t)chain * dim;
#pragma unroll
  for (int i = 0; i < MAXD; ++i)
    if (i < dim) out[i] = x[i];
}

}  // namespace tsu_langevin
