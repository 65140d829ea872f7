// Fused overdamped-Langevin sampler for built-in analytic energies (sm_100a).
//
// Replaces the Python loop of ThermalSamplingUnit.sample_from_energy (tsu/core.py:100-162):
//   for every sample: restart at x_init (+ 0.1 N(0,I) for sample_idx > 0, core.py:142-143),
//   n_burnin + n_steps Euler-Maruyama steps (core.py:64-80)
//       x <- x - grad E(x) * dt / gamma + sqrt(2 T dt / gamma) * N(0, I)
//   with the central-difference gradient (core.py:82-98) replaced by the analytic gradient of the
//   built-in energy.  Every sample is an independent chain, so one thread runs one chain with the
//   state in registers: gradient + noise + update are one fused loop, HBM is touched only for the
//   final state (and the optional trajectory).
//
// Noise: Philox4x32-10 + Box-Muller, counter = (chain lo, chain hi & 0xFFFF | block << 16, step, 'LANG'); block b of a
// chain holds coordinates b * PER .. b * PER + PER - 1 (PER = 2 in float64, 4 in float32).
// dim <= 64 runs here; dim > 64 (built-in energies only) runs on the kernels of langevin_wide.cu, which draw the same
// normal for every coordinate and evaluate the per-coordinate expressions of langevin_body.cuh in the same order (caps
// in langevin_wide.cuh and include/tsu_b200.h).
// Parity mode reads the N(0,1) draws from a caller tensor so that the reference (with
// numpy.random.randn patched to the same draws) can be compared step for step.

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"
#include "jit.cuh"
#include "langevin_body.cuh"
#include "langevin_wide.cuh"

namespace {

enum { ENERGY_QUADRATIC = 0, ENERGY_MIXTURE = 1, ENERGY_DOUBLE_WELL = 2, ENERGY_QUADRATIC_FORM = 3 };

using tsu_langevin::kMaxDynDim;
using tsu_langevin::LangevinParams;

// gradient of the built-in energies; sp = parameters staged in shared memory as `real`
template <typename real, int DIM>
__device__ __forceinline__ void gradient(int kind, int dim, const real* __restrict__ sp, const real* x, real* g) {
  constexpr int MAXD = DIM > 0 ? DIM : kMaxDynDim;
  if (kind == ENERGY_QUADRATIC) {
    // E = a sum (x - mu)^2 w ; sp = [a, mu[dim], w[dim]]
    const real two_a = (real)2 * sp[0];
#pragma unroll
    for (int i = 0; i < MAXD; ++i)
      if (i < dim) g[i] = tsu_langevin::grad_quadratic(two_a, sp[1 + dim + i], x[i], sp[1 + i]);
  } else if (kind == ENERGY_DOUBLE_WELL) {
    // E = sum a (x^2 - b)^2
    const real a4 = (real)4 * sp[0], b = sp[1];
#pragma unroll
    for (int i = 0; i < MAXD; ++i)
      if (i < dim) g[i] = tsu_langevin::grad_double_well(a4, b, x[i]);
  } else if (kind == ENERGY_QUADRATIC_FORM) {
    // E = 1/2 x^T A x - b^T x ; sp = [A[dim][dim], b[dim]] ; grad = A x - b
#pragma unroll
    for (int i = 0; i < MAXD; ++i)
      if (i < dim) {
        real acc = -sp[dim * dim + i];
#pragma unroll
        for (int j = 0; j < MAXD; ++j)
          if (j < dim) acc = tsu_langevin::qform_term(acc, sp[i * dim + j], x[j]);
        g[i] = acc;
      }
  } else {
    // E = -log(sum_k p_k exp(-|x - c_k|^2 / 2) + 1e-10); grad = sum_k p_k e_k (x - c_k) / (sum_k p_k e_k + 1e-10)
    const int K = (int)sp[0];
    real tot = (real)0;
#pragma unroll
    for (int i = 0; i < MAXD; ++i)
      if (i < dim) g[i] = (real)0;
    for (int k = 0; k < K; ++k) {
      const real* c = sp + 1 + K + (size_t)k * dim;
      real d2 = (real)0;
#pragma unroll
      for (int i = 0; i < MAXD; ++i)
        if (i < dim) d2 = tsu_langevin::mixture_d2_term(d2, x[i], c[i]);
      const real e = tsu_langevin::mixture_weight(sp[1 + k], d2);
      tot += e;
#pragma unroll
      for (int i = 0; i < MAXD; ++i)
        if (i < dim) g[i] = tsu_langevin::mixture_grad_term(g[i], e, x[i], c[i]);
    }
    const real inv = tsu_langevin::mixture_inv(tot);
#pragma unroll
    for (int i = 0; i < MAXD; ++i)
      if (i < dim) g[i] *= inv;
  }
}

template <typename real, int DIM>
struct BuiltinGrad {
  int kind;
  const real* sp;
  __device__ __forceinline__ void operator()(int dim, const real* x, real* g) const {
    gradient<real, DIM>(kind, dim, sp, x, g);
  }
};

template <typename real, int DIM>
__global__ void __launch_bounds__(128) langevin_kernel(LangevinParams P) {
  extern __shared__ double smem_raw[];
  real* sp = reinterpret_cast<real*>(smem_raw);
  for (int i = threadIdx.x; i < P.n_params; i += blockDim.x) sp[i] = (real)P.params[i];
  __syncthreads();
  tsu_langevin::langevin_chain<real, DIM>(P, BuiltinGrad<real, DIM>{P.energy_kind, sp});
}

template <typename real, int DIM>
int launch(const LangevinParams& P, cudaStream_t st) {
  const unsigned grid = (unsigned)((P.n_chains + 127) / 128);
  const size_t smem = sizeof(double) * (size_t)((P.n_params + 1) & ~1);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(langevin_kernel<real, DIM>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  langevin_kernel<real, DIM><<<grid, 128, smem, st>>>(P);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? TSU_OK : (int)e;
}

template <typename real>
int dispatch_dim(const LangevinParams& P, cudaStream_t st) {
  switch (P.dim) {
    case 1: return launch<real, 1>(P, st);
    case 2: return launch<real, 2>(P, st);
    case 3: return launch<real, 3>(P, st);
    case 4: return launch<real, 4>(P, st);
    case 8: return launch<real, 8>(P, st);
    case 10: return launch<real, 10>(P, st);
    case 16: return launch<real, 16>(P, st);
    default: return launch<real, 0>(P, st);
  }
}

}  // namespace

extern "C" int tsu_langevin_run(void* d_x, int dtype, int64_t n_chains, int dim, int energy_kind,
                                const double* d_params, int n_params, const void* d_x_init, double jitter,
                                int first_chain_exact, double T, double dt, double gamma, int n_burnin, int n_steps, uint64_t seed, uint64_t chain0,
                                const void* d_normals, void* d_traj, uintptr_t stream) {
  TSU_CHECK_ARG(d_x && d_params && n_chains > 0 && dim > 0);
  TSU_CHECK_ARG(dtype == 0 || dtype == 1);
  TSU_CHECK_ARG(T > 0 && dt > 0 && gamma > 0 && n_burnin >= 0 && n_steps >= 0);
  TSU_CHECK_ARG(energy_kind >= 0 && energy_kind <= 3);
  const bool wide = dim > kMaxDynDim;
  // dim > 64: the wide kernels (langevin_wide.cu), capped by the 16-bit Philox block field and, for QUADRATIC_FORM, by
  // the shared-memory chain tile
  if (wide) TSU_CHECK_ARG(dim <= (dtype == 1 ? tsu_langevin::kWideMaxDimF64 : tsu_langevin::kWideMaxDimF32));
  if (wide && energy_kind == ENERGY_QUADRATIC_FORM) TSU_CHECK_ARG(dim <= tsu_langevin::kWideMaxDimQForm);
  if (energy_kind == ENERGY_QUADRATIC_FORM) TSU_CHECK_ARG(n_params == dim * dim + dim);
  if (energy_kind == ENERGY_QUADRATIC) TSU_CHECK_ARG(n_params == 1 + 2 * dim);
  if (energy_kind == ENERGY_DOUBLE_WELL) TSU_CHECK_ARG(n_params == 2);
  if (energy_kind == ENERGY_MIXTURE && !wide) TSU_CHECK_ARG(n_params >= 2 + dim && n_params <= 20000);
  int mixture_k = 0;  // wide MIXTURE: params = [K, p[K], c[K][dim]] fixes K = (n_params - 1) / (dim + 1)
  if (energy_kind == ENERGY_MIXTURE && wide) {
    TSU_CHECK_ARG(n_params > 1 && (n_params - 1) % (dim + 1) == 0);
    mixture_k = (n_params - 1) / (dim + 1);
    TSU_CHECK_ARG(mixture_k <= tsu_langevin::kWideMaxCentres);
  }
  LangevinParams P;
  P.x = d_x;
  P.x_init = d_x_init;
  P.normals = d_normals;
  P.traj = d_traj;
  P.params = d_params;
  P.n_chains = n_chains;
  P.chain0 = chain0;
  P.dim = dim;
  P.energy_kind = energy_kind;
  P.n_params = n_params;
  P.n_burnin = n_burnin;
  P.n_steps = n_steps;
  P.jitter = jitter;
  P.first_chain_exact = first_chain_exact;
  P.drift = dt / gamma;
  P.noise = sqrt(2.0 * T * dt / gamma);
  P.k0 = (uint32_t)seed;
  P.k1 = (uint32_t)(seed >> 32);
  if (wide) return tsu_langevin::langevin_wide_launch(P, dtype, mixture_k, stream);
  return dtype == 0 ? dispatch_dim<float>(P, tsu_stream(stream)) : dispatch_dim<double>(P, tsu_stream(stream));
}


// ---- traced Python energies: the gradient arrives as CUDA source (tsu_emulator_b200/trace.py) -------------------
namespace {
struct LangevinJit {
  void* fn;
  int dtype, dim;
};
std::mutex g_lj_mutex;
std::map<std::string, int> g_lj_cache;
std::vector<LangevinJit> g_lj;
}  // namespace

extern "C" int tsu_langevin_jit_prepare(const char* grad_source, int dtype, int dim, const char* src_dir, char* log_buf,
                                        int log_len) {
  TSU_CHECK_ARG(grad_source && src_dir && (dtype == 0 || dtype == 1) && dim > 0 && dim <= kMaxDynDim);
  if (log_buf && log_len > 0) log_buf[0] = 0;
  std::lock_guard<std::mutex> lock(g_lj_mutex);
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  const std::string key = std::to_string(dev) + ":" + std::to_string(dtype) + ":" + std::to_string(dim) + ":" + grad_source;
  auto it = g_lj_cache.find(key);
  if (it != g_lj_cache.end()) return it->second;
  std::string src = "#include \"langevin_body.cuh\"\n";
  src += grad_source;
  src += "\nstruct TsuUserGrad {\n  template <typename real>\n  __device__ __forceinline__ void operator()(int, const real* x, "
         "real* g) const { tsu_user_grad<real>(x, g); }\n};\n";
  src += std::string("extern \"C\" __global__ void __launch_bounds__(128) tsu_jit_langevin(tsu_langevin::LangevinParams P) {\n") +
         "  tsu_langevin::langevin_chain<" + (dtype == 0 ? "float" : "double") + ", " + std::to_string(dim) +
         ">(P, TsuUserGrad());\n}\n";
  std::string log;
  void* fn = tsu_jit::compile(src, "tsu_jit_langevin.cu", "tsu_jit_langevin", src_dir, log);
  if (!fn) {
    if (log_buf && log_len > 0) snprintf(log_buf, log_len, "%s", log.c_str());
    g_lj_cache[key] = 0;
    return 0;
  }
  g_lj.push_back(LangevinJit{fn, dtype, dim});
  const int handle = (int)g_lj.size();
  g_lj_cache[key] = handle;
  return handle;
}

extern "C" int tsu_langevin_run_jit(int handle, void* d_x, int64_t n_chains, const void* d_x_init, double jitter,
                                    int first_chain_exact, double T, double dt, double gamma, int n_burnin, int n_steps,
                                    uint64_t seed, uint64_t chain0, const void* d_normals, void* d_traj, uintptr_t stream) {
  LangevinJit k;
  {
    std::lock_guard<std::mutex> lock(g_lj_mutex);
    TSU_CHECK_ARG(handle >= 1 && handle <= (int)g_lj.size());
    k = g_lj[handle - 1];
  }
  TSU_CHECK_ARG(d_x && n_chains > 0 && T > 0 && dt > 0 && gamma > 0 && n_burnin >= 0 && n_steps >= 0);
  LangevinParams P;
  P.x = d_x;
  P.x_init = d_x_init;
  P.normals = d_normals;
  P.traj = d_traj;
  P.params = nullptr;
  P.n_chains = n_chains;
  P.chain0 = chain0;
  P.dim = k.dim;
  P.energy_kind = -1;
  P.n_params = 0;
  P.n_burnin = n_burnin;
  P.n_steps = n_steps;
  P.jitter = jitter;
  P.first_chain_exact = first_chain_exact;
  P.drift = dt / gamma;
  P.noise = sqrt(2.0 * T * dt / gamma);
  P.k0 = (uint32_t)seed;
  P.k1 = (uint32_t)(seed >> 32);
  void* args[] = {&P};
  return tsu_jit::launch(k.fn, (unsigned)((n_chains + 127) / 128), 128, 0, (void*)tsu_stream(stream), args);
}
