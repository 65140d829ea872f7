// Houdayer cluster moves of chain pairs on SPARSE couplings (sm_100a): the overlap-cluster half of the isoenergetic
// cluster move (ICM, Zhu, Ochoa & Katzgraber, PRL 115, 077201, 2015) on any CSR graph, for the chains of the chromatic
// sweep kernel (sparse_gibbs.cu).  The contract is stated at tsu_sparse_houdayer in include/tsu_b200.h.
//
// One CTA per pair runs every step of the call.  A step: d = x^a xor x^b; labels[i] = i; every thread takes the d = 1
// sites of a strided range and unions each with its CSR neighbours j > i that have d_j = 1 and J_ij != 0 (lock-free,
// the larger root hangs under the smaller: union_find.cuh); full path compression; one Philox call per root (the
// cluster's smallest site), its flip bit parked in bit 31 of the root's label; every d = 1 site then XORs its root's
// bit into both rows.  With the labels in shared memory (N <= kResidentSites) the two rows are staged there as well;
// above that, labels go to the caller's workspace and the rows are read and written in place.  Both paths compute the
// same labels, roots and bits.  Energies come from sparse_energy with the sweep kernel's thread count, so they equal
// the sweep kernel's bit for bit.

#include "common.cuh"
#include "philox.cuh"
#include "sparse_energy.cuh"
#include "union_find.cuh"

namespace {

constexpr int kMaxSites = 204800;       // the sweep kernel's cap (one byte per site in shared memory)
constexpr int kResidentSites = 32768;   // 2 rows + int32 labels: 6 bytes per site, 192 KB of shared memory at most
constexpr uint32_t kFlipBit = 0x80000000u;

__host__ __device__ inline size_t pad16(size_t n) { return (n + 15) / 16 * 16; }
__host__ __device__ inline size_t resident_smem(int N) { return 2 * pad16((size_t)N) + 4 * pad16((size_t)N); }
__host__ __device__ inline size_t labels_bytes(int N) { return pad16(4 * (size_t)N); }

struct HoudayerParams {
  const int32_t* rowptr;
  const int32_t* col;
  const double* val;
  const double* bias;
  uint8_t* state;        // [n_chains][N]
  const int32_t* pairs;  // [n_pairs][2]; this launch serves pairs pair0 .. pair0 + gridDim.x - 1
  double* energy;        // [n_chains] or nullptr
  char* work;            // global-label path: labels_bytes(N) per CTA
  int n_chains, N, pair0, n_steps;
  uint32_t k0, k1, step0, chain0;
};

// root of x without writing: another thread may be storing x's own root meanwhile, and a stale read still leads there
__device__ __forceinline__ int find_root(const int32_t* L, int x) {
  const volatile int32_t* V = L;
  int y = V[x];
  while (y != x) {
    x = y;
    y = V[x];
  }
  return x;
}

template <bool kResident>
__global__ void __launch_bounds__(256) sparse_houdayer_kernel(HoudayerParams P) {
  extern __shared__ __align__(16) unsigned char smem_h[];
  __shared__ double red[32];
  const int N = P.N, q = P.pair0 + blockIdx.x;
  const int a = P.pairs[2 * q], b = P.pairs[2 * q + 1];
  if (a < 0 || a >= P.n_chains || b < 0 || b >= P.n_chains || a == b) return;  // skipped: rows neither read nor written
  uint8_t* ga = P.state + (size_t)a * N;
  uint8_t* gb = P.state + (size_t)b * N;
  uint8_t *xa = ga, *xb = gb;
  int32_t* L;
  if (kResident) {
    xa = smem_h;
    xb = smem_h + pad16((size_t)N);
    L = reinterpret_cast<int32_t*>(smem_h + 2 * pad16((size_t)N));
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      xa[i] = ga[i] ? 1 : 0;
      xb[i] = gb[i] ? 1 : 0;
    }
  } else {
    L = reinterpret_cast<int32_t*>(P.work + (size_t)blockIdx.x * labels_bytes(N));
  }
  const uint32_t chain = P.chain0 + (uint32_t)a;
  for (int s = 0; s < P.n_steps; ++s) {
    for (int i = threadIdx.x; i < N; i += blockDim.x) L[i] = i;
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      if ((xa[i] != 0) == (xb[i] != 0)) continue;
      for (int k = P.rowptr[i]; k < P.rowptr[i + 1]; ++k) {
        const int j = P.col[k];
        if (j > i && (xa[j] != 0) != (xb[j] != 0) && P.val[k] != 0.0) cluster_union(L, i, j);
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x)
      if ((xa[i] != 0) != (xb[i] != 0)) L[i] = find_root(L, i);
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      if (L[i] != i || (xa[i] != 0) == (xb[i] != 0)) continue;
      const tsu_u32x4 o = tsu_philox4x32_10((uint32_t)i, chain, P.step0 + (uint32_t)s, TSU_STREAM_HOUDAYER, P.k0, P.k1);
      if (o.x & 1u) L[i] = (int32_t)((uint32_t)i | kFlipBit);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      const bool da = xa[i] != 0, db = xb[i] != 0;
      if (da == db) continue;
      const int r = (int)((uint32_t)L[i] & ~kFlipBit);
      if ((uint32_t)L[r] & kFlipBit) {  // (0, 1) <-> (1, 0): the two chains swap their bits here
        xa[i] = db ? 1 : 0;
        xb[i] = da ? 1 : 0;
      }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < N; i += blockDim.x) {  // the resident rows, or 0 / 1 bytes in place, as the sweep writes
    ga[i] = xa[i] ? 1 : 0;
    gb[i] = xb[i] ? 1 : 0;
  }
  if (P.energy) {
    __syncthreads();
    const double ea = sparse_energy(P.rowptr, P.col, P.val, P.bias, P.N, xa, red);
    const double eb = sparse_energy(P.rowptr, P.col, P.val, P.bias, P.N, xb, red);
    if (threadIdx.x == 0) {
      P.energy[a] = ea;
      P.energy[b] = eb;
    }
  }
}

}  // namespace

extern "C" {

int64_t tsu_sparse_houdayer_work_bytes(int n_pairs, int N) {
  if (n_pairs < 1 || N < 1 || N > kMaxSites || N <= kResidentSites) return 0;
  return (int64_t)n_pairs * (int64_t)labels_bytes(N);
}

int tsu_sparse_houdayer(const int32_t* d_rowptr, const int32_t* d_col, const double* d_val, const double* d_bias,
                        uint8_t* d_state, int n_chains, int N, const int32_t* d_pairs, int n_pairs, uint64_t seed,
                        uint32_t step0, int n_steps, uint32_t chain0, double* d_energy, void* d_work,
                        size_t work_bytes, uintptr_t stream) {
  TSU_CHECK_ARG(d_rowptr && d_col && d_val && d_state && d_pairs);
  TSU_CHECK_ARG(N > 0 && N <= kMaxSites && n_steps >= 0 && n_pairs >= 1 && 2LL * n_pairs <= n_chains);
  const bool resident = N <= kResidentSites;
  const size_t per_pair = resident ? 0 : labels_bytes(N);
  TSU_CHECK_ARG(resident || (d_work && ((uintptr_t)d_work & 15) == 0 && work_bytes >= per_pair));
  if (n_steps == 0) return TSU_OK;
  HoudayerParams P;
  P.rowptr = d_rowptr;
  P.col = d_col;
  P.val = d_val;
  P.bias = d_bias;
  P.state = d_state;
  P.pairs = d_pairs;
  P.energy = d_energy;
  P.work = static_cast<char*>(d_work);
  P.n_chains = n_chains;
  P.N = N;
  P.pair0 = 0;
  P.n_steps = n_steps;
  P.k0 = (uint32_t)seed;
  P.k1 = (uint32_t)(seed >> 32);
  P.step0 = step0;
  P.chain0 = chain0;
  const cudaStream_t st = tsu_stream(stream);
  const int threads = sparse_threads(N);  // the sweep kernel's: the energies' summation order depends on it
  if (resident) {
    const size_t smem = resident_smem(N);
    if (smem > 48 * 1024) {
      const cudaError_t e = cudaFuncSetAttribute(sparse_houdayer_kernel<true>,
                                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
    }
    sparse_houdayer_kernel<true><<<n_pairs, threads, smem, st>>>(P);
    TSU_RETURN_LAUNCH_STATUS();
  }
  // chunks one after the other, each through all its steps: pairs are disjoint, so the bits depend on no chunk size
  const long long fit = (long long)(work_bytes / per_pair);
  const int chunk = fit < n_pairs ? (int)fit : n_pairs;
  for (int p0 = 0; p0 < n_pairs; p0 += chunk) {
    P.pair0 = p0;
    sparse_houdayer_kernel<false><<<p0 + chunk < n_pairs ? chunk : n_pairs - p0, threads, 0, st>>>(P);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
  }
  return TSU_OK;
}

}  // extern "C"
