// Population-annealing resampling shared by the lattice (tsu_ising2d_population_anneal, ising2d.cu) and by any back
// end's chain states (tsu_population_resample, population.cu): quantised weights, their prefix sums, one Philox draw per
// population, systematic parents by bisection and the gather.  Nothing here knows how a state is laid out: a row is
// rep_vecs elements of V (uint4 for 16-byte aligned rows, uint8_t otherwise).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"
#include "philox.cuh"

namespace {

// The population is n_pop contiguous blocks of rp replicas, each resampled on its own.  Everything after the weights'
// exp is integer arithmetic, so any decomposition of the sums gives the same bits.  The caller's work buffer holds
// (uint64): prefix[n_replicas] (inclusive prefix sums of the quantised weights within each tile of kPaTile replicas),
// tile_off[n_pop][nt] (tile totals, then their exclusive prefix sums within the population), min_key[n_pop] (order key
// of E_ref) and draw[n_pop] (the step's U).
constexpr int kPaThreads = 256, kPaPerThread = 4, kPaTile = kPaThreads * kPaPerThread, kPaScanThreads = 1024;

struct PopParams {
  int rp, n_pop, nt, s;  // replicas per population, populations, tiles per population, weight shift 62 - ceil(log2 rp)
  unsigned long long* prefix;
  unsigned long long* tile_off;
  unsigned long long* min_key;
  unsigned long long* draw;
};

// the work buffer of tsu_ising2d_population_work_bytes(n_replicas, n_pop) carved as above
inline PopParams pop_params(void* work, int n_replicas, int n_pop) {
  PopParams Q;
  Q.rp = n_replicas / n_pop;
  Q.n_pop = n_pop;
  Q.nt = (Q.rp + kPaTile - 1) / kPaTile;
  int lg = 0;
  while ((1LL << lg) < Q.rp) ++lg;
  Q.s = 62 - lg;
  Q.prefix = static_cast<unsigned long long*>(work);
  Q.tile_off = Q.prefix + n_replicas;
  Q.min_key = Q.tile_off + (size_t)n_pop * Q.nt;
  Q.draw = Q.min_key + n_pop;
  return Q;
}

// float64 -> uint64 with the same order, so that the lowest E is an integer atomicMin
__device__ __forceinline__ unsigned long long order_key(double e) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(e);
  return (b >> 63) ? ~b : b | 0x8000000000000000ull;
}

__device__ __forceinline__ double key_value(unsigned long long k) {
  return __longlong_as_double((long long)((k >> 63) ? k & 0x7fffffffffffffffull : ~k));
}

__device__ __forceinline__ unsigned long long warp_min(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ unsigned long long warp_inclusive_scan(unsigned long long v) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned long long y = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += y;
  }
  return v;
}

// dst[t] = src[t] for t = t0, t0 + stride, ... below n_vecs: accesses of sizeof(V) bytes, four in flight per thread
template <typename V>
__device__ __forceinline__ void copy_vecs(const V* src, V* dst, long long n_vecs, long long t0, long long stride) {
  long long t = t0;
  for (; t + 3 * stride < n_vecs; t += 4 * stride) {
    const V a = src[t], b = src[t + stride], c = src[t + 2 * stride], d = src[t + 3 * stride];
    dst[t] = a;
    dst[t + stride] = b;
    dst[t + 2 * stride] = c;
    dst[t + 3 * stride] = d;
  }
  for (; t < n_vecs; t += stride) dst[t] = src[t];
}

// exp(-x) for x >= 0 with every rounding spelled out (oracle/population_oracle.py, exp_neg, repeats it): n = rint(x / ln 2),
// r = x - n ln 2 with a two-part ln 2, exp(-r) by a degree-13 Horner polynomial in -r, times 2^(s - n).  Only float64
// multiplies and adds rounded to nearest, never contracted: within 1 ulp of exp on [0, 45] and exactly 1 at x = 0.
// q = floor(exp(-x) 2^s); 0 when n > s + 1.
__device__ __forceinline__ unsigned long long quantised_weight(double x, int s) {
  constexpr double kInvLn2 = 0x1.71547652b82fep+0, kLn2Hi = 0x1.62e42fee00000p-1, kLn2Lo = 0x1.a39ef35793c76p-33;
  constexpr double c[14] = {0x1.0p+0, 0x1.0p+0, 0x1.0p-1, 0x1.5555555555555p-3, 0x1.5555555555555p-5,
                            0x1.1111111111111p-7, 0x1.6c16c16c16c17p-10, 0x1.a01a01a01a01ap-13, 0x1.a01a01a01a01ap-16,
                            0x1.71de3a556c734p-19, 0x1.27e4fb7789f5cp-22, 0x1.ae64567f544e4p-26, 0x1.1eed8eff8d898p-29,
                            0x1.6124613a86d09p-33};  // 1/k!
  const double n = rint(__dmul_rn(x, kInvLn2));
  if (n > (double)(s + 1)) return 0ull;
  const double t = -__dsub_rn(__dsub_rn(x, __dmul_rn(n, kLn2Hi)), __dmul_rn(n, kLn2Lo));
  double p = c[13];
#pragma unroll
  for (int k = 12; k >= 0; --k) p = __dadd_rn(__dmul_rn(p, t), c[k]);
  return __double2ull_rz(ldexp(p, s - (int)n));
}

// Quantised weights of one tile of kPaTile replicas of population blockIdx.y (x = dbeta (E - E_ref)), their inclusive
// prefix sums within the tile into Q.prefix and the tile total into Q.tile_off.
__global__ void __launch_bounds__(kPaThreads) pa_weights_kernel(const double* __restrict__ energy,
                                                                const double* __restrict__ dbeta, PopParams Q) {
  const int p = blockIdx.y, tile = blockIdx.x;
  const double db = *dbeta, e_ref = key_value(Q.min_key[p]);
  const size_t base = (size_t)p * Q.rp;
  const int j0 = tile * kPaTile + threadIdx.x * kPaPerThread;
  unsigned long long q[kPaPerThread], run = 0;
#pragma unroll
  for (int m = 0; m < kPaPerThread; ++m) {
    const int j = j0 + m;
    run += j < Q.rp ? quantised_weight(__dmul_rn(db, __dsub_rn(energy[base + j], e_ref)), Q.s) : 0ull;
    q[m] = run;
  }
  __shared__ unsigned long long warp_tot[kPaThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned long long incl = warp_inclusive_scan(run);
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const unsigned long long v = warp_inclusive_scan(lane < kPaThreads / 32 ? warp_tot[lane] : 0ull);
    if (lane < kPaThreads / 32) warp_tot[lane] = v;
  }
  __syncthreads();
  const unsigned long long excl = incl - run + (warp > 0 ? warp_tot[warp - 1] : 0ull);
#pragma unroll
  for (int m = 0; m < kPaPerThread; ++m)
    if (j0 + m < Q.rp) Q.prefix[base + j0 + m] = excl + q[m];
  if (threadIdx.x == kPaThreads - 1) Q.tile_off[(size_t)p * Q.nt + tile] = excl + run;
}

// One block per population: the tile totals become exclusive prefix sums, W = their sum goes to weight_sum[p], E_ref to
// energy_ref[p] (min_key is reset for the next step), and the population's Philox draw u (kind 3) gives
// U = floor(u W / 2^64) in Q.draw[p].
__global__ void __launch_bounds__(kPaScanThreads) pa_scan_kernel(PopParams Q, uint32_t k0, uint32_t k1, uint32_t sweep,
                                                                 uint32_t replica0, unsigned long long* weight_sum,
                                                                 double* energy_ref) {
  const int p = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long* off = Q.tile_off + (size_t)p * Q.nt;
  __shared__ unsigned long long warp_tot[kPaScanThreads / 32];
  unsigned long long carry = 0;  // the same in every thread
  for (int c0 = 0; c0 < Q.nt; c0 += kPaScanThreads) {
    const int t = c0 + threadIdx.x;
    const unsigned long long v = t < Q.nt ? off[t] : 0ull;
    const unsigned long long incl = warp_inclusive_scan(v);
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) warp_tot[lane] = warp_inclusive_scan(warp_tot[lane]);
    __syncthreads();
    if (t < Q.nt) off[t] = carry + incl - v + (warp > 0 ? warp_tot[warp - 1] : 0ull);
    carry += warp_tot[kPaScanThreads / 32 - 1];
    __syncthreads();  // warp_tot is overwritten by the next chunk
  }
  if (threadIdx.x == 0) {
    const unsigned long long W = carry;
    weight_sum[p] = W;
    energy_ref[p] = key_value(Q.min_key[p]);
    Q.min_key[p] = ~0ull;
    const tsu_u32x4 o = tsu_lattice_philox(0u, 0u, TSU_KIND_RESAMPLE, 0u, sweep, replica0 + (uint32_t)p * (uint32_t)Q.rp,
                                           k0, k1);
    Q.draw[p] = __umul64hi((unsigned long long)o.x | ((unsigned long long)o.y << 32), W);
  }
}

// Parent of child j of population p: the smallest i with rp C_i > j W + U (128-bit products), C_i the inclusive prefix
// sum prefix[i] + tile_off[i / kPaTile].  C is non-decreasing and rp C_{rp-1} = rp W > j W + U, so a bisection finds it.
__device__ __forceinline__ int pa_parent(const PopParams& Q, int p, int j, unsigned long long W) {
  const unsigned long long U = Q.draw[p];
  unsigned long long t_lo = (unsigned long long)j * W, t_hi = __umul64hi((unsigned long long)j, W);
  t_lo += U;
  t_hi += t_lo < U ? 1ull : 0ull;
  const unsigned long long* pre = Q.prefix + (size_t)p * Q.rp;
  const unsigned long long* off = Q.tile_off + (size_t)p * Q.nt;
  const unsigned long long rp = (unsigned long long)Q.rp;
  int lo = 0, hi = Q.rp - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const unsigned long long c = pre[mid] + off[mid / kPaTile];
    const unsigned long long c_lo = rp * c, c_hi = __umul64hi(rp, c);
    if (c_hi > t_hi || (c_hi == t_hi && c_lo > t_lo))
      hi = mid;
    else
      lo = mid + 1;
  }
  return lo;
}

// state'[c] = state[parent(c)] and family'[c] = family[parent(c)], a row being rep_vecs elements of V.  group < 256:
// `group` threads (a power of two) per child, 256 / group children per block along x; group == 256: blockIdx.y walks
// the children and blockIdx.x tiles one.
template <typename V>
__global__ void __launch_bounds__(256) pa_gather_kernel(const V* __restrict__ src, V* dst,
                                                        const int32_t* __restrict__ fam_src, int32_t* fam_dst,
                                                        PopParams Q, const unsigned long long* __restrict__ weight_sum,
                                                        long long rep_vecs, int group) {
  const int n = Q.rp * Q.n_pop;
  if (group < 256) {
    const long long c = (long long)blockIdx.x * (256 / group) + threadIdx.x / group;
    if (c >= n) return;
    const int p = (int)(c / Q.rp);
    const size_t parent = (size_t)p * Q.rp + pa_parent(Q, p, (int)(c - (long long)p * Q.rp), weight_sum[p]);
    const int t0 = threadIdx.x & (group - 1);
    copy_vecs(src + parent * rep_vecs, dst + c * rep_vecs, rep_vecs, t0, group);
    if (t0 == 0) fam_dst[c] = fam_src[parent];
    return;
  }
  for (int c = blockIdx.y; c < n; c += gridDim.y) {
    const int p = c / Q.rp;
    const size_t parent = (size_t)p * Q.rp + pa_parent(Q, p, c - p * Q.rp, weight_sum[p]);
    copy_vecs(src + parent * rep_vecs, dst + (size_t)c * rep_vecs, rep_vecs,
              (long long)blockIdx.x * blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x);
    if (blockIdx.x == 0 && threadIdx.x == 0) fam_dst[c] = fam_src[parent];
  }
}

// Steps 2-4 of a resampling step once min_key holds each population's E_ref: the weights of energy[] at *dbeta, the scan
// and draw (lattice stream kind 3 at (sweep, chain0 + p rp)), and the gather of rows of rep_vecs elements of V from src
// to dst with their family entries.  A group of threads per child (at least 4 elements per thread), or whole blocks of
// threads per child for long rows.
template <typename V>
int launch_pa_resample(const PopParams& Q, const double* energy, const double* dbeta, uint64_t seed, uint32_t sweep,
                       uint32_t chain0, unsigned long long* weight_sum, double* energy_ref, const V* src, V* dst,
                       const int32_t* fam_src, int32_t* fam_dst, long long rep_vecs, cudaStream_t st) {
  const long long n = (long long)Q.rp * Q.n_pop;
  int group = 1;
  while (group < 256 && 4LL * group < rep_vecs) group <<= 1;
  dim3 gather_grid;
  if (group < 256) {
    gather_grid = dim3((unsigned)((n + 256 / group - 1) / (256 / group)));
  } else {
    long long bx = (rep_vecs + 4 * 256 - 1) / (4 * 256);
    const long long cap = (148LL * 8 + n - 1) / n;  // about 8 CTAs per SM in total
    if (bx > cap) bx = cap;
    gather_grid = dim3((unsigned)bx, (unsigned)(n < 65535 ? n : 65535));
  }
  pa_weights_kernel<<<dim3((unsigned)Q.nt, (unsigned)Q.n_pop), kPaThreads, 0, st>>>(energy, dbeta, Q);
  pa_scan_kernel<<<Q.n_pop, kPaScanThreads, 0, st>>>(Q, (uint32_t)seed, (uint32_t)(seed >> 32), sweep, chain0,
                                                    weight_sum, energy_ref);
  pa_gather_kernel<V><<<gather_grid, 256, 0, st>>>(src, dst, fam_src, fam_dst, Q, weight_sum, rep_vecs, group);
  TSU_RETURN_LAUNCH_STATUS();
}

}  // namespace
