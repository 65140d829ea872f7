// Dense-coupling Gibbs sampler on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), sm_100a.
//
// Replaces, for a batch of chains that share one coupling matrix (BASELINE config 3: N = 4096 spins,
// 2048 chains), the local-field evaluation of the reference
//     h_i = np.dot(coupling[i, :], state) + bias[i]                 tsu/gibbs.py:79-100
// inside the sequential sweep of tsu/gibbs.py:128-162.
//
// Exact sequential Gibbs, blocked on two levels.  The N sites are visited in index order.
//   * PANEL (128 sites): the fields of a panel's sites for the CTA's chains are one M x 128 x N GEMM
//     H = S . J[panel, :]^T  (S: current bits as bf16, J: bf16, fp32 accumulation in TMEM), issued as
//     tcgen05.mma M128 (or M64) N128 K16 instructions by one elected thread.  The K-chunk that holds the previous
//     panel is multiplied last, after that panel's update; all other chunks overlap with it.
//   * BLOCK (32 sites, four per panel): the epilogue thread of each chain reads the block's 32 fields out of
//     TMEM, walks the sites in order, draws the heat-bath bit and applies the rank-1 correction
//     h_i' += J[i', i] * (new_i - old_i) to the not yet visited sites of the block in registers (packed dual-fp32
//     FMAs, fma.rn.f32x2 -> FFMA2: the chain is bound by the FMA pipe).  The flips of the block are then
//     written to TMEM as an M x 32 operand (-2 / 0 / +2) and ONE small MMA
//     H[:, later blocks of the panel] += delta . J[later, block]^T  corrects the rest of the panel.
// The result is identical to a site-by-site sweep with the same fields.
//
// One CTA owns M = 128 chains (TMEM lane = chain), or 64 while 64-chain tiles still fit in one wave of the SMs.
// The chain states stay resident in shared memory as bits for the whole call.  Each K-chunk of 128 sites is
// expanded to bf16 by the thread that owns the chain and written straight into TENSOR MEMORY (tcgen05.st,
// lane = chain, column = K pair): the spin operand A never touches shared memory.  A spin is encoded as 0.0 / 2.0:
// bf16 2.0 = 0x4000 has ONE set bit, so a packed pair of spins is (word << s) & 0x40004000 - two integer
// instructions per register - and the accumulated field is halved (exactly) in the epilogue.  The matching J
// tile (operand B, 128 x 128, K-major) is fetched by TMA (cp.async.bulk.tensor.2d, two 64-column boxes with the
// 128-byte swizzle the UMMA descriptor expects) into a 3-stage ring; J (32 MB at N = 4096) stays L2-resident.
//
// Acceptance: u < sigmoid(h / T)  <=>  h > T * logit(u) (strict, gibbs.py:126), thresholds T * logit(u) clamped to
// +-20 T (the reference's sigmoid clamp, gibbs.py:65-70), u = 24-bit Philox uniform, logit via lg2.approx in fp32,
// produced one block ahead by two dedicated warps.  Against the float64 rule the kernel can only disagree where u
// lies within ~5e-6 (exactly representable J) / ~5e-5 (Gaussian J, N <= 4096) of the acceptance probability; the
// tests count those sites and check the bound (tests/test_dense_gpu.py, tests/test_dense_tc_kernel_gpu.py).
//
// Warp roles (16 warps): 0-7 two producer groups (TMA requests + spin expansion), 8-11 epilogue, 12 main MMA
// issuer, 13 in-panel correction issuer, 14-15 thresholds.

#include <cstdlib>
#include <type_traits>
#include <cuda.h>  // CUtensorMap (types only; the encoder is fetched through cudaGetDriverEntryPoint)
#include <cuda_bf16.h>

#include "common.cuh"
#include "philox.cuh"

namespace {

constexpr int kChains = 128;  // TMEM lanes = threads per role group; chains per CTA = UMMA M = kM (128 or 64, template parameter)
constexpr int kBlk = 32;      // sites per block (sequential update unit of the epilogue)
constexpr int kKC = 128;      // K-chunk (sites) per pipeline stage
constexpr int kPanel = 128;   // sites per panel = UMMA N of the main GEMM; a panel is also exactly one K-chunk
constexpr int kStages = 3;    // ring: expanded spin tile in tensor memory (64 columns) + J tile in shared memory (32 KB)
constexpr int kGroups = 2;    // producer groups: chunk g of the global sequence goes to group g % kGroups
constexpr int kACols = kKC / 2;              // 32-bit columns of one expanded spin tile
constexpr int kAccCols = 2 * kPanel;         // two panel accumulators (fp32, 128 columns each)
constexpr int kDeltaCol = kAccCols + kStages * kACols;  // 16 columns: flips of one block as bf16 pairs
static_assert(kDeltaCol + kBlk / 2 <= 512, "tensor memory budget");
static_assert(kPanel == kKC && kPanel == 4 * kBlk, "panel = chunk = four blocks");

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor for the 128-byte swizzled K-major layout TMA writes (rows of 64 bf16 = 128 bytes,
// 8-row groups of 1024 bytes):
// SBO = 1024, LBO unused, layout type 2 = SWIZZLE_128B; a K = 16 step advances the start address by 32 bytes
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// instruction descriptor: D = F32, A = B = BF16, both K-major, M x N
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// tcgen05.mma, A operand in tensor memory (lane = row, one 32-bit column = two consecutive K elements), B from shared memory
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}

// 16 consecutive 32-bit columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n"
      :
      : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}\n" : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// one 64 x 128 box (K x rows) of the bf16 matrix behind `tmap` -> 16 KB of shared memory, completion on `bar`
__device__ __forceinline__ void tma_load_2d(void* smem, const CUtensorMap* tmap, int x, int y, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(smem)),
      "l"(tmap), "r"(x), "r"(y), "r"(smem_u32(bar))
      : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!done);
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 32 consecutive fp32 accumulator columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

#ifdef TSU_TC_TIMING  // per-role stall accounting, see tools/tc_timing.py
__device__ unsigned long long g_tc_timing[32];
#define TC_T0() long long t0__ = clock64()
#define TC_ACC(i) do { if (blockIdx.x == 0 && (threadIdx.x & 31) == 0) atomicAdd(&g_tc_timing[i], (unsigned long long)(clock64() - t0__)); } while (0)
#define TC_NEXT(i) do { const long long t1__ = clock64(); if (blockIdx.x == 0 && (threadIdx.x & 31) == 0) atomicAdd(&g_tc_timing[i], (unsigned long long)(t1__ - t0__)); t0__ = t1__; } while (0)
#else
#define TC_NEXT(i) do {} while (0)
#define TC_T0() do {} while (0)
#define TC_ACC(i) do {} while (0)
#endif

#ifdef TSU_TC_DEBUG_SWITCHES
#define TC_DBG(P, bit) ((P).dbg & (bit))
#else
#define TC_DBG(P, bit) 0
#endif

struct TcParams {
  const __nv_bfloat16* J;   // [N][N] row-major coupling matrix (row i = couplings INTO site i)
  const float* bias;        // [N] or nullptr
  uint8_t* state;           // [n_chains][N] bits, updated in place
  float* fields_out;        // diagnostics: [n_chains][N] field of every site at the time it was visited
  const double* T_chain;    // [n_chains] or nullptr
  int n_chains, N, n_sweeps;
  float T;
  uint32_t k0, k1, sweep0, chain0;
  int gemm_only;            // diagnostics: no spin update (fields of the initial state for every site)
  int dbg;                  // knock-out switches of timing experiments; always 0 unless built with -DTSU_TC_DEBUG_SWITCHES
  // energy pass (dense_tc_kernel<kM, true>): read by that instantiation only
  double* energy;           // [n_chains] -1/2 s^T J s - b^T s of the state
  double* best_energy;      // [n_chains] lowest energy so far, or nullptr (then best_state is nullptr too)
  uint8_t* best_state;      // [n_chains][N] the state that had it
};

constexpr int kProducers = 128 * kGroups;           // warps 0-7: 4 warps (128 chains) per group
constexpr int kEpilogue0 = kProducers / 32;         // warps 8-11: epilogue (thread = chain = TMEM lane)
constexpr int kIssuer0 = kEpilogue0 + 4;            // warp 12: main GEMM issuer, warp 13: in-panel correction issuer
constexpr int kThresh0 = kIssuer0 + 2;              // warps 14-15: acceptance thresholds (Philox + logit), two chains per thread
constexpr int kThreads = 32 * (kThresh0 + 2);       // 512

// position of site i (0-31 of a block) inside a state word: even sites in the low half, odd sites in the high
// half, so that (word >> j) & 0x00010001 is the pair (2j, 2j+1)
__host__ __device__ constexpr int site_bit(int i) { return (i >> 1) + 16 * (i & 1); }

// J tile in shared memory as TMA writes it: two K halves of 64 sites, each 128 rows (sites n) x 128 bytes, 128-byte swizzle
constexpr int kTileBytes = kPanel * kKC * 2;   // 32 KB
constexpr int kHalfBytes = kTileBytes / 2;     // one TMA box
struct __align__(1024) JTile {
  unsigned char bytes[kTileBytes];
};

// shared memory carve-up (~213 KB; the J tiles need 1024-byte alignment for the swizzle)
struct TcSmem {
  uint32_t sbits[4096 / 32][kChains];        // chain states, word-major: sbits[w][chain], bit order = site_bit()
  JTile b[kStages];                          // J[panel rows, chunk columns]
  JTile jdiag;                               // J[panel rows, panel columns]: operand of the in-panel corrections
  __align__(16) float jblk[2][kBlk][kBlk + 4];  // J[blk, blk] as fp32, transposed: jblk[.][i][i'] = J[i0+i'][i0+i]; block g in buffer g & 1
  float thr[kBlk][kChains];                  // acceptance thresholds T * logit(u) of one block, thr[site][chain]
  __align__(8) uint64_t full[kStages];       // producers -> issuer: A slot written (one arrival per warp) + J tile landed (TMA bytes)
  __align__(8) uint64_t empty[kStages];      // issuer -> producers: the MMAs reading the stage are done        (commit)
  __align__(8) uint64_t acc_full[2];         // issuer -> epilogue: main GEMM of the panel complete             (commit)
  __align__(8) uint64_t acc_free[2];         // epilogue -> issuer: accumulator buffer read out     (one arrival per warp)
  __align__(8) uint64_t panel_done[4];       // epilogue -> producers: bits of panel gp written (ring, one arrival per warp)
  __align__(8) uint64_t delta_ready;         // epilogue -> correction issuer: flips of a block are in TMEM (per warp)
  __align__(8) uint64_t thr_full;            // threshold warps -> epilogue: thresholds of the next block written (per warp)
  __align__(8) uint64_t thr_free;            // epilogue -> threshold warps: thresholds are in registers       (per warp)
  __align__(8) uint64_t jdiag_full;          // TMA -> correction issuer: jdiag of the panel landed
  __align__(8) uint64_t corr_done;           // correction issuer -> epilogue: the rest of the panel is corrected (commit)
  uint32_t tmem_base;
};

// acc[ip] += row[ip] * s for ip = first .. 31 (the rank-1 corrections of the sequential block update) with the packed
// dual-fp32 FMA of sm_100 (fma.rn.f32x2 -> FFMA2: two IEEE fp32 FMAs per instruction, same rounding as fmaf): half the
// instructions on the pipe the epilogue shares with everybody else.  `row` is a 16-byte aligned shared-memory row.
__device__ __forceinline__ void ffma2(float& a0, float& a1, float j0, float j1, unsigned long long ss) {
  unsigned long long jj, aa;
  asm("mov.b64 %0, {%1, %2};" : "=l"(jj) : "f"(j0), "f"(j1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(aa) : "f"(a0), "f"(a1));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(aa) : "l"(jj), "l"(ss));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(aa));
}

template <int kFirst>
__device__ __forceinline__ void axpy_tail(float (&acc)[32], const float* __restrict__ row, float s) {
  if constexpr ((kFirst & 1) != 0) acc[kFirst] = fmaf(row[kFirst], s, acc[kFirst]);
  constexpr int kPair0 = (kFirst + 1) & ~1;       // first even index
  constexpr int kQuad0 = (kPair0 + 3) & ~3;       // first index that is a multiple of 4
  unsigned long long ss;
  asm("mov.b64 %0, {%1, %1};" : "=l"(ss) : "f"(s));
  if constexpr (kPair0 < kQuad0 && kPair0 < 32) {  // one 8-byte load up to the 16-byte boundary
    const float2 j2 = *reinterpret_cast<const float2*>(row + kPair0);
    ffma2(acc[kPair0], acc[kPair0 + 1], j2.x, j2.y, ss);
  }
#pragma unroll
  for (int ip = kQuad0; ip < 32; ip += 4) {       // 16-byte loads: one LDS.128 feeds two FFMA2
    const float4 j4 = *reinterpret_cast<const float4*>(row + ip);
    ffma2(acc[ip], acc[ip + 1], j4.x, j4.y, ss);
    ffma2(acc[ip + 2], acc[ip + 3], j4.z, j4.w, ss);
  }
}

// compile-time loop over the 32 sites of a block: f(integral_constant<i>)
template <int I, typename F>
__device__ __forceinline__ void for_each_site(F&& f) {
  if constexpr (I < 32) {
    f(std::integral_constant<int, I>{});
    for_each_site<I + 1>(f);
  }
}

// log2 without the denormal pre-scaling of __log2f (the arguments are 0 or >= 2^-24)
__device__ __forceinline__ float lg2_ftz(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// all lanes have done their part: one lane arrives for the warp (__syncwarp orders the lanes' writes before it)
__device__ __forceinline__ void warp_arrive(uint64_t* bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}
__device__ __forceinline__ void named_bar_sync(int id, int n) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory");
}

// chain (row of the M x N tile) served by thread t (0..127) of a role group.  UMMA M = 128: TMEM lane = row.
// UMMA M = 64: row m lives in lane 32 (m / 16) + m % 16, i.e. the lower half of every 32-lane quarter; the
// upper-half threads shadow their lower twins (same loads, same arithmetic, no stores).
template <int kM>
__device__ __forceinline__ int chain_row(int t) {
  return kM == 128 ? t : 16 * (t >> 5) + (t & 15);
}
template <int kM>
__device__ __forceinline__ bool chain_lane_active(int t) {
  return kM == 128 || (t & 31) < 16;
}

// bits of row `row` of sm.sbits -> dst[0 .. N-1] as uint8 (the layout of the state arrays).  The sweep's final-state
// write keeps its own copy of this loop: calling this function there changes the sweep's instruction schedule.
__device__ __forceinline__ void unpack_bits(const TcSmem& sm, int row, int N, uint8_t* dst) {
  for (int w = 0; w < N / 32; ++w) {
    const uint32_t x = sm.sbits[w][row];
    uint8_t* d = dst + 32 * w;
#pragma unroll
    for (int b = 0; b < 32; b += 4) {
      const uint32_t e2 = x >> (b >> 1), o2 = x >> (16 + (b >> 1));
      *reinterpret_cast<uint32_t*>(d + b) = (e2 & 1u) | ((o2 & 1u) << 8) | ((e2 & 2u) << 15) | ((o2 & 2u) << 23);
    }
  }
}

// kEnergy = false: the sweep (or, with P.gemm_only, the fields of the initial state for diagnostics).
// kEnergy = true: the energy pass - the main GEMM of every panel (as gemm_only) and, per chain, the energy
// -1/2 s.f - s.b summed in float64 over the sites in index order, with optional best-state tracking.  A separate
// instantiation, so that none of it costs the register-bound sweep anything.
template <int kM, bool kEnergy>
__global__ void __launch_bounds__(kThreads, 1) dense_tc_kernel(TcParams P, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // round the base up to 1024 bytes in the SHARED address space (keeps the compiler on LDS/STS)
  TcSmem& sm = *reinterpret_cast<TcSmem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
  const int tid = threadIdx.x, warp = tid >> 5;
  const int N = P.N;
  const int n_panels = N / kPanel;  // = number of K-chunks
  const int total_panels = n_panels * P.n_sweeps;
  const bool gemm_only = kEnergy || P.gemm_only;

  // ---- one-time setup -------------------------------------------------------------------------
  if (tid < kM) {  // pack this chain's bits
    const int chain = blockIdx.x * kM + tid;
    for (int w = 0; w < N / 32; ++w) {
      uint32_t x = 0;
      if (chain < P.n_chains) {
        const uint8_t* src = P.state + (size_t)chain * N + 32 * w;
#pragma unroll
        for (int b = 0; b < 32; b += 4) {
          const uint32_t v = *reinterpret_cast<const uint32_t*>(src + b);  // sites b .. b+3
          x |= ((v & 1u) | ((v >> 15) & 2u)) << (b >> 1);                  // even sites b, b+2
          x |= (((v >> 8) & 1u) | ((v >> 23) & 2u)) << (16 + (b >> 1));    // odd sites b+1, b+3
        }
      }
      sm.sbits[w][tid] = x;
    }
  }
  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&sm.full[s], 5);
      mbar_init(&sm.empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&sm.acc_full[s], 1);
      mbar_init(&sm.acc_free[s], 4);
    }
    for (int s = 0; s < 4; ++s) mbar_init(&sm.panel_done[s], 4);
    mbar_init(&sm.delta_ready, 4);
    mbar_init(&sm.corr_done, 1);
    mbar_init(&sm.jdiag_full, 1);
    mbar_init(&sm.thr_full, 2);
    mbar_init(&sm.thr_free, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kIssuer0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&sm.tmem_base)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = sm.tmem_base;

  if (warp < kEpilogue0) {
    // ===================== producers: stream J tiles, expand spins to bf16 A tiles ======================
    // group q = warp / 4 handles the chunks g = q, q + kGroups, ... of the global sequence (panel-major);
    // thread = chain (TMEM lane)
    const int q = warp >> 2, row = chain_row<kM>(tid & (kChains - 1));
    int done_seen = 0;  // number of panel_done phases consumed
    long long g = 0;
    int s = 0;          // stage of chunk g
    uint32_t round = 0; // g / kStages: how often the ring has wrapped
    for (int gp = 0; gp < total_panels; ++gp) {
      const int p = gp % n_panels;
      for (int cc = 0; cc < n_panels; ++cc, ++g) {
        if ((int)(g % kGroups) == q) {
          // chunk order: own, own + 1, ..., own - 2 and LAST own - 1, the previous panel, which has to be
          // updated first; everything earlier only needs the state as of two panels ago
          int kc = p + cc;
          if (kc >= n_panels) kc -= n_panels;
          if (round > 0) {  // the MMAs of chunk g - kStages (the other group's, for an odd ring) are done: the stage is free
            TC_T0();
            mbar_wait(&sm.empty[s], (round - 1u) & 1u);  // completion number `round` of this stage's barrier
            if ((warp & 3) == 0) TC_ACC(3 + 4 * q);
          }
          TC_T0();
          if ((tid & (kChains - 1)) == 0) {  // J[panel p rows, chunk kc columns]: two 16 KB boxes, bytes counted on the stage's full barrier
            if (TC_DBG(P, 4)) {
              mbar_arrive(&sm.full[s]);
            } else {
              mbar_arrive_expect_tx(&sm.full[s], kTileBytes);
              tma_load_2d(sm.b[s].bytes, &tmap, kc * kKC, p * kPanel, &sm.full[s]);
              tma_load_2d(sm.b[s].bytes + kHalfBytes, &tmap, kc * kKC + 64, p * kPanel, &sm.full[s]);
            }
          }
          if (warp == 0) TC_NEXT(16);
          const int need = (cc == n_panels - 1) ? gp : gp - 1;
          while (done_seen < need) {
            mbar_wait(&sm.panel_done[done_seen & 3], (uint32_t)((done_seen >> 2) & 1));
            ++done_seen;
          }
          if (warp == 0) TC_NEXT(4);
          // 128 bits of this chain -> 64 packed bf16 pairs -> 64 TMEM columns of the chain's lane
          const uint32_t a_col = tmem_d + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(kAccCols + s * kACols);
#pragma unroll
          for (int w4 = 0; w4 < kKC / 32 && !(TC_DBG(P, 2)); ++w4) {
            const uint32_t w = sm.sbits[(kKC / 32) * kc + w4][row];
            uint32_t r[16];
#pragma unroll
            for (int j = 0; j < 15; ++j) r[j] = (w << (14 - j)) & 0x40004000u;  // sites 2j (low half), 2j+1 (high half)
            r[15] = (w >> 1) & 0x40004000u;
            tmem_st16(a_col + 16 * w4, r);
          }
          if (warp == 0) TC_NEXT(17);
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
          if (warp == 0) TC_NEXT(18);
          tc_fence_before();
          warp_arrive(&sm.full[s]);
          if (warp == 0) TC_NEXT(20);
        }
        if (++s == kStages) {
          s = 0;
          ++round;
        }
      }
    }
  } else if (warp == kIssuer0) {
    // ===================== main GEMM issuer: one elected lane feeds the tensor core ======================
    // The whole warp runs the loop (uniform control flow keeps counters and descriptors in uniform registers);
    // only the tcgen05.mma / commit instructions are issued by the elected lane.
    const uint32_t idesc = umma_idesc(kM, kPanel);
    const uint64_t b_desc0 = umma_desc_sw128(smem_u32(sm.b[0].bytes));
    constexpr uint32_t kSlotUnits = (uint32_t)(kTileBytes >> 4);  // 16-byte units per ring slot
    uint32_t full_phase = 0, free_phase = 0;
    int s = 0;
    for (int gp = 0; gp < total_panels; ++gp) {
      const int buf = gp & 1;
      if (gp >= 2) {  // the epilogue has read this accumulator buffer out
        TC_T0();
        mbar_wait(&sm.acc_free[buf], (free_phase >> buf) & 1u);
        free_phase ^= 1u << buf;
        TC_ACC(2);
      }
      const uint32_t d0 = tmem_d + (uint32_t)(buf * kPanel);
      for (int cc = 0; cc < n_panels; ++cc) {
        {
          TC_T0();
          mbar_wait(&sm.full[s], (full_phase >> s) & 1u);
          TC_ACC(0);
        }
        full_phase ^= 1u << s;
        TC_T0();
        tc_fence_after();
        TC_NEXT(21);
        if (elect_one()) {
          const uint64_t bd0 = b_desc0 + (uint64_t)((uint32_t)s * kSlotUnits);
          const uint32_t a0 = tmem_d + (uint32_t)(kAccCols + s * kACols);
#pragma unroll
          for (int j = 0; j < kKC / 16 && !(TC_DBG(P, 1)); ++j)
            umma_bf16_ts(d0, a0 + 8u * j, bd0 + (uint64_t)(((j >> 2) * kHalfBytes + (j & 3) * 32) >> 4), idesc,
                         (cc > 0 || j > 0) ? 1u : 0u);
          umma_commit(&sm.empty[s]);
          if (cc == n_panels - 1) umma_commit(&sm.acc_full[buf]);
        }
        __syncwarp();
        TC_NEXT(22);
        if (++s == kStages) s = 0;
      }
    }
  } else if (warp == kIssuer0 + 1) {
    // ===================== correction issuer: H[:, later blocks] += delta(block b) . J[later, block b]^T ====
    if (!gemm_only) {
      const uint64_t jd_desc0 = umma_desc_sw128(smem_u32(sm.jdiag.bytes));
      uint32_t ready_phase = 0;
      for (int gp = 0; gp < total_panels; ++gp) {
        const uint32_t d0 = tmem_d + (uint32_t)((gp & 1) * kPanel);
        for (int b = 0; b < 3; ++b) {
          TC_T0();
          mbar_wait(&sm.delta_ready, ready_phase);
          ready_phase ^= 1u;
          if (b == 0) mbar_wait(&sm.jdiag_full, (uint32_t)(gp & 1));  // J[panel, panel] has landed
          TC_NEXT(23);
          tc_fence_after();
          if (elect_one()) {
            const int n_cols = kPanel - kBlk * (b + 1);               // columns (sites) of the blocks still to come
            const uint32_t idesc = umma_idesc(kM, n_cols);
            // rows (sites) 32 (b+1) .. 127 of jdiag (8-row groups of 1024 bytes), K = sites 32 b .. 32 b + 31 of the panel
            const uint64_t bd = jd_desc0 + (uint64_t)(((uint32_t)(b >> 1) * kHalfBytes + (uint32_t)(4 * (b + 1)) * 1024u + (uint32_t)(b & 1) * 64u) >> 4);
#pragma unroll
            for (int j = 0; j < kBlk / 16; ++j)
              umma_bf16_ts(d0 + (uint32_t)(kBlk * (b + 1)), tmem_d + (uint32_t)(kDeltaCol + 8 * j), bd + (uint64_t)(2 * j), idesc, 1u);
            umma_commit(&sm.corr_done);
          }
          __syncwarp();
          TC_NEXT(24);
        }
      }
    }
  } else if (warp >= kThresh0) {
    // ===================== threshold warps: T * logit(u) for every (chain, site), one block ahead ===========
    //   u < sigmoid(h / T)  <=>  h > T * logit(u)          (gibbs.py:61-77,126; strict <)
    // and the clamp of gibbs.py:65-70 (|h/T| > 20 -> p = 1 / 0) is the clamp of the threshold to +-20 T.
    // This takes Philox, exp and the division off the epilogue's site-to-site dependency chain.
    if (!gemm_only) {
      const int t = tid - 32 * kThresh0;  // 0..63: chains t and (M = 128) t + 64 of the tile
      constexpr int kPer = kM / 64;
      float Tc[kPer];
      uint32_t cg[kPer];
#pragma unroll
      for (int c = 0; c < kPer; ++c) {
        const int chain = blockIdx.x * kM + t + 64 * c;
        Tc[c] = P.T_chain ? (float)P.T_chain[chain < P.n_chains ? chain : 0] : P.T;
        cg[c] = P.chain0 + (uint32_t)chain;
      }
      const int total_blk = total_panels * 4;
      for (int gblk = 0; gblk < total_blk; ++gblk) {
        const int gp = gblk >> 2, p = gp % n_panels, sweep = gp / n_panels;
        const int i0 = (4 * p + (gblk & 3)) * kBlk;
        // compute into registers first: this overlaps with the epilogue still using the previous block's thresholds
        float v[kPer][kBlk];
#pragma unroll
        for (int c = 0; c < kPer; ++c) {
#pragma unroll
          for (int i = 0; i < kBlk && (TC_DBG(P, 16)); ++i) v[c][i] = 0.0f;
#pragma unroll
          for (int i = 0; i < kBlk && !(TC_DBG(P, 16)); i += 4) {
            const tsu_u32x4 o = tsu_philox4x32_10((uint32_t)((i0 + i) >> 2), cg[c], P.sweep0 + (uint32_t)sweep,
                                                  TSU_STREAM_DENSE_TC, P.k0, P.k1);
            const uint32_t r4[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float u = (float)(r4[k] >> 8) * (1.0f / 16777216.0f);  // 24-bit uniform, exact in fp32
              const float lg = (lg2_ftz(u) - lg2_ftz(1.0f - u)) * 0.69314718056f;  // u = 0 -> -inf -> clamped
              v[c][i + k] = fminf(fmaxf(lg, -20.0f), 20.0f) * Tc[c];
            }
          }
        }
        if (gblk > 0) mbar_wait(&sm.thr_free, (uint32_t)((gblk - 1) & 1));  // the previous block's thresholds are in registers
#pragma unroll
        for (int c = 0; c < kPer; ++c) {
#pragma unroll
          for (int i = 0; i < kBlk; ++i) sm.thr[i][t + 64 * c] = v[c][i];
        }
        warp_arrive(&sm.thr_full);
      }
    }
  } else {
    // ===================== epilogue: fields out of TMEM, sequential update block by block ================
    const int t128 = tid - kProducers;                   // thread of the role group = TMEM lane
    const int row = chain_row<kM>(t128);                 // chain within the tile
    const int chain = blockIdx.x * kM + row;
    const bool chain_ok = chain < P.n_chains && chain_lane_active<kM>(t128);
    const uint32_t tmem_lane = tmem_d + ((uint32_t)((warp & 3) * 32) << 16);
    uint32_t accf_phase = 0, corr_phase = 0, thr_phase = 0;
    double e1 = 0.0, e2 = 0.0;  // energy pass: sum of s_i f_i and of s_i b_i over the sites visited so far
    // diagonal block J[blk, blk]: 8 bf16 per thread (row i0 + t128/4, columns i0 + 8 (t128%4) ..), fetched one
    // block ahead so that the load latency hides behind the previous block's update
    auto load_diag = [&](int blk) {
      const int i0 = blk * kBlk;
      return __ldg(reinterpret_cast<const uint4*>(P.J + (size_t)(i0 + (t128 >> 2)) * N + i0 + 8 * (t128 & 3)));
    };
    const int n_blocks = N / kBlk;
    auto stage_jblk = [&](int buf2, const uint4& v) {  // diagonal block as fp32, transposed: jblk[i][i'] = J[i0 + i', i0 + i]
      const uint32_t jw[4] = {v.x, v.y, v.z, v.w};
      const int r = t128 >> 2, c0 = 8 * (t128 & 3);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        sm.jblk[buf2][c0 + 2 * e][r] = __uint_as_float(jw[e] << 16);  // bf16 -> fp32 is a 16-bit shift
        sm.jblk[buf2][c0 + 2 * e + 1][r] = __uint_as_float(jw[e] & 0xffff0000u);
      }
    };
    stage_jblk(0, load_diag(0));
    uint4 jd = load_diag(1 % n_blocks);  // always one block ahead of the staged one
    named_bar_sync(1, kChains);
    int gblk = 0;
    for (int gp = 0; gp < total_panels; ++gp) {
      const int p = gp % n_panels, buf = gp & 1;
      // J[panel, panel] for this panel's corrections; the previous panel's corrections are all complete
      if (!gemm_only && t128 == 0) {
        mbar_arrive_expect_tx(&sm.jdiag_full, kTileBytes);
        tma_load_2d(sm.jdiag.bytes, &tmap, p * kPanel, p * kPanel, &sm.jdiag_full);
        tma_load_2d(sm.jdiag.bytes + kHalfBytes, &tmap, p * kPanel + 64, p * kPanel, &sm.jdiag_full);
      }
      for (int b = 0; b < 4; ++b, ++gblk) {
        const int blk = 4 * p + b, i0 = blk * kBlk, jb = gblk & 1;
#ifdef TSU_TC_TIMING
        long long tb__ = clock64();
#define TC_B(i) do { const long long t1__ = clock64(); if (blockIdx.x == 0 && tid == kProducers) atomicAdd(&g_tc_timing[i], (unsigned long long)(t1__ - tb__)); tb__ = t1__; } while (0)
#else
#define TC_B(i) do {} while (0)
#endif
        // Thresholds of the block (threshold warps) -> registers.  The site-to-site dependency chain of the update is:
        // compare -> new - old -> packed fma into the fields of the sites still to come.
        float thr[kBlk];
        const uint32_t w_old = sm.sbits[blk][row];
        if (!gemm_only) {
          mbar_wait(&sm.thr_full, thr_phase);
          thr_phase ^= 1u;
#pragma unroll
          for (int i = 0; i < kBlk; ++i) thr[i] = sm.thr[i][row];
          warp_arrive(&sm.thr_free);
        }
        TC_B(26);
        {
          TC_T0();
          if (b == 0) {
            mbar_wait(&sm.acc_full[buf], (accf_phase >> buf) & 1u);  // main GEMM of the panel
            accf_phase ^= 1u << buf;
            if (warp == kEpilogue0) TC_ACC(11);
          } else if (!gemm_only) {
            mbar_wait(&sm.corr_done, corr_phase);  // flips of block b - 1 are in the fields of this block
            corr_phase ^= 1u;
            if (warp == kEpilogue0) TC_ACC(13);
          }
        }
        TC_T0();
        TC_B(27);
        tc_fence_after();
        float h[kBlk];
        tmem_ld32(tmem_lane + (uint32_t)(buf * kPanel + b * kBlk), h);
        TC_B(28);
        if (b == 3) {
          tc_fence_before();
          warp_arrive(&sm.acc_free[buf]);  // the tensor core may overwrite this buffer (panel gp + 2)
        }
        // the next block's diagonal couplings go to the other jblk buffer (its previous user, block gblk - 1, is done)
        stage_jblk(jb ^ 1, jd);
        jd = load_diag((blk + 2) % n_blocks);
        if constexpr (kEnergy) {
          // sites in index order: f_i = the field without bias (x0.5 is exact), s_i = the bit as the GEMM saw it
#pragma unroll
          for (int i = 0; i < kBlk; ++i) {
            const bool s = (w_old >> site_bit(i)) & 1u;
            e1 += s ? (double)(h[i] * 0.5f) : 0.0;
            e2 += s && P.bias ? (double)__ldg(P.bias + i0 + i) : 0.0;
          }
        } else {
#pragma unroll
          for (int i = 0; i < kBlk; ++i) h[i] = fmaf(h[i], 0.5f, P.bias ? __ldg(P.bias + i0 + i) : 0.0f);  // spins were 0 / 2
        }
        if (gemm_only) {
          if (!kEnergy && P.fields_out && chain_ok) {
#pragma unroll
            for (int i = 0; i < kBlk; ++i) P.fields_out[(size_t)chain * N + i0 + i] = h[i];
          }
        } else {
          // sequential heat-bath update of the 32 sites of this block for this thread's chain (gibbs.py:153-160)
          static_assert(kBlk == 32, "one state word per block");
          uint32_t w_new = 0;
          for_each_site<0>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
            if (P.fields_out && chain_ok) P.fields_out[(size_t)chain * N + i0 + i] = h[i];  // as compared (diagnostics)
            const bool up = h[i] > thr[i];
            float s_new = up ? 1.0f : 0.0f;
            s_new -= ((w_old >> site_bit(i)) & 1u) ? 1.0f : 0.0f;   // the correction carries new - old: -1, 0 or +1
            w_new |= up ? (1u << site_bit(i)) : 0u;
            // not yet visited sites of the block see the new value (rank-1 correction, branch free)
            if (!(TC_DBG(P, 8))) axpy_tail<i + 1>(h, sm.jblk[jb][i], s_new);
          });
          if (chain_lane_active<kM>(t128)) sm.sbits[blk][row] = w_new;
          TC_B(29);
          if (b < 3) {
            // flips of the block as a bf16 operand in the accumulator's units (spins are 0 / 2): +2 = 0x4000, -2 = 0xC000
            const uint32_t chg = w_new ^ w_old, neg = w_old & ~w_new;
            uint32_t r[16];
#pragma unroll
            for (int j = 0; j < 15; ++j) r[j] = ((chg << (14 - j)) & 0x40004000u) | ((neg << (15 - j)) & 0x80008000u);
            r[15] = ((chg >> 1) & 0x40004000u) | (neg & 0x80008000u);
            tmem_st16(tmem_lane + (uint32_t)kDeltaCol, r);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tc_fence_before();
            warp_arrive(&sm.delta_ready);
            TC_B(30);
          }
        }
        if (b == 3) warp_arrive(&sm.panel_done[gp & 3]);  // release: the producers may expand the chunk holding this panel
        named_bar_sync(1, kChains);  // the next block's jblk is complete, everybody is done with this block's
            if (warp == kEpilogue0) TC_ACC(12);
      }  // release: the producers may expand the chunk holding this panel
    }
    if (!gemm_only && chain_ok) {  // unpack the final bits of this chain
      for (int w = 0; w < N / 32; ++w) {
        const uint32_t x = sm.sbits[w][row];
        uint8_t* dst = P.state + (size_t)chain * N + 32 * w;
#pragma unroll
        for (int b = 0; b < 32; b += 4) {
          const uint32_t e2 = x >> (b >> 1), o2 = x >> (16 + (b >> 1));
          *reinterpret_cast<uint32_t*>(dst + b) = (e2 & 1u) | ((o2 & 1u) << 8) | ((e2 & 2u) << 15) | ((o2 & 2u) << 23);
        }
      }
    }
    if constexpr (kEnergy) {
      if (chain_ok) {
        const double E = -0.5 * e1 - e2;
        P.energy[chain] = E;
        if (P.best_energy && E < P.best_energy[chain]) {  // strict: an equal energy keeps the earlier state (gibbs.py:387-391)
          P.best_energy[chain] = E;
          unpack_bits(sm, row, N, P.best_state + (size_t)chain * N);
        }
      }
    }
  }
  // ---- teardown ----------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == kIssuer0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_d) : "memory");
  }
}

}  // namespace

// 2-D tensor map of the bf16 coupling matrix: box = 64 columns (128 bytes, 128-byte swizzle) x 128 rows
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_j_tensor_map(CUtensorMap* tmap, const void* J, int N) {
  static EncodeTiledFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) return TSU_ERR_UNSUPPORTED;
    encode = reinterpret_cast<EncodeTiledFn>(fn);
  }
  const cuuint64_t dims[2] = {(cuuint64_t)N, (cuuint64_t)N};
  const cuuint64_t strides[1] = {(cuuint64_t)N * 2};
  const cuuint32_t box[2] = {64, (cuuint32_t)kPanel};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(J), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? TSU_OK : TSU_ERR_UNSUPPORTED;
}

template <int kM, bool kEnergy>
static cudaError_t launch_tiles(const TcParams& P, const CUtensorMap& tmap, size_t smem, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(dense_tc_kernel<kM, kEnergy>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  dense_tc_kernel<kM, kEnergy><<<(P.n_chains + kM - 1) / kM, kThreads, smem, st>>>(P, tmap);
  return cudaGetLastError();
}

template <bool kEnergy>
static int launch_tc(const TcParams& P, cudaStream_t st) {
  const size_t smem = sizeof(TcSmem) + 1024;  // slack: the dynamic shared memory base is only guaranteed 16-byte aligned
  CUtensorMap tmap;
  int rc = make_j_tensor_map(&tmap, P.J, P.N);
  if (rc != TSU_OK) return rc;
  // chains per CTA: 128 fills the tensor core's M; with few chains 64 per CTA puts twice as many SMs to work (a
  // tcgen05.mma with M = 64 takes as long as one with M = 128, so this only pays while SMs would otherwise idle).
  // One CTA fits an SM, so 64 is chosen only while its tiles fit one wave: from sm_count * 64 + 1 chains on (9473 on
  // a B200), 64-chain tiles need two waves where 128-chain tiles need one (B200 at its 1000 W power limit, N = 4096,
  // 10 sweeps: 12000 chains 8.05 ms at M = 64, 4.38 ms at M = 128; tools/tc_tile_height.py)
  int sm_count = 0, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
  int m = (P.n_chains + 63) / 64 <= sm_count ? 64 : 128;
  if (const char* env = getenv("TSU_TC_M")) m = atoi(env) == 64 ? 64 : 128;  // tile height override (tests; same bits)
  const cudaError_t e = m == 64 ? launch_tiles<64, kEnergy>(P, tmap, smem, st) : launch_tiles<128, kEnergy>(P, tmap, smem, st);
  return e == cudaSuccess ? TSU_OK : (int)e;
}

extern "C" int tsu_dense_gibbs_tc_run(const void* d_J_bf16, const float* d_bias, uint8_t* d_state, int n_chains, int N,
                                      double T, const double* d_T_chain, int n_sweeps, uint64_t seed, uint32_t sweep0,
                                      uint32_t chain0, float* d_fields_or_null, uintptr_t stream) {
  TSU_CHECK_ARG(d_J_bf16 && d_state && n_chains > 0 && N > 0 && N % 128 == 0 && N <= 4096 && n_sweeps >= 0);
  TSU_CHECK_ARG(d_T_chain || T > 0);
  TcParams P = {};
  P.J = reinterpret_cast<const __nv_bfloat16*>(d_J_bf16);
  P.bias = d_bias;
  P.state = d_state;
  P.fields_out = d_fields_or_null;
  P.T_chain = d_T_chain;
  P.n_chains = n_chains;
  P.N = N;
  P.n_sweeps = n_sweeps;
  P.T = (float)T;
  P.k0 = (uint32_t)seed;
  P.k1 = (uint32_t)(seed >> 32);
  P.sweep0 = sweep0;
  P.chain0 = chain0;
  P.gemm_only = 0;
#ifdef TSU_TC_DEBUG_SWITCHES  // knock-out timing experiments (tools/tc_dbg.py); results are wrong with any bit set
  if (const char* e = getenv("TSU_TC_DEBUG")) P.dbg = atoi(e);
#endif
  return launch_tc<false>(P, tsu_stream(stream));
}

#ifdef TSU_TC_TIMING
extern "C" int tsu_dense_tc_debug_timing(unsigned long long* h_out16, int reset) {
  if (reset) {
    unsigned long long z[32] = {0};
    return (int)cudaMemcpyToSymbol(g_tc_timing, z, sizeof z);
  }
  return (int)cudaMemcpyFromSymbol(h_out16, g_tc_timing, sizeof(unsigned long long) * 32);
}
#endif

extern "C" int tsu_dense_tc_debug_fields(const void* d_J_bf16, const uint8_t* d_state, int n_chains, int N,
                                         float* d_fields, uintptr_t stream) {
  TSU_CHECK_ARG(d_J_bf16 && d_state && d_fields && n_chains > 0 && N > 0 && N % 128 == 0 && N <= 4096);
  TcParams P = {};
  P.J = reinterpret_cast<const __nv_bfloat16*>(d_J_bf16);
  P.state = const_cast<uint8_t*>(d_state);
  P.fields_out = d_fields;
  P.n_chains = n_chains;
  P.N = N;
  P.n_sweeps = 1;
  P.T = 1.0f;
  P.gemm_only = 1;
#ifdef TSU_TC_DEBUG_SWITCHES  // knock-out timing experiments (tools/tc_dbg.py); results are wrong with any bit set
  if (const char* e = getenv("TSU_TC_DEBUG")) P.dbg = atoi(e);
#endif
  return launch_tc<false>(P, tsu_stream(stream));
}

extern "C" int tsu_dense_tc_energy(const void* d_J_bf16, const float* d_bias, const uint8_t* d_state, int n_chains, int N,
                                   double* d_energy, double* d_best_energy, uint8_t* d_best_state, uintptr_t stream) {
  TSU_CHECK_ARG(d_J_bf16 && d_state && d_energy && n_chains > 0 && N > 0 && N % 128 == 0 && N <= 4096);
  TSU_CHECK_ARG((d_best_energy == nullptr) == (d_best_state == nullptr));
  TcParams P = {};
  P.J = reinterpret_cast<const __nv_bfloat16*>(d_J_bf16);
  P.bias = d_bias;
  P.state = const_cast<uint8_t*>(d_state);  // read only: the energy pass never writes the state
  P.n_chains = n_chains;
  P.N = N;
  P.n_sweeps = 1;
  P.T = 1.0f;
  P.gemm_only = 1;
  P.energy = d_energy;
  P.best_energy = d_best_energy;
  P.best_state = d_best_state;
  return launch_tc<true>(P, tsu_stream(stream));
}
