// 2-D nearest-neighbour Ising lattice: bit-packed checkerboard heat-bath Gibbs update for sm_100a.
//
// Replaces the per-spin Python loop of the reference
//   GibbsSampler.gibbs_sweep / sample_conditional   tsu/gibbs.py:102-162
// for the lattice wired by IsingGrid                 tsu/models/ising.py:320-361
// (and README's IsingModel2D.gibbs_update, README.md:116-131).
//
// Multi-spin coding: one uint32 word = 32 spins of one colour of one row.  For a word the four
// neighbour words (north, south, centre, side-shifted) are reduced to a bit-sliced up-count
// (c2 c1 c0) with 6 LOP3 + 1 funnel shift.  The acceptance test  u < t[class]  (u: 32-bit uniform
// per spin, t: integer threshold = ceil(sigmoid(h/T) * 2^32) from the host LUT) is evaluated
// bit-sliced as well: the top 8 bits of all 32 uniforms are 8 random bit-planes = 2 Philox calls;
// a borrow chain gives "less than" and "equal so far" masks.  Only lanes whose top 8 bits tie with
// the threshold (probability 2^-8) need the low 24 bits, which come from a per-lane-group Philox
// call.  The result is identical to a full 32-bit compare per spin, so it is bit-exact with the
// CPU oracle (oracle/ising2d_oracle.py) and with the reference's `rand() < prob`.
//
// HBM traffic per half-sweep: read the opposite colour once (+2 halo rows per strip), write the
// updated colour once = 2 bits per spin update; the kernel is integer-issue bound, not DRAM bound
// (see DESIGN.md for the roofline arithmetic).

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "common.cuh"
#include "philox.cuh"
#include "ising2d_fast.cuh"
#include "jit.cuh"

namespace {

using tsu_fast::Geom;
using tsu_fast::colour_count;
using tsu_fast::words_per_row;
using tsu_fast::Planes;
using tsu_fast::opp_row;
using tsu_fast::Coords;
using tsu_fast::lattice_call;
using tsu_fast::SweepParams;
using tsu_fast::BondParams;
using tsu_fast::kBondN;
using tsu_fast::kBondS;
using tsu_fast::kBondW;
using tsu_fast::kBondE;

constexpr BondParams kNoBonds = {nullptr, nullptr};

__device__ __forceinline__ uint32_t lane_mask_lt(int n) {  // lanes [0, n), n clamped to [0, 32]
  return n >= 32 ? 0xffffffffu : (n <= 0 ? 0u : ((1u << n) - 1u));
}

// pointers to the two colour planes of one replica
struct Hood {
  uint32_t n, s, c, side;  // neighbour bit words (missing neighbours read 0)
  uint32_t valid;          // own lanes that exist
  uint32_t missW, missE;   // own lanes without a west / east neighbour (open columns)
  int has_n, has_s;
};

__device__ __forceinline__ Hood load_hood(const Planes& P, const Geom& g, int colour, int i, int w) {
  Hood h;
  const int p = (g.row0 + i + colour) & 1;  // column offset of the own colour in this row
  const int nk_own = colour_count(g.cols, p);
  const int nk_opp = colour_count(g.cols, 1 - p);
  h.valid = lane_mask_lt(nk_own - 32 * w);
  const uint32_t* rn = opp_row(P, g, i - 1);
  const uint32_t* rs = opp_row(P, g, i + 1);
  const uint32_t* rc = P.opp + (size_t)i * g.wpr;
  h.has_n = rn != nullptr;
  h.has_s = rs != nullptr;
  h.n = rn ? rn[w] : 0u;
  h.s = rs ? rs[w] : 0u;
  h.c = rc[w];
  h.missW = 0u;
  h.missE = 0u;
  const int last = nk_own - 1;  // last own lane index in the row
  if (p) {
    // own col = 2k+1: west = opp k (centre), east = opp k+1
    uint32_t nx = (w + 1 < g.wpr) ? rc[w + 1] : 0u;
    h.side = (h.c >> 1) | (nx << 31);
    if (last >= 0 && (last >> 5) == w && 2 * last + 2 >= g.cols) {  // east neighbour would be col >= cols
      if (g.wrap_cols)
        h.side |= (rc[0] & 1u) << (last & 31);
      else
        h.missE = 1u << (last & 31);
    }
  } else {
    // own col = 2k: east = opp k (centre), west = opp k-1
    uint32_t pv = (w > 0) ? rc[w - 1] : 0u;
    h.side = (h.c << 1) | (pv >> 31);
    if (w == 0) {
      if (g.wrap_cols) {
        int lo = nk_opp - 1;
        h.side |= (rc[lo >> 5] >> (lo & 31)) & 1u;
      } else {
        h.missW = 1u;
      }
    }
    if (last >= 0 && (last >> 5) == w && 2 * last + 1 >= g.cols) h.missE = 1u << (last & 31);  // odd cols
  }
  return h;
}

// Bonded lattices: XOR the four neighbour words of (colour, local row i, word w) with their bond words, so that every
// count taken from the hood counts bond-satisfying neighbours (absent neighbours keep reading 0: their bits are 0)
__device__ __forceinline__ void apply_bonds(Hood& h, const BondParams& B, const Geom& g, int rep, int colour, int i, int w) {
  const size_t plane = (size_t)g.rows * g.wpr;
  const uint32_t* b = tsu_fast::bond_base(B, g, rep, colour) + (size_t)i * g.wpr + w;
  const int p = (g.row0 + i + colour) & 1;  // own columns odd: the centre word is the west neighbour
  h.n ^= b[kBondN * plane];
  h.s ^= b[kBondS * plane];
  h.c ^= b[(p ? kBondW : kBondE) * plane];
  h.side ^= b[(p ? kBondE : kBondW) * plane];
}

// ---- bit-sliced acceptance -------------------------------------------------------------
struct LutRegs {
  uint32_t K[8][5];  // K[k][u] = all-ones iff bit (31-k) of threshold(d, u) is set
  uint32_t always;   // bit u set: class (d, u) accepts with probability 1 (threshold 2^32)
};

__device__ __forceinline__ void load_lut_regs(LutRegs& L, const uint32_t* __restrict__ lut, int d) {
#pragma unroll
  for (int u = 0; u < 5; ++u) {
    uint32_t t = __ldg(lut + d * 5 + u);
#pragma unroll
    for (int k = 0; k < 8; ++k) L.K[k][u] = 0u - ((t >> (31 - k)) & 1u);
  }
  L.always = (__ldg(lut + 25) >> (d * 5)) & 31u;
}

__device__ __forceinline__ uint32_t bitsel(uint32_t m, uint32_t a, uint32_t b) {  // m ? a : b  (bitwise)
  return (m & a) | (~m & b);
}

// lane j's 32-bit uniform: the top 8 bits from the bit-planes r, the low 24 from call low0 + (j >> 2)
__device__ __forceinline__ uint32_t lane_uniform(const uint32_t r[8], const Coords& q, uint32_t w, uint32_t row_g, int j,
                                                 uint32_t low0 = TSU_KIND_LOW0) {
  uint32_t u = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) u |= ((r[k] >> j) & 1u) << (31 - k);
  tsu_u32x4 lo = lattice_call(q, w, row_g, low0 + (uint32_t)(j >> 2));
  int sel = j & 3;
  uint32_t v = sel == 0 ? lo.x : (sel == 1 ? lo.y : (sel == 2 ? lo.z : lo.w));
  return u | (v >> 8);
}

__device__ __forceinline__ uint32_t lane_accept(const uint32_t* __restrict__ lut, int d, int up, uint32_t u) {
  int cls = d * 5 + up;
  if ((__ldg(lut + 25) >> cls) & 1u) return 1u;
  return u < __ldg(lut + cls) ? 1u : 0u;
}

// New value of one word of the colour being updated.
//   a,b,c,s: neighbour words; d_row: number of neighbours of a regular lane (2 + has_n + has_s);
//   special: lanes with fewer neighbours than d_row (missW | missE), resolved one by one.
template <bool FAST>
__device__ __forceinline__ uint32_t update_word(uint32_t a, uint32_t b, uint32_t c, uint32_t s, const LutRegs& L,
                                                const uint32_t* __restrict__ lut, int d_row, uint32_t valid,
                                                uint32_t missW, uint32_t missE, const Coords& q, uint32_t w,
                                                uint32_t row_g) {
  // bit-sliced count of up neighbours: c2 c1 c0
  const uint32_t s1 = a ^ b ^ c;
  const uint32_t m1 = tsu_lop3_maj(a, b, c);
  const uint32_t c0 = s1 ^ s;
  const uint32_t k2 = s1 & s;
  const uint32_t c1 = m1 ^ k2;
  const uint32_t c2 = m1 & k2;

  uint32_t r[8];
  {
    tsu_u32x4 p0 = lattice_call(q, w, row_g, TSU_KIND_PLANE0);
    tsu_u32x4 p1 = lattice_call(q, w, row_g, TSU_KIND_PLANE1);
    r[0] = p0.x; r[1] = p0.y; r[2] = p0.z; r[3] = p0.w;
    r[4] = p1.x; r[5] = p1.y; r[6] = p1.z; r[7] = p1.w;
  }
  uint32_t lt = 0u, eq = 0xffffffffu;
#pragma unroll
  for (int k = 7; k >= 0; --k) {  // least significant of the 8 planes first
    const uint32_t tk = bitsel(c2, L.K[k][4], bitsel(c1, bitsel(c0, L.K[k][3], L.K[k][2]), bitsel(c0, L.K[k][1], L.K[k][0])));
    const uint32_t x = r[k] ^ tk;
    lt = (~r[k] & tk) | (~x & lt);
    eq &= ~x;
  }
  const uint32_t always = L.always;
  if (always) {  // classes with p == 1.0 (threshold 2^32 does not fit 32 bits)
    uint32_t am = 0u;
    if (always & 1u) am |= ~c2 & ~c1 & ~c0;
    if (always & 2u) am |= ~c2 & ~c1 & c0;
    if (always & 4u) am |= ~c2 & c1 & ~c0;
    if (always & 8u) am |= ~c2 & c1 & c0;
    if (always & 16u) am |= c2;
    lt |= am;
    eq &= ~am;
  }
  uint32_t special = 0u;
  if (!FAST) {
    special = (missW | missE) & valid;
    eq &= valid & ~special;
  }
  // lanes whose top 8 bits tie with the threshold: decide on the full 32-bit uniform
  while (eq) {
    const int j = __ffs(eq) - 1;
    eq &= eq - 1u;
    const int up = ((c0 >> j) & 1u) | (((c1 >> j) & 1u) << 1) | (((c2 >> j) & 1u) << 2);
    const uint32_t bit = lane_accept(lut, d_row, up, lane_uniform(r, q, w, row_g, j));
    lt = (lt & ~(1u << j)) | (bit << j);
  }
  if (!FAST) {
    while (special) {
      const int j = __ffs(special) - 1;
      special &= special - 1u;
      const int up = ((c0 >> j) & 1u) | (((c1 >> j) & 1u) << 1) | (((c2 >> j) & 1u) << 2);
      const int d = d_row - (int)((missW >> j) & 1u) - (int)((missE >> j) & 1u);
      const uint32_t bit = lane_accept(lut, d, up, lane_uniform(r, q, w, row_g, j));
      lt = (lt & ~(1u << j)) | (bit << j);
    }
    lt &= valid;
  }
  return lt;
}

#ifdef TSU_LATTICE_TRACE  // diagnosis build (tools/lattice_trace.py): when and where every CTA of the last launches ran
constexpr int kTraceCtas = 8192;
__device__ unsigned long long g_lat_trace[4][3 * kTraceCtas];  // [launch & 3][cta] = start ns, end ns, SM id
__device__ __forceinline__ unsigned long long trace_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#endif

template <int W, int MINB, bool BONDED>
__global__ void __launch_bounds__(128, MINB) half_sweep_fast_kernel(SweepParams P, BondParams B) {
#ifdef TSU_LATTICE_TRACE
  const unsigned long long t_start = trace_now();
#endif
  tsu_fast::half_sweep_fast_body<W, BONDED>(P, B);
#ifdef TSU_LATTICE_TRACE
  __syncthreads();
  if (threadIdx.x == 0 && blockIdx.x < kTraceCtas) {
    unsigned smid;
    asm("mov.u32 %0, %%smid;" : "=r"(smid));
    unsigned long long* t = g_lat_trace[(P.sweep * 2 + P.colour) & 3] + 3 * blockIdx.x;
    t[0] = t_start;
    t[1] = trace_now();
    t[2] = smid;
  }
#endif
}

// One word of (replica rep, colour, local row i): any size, open or periodic edges, ragged last word.
template <bool BONDED>
__device__ __forceinline__ void generic_update_one(const SweepParams& P, const BondParams& B, int colour, uint32_t sweep,
                                                   int rep, int i, int w) {
  const Geom& g = P.g;
  const size_t plane = (size_t)g.rows * g.wpr;
  uint32_t* own = P.state + ((size_t)rep * 2 + colour) * plane;
  Planes pl;
  pl.opp = P.state + ((size_t)rep * 2 + (1 - colour)) * plane;
  pl.halo_top = P.halo_top ? P.halo_top + (size_t)rep * g.wpr : nullptr;
  pl.halo_bot = P.halo_bot ? P.halo_bot + (size_t)rep * g.wpr : nullptr;
  const uint32_t* lut = P.lut + (P.lut_index ? (size_t)P.lut_index[rep] * 32 : 0);

  Hood h = load_hood(pl, g, colour, i, w);
  if (h.valid == 0u) return;  // padding word (stays 0)
  if constexpr (BONDED) apply_bonds(h, B, g, rep, colour, i, w);
  const int d_row = 2 + h.has_n + h.has_s;
  LutRegs L;
  load_lut_regs(L, lut, d_row);
  Coords q;
  q.colour = (uint32_t)colour;
  q.sweep = sweep;
  q.replica = P.replica0 + (uint32_t)rep;
  q.k0 = P.k0;
  q.k1 = P.k1;
  own[(size_t)i * g.wpr + w] = update_word<false>(h.n, h.s, h.c, h.side, L, lut, d_row, h.valid, h.missW, h.missE, q,
                                                  (uint32_t)w, (uint32_t)(g.row0 + i));
}

// Generic path: one thread per word, one launch per half-sweep.
template <bool BONDED>
__global__ void __launch_bounds__(128) half_sweep_generic_kernel(SweepParams P, BondParams B) {
  // rows [P.row_begin, P.row_end) of every replica
  const Geom& g = P.g;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_rep = (long long)(P.row_end - P.row_begin) * g.wpr;
  if (tid >= per_rep * g.n_replicas) return;
  const int rep = (int)(tid / per_rep);
  const int rem = (int)(tid - (long long)rep * per_rep);
  const int i = rem / g.wpr;
  generic_update_one<BONDED>(P, B, P.colour, P.sweep, rep, P.row_begin + i, rem - i * g.wpr);
}

// Small lattices (C1: 50 x 50): the whole replica belongs to ONE thread block, which runs both colours of
// n_sweeps sweeps in a single launch with a block barrier between half-sweeps.  Same words, same Philox
// coordinates, same bits as the per-half-sweep launches - it only removes 2 n_sweeps - 1 kernel launches,
// which is all the time there is at this size.
constexpr int kResidentThreads = 256;
template <bool BONDED>
__global__ void __launch_bounds__(kResidentThreads) sweeps_resident_kernel(SweepParams P, int n_sweeps, BondParams B) {
  const Geom& g = P.g;
  const int rep = blockIdx.x;
  const int per_rep = g.rows * g.wpr;
  for (int t = 0; t < n_sweeps; ++t) {
    for (int colour = 0; colour < 2; ++colour) {
      for (int rem = threadIdx.x; rem < per_rep; rem += kResidentThreads) {
        const int i = rem / g.wpr;
        generic_update_one<BONDED>(P, B, colour, P.sweep + (uint32_t)t, rep, i, rem - i * g.wpr);
      }
      __syncthreads();  // the other colour reads what this half-sweep wrote (same SM: L1 is coherent for its own stores)
    }
  }
}

// Open boundaries and / or ragged rows: the wide kernel updates, in every row that has both vertical neighbours, the
// 4-word groups whose lanes all exist, as if the columns wrapped at a word boundary; this pass then recomputes, with the true geometry and degree tables, the rim it
// got wrong or skipped: rows [0, rb) and [re, rows) completely and, for open columns, the first and last word of the
// rows in between.  Both passes read only the other colour, so the order of the two launches is the only dependency.
struct RimRows {
  int a0, a1;  // rows [a0, a1) and [b0, b1) are recomputed completely
  int b0, b1;
  int p0, p1;  // of the rows [p0, p1): word 0 if `head`, and the words tail_begin .. wpr-1
  int head, tail_begin;
};

template <bool BONDED>
__global__ void __launch_bounds__(128) half_sweep_rim_kernel(SweepParams P, RimRows R, BondParams B) {
  const Geom& g = P.g;
  const int na = R.a1 - R.a0, nb = R.b1 - R.b0;
  const int full_rows = na + nb;
  const int per_row = R.head + (g.wpr - R.tail_begin);
  const long long per_rep = (long long)full_rows * g.wpr + (long long)per_row * (R.p1 - R.p0);
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= per_rep * g.n_replicas) return;
  const int rep = (int)(tid / per_rep);
  const int rem = (int)(tid - (long long)rep * per_rep);
  int i, w;
  if (rem < full_rows * g.wpr) {
    const int r = rem / g.wpr;
    w = rem - r * g.wpr;
    i = r < na ? R.a0 + r : R.b0 + (r - na);
  } else {
    const int e = rem - full_rows * g.wpr;
    const int r = e / per_row, k = e - r * per_row;
    i = R.p0 + r;
    w = (R.head && k == 0) ? 0 : R.tail_begin + (k - R.head);
  }
  generic_update_one<BONDED>(P, B, P.colour, P.sweep, rep, i, w);
}

// Parity mode: uniforms injected per site.  One thread per word, one lane at a time.
template <bool BONDED>
__global__ void __launch_bounds__(128) half_sweep_injected_kernel(SweepParams P, const uint32_t* __restrict__ uniforms,
                                                                  BondParams B) {
  const Geom& g = P.g;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_rep = (long long)g.rows * g.wpr;
  if (tid >= per_rep * g.n_replicas) return;
  const int rep = (int)(tid / per_rep);
  const int rem = (int)(tid - (long long)rep * per_rep);
  const int i = rem / g.wpr;
  const int w = rem - i * g.wpr;
  const size_t plane = (size_t)g.rows * g.wpr;
  uint32_t* own = P.state + ((size_t)rep * 2 + P.colour) * plane;
  Planes pl;
  pl.opp = P.state + ((size_t)rep * 2 + (1 - P.colour)) * plane;
  pl.halo_top = P.halo_top ? P.halo_top + (size_t)rep * g.wpr : nullptr;
  pl.halo_bot = P.halo_bot ? P.halo_bot + (size_t)rep * g.wpr : nullptr;
  const uint32_t* lut = P.lut + (P.lut_index ? (size_t)P.lut_index[rep] * 32 : 0);
  Hood h = load_hood(pl, g, P.colour, i, w);
  if (h.valid == 0u) return;
  if constexpr (BONDED) apply_bonds(h, B, g, rep, P.colour, i, w);
  const int p = (g.row0 + i + P.colour) & 1;
  const uint32_t* urow = uniforms + ((size_t)rep * g.rows + i) * g.cols;
  uint32_t out = 0u;
  uint32_t m = h.valid;
  while (m) {
    const int j = __ffs(m) - 1;
    m &= m - 1u;
    const int up = ((h.n >> j) & 1u) + ((h.s >> j) & 1u) + ((h.c >> j) & 1u) + ((h.side >> j) & 1u);
    const int d = 2 + h.has_n + h.has_s - (int)((h.missW >> j) & 1u) - (int)((h.missE >> j) & 1u);
    const int col = 2 * (32 * w + j) + p;
    out |= lane_accept(lut, d, up, urow[col]) << j;
  }
  own[(size_t)i * g.wpr + w] = out;
}

__global__ void init_random_kernel(uint32_t* state, Geom g, uint32_t replica0, uint32_t k0, uint32_t k1) {
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_rep = 2LL * g.rows * g.wpr;
  if (tid >= per_rep * g.n_replicas) return;
  const int rep = (int)(tid / per_rep);
  long long rem = tid - (long long)rep * per_rep;
  const int colour = (int)(rem / ((long long)g.rows * g.wpr));
  rem -= (long long)colour * g.rows * g.wpr;
  const int i = (int)(rem / g.wpr);
  const int w = (int)(rem - (long long)i * g.wpr);
  const int p = (g.row0 + i + colour) & 1;
  const uint32_t valid = lane_mask_lt(colour_count(g.cols, p) - 32 * w);
  tsu_u32x4 o = tsu_lattice_philox((uint32_t)w, (uint32_t)colour, TSU_KIND_INIT, (uint32_t)(g.row0 + i), 0u,
                                   replica0 + (uint32_t)rep, k0, k1);
  state[tid] = o.x & valid;
}

__global__ void pack_kernel(const int8_t* __restrict__ spins, uint32_t* state, Geom g) {
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_rep = 2LL * g.rows * g.wpr;
  if (tid >= per_rep * g.n_replicas) return;
  const int rep = (int)(tid / per_rep);
  long long rem = tid - (long long)rep * per_rep;
  const int colour = (int)(rem / ((long long)g.rows * g.wpr));
  rem -= (long long)colour * g.rows * g.wpr;
  const int i = (int)(rem / g.wpr);
  const int w = (int)(rem - (long long)i * g.wpr);
  const int p = (g.row0 + i + colour) & 1;
  const int nk = colour_count(g.cols, p);
  const int8_t* row = spins + ((size_t)rep * g.rows + i) * g.cols;
  uint32_t x = 0u;
  for (int j = 0; j < 32; ++j) {
    int k = 32 * w + j;
    if (k < nk && row[2 * k + p] > 0) x |= 1u << j;
  }
  state[tid] = x;
}

__global__ void unpack_kernel(const uint32_t* __restrict__ state, int8_t* spins, Geom g, int as_pm1) {
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_rep = 2LL * g.rows * g.wpr;
  if (tid >= per_rep * g.n_replicas) return;
  const int rep = (int)(tid / per_rep);
  long long rem = tid - (long long)rep * per_rep;
  const int colour = (int)(rem / ((long long)g.rows * g.wpr));
  rem -= (long long)colour * g.rows * g.wpr;
  const int i = (int)(rem / g.wpr);
  const int w = (int)(rem - (long long)i * g.wpr);
  const int p = (g.row0 + i + colour) & 1;
  const int nk = colour_count(g.cols, p);
  int8_t* row = spins + ((size_t)rep * g.rows + i) * g.cols;
  const uint32_t x = state[tid];
  for (int j = 0; j < 32; ++j) {
    int k = 32 * w + j;
    if (k < nk) {
      int b = (x >> j) & 1u;
      row[2 * k + p] = (int8_t)(as_pm1 ? 2 * b - 1 : b);
    }
  }
}

// Adds to ups / anti the up spins and the anti-aligned (right + down) bonds of word (rep, colour, local row i, w);
// bonded: unsatisfied bonds (sigma s_i s_j = -1) instead of anti-aligned ones.  plane = rows * wpr.
template <bool BONDED>
__device__ __forceinline__ void count_word(const uint32_t* state, const Geom& g, size_t plane, const uint32_t* next_rows,
                                           const BondParams& B, int rep, int colour, int i, int w,
                                           unsigned long long& ups, unsigned long long& anti) {
  const uint32_t* own = state + ((size_t)rep * 2 + colour) * plane;
  Planes pl;
  pl.opp = state + ((size_t)rep * 2 + (1 - colour)) * plane;
  pl.halo_top = nullptr;
  pl.halo_bot = next_rows ? next_rows + ((size_t)rep * 2 + (1 - colour)) * g.wpr : nullptr;
  Hood h = load_hood(pl, g, colour, i, w);
  if (h.valid == 0u) return;
  if constexpr (BONDED) apply_bonds(h, B, g, rep, colour, i, w);
  const uint32_t x = own[(size_t)i * g.wpr + w];
  const int p = (g.row0 + i + colour) & 1;
  ups += __popc(x & h.valid);
  // east neighbour: centre word if own col is even (p == 0), shifted word otherwise
  const uint32_t east = p ? h.side : h.c;
  anti += __popc((x ^ east) & h.valid & ~h.missE);
  if (h.has_s) anti += __popc((x ^ h.s) & h.valid);
}

// up-spin count and anti-aligned (right + down) bond count per replica; bonded: unsatisfied bonds (sigma s_i s_j = -1)
template <bool BONDED>
__global__ void __launch_bounds__(256) observables_kernel(const uint32_t* __restrict__ state, Geom g,
                                                         const uint32_t* __restrict__ next_rows,
                                                         unsigned long long* out, BondParams B) {
  const int rep = blockIdx.y;
  const size_t plane = (size_t)g.rows * g.wpr;
  const long long n_words = 2LL * g.rows * g.wpr;
  unsigned long long ups = 0, anti = 0;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n_words;
       t += (long long)gridDim.x * blockDim.x) {
    const int colour = (int)(t / ((long long)g.rows * g.wpr));
    const long long rem = t - (long long)colour * g.rows * g.wpr;
    const int i = (int)(rem / g.wpr);
    const int w = (int)(rem - (long long)i * g.wpr);
    count_word<BONDED>(state, g, plane, next_rows, B, rep, colour, i, w, ups, anti);
  }
  ups = tsu_warp_sum(ups);
  anti = tsu_warp_sum(anti);
  if ((threadIdx.x & 31) == 0) {
    if (ups) atomicAdd(out + 2 * rep, ups);
    if (anti) atomicAdd(out + 2 * rep + 1, anti);
  }
}

// Same counts for lattices with full words (cols % 256 == 0; periodic or open), at HBM speed: a thread owns a 4-word column
// strip of BOTH colour planes and walks down its rows with a rolling (row i, row i+1) window, so every word is
// loaded once as a 16-byte vector.  In a row exactly one colour has odd own columns (east neighbour = next lane of
// the other plane, i.e. a 1-bit funnel shift that needs one extra word); the other colour's east neighbour is the
// same lane.  The south neighbour of (colour, row i, lane) is (other colour, row i+1, same lane).
// Bonded: the east and south bond words of both colours are XOR-ed into the pairs, which counts unsatisfied bonds.
template <bool BONDED>
__global__ void __launch_bounds__(128) observables_fast_kernel(const uint32_t* __restrict__ state, Geom g,
                                                              const uint32_t* __restrict__ next_rows, int strip_rows,
                                                              int n_strips, unsigned long long* out, BondParams B) {
  const int nvec = g.wpr >> 2;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int per_rep = n_strips * nvec;
  const int per_rep_pad = (per_rep + 31) & ~31;  // warps never straddle replicas
  const int rep = (int)(tid / per_rep_pad);
  if (rep >= g.n_replicas) return;
  const int rem = (int)(tid - (long long)rep * per_rep_pad);
  unsigned ups = 0, anti = 0;
  if (rem < per_rep) {
    const int strip = rem / nvec, w0 = 4 * (rem - strip * nvec);
    const int r_begin = strip * strip_rows, r_end = min(g.rows, r_begin + strip_rows);
    const int w_next = (w0 + 4 == g.wpr) ? 0 : w0 + 4;
    const size_t plane = (size_t)g.rows * g.wpr;
    const uint32_t* pl[2] = {state + (size_t)rep * 2 * plane, state + ((size_t)rep * 2 + 1) * plane};
    Planes opp[2];  // opp[c] = the plane that is NOT colour c (south rows beyond the local rows come from next_rows)
    for (int c = 0; c < 2; ++c) {
      opp[c].opp = pl[1 - c];
      opp[c].halo_top = nullptr;
      opp[c].halo_bot = next_rows ? next_rows + ((size_t)rep * 2 + (1 - c)) * g.wpr : nullptr;
    }
    uint4 a[2];
    a[0] = *reinterpret_cast<const uint4*>(pl[0] + (size_t)r_begin * g.wpr + w0);
    a[1] = *reinterpret_cast<const uint4*>(pl[1] + (size_t)r_begin * g.wpr + w0);
    for (int i = r_begin; i < r_end; ++i) {
      // row i + 1 of both planes (the south neighbours), or nothing below an open last row
      const uint32_t* s1 = opp_row(opp[0], g, i + 1);  // plane 1 at row i+1 = south of colour 0
      const uint32_t* s0 = opp_row(opp[1], g, i + 1);  // plane 0 at row i+1 = south of colour 1
      uint4 b[2] = {a[0], a[1]};
      if (s0) b[0] = *reinterpret_cast<const uint4*>(s0 + w0);
      if (s1) b[1] = *reinterpret_cast<const uint4*>(s1 + w0);
      const int odd = 1 - ((g.row0 + i) & 1);  // colour `odd` has odd own columns in this row: col = 2 lane + 1
      const uint32_t extra = pl[1 - odd][(size_t)i * g.wpr + w_next];  // next word of the plane the odd colour looks at
      const uint32_t x0[4] = {a[0].x, a[0].y, a[0].z, a[0].w}, x1[4] = {a[1].x, a[1].y, a[1].z, a[1].w};
      const uint32_t* own_odd = odd ? x1 : x0;   // colour with the shifted east neighbour
      const uint32_t* own_even = odd ? x0 : x1;
      // bond words of row i: east of either colour, south of colour 0 / 1 (all 0 for the ferromagnet)
      uint4 be_odd = make_uint4(0u, 0u, 0u, 0u), be_even = be_odd, bs0 = be_odd, bs1 = be_odd;
      if constexpr (BONDED) {
        const size_t off = (size_t)i * g.wpr + w0;
        const uint32_t* b0 = tsu_fast::bond_base(B, g, rep, 0) + off;
        const uint32_t* b1 = tsu_fast::bond_base(B, g, rep, 1) + off;
        be_odd = *reinterpret_cast<const uint4*>((odd ? b1 : b0) + kBondE * plane);
        be_even = *reinterpret_cast<const uint4*>((odd ? b0 : b1) + kBondE * plane);
        bs0 = *reinterpret_cast<const uint4*>(b0 + kBondS * plane);
        bs1 = *reinterpret_cast<const uint4*>(b1 + kBondS * plane);
      }
      const uint32_t eo[4] = {be_odd.x, be_odd.y, be_odd.z, be_odd.w}, ee[4] = {be_even.x, be_even.y, be_even.z, be_even.w};
      // (own_even is also the plane the odd colour looks at, and vice versa)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t nxt = k < 3 ? own_even[k + 1] : extra;
        const uint32_t east_odd = __funnelshift_r(own_even[k], nxt, 1);
        // open columns: the last site of a row with odd own columns has no east neighbour
        const uint32_t has_east = (k == 3 && !g.wrap_cols && w0 + 4 == g.wpr) ? 0x7fffffffu : 0xffffffffu;
        ups += __popc(x0[k]) + __popc(x1[k]);
        if constexpr (BONDED)
          anti += __popc((own_odd[k] ^ east_odd ^ eo[k]) & has_east) + __popc(own_even[k] ^ own_odd[k] ^ ee[k]);
        else
          anti += __popc((own_odd[k] ^ east_odd) & has_east) + __popc(own_even[k] ^ own_odd[k]);
      }
      if constexpr (BONDED) {
        if (s1) anti += __popc(a[0].x ^ b[1].x ^ bs0.x) + __popc(a[0].y ^ b[1].y ^ bs0.y) + __popc(a[0].z ^ b[1].z ^ bs0.z) + __popc(a[0].w ^ b[1].w ^ bs0.w);
        if (s0) anti += __popc(a[1].x ^ b[0].x ^ bs1.x) + __popc(a[1].y ^ b[0].y ^ bs1.y) + __popc(a[1].z ^ b[0].z ^ bs1.z) + __popc(a[1].w ^ b[0].w ^ bs1.w);
      } else {
        if (s1) anti += __popc(a[0].x ^ b[1].x) + __popc(a[0].y ^ b[1].y) + __popc(a[0].z ^ b[1].z) + __popc(a[0].w ^ b[1].w);
        if (s0) anti += __popc(a[1].x ^ b[0].x) + __popc(a[1].y ^ b[0].y) + __popc(a[1].z ^ b[0].z) + __popc(a[1].w ^ b[0].w);
      }
      a[0] = b[0];
      a[1] = b[1];
    }
  }
  const unsigned long long u64 = tsu_warp_sum((unsigned long long)ups), a64 = tsu_warp_sum((unsigned long long)anti);
  if ((threadIdx.x & 31) == 0) {
    if (u64) atomicAdd(out + 2 * rep, u64);
    if (a64) atomicAdd(out + 2 * rep + 1, a64);
  }
}

// E = -J (n_bonds - 2 anti) - h (2 up - n_sites).  The two differences are exact (integers below 2^53); the rounding
// is spelled out as one product and one fused multiply-add, so that every kernel computing E rounds the same way.
__device__ __forceinline__ double energy_of_counts(double up, double anti, double J, double h, long long n_bonds,
                                                   long long n_sites) {
  return fma(-J, (double)n_bonds - 2.0 * anti, -__dmul_rn(h, 2.0 * up - (double)n_sites));
}

__global__ void energy_from_obs_kernel(const unsigned long long* __restrict__ obs, int n, double J, double h,
                                       long long n_bonds, long long n_sites, double* energy) {
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  energy[r] = energy_of_counts((double)obs[2 * r], (double)obs[2 * r + 1], J, h, n_bonds, n_sites);
}

// ---- simulated annealing (tsu_ising2d_anneal) -----------------------------------------------------------------
// What an anneal step does after its sweep: E of every replica from its counts, and the strict best-so-far update.
struct AnnealOut {
  double J, h;
  long long n_bonds, n_sites;
  double* energy;       // [replicas] E of the current state
  double* best_energy;  // [replicas] in/out, or NULL (then best_state is NULL too)
  uint32_t* best_state; // [replicas][2][rows][wpr]
};

// obs[r] = (up, anti) -> energy[r]; replicas with E < best_energy[r] take E, and obs[2r] becomes 1 if they did, else 0
// (the flag anneal_copy_kernel reads)
__global__ void anneal_select_kernel(unsigned long long* obs, int n, AnnealOut A) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const double e = energy_of_counts((double)obs[2 * r], (double)obs[2 * r + 1], A.J, A.h, A.n_bonds, A.n_sites);
  A.energy[r] = e;
  if (!A.best_energy) return;
  const bool better = e < A.best_energy[r];
  if (better) A.best_energy[r] = e;
  obs[2 * r] = better ? 1ull : 0ull;
}

// dst[t] = src[t] for t = t0, t0 + stride, ... below n_vecs: 16-byte accesses, four in flight per thread
__device__ __forceinline__ void copy_vecs(const uint4* src, uint4* dst, long long n_vecs, long long t0, long long stride) {
  long long t = t0;
  for (; t + 3 * stride < n_vecs; t += 4 * stride) {
    const uint4 a = src[t], b = src[t + stride], c = src[t + 2 * stride], d = src[t + 3 * stride];
    dst[t] = a;
    dst[t + stride] = b;
    dst[t + 2 * stride] = c;
    dst[t + 3 * stride] = d;
  }
  for (; t < n_vecs; t += stride) dst[t] = src[t];
}

// best_state[r] = state[r] for the replicas flagged by anneal_select_kernel; blockIdx.y walks the replicas, so the
// blocks of replicas that did not improve leave at once.
__global__ void __launch_bounds__(256) anneal_copy_kernel(const uint4* __restrict__ state, uint4* best_state,
                                                          const unsigned long long* __restrict__ flags, int n,
                                                          long long rep_vecs) {
  for (int r = blockIdx.y; r < n; r += gridDim.y) {
    if (!flags[2 * r]) continue;
    const uint4* src = state + (size_t)r * rep_vecs;
    uint4* dst = best_state + (size_t)r * rep_vecs;
    const long long stride = (long long)gridDim.x * blockDim.x;
    copy_vecs(src, dst, rep_vecs, (long long)blockIdx.x * blockDim.x + threadIdx.x, stride);
  }
}

// Small lattices: the whole anneal in one launch, one thread block per replica (as sweeps_resident_kernel).  Step k
// sweeps with table luts[k] and sweep index P.sweep + k; before the first step and after every step the block counts
// its replica as count_word does, and takes E and the best state as anneal_select_kernel / anneal_copy_kernel do.
template <bool BONDED>
__global__ void __launch_bounds__(kResidentThreads) anneal_resident_kernel(SweepParams P, const uint32_t* __restrict__ luts,
                                                                           int n_steps, BondParams B, AnnealOut A) {
  const Geom& g = P.g;
  const int rep = blockIdx.x;
  const int per_rep = g.rows * g.wpr;
  __shared__ unsigned long long part[2][kResidentThreads / 32];
  __shared__ int better;
  for (int k = -1; k < n_steps; ++k) {
    if (k >= 0) {
      SweepParams Q = P;
      Q.lut = luts + 32 * (size_t)k;
      for (int colour = 0; colour < 2; ++colour) {
        for (int rem = threadIdx.x; rem < per_rep; rem += kResidentThreads) {
          const int i = rem / g.wpr;
          generic_update_one<BONDED>(Q, B, colour, P.sweep + (uint32_t)k, rep, i, rem - i * g.wpr);
        }
        __syncthreads();
      }
    }
    unsigned long long ups = 0, anti = 0;
    for (int t = threadIdx.x; t < 2 * per_rep; t += kResidentThreads) {
      const int colour = t / per_rep, rem = t - colour * per_rep, i = rem / g.wpr;
      count_word<BONDED>(P.state, g, (size_t)per_rep, nullptr, B, rep, colour, i, rem - i * g.wpr, ups, anti);
    }
    ups = tsu_warp_sum(ups);
    anti = tsu_warp_sum(anti);
    if ((threadIdx.x & 31) == 0) {
      part[0][threadIdx.x >> 5] = ups;
      part[1][threadIdx.x >> 5] = anti;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      ups = 0;
      anti = 0;
      for (int j = 0; j < kResidentThreads / 32; ++j) {
        ups += part[0][j];
        anti += part[1][j];
      }
      const double e = energy_of_counts((double)ups, (double)anti, A.J, A.h, A.n_bonds, A.n_sites);
      A.energy[rep] = e;
      better = A.best_energy && e < A.best_energy[rep];
      if (better) A.best_energy[rep] = e;
    }
    __syncthreads();
    if (better) {
      const uint4* src = reinterpret_cast<const uint4*>(P.state + (size_t)rep * 2 * per_rep);
      uint4* dst = reinterpret_cast<uint4*>(A.best_state + (size_t)rep * 2 * per_rep);
      for (int t = threadIdx.x; t < per_rep / 2; t += kResidentThreads) dst[t] = src[t];  // 2 per_rep words
    }
    __syncthreads();  // the next half-sweep overwrites what the counts and the copy read
  }
}

// ---- population annealing (tsu_ising2d_population_anneal) -------------------------------------------------------
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

// More replicas than the word-by-word observables kernel's grid takes (gridDim.y <= 65535): one warp per replica counts
// its words with count_word and writes out[rep] (no atomics, no zeroing).
template <bool BONDED>
__global__ void __launch_bounds__(256) pa_count_kernel(const uint32_t* __restrict__ state, Geom g,
                                                      unsigned long long* out, BondParams B) {
  const long long rep = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (rep >= g.n_replicas) return;
  const long long plane = (long long)g.rows * g.wpr;
  unsigned long long ups = 0, anti = 0;
  for (long long t = threadIdx.x & 31; t < 2 * plane; t += 32) {
    const int colour = (int)(t / plane);
    const long long rem = t - colour * plane;
    const int i = (int)(rem / g.wpr);
    count_word<BONDED>(state, g, (size_t)plane, nullptr, B, (int)rep, colour, i, (int)(rem - (long long)i * g.wpr), ups,
                       anti);
  }
  ups = tsu_warp_sum(ups);
  anti = tsu_warp_sum(anti);
  if ((threadIdx.x & 31) == 0) {
    out[2 * rep] = ups;
    out[2 * rep + 1] = anti;
  }
}

// E of every replica from its counts (energy_of_counts) into A.energy; per population the sums of the counts
// (sums[p][2]) and the order key of the lowest E (Q.min_key[p]).  Grid (x, n_pop): blockIdx.x strides over a population.
__global__ void __launch_bounds__(kPaThreads) pa_reduce_kernel(const unsigned long long* __restrict__ obs, PopParams Q,
                                                               AnnealOut A, unsigned long long* sums) {
  const int p = blockIdx.y;
  unsigned long long ups = 0, anti = 0, key = ~0ull;
  for (int j = blockIdx.x * kPaThreads + threadIdx.x; j < Q.rp; j += gridDim.x * kPaThreads) {
    const size_t r = (size_t)p * Q.rp + j;
    const unsigned long long u = obs[2 * r], a = obs[2 * r + 1];
    const double e = energy_of_counts((double)u, (double)a, A.J, A.h, A.n_bonds, A.n_sites);
    A.energy[r] = e;
    ups += u;
    anti += a;
    key = min(key, order_key(e));
  }
  __shared__ unsigned long long part[3][kPaThreads / 32];
  ups = tsu_warp_sum(ups);
  anti = tsu_warp_sum(anti);
  key = warp_min(key);
  if ((threadIdx.x & 31) == 0) {
    part[0][threadIdx.x >> 5] = ups;
    part[1][threadIdx.x >> 5] = anti;
    part[2][threadIdx.x >> 5] = key;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kPaThreads / 32; ++w) {
      ups += part[0][w];
      anti += part[1][w];
      key = min(key, part[2][w]);
    }
    atomicAdd(sums + 2 * p, ups);
    atomicAdd(sums + 2 * p + 1, anti);
    atomicMin(Q.min_key + p, key);
  }
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

// state'[c] = state[parent(c)] and family'[c] = family[parent(c)].  group < 256: `group` threads (a power of two) per
// child, 256 / group children per block along x; group == 256: blockIdx.y walks the children and blockIdx.x tiles one.
__global__ void __launch_bounds__(256) pa_gather_kernel(const uint4* __restrict__ src, uint4* dst,
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

// ---- Swendsen-Wang cluster updates (tsu_ising2d_swendsen_wang) ------------------------------------------------
// Per replica the caller's work buffer holds (ClusterParams::rep_bytes apart) labels int32 [rows * cols] (site index
// row * cols + col, padded to 16 bytes), the activation words uint32 [2 colours][east, south][rows][wpr] and the flip
// words uint32 [2 colours][rows][wpr], both in the layout of the state.  Labels form a union-find forest in which a
// site's parent never has a larger index; unions always hang the larger root under the smaller, so every tree's root
// is its cluster's smallest site index, whatever order the unions run in.
constexpr int kClusterThreads = 256;
constexpr int kClusterTileRows = 32, kClusterTileWords = 4;  // tiles of the local pass: 32 rows x 256 columns
constexpr int kClusterTileCols = 64 * kClusterTileWords;
constexpr int kClusterResidentSites = 12288;  // labels of a replica in 48 KB of shared memory: one launch per call

struct ClusterParams {
  const unsigned long long* thresholds;  // [n_tables] t = ceil(p 2^32), p = 1 - exp(-2|J|/T); 2^32: always active
  int sign;                              // sign of J: +1 satisfied = aligned (after the bond sign), -1 anti-aligned
  char* work;
  size_t rep_bytes, act_offset, flip_offset;  // per replica: its share of the work buffer, where its words start
};

__device__ __forceinline__ int32_t* cluster_labels(const ClusterParams& C, int rep) {
  return reinterpret_cast<int32_t*>(C.work + (size_t)rep * C.rep_bytes);
}
__device__ __forceinline__ uint32_t* cluster_act(const ClusterParams& C, int rep) {  // [colour][dir][rows][wpr]
  return reinterpret_cast<uint32_t*>(C.work + (size_t)rep * C.rep_bytes + C.act_offset);
}
__device__ __forceinline__ uint32_t* cluster_flip(const ClusterParams& C, int rep) {  // [colour][rows][wpr]
  return reinterpret_cast<uint32_t*>(C.work + (size_t)rep * C.rep_bytes + C.flip_offset);
}

// lanes of `sat` whose bond uniform u (bit-planes of kinds plane0, plane0 + 1, low bits of kinds low0 ..) is below t:
// the borrow chain of update_word against one threshold, with the low words drawn only on ties
__device__ __forceinline__ uint32_t activate_bonds(uint32_t sat, unsigned long long t, const Coords& q, uint32_t w,
                                                   uint32_t row_g, uint32_t plane0, uint32_t low0) {
  if (sat == 0u || t >= (1ull << 32)) return sat;
  const uint32_t t32 = (uint32_t)t;
  uint32_t r[8];
  {
    tsu_u32x4 p0 = lattice_call(q, w, row_g, plane0);
    tsu_u32x4 p1 = lattice_call(q, w, row_g, plane0 + 1u);
    r[0] = p0.x; r[1] = p0.y; r[2] = p0.z; r[3] = p0.w;
    r[4] = p1.x; r[5] = p1.y; r[6] = p1.z; r[7] = p1.w;
  }
  uint32_t lt = 0u, eq = 0xffffffffu;
#pragma unroll
  for (int k = 7; k >= 0; --k) {
    const uint32_t tk = 0u - ((t32 >> (31 - k)) & 1u);
    const uint32_t x = r[k] ^ tk;
    lt = (~r[k] & tk) | (~x & lt);
    eq &= ~x;
  }
  eq &= sat;
  while (eq) {
    const int j = __ffs(eq) - 1;
    eq &= eq - 1u;
    const uint32_t bit = lane_uniform(r, q, w, row_g, j, low0) < t32 ? 1u : 0u;
    lt = (lt & ~(1u << j)) | (bit << j);
  }
  return lt & sat;
}

// Step `sweep` of word (rep, colour, row i, w): its east and south activation words and its flip word.  The hood's
// neighbour words carry the bond signs (apply_bonds), so x ^ neighbour is 1 where sigma s_i s_j = -1, as count_word counts.
template <bool BONDED>
__device__ __forceinline__ void cluster_bond_word(const SweepParams& P, const BondParams& B, const ClusterParams& C,
                                                  uint32_t sweep, int rep, int colour, int i, int w) {
  const Geom& g = P.g;
  const size_t plane = (size_t)g.rows * g.wpr;
  Planes pl;
  pl.opp = P.state + ((size_t)rep * 2 + (1 - colour)) * plane;
  pl.halo_top = nullptr;
  pl.halo_bot = nullptr;
  Hood h = load_hood(pl, g, colour, i, w);
  const size_t off = (size_t)i * g.wpr + w;
  uint32_t* act = cluster_act(C, rep) + (size_t)colour * 2 * plane + off;
  uint32_t* flip = cluster_flip(C, rep) + (size_t)colour * plane + off;
  if (h.valid == 0u) {  // padding word
    act[0] = 0u;
    act[plane] = 0u;
    *flip = 0u;
    return;
  }
  if constexpr (BONDED) apply_bonds(h, B, g, rep, colour, i, w);
  const uint32_t x = P.state[((size_t)rep * 2 + colour) * plane + off];
  const int p = (g.row0 + i + colour) & 1;
  const uint32_t aligned = C.sign > 0 ? 0xffffffffu : 0u;
  const uint32_t sat_e = (x ^ (p ? h.side : h.c) ^ aligned) & h.valid & ~h.missE;
  const uint32_t sat_s = h.has_s ? (x ^ h.s ^ aligned) & h.valid : 0u;
  Coords q;
  q.colour = (uint32_t)colour;
  q.sweep = sweep;
  q.replica = P.replica0 + (uint32_t)rep;
  q.k0 = P.k0;
  q.k1 = P.k1;
  const unsigned long long t = C.thresholds[P.lut_index ? P.lut_index[rep] : 0];
  const uint32_t row_g = (uint32_t)(g.row0 + i);
  act[0] = activate_bonds(sat_e, t, q, (uint32_t)w, row_g, TSU_KIND_BOND_E_PLANE0, TSU_KIND_BOND_E_LOW0);
  act[plane] = activate_bonds(sat_s, t, q, (uint32_t)w, row_g, TSU_KIND_BOND_S_PLANE0, TSU_KIND_BOND_S_LOW0);
  *flip = lattice_call(q, (uint32_t)w, row_g, TSU_KIND_CLUSTER_FLIP).x & h.valid;
}

// root of x, halving the path on the way (every site then points at its former grandparent).  A label only ever
// points at a smaller site of the same cluster, so a stale read or an overwritten link still leads to the root
// (the pointer jumping of ECL-CC, Jaiganesh & Burtscher 2018).
__device__ __forceinline__ int cluster_find(int32_t* L, int x) {
  volatile int32_t* V = L;
  int y = V[x];
  while (y != x) {
    const int z = V[y];
    if (z != y) V[x] = z;
    x = y;
    y = z;
  }
  return x;
}

// joins the trees of a and b, hanging the larger root under the smaller (Playne & Hawick's lock-free union)
__device__ __forceinline__ void cluster_union(int32_t* L, int a, int b) {
  while (true) {
    a = cluster_find(L, a);
    b = cluster_find(L, b);
    if (a == b) return;
    if (a > b) {
      const int t = a;
      a = b;
      b = t;
    }
    const int old = atomicMin(L + b, a);
    if (old == b) return;
    b = old;  // b was no longer a root: join its parent (b itself now points to min(old, a)) to a
  }
}

// Unions in the forest L of one tile every active bond whose two sites both lie in it.  The tile is rows
// [r0, r0 + nr) and columns [c0, c0 + nc) with c0 = 64 w0; its words are w0 .. w0 + nw - 1 of both colours, and its
// site (i, col) is L[(i - r0) * nc + col - c0].  Wrapped neighbours count when they lie in the tile.
__device__ __forceinline__ void cluster_tile_unions(int32_t* L, const uint32_t* act, const Geom& g, int r0, int nr,
                                                    int w0, int nw, int c0, int nc) {
  const size_t plane = (size_t)g.rows * g.wpr;
  for (int t = threadIdx.x; t < 2 * nr * nw; t += blockDim.x) {
    const int colour = t / (nr * nw), rem = t - colour * nr * nw, r = rem / nw, w = w0 + rem - r * nw, i = r0 + r;
    const int p = (g.row0 + i + colour) & 1;
    const uint32_t* a = act + (size_t)colour * 2 * plane + (size_t)i * g.wpr + w;
    uint32_t e = a[0], s = a[plane];
    const int ni = i + 1 == g.rows ? 0 : i + 1;
    if (ni < r0 || ni >= r0 + nr) s = 0u;
    while (e | s) {
      const int j = __ffs(e | s) - 1;
      const uint32_t bit = 1u << j;
      const int col = 2 * (32 * w + j) + p, x = r * nc + col - c0;
      if (e & bit) {
        const int ncol = col + 1 == g.cols ? 0 : col + 1;
        if (ncol >= c0 && ncol < c0 + nc) cluster_union(L, x, r * nc + ncol - c0);
      }
      if (s & bit) cluster_union(L, x, (ni - r0) * nc + col - c0);
      e &= ~bit;
      s &= ~bit;
    }
  }
}

// XORs into word (rep, colour, row i, w) the flip bit of every site's cluster root; `L` is the label forest of the
// whole replica (site index row * cols + col).  Path compression: each site then points at its root.
__device__ __forceinline__ void cluster_flip_word(const SweepParams& P, const ClusterParams& C, int32_t* L, int rep,
                                                  int colour, int i, int w) {
  const Geom& g = P.g;
  const int p = (g.row0 + i + colour) & 1;
  uint32_t m = lane_mask_lt(colour_count(g.cols, p) - 32 * w);
  if (m == 0u) return;
  const size_t plane = (size_t)g.rows * g.wpr;
  const uint32_t* flip = cluster_flip(C, rep);
  uint32_t out = 0u;
  while (m) {
    const int j = __ffs(m) - 1;
    m &= m - 1u;
    const int x = i * g.cols + 2 * (32 * w + j) + p;
    const int root = cluster_find(L, x);
    if (L[x] != root) L[x] = root;
    const int ri = root / g.cols, rc = root - ri * g.cols, rk = rc >> 1;
    out |= ((flip[(size_t)((g.row0 + ri + rc) & 1) * plane + (size_t)ri * g.wpr + (rk >> 5)] >> (rk & 31)) & 1u) << j;
  }
  P.state[((size_t)rep * 2 + colour) * plane + (size_t)i * g.wpr + w] ^= out;
}

// One thread per state word of every replica: activation and flip words of step P.sweep.
template <bool BONDED>
__global__ void __launch_bounds__(kClusterThreads) cluster_bonds_kernel(SweepParams P, BondParams B, ClusterParams C) {
  const Geom& g = P.g;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_rep = 2LL * g.rows * g.wpr;
  if (tid >= per_rep * g.n_replicas) return;
  const int rep = (int)(tid / per_rep);
  const int rem = (int)(tid - (long long)rep * per_rep), colour = rem / (g.rows * g.wpr);
  const int rw = rem - colour * g.rows * g.wpr, i = rw / g.wpr;
  cluster_bond_word<BONDED>(P, B, C, P.sweep, rep, colour, i, rw - i * g.wpr);
}

// One block per tile of kClusterTileRows x kClusterTileCols sites: unions in shared memory, then every site's label is
// the site index of its root within the tile.
__global__ void __launch_bounds__(kClusterThreads) cluster_local_kernel(SweepParams P, ClusterParams C, int tiles_x,
                                                                        int tiles_per_rep) {
  __shared__ int32_t L[kClusterTileRows * kClusterTileCols];
  const Geom& g = P.g;
  const int rep = (int)(blockIdx.x / (unsigned)tiles_per_rep), tile = (int)(blockIdx.x % (unsigned)tiles_per_rep);
  const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
  const int r0 = ty * kClusterTileRows, nr = min(kClusterTileRows, g.rows - r0);
  const int c0 = tx * kClusterTileCols, nc = min(kClusterTileCols, g.cols - c0);
  for (int t = threadIdx.x; t < nr * nc; t += kClusterThreads) L[t] = t;
  __syncthreads();
  cluster_tile_unions(L, cluster_act(C, rep), g, r0, nr, tx * kClusterTileWords, kClusterTileWords, c0, nc);
  __syncthreads();
  int32_t* labels = cluster_labels(C, rep);
  for (int t = threadIdx.x; t < nr * nc; t += kClusterThreads) {
    const int root = cluster_find(L, t), r = t / nc, rr = root / nc;
    labels[(r0 + r) * g.cols + c0 + t - r * nc] = (r0 + rr) * g.cols + c0 + root - rr * nc;
  }
}

// active bond of site (i, col) in direction dir (0 east, 1 south)
__device__ __forceinline__ bool cluster_bond_active(const uint32_t* act, const Geom& g, int i, int col, int dir) {
  const int colour = (g.row0 + i + col) & 1, k = col >> 1;
  return (act[((size_t)colour * 2 + dir) * g.rows * g.wpr + (size_t)i * g.wpr + (k >> 5)] >> (k & 31)) & 1u;
}

// The bonds between tiles: south bonds of the last row of every tile row (n_brows of them) and east bonds of the last
// column of every tile column (n_bcols), including the wraps; unions in global memory.
__global__ void __launch_bounds__(kClusterThreads) cluster_merge_kernel(SweepParams P, ClusterParams C, int n_brows,
                                                                        int n_bcols) {
  const Geom& g = P.g;
  const long long per_rep = (long long)n_brows * g.cols + (long long)g.rows * n_bcols;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= per_rep * g.n_replicas) return;
  const int rep = (int)(tid / per_rep);
  const long long t = tid - (long long)rep * per_rep;
  int i, col, ni, ncol, dir;
  if (t < (long long)n_brows * g.cols) {
    const int b = (int)(t / g.cols);
    col = (int)(t - (long long)b * g.cols);
    i = min(b * kClusterTileRows + kClusterTileRows - 1, g.rows - 1);
    ni = i + 1 == g.rows ? 0 : i + 1;
    ncol = col;
    dir = 1;
    if (ni / kClusterTileRows == i / kClusterTileRows) return;  // one tile row: the local pass took the wrap
  } else {
    const long long u = t - (long long)n_brows * g.cols;
    i = (int)(u / n_bcols);
    const int b = (int)(u - (long long)i * n_bcols);
    col = min(b * kClusterTileCols + kClusterTileCols - 1, g.cols - 1);
    ncol = col + 1 == g.cols ? 0 : col + 1;
    ni = i;
    dir = 0;
    if (ncol / kClusterTileCols == col / kClusterTileCols) return;
  }
  if (cluster_bond_active(cluster_act(C, rep), g, i, col, dir))
    cluster_union(cluster_labels(C, rep), i * g.cols + col, ni * g.cols + ncol);
}

__global__ void __launch_bounds__(kClusterThreads) cluster_flip_kernel(SweepParams P, ClusterParams C) {
  const Geom& g = P.g;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_rep = 2LL * g.rows * g.wpr;
  if (tid >= per_rep * g.n_replicas) return;
  const int rep = (int)(tid / per_rep);
  const int rem = (int)(tid - (long long)rep * per_rep), colour = rem / (g.rows * g.wpr);
  const int rw = rem - colour * g.rows * g.wpr, i = rw / g.wpr;
  cluster_flip_word(P, C, cluster_labels(C, rep), rep, colour, i, rw - i * g.wpr);
}

// Lattices of at most kClusterResidentSites sites: every step of the call in one launch, one block per replica, the
// labels in shared memory (the whole lattice is one tile of cluster_tile_unions).  The activation and flip words go
// through the work buffer; the block's barriers make its own global stores visible to it.
template <bool BONDED>
__global__ void __launch_bounds__(kClusterThreads) cluster_resident_kernel(SweepParams P, BondParams B, ClusterParams C,
                                                                           int n_steps) {
  extern __shared__ int32_t L[];
  const Geom& g = P.g;
  const int rep = blockIdx.x, per_rep = g.rows * g.wpr, n_sites = g.rows * g.cols;
  for (int s = 0; s < n_steps; ++s) {
    for (int t = threadIdx.x; t < 2 * per_rep; t += kClusterThreads) {
      const int colour = t / per_rep, rem = t - colour * per_rep, i = rem / g.wpr;
      cluster_bond_word<BONDED>(P, B, C, P.sweep + (uint32_t)s, rep, colour, i, rem - i * g.wpr);
    }
    for (int t = threadIdx.x; t < n_sites; t += kClusterThreads) L[t] = t;
    __syncthreads();
    cluster_tile_unions(L, cluster_act(C, rep), g, 0, g.rows, 0, g.wpr, 0, g.cols);
    __syncthreads();
    for (int t = threadIdx.x; t < 2 * per_rep; t += kClusterThreads) {
      const int colour = t / per_rep, rem = t - colour * per_rep, i = rem / g.wpr;
      cluster_flip_word(P, C, L, rep, colour, i, rem - i * g.wpr);
    }
    __syncthreads();  // the next step's bonds read the flipped words
  }
}

// ---- Edwards-Anderson bonds ---------------------------------------------------------------------------------
// int8 signs[k][2][rows][cols] ([.,0,i,j]: bond (i,j)-(i,j+1 mod cols), [.,1,i,j]: bond (i,j)-(i+1 mod rows,j); < 0
// = antiferromagnetic) -> bond words[k][colour][N,S,W,E][rows][wpr].  Bonds the wiring does not create (open edges;
// a wrap that is off) leave their bits 0, and so do padding lanes.  One thread per word.
__global__ void pack_bonds_kernel(const int8_t* __restrict__ signs, uint32_t* bonds, int n_real, Geom g) {
  const long long plane = (long long)g.rows * g.wpr;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= (long long)n_real * 8 * plane) return;
  const int k = (int)(tid / (8 * plane));
  long long rem = tid - (long long)k * 8 * plane;
  const int colour = (int)(rem / (4 * plane));
  rem -= (long long)colour * 4 * plane;
  const int dir = (int)(rem / plane);
  rem -= (long long)dir * plane;
  const int i = (int)(rem / g.wpr);
  const int w = (int)(rem - (long long)i * g.wpr);
  const int p = (i + colour) & 1;
  const int nk = colour_count(g.cols, p);
  const int8_t* horiz = signs + ((size_t)k * 2 * g.rows) * g.cols;
  const int8_t* vert = horiz + (size_t)g.rows * g.cols;
  uint32_t x = 0u;
  for (int j = 0; j < 32; ++j) {
    const int kk = 32 * w + j;
    if (kk >= nk) break;
    const int col = 2 * kk + p;
    int8_t sgn = 1;
    if (dir == kBondN) {
      if (i > 0 || g.wrap_rows) sgn = vert[(size_t)(i > 0 ? i - 1 : g.rows - 1) * g.cols + col];
    } else if (dir == kBondS) {
      if (i + 1 < g.rows || g.wrap_rows) sgn = vert[(size_t)i * g.cols + col];
    } else if (dir == kBondW) {
      if (col > 0 || g.wrap_cols) sgn = horiz[(size_t)i * g.cols + (col > 0 ? col - 1 : g.cols - 1)];
    } else {
      if (col + 1 < g.cols || g.wrap_cols) sgn = horiz[(size_t)i * g.cols + col];
    }
    if (sgn < 0) x |= 1u << j;
  }
  bonds[tid] = x;
}

// number of sites at which replicas pairs[2q] and pairs[2q+1] differ, for every pair q (padding bits are 0 in both)
__global__ void __launch_bounds__(256) overlap_kernel(const uint32_t* __restrict__ state, long long rep_vecs,
                                                      const int32_t* __restrict__ pairs, unsigned long long* out) {
  const int q = blockIdx.y;
  const uint4* a = reinterpret_cast<const uint4*>(state) + (size_t)pairs[2 * q] * rep_vecs;
  const uint4* b = reinterpret_cast<const uint4*>(state) + (size_t)pairs[2 * q + 1] * rep_vecs;
  unsigned long long diff = 0;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < rep_vecs; t += (long long)gridDim.x * blockDim.x) {
    const uint4 x = a[t], y = b[t];
    diff += __popc(x.x ^ y.x) + __popc(x.y ^ y.y) + __popc(x.z ^ y.z) + __popc(x.w ^ y.w);
  }
  diff = tsu_warp_sum(diff);
  if ((threadIdx.x & 31) == 0 && diff) atomicAdd(out + q, diff);
}

// ---- row slabs with peer-mapped halos (tsu_ising2d_slab_sweeps_p2p) ---------------------------------------
// copy one row of `colour` of every replica into a halo buffer that may live on another GPU (NVLink peer mapping)
__global__ void __launch_bounds__(256) slab_send_rows_kernel(const uint32_t* __restrict__ state, int n_replicas, int rows,
                                                           int wpr, int colour, uint32_t* up_dst, uint32_t* down_dst) {
  // up_dst   <- my first row (the row below the upper neighbour's last row)
  // down_dst <- my last row  (the row above the lower neighbour's first row)
  const int nvec = wpr >> 2;
  const long long per_side = (long long)n_replicas * nvec;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < 2 * per_side; t += (long long)gridDim.x * blockDim.x) {
    const int side = t >= per_side;
    uint32_t* dst = side ? down_dst : up_dst;
    if (!dst) continue;
    const long long u = t - side * per_side;
    const int rep = (int)(u / nvec), v = (int)(u - (long long)rep * nvec);
    const size_t row = side ? (size_t)(rows - 1) : 0;
    const uint4 x = *reinterpret_cast<const uint4*>(state + (((size_t)rep * 2 + colour) * rows + row) * wpr + 4 * v);
    *reinterpret_cast<uint4*>(dst + (size_t)rep * wpr + 4 * v) = x;
  }
}

// the rows sent before this kernel (stream order) are complete: publish their message number to the receivers
__global__ void slab_signal_kernel(uint32_t* up_flag, uint32_t* down_flag, uint32_t value) {
  __threadfence_system();
  if (up_flag) *reinterpret_cast<volatile uint32_t*>(up_flag) = value;
  if (down_flag) *reinterpret_cast<volatile uint32_t*>(down_flag) = value;
}

// hold the stream until both neighbours' rows with message number >= need have arrived (they write the counters
// through their peer mapping).  Gives up after ~20 s and raises the status word instead of hanging the GPU.
__global__ void slab_wait_kernel(const uint32_t* flag_a, const uint32_t* flag_b, uint32_t need, uint32_t* status) {
  const long long t0 = clock64();
  const volatile uint32_t* fa = flag_a;
  const volatile uint32_t* fb = flag_b;
  while (true) {
    const bool a_ok = !fa || (int32_t)(*fa - need) >= 0;
    const bool b_ok = !fb || (int32_t)(*fb - need) >= 0;
    if (a_ok && b_ok) return;
    if (clock64() - t0 > 40000000000LL) {
      *status = 1u;
      return;
    }
    __nanosleep(200);
  }
}

// streams the slab driver launches its extra interior row ranges on: created once per device, never destroyed
std::mutex g_slab_stream_mutex;
std::map<int, std::vector<cudaStream_t>> g_slab_streams;
cudaStream_t slab_stream(int dev, int idx) {
  std::lock_guard<std::mutex> lock(g_slab_stream_mutex);
  std::vector<cudaStream_t>& v = g_slab_streams[dev];
  while ((int)v.size() <= idx) {
    cudaStream_t s = nullptr;
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    v.push_back(s);
  }
  return v[idx];
}

bool geom_ok(int n_replicas, int rows, int cols) {
  // counter word 1 of the lattice stream keeps the global row in 24 bits, counter word 0 the 4-word group in 24
  return n_replicas > 0 && rows > 0 && cols > 0 && cols < (1 << 26) && rows <= TSU_LATTICE_MAX_ROWS;
}

bool rows_ok(int rows, int row0) { return row0 >= 0 && (long long)row0 + rows <= TSU_LATTICE_MAX_ROWS; }

// Tuning knobs (never change results), read once per process:
//   TSU_LATTICE_STRIP  rows per thread strip of the wide kernel (default: 128, shortened until the grid fills the GPU)
//   TSU_LATTICE_SPLIT  row ranges a half-sweep is cut into (split_ranges(); 1 = one launch per half-sweep)
//   TSU_LATTICE_W      words per thread of the prebuilt wide kernel (2 or 4)
//   TSU_LATTICE_OPEN_GENERIC / TSU_LATTICE_OBS_GENERIC / TSU_LATTICE_RESIDENT=0  force the one-thread-per-word kernels
//   TSU_JIT_THREADS (32 / 64 / 128 threads per CTA),
//   TSU_JIT_W, TSU_JIT_MINB, TSU_JIT_UNROLL   words per thread, CTAs per SM and row-loop unrolling the run-time
//                                             specialised kernel is compiled for
struct Tuning {
  int strip = 0, w = 0, open_generic = 0, obs_generic = 0, resident = 1, jit_w = 0, jit_minb = 0, jit_unroll = 0, jit_threads = 0, split = -1;
  Tuning() {
    auto num = [](const char* name, int dflt) {
      const char* e = getenv(name);
      return e ? atoi(e) : dflt;
    };
    strip = num("TSU_LATTICE_STRIP", 0);
    w = num("TSU_LATTICE_W", 0);
    open_generic = getenv("TSU_LATTICE_OPEN_GENERIC") != nullptr;
    obs_generic = getenv("TSU_LATTICE_OBS_GENERIC") != nullptr;
    resident = num("TSU_LATTICE_RESIDENT", 1);
    jit_w = num("TSU_JIT_W", 0);
    jit_minb = num("TSU_JIT_MINB", 0);
    jit_unroll = num("TSU_JIT_UNROLL", 0);
    jit_threads = num("TSU_JIT_THREADS", 0);
    split = num("TSU_LATTICE_SPLIT", -1);
  }
};
Tuning g_tuning;  // read when the library is loaded; tsu_ising2d_reload_tuning() reads the environment again
const Tuning& tuning() { return g_tuning; }
constexpr int kDefaultW = 4, kDefaultJitW = 4, kDefaultJitMinB = 5, kDefaultJitThreads = 128;
constexpr int kDefaultSplit = 8, kMaxSplit = 8;  // row ranges of one half-sweep launched on streams of their own  // 5 CTAs/SM (93 registers): +1 % over 4, measured

Geom make_geom(int n_replicas, int rows, int cols, int wrap_rows, int wrap_cols, int row0) {
  Geom g;
  g.rows = rows;
  g.cols = cols;
  g.wpr = words_per_row(cols);
  g.wrap_rows = wrap_rows ? 1 : 0;
  g.wrap_cols = wrap_cols ? 1 : 0;
  g.row0 = row0;
  g.n_replicas = n_replicas;
  return g;
}

unsigned blocks_for(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

// ---- run-time specialisation of the fast kernel (NVRTC) ------------------------------------------------
// For a launch whose replicas all share one threshold table, ising2d_fast.cuh is compiled once per table set
// with the eight 5-bit truth tables as literals.  libnvrtc and libcuda are opened with dlopen so that the
// library has no link-time dependency on them; any failure simply leaves the prebuilt jump-table kernel in use.
std::mutex g_jit_mutex;
std::map<std::string, int> g_jit_cache;  // "device:t0,..,t7" -> handle
struct JitKernel {
  void* fn;
  int w;        // words per thread it was compiled for
  int threads;  // threads per CTA it was compiled for
};
std::vector<JitKernel> g_jit_functions;  // handle - 1 -> kernel

// the kernel of `handle` where it can serve a call: one threshold table for all replicas and no bonds (it has no
// bonded form); fn == nullptr: the prebuilt kernels
JitKernel jit_function(int handle, const int32_t* d_lut_index, const uint32_t* d_bonds) {
  if (handle < 1 || d_lut_index || d_bonds) return JitKernel{nullptr, 0, 0};
  std::lock_guard<std::mutex> lock(g_jit_mutex);
  if (handle > (int)g_jit_functions.size()) return JitKernel{nullptr, 0, 0};
  return g_jit_functions[handle - 1];
}

// What stays fixed over one call of a lattice entry point.
struct Lattice {
  uint32_t* state;
  Geom g;  // geometry, wraps, row0, number of replicas
  const uint32_t* lut;
  const int32_t* lut_index;
  BondParams B;  // B.words == nullptr: ferromagnet
  uint64_t seed;
  uint32_t replica0;
  JitKernel jit;  // jit.fn == nullptr: the prebuilt kernels

  // the same lattices restricted to replicas [r0, r1)
  Lattice replicas(int r0, int r1) const {
    Lattice c = *this;
    c.state += (size_t)r0 * 2 * g.rows * g.wpr;
    c.g.n_replicas = r1 - r0;
    if (lut_index) c.lut_index += r0;
    if (B.index) c.B.index += r0;
    c.replica0 += (uint32_t)r0;
    return c;
  }
};

// The argument rules of the lattice entry points, checked before any CUDA call.  `halo`: rows next to the local ones
// are given (halo rows, or the row after the last for the observables); they take the place of a row wrap.  Bond words
// are indexed by local row, so bonds serve whole lattices only; a bond index needs bond words.
bool args_ok(const Geom& g, const BondParams& B, bool halo, int colour, int row_begin, int row_end) {
  return geom_ok(g.n_replicas, g.rows, g.cols) && rows_ok(g.rows, g.row0) && (colour == 0 || colour == 1) &&
         row_begin >= 0 && row_begin <= row_end && row_end <= g.rows &&
         (!g.wrap_cols || (g.cols % 2 == 0 && g.cols > 2)) &&
         (!g.wrap_rows || (g.rows % 2 == 0 && g.rows > 2) || halo) &&
         (B.words ? !halo && g.row0 == 0 : !B.index);
}

// kernel parameters of a half-sweep of every local row; the wide path narrows the rows and sets its strips
SweepParams sweep_params(const Lattice& L, int colour, uint32_t sweep, const uint32_t* halo_top,
                         const uint32_t* halo_bot) {
  SweepParams P = {};
  P.state = L.state;
  P.lut = L.lut;
  P.lut_index = L.lut_index;
  P.halo_top = halo_top;
  P.halo_bot = halo_bot;
  P.g = L.g;
  P.colour = colour;
  P.sweep = sweep;
  P.replica0 = L.replica0;
  P.k0 = (uint32_t)L.seed;
  P.k1 = (uint32_t)(L.seed >> 32);
  P.keys = tsu_philox_key_schedule(P.k0, P.k1);
  P.strip_rows = 1;
  P.n_strips = L.g.rows;
  P.row_begin = 0;
  P.row_end = L.g.rows;
  P.nvec_fast = L.g.wpr / 4;
  return P;
}

// One half-sweep of `colour` over the local rows [upd_begin, upd_end).  pieces: this launch is one of `pieces` row
// ranges or replica chunks of a half-sweep that run concurrently (split_ranges(), split_replicas()).
int launch_half_sweep(const Lattice& L, int colour, uint32_t sweep, const uint32_t* halo_top, const uint32_t* halo_bot,
                      int upd_begin, int upd_end, int pieces, cudaStream_t st) {
  if (upd_begin >= upd_end) return TSU_OK;
  const Geom& g = L.g;
  const int rows = g.rows, cols = g.cols;
  const bool bonded = L.B.words != nullptr;
  SweepParams P = sweep_params(L, colour, sweep, halo_top, halo_bot);
  // rows that have a north / south neighbour (exactly the cases opp_row() resolves): the wide kernel takes those,
  // columns treated as periodic; what that gets wrong on open lattices is redone by the rim pass
  const bool north_ok = halo_top || g.wrap_rows, south_ok = halo_bot || g.wrap_rows;
  const int rb0 = north_ok ? 0 : 1, re0 = south_ok ? rows : rows - 1;
  const int rb = rb0 > upd_begin ? rb0 : upd_begin, re = re0 < upd_end ? re0 : upd_end;  // rows of the wide kernel
  // words that are full for both row parities: floor(cols / 2) lanes exist in every row of either colour
  const int full_words = (cols / 2) / 32;
  const bool ragged = cols % 256 != 0;
  const int nvec_f = ragged ? full_words / 4 : g.wpr / 4;
  const bool need_rim = rb > upd_begin || re < upd_end || !g.wrap_cols || ragged;
  bool fast = nvec_f >= 1 && re - rb >= 1;
  if (need_rim && tuning().open_generic) fast = false;
  if (fast) {
    const JitKernel& jit = L.jit;
    const int W = jit.fn ? jit.w : (tuning().w == 2 ? 2 : kDefaultW);
    const int nvec = nvec_f * (4 / W);  // W-word groups per row
    const int frows = re - rb;
    P.nvec_fast = nvec_f;
    // strips long enough to amortise the two halo rows and the warp prologue, short enough to fill 148 SMs x 16 warps
    const long long target_threads = 148LL * 2048;
    int strip = 128;
    const long long srows = (long long)frows * pieces;
    while (strip > 1 && (long long)g.n_replicas * nvec * ((srows + strip - 1) / strip) < target_threads) strip >>= 1;
    // the tail of one range is filled by the next: longer strips (less set-up per row) cost nothing there
    if (pieces >= 4) strip = strip * 4 < 128 ? strip * 4 : 128;
    if (tuning().strip > 0) strip = tuning().strip;
    P.strip_rows = strip;
    P.n_strips = (frows + strip - 1) / strip;
    P.row_begin = rb;
    P.row_end = re;
    const long long per_rep_pad = ((long long)P.n_strips * nvec + 31) / 32 * 32;  // warps never straddle replicas
    const long long total = (long long)g.n_replicas * per_rep_pad;
    const unsigned grid = blocks_for(total, 128);
    if (jit.fn) {  // table-specialised build of the same kernel body
      void* args[] = {&P};
      if (tsu_jit::launch(jit.fn, blocks_for(total, jit.threads), jit.threads, 0, (void*)st, args) != 0) return 999;  // driver-API launch failure
    } else if (bonded) {  // one CTA per SM fewer: the next row's 4 W bond words stay in registers without spills
      if (W == 2)
        half_sweep_fast_kernel<2, 6, true><<<grid, 128, 0, st>>>(P, L.B);
      else
        half_sweep_fast_kernel<4, 3, true><<<grid, 128, 0, st>>>(P, L.B);
    } else if (W == 2) {
      half_sweep_fast_kernel<2, 8, false><<<grid, 128, 0, st>>>(P, kNoBonds);
    } else {
      half_sweep_fast_kernel<4, 4, false><<<grid, 128, 0, st>>>(P, kNoBonds);
    }
    if (need_rim) {
      RimRows R;
      R.a0 = upd_begin; R.a1 = rb;   // updated rows above / below the wide kernel's range (no north / south neighbour)
      R.b0 = re; R.b1 = upd_end;
      R.p0 = rb; R.p1 = re;
      R.head = (ragged || !g.wrap_cols) ? 1 : 0;
      R.tail_begin = ragged ? 4 * nvec_f : (g.wrap_cols ? g.wpr : g.wpr - 1);
      const long long per_rep = (long long)((R.a1 - R.a0) + (R.b1 - R.b0)) * g.wpr +
                                (long long)(R.head + g.wpr - R.tail_begin) * frows;
      if (per_rep > 0) {
        if (bonded)
          half_sweep_rim_kernel<true><<<blocks_for(per_rep * g.n_replicas, 128), 128, 0, st>>>(P, R, L.B);
        else
          half_sweep_rim_kernel<false><<<blocks_for(per_rep * g.n_replicas, 128), 128, 0, st>>>(P, R, kNoBonds);
      }
    }
  } else {
    P.row_begin = upd_begin;
    P.row_end = upd_end;
    const long long total = (long long)g.n_replicas * (upd_end - upd_begin) * g.wpr;
    if (bonded)
      half_sweep_generic_kernel<true><<<blocks_for(total, 128), 128, 0, st>>>(P, L.B);
    else
      half_sweep_generic_kernel<false><<<blocks_for(total, 128), 128, 0, st>>>(P, kNoBonds);
  }
  TSU_RETURN_LAUNCH_STATUS();
}

// Row ranges a half-sweep is cut into.  One launch per half-sweep loses ~15 us to its tail (launch gap, the last warps
// finishing alone: measured, tools/lattice_trace.py); ranges on streams of their own, each depending only on its
// neighbours' previous half-sweep, let the next half-sweep start while this one drains.  Pays between ~0.1 and ~5 ms
// per half-sweep (6.8 % on a 16384 x 131072 slab, 2.5 % on 131072^2); TSU_LATTICE_SPLIT overrides (1 = never).
int split_ranges(int n_replicas, int rows, int cols) {
  int K;
  if (tuning().split >= 1) {
    K = tuning().split < kMaxSplit ? tuning().split : kMaxSplit;
  } else {
    const double sites = (double)n_replicas * rows * cols;
    K = (sites >= 1e9 && sites <= 6e10) ? kDefaultSplit : 1;
  }
  while (K > 1 && rows / K < 256) --K;  // short ranges would only add launches
  return K;
}

// Chunks of replicas a batch of lattices is cut into for the same reason (replicas do not depend on each other, so
// every chunk simply runs its half-sweeps back to back on its own stream).  TSU_LATTICE_SPLIT=1 disables.
int split_replicas(int n_replicas, int rows, int cols) {
  if (tuning().split == 1 || n_replicas < 2 * kDefaultSplit) return 1;
  const double sites = (double)n_replicas * rows * cols;
  if (tuning().split < 1 && !(sites >= 5e8 && sites <= 6e10)) return 1;
  return tuning().split > 1 ? (tuning().split < kMaxSplit ? tuning().split : kMaxSplit) : kDefaultSplit;
}

// The streams of one call that runs row ranges or replica chunks concurrently: s[0] is the caller's stream,
// s[1 .. K-1] are library streams (slab_stream) and s[K] is the caller's `side` stream if one is given.  They all start
// after what the caller queued before the call.  join() makes the caller's stream wait for all of them, so that to
// the caller the call stays ordered on its own stream; the destructor does the same on any other way out.
// ev[k][j] is for stream k to record after its half-sweep of colour j.
struct StreamFork {
  cudaStream_t s[kMaxSplit + 1];
  cudaEvent_t ev[kMaxSplit + 1][2] = {};
  cudaEvent_t fork = nullptr;
  int n = 0;            // streams forked, joined back by release()
  int status = TSU_OK;  // otherwise nothing was forked: the call returns this

  StreamFork(cudaStream_t caller, int K, const cudaStream_t* side = nullptr) {
    int dev = 0;
    cudaGetDevice(&dev);
    s[0] = caller;
    bool ok = true;
    for (int k = 1; k < K && ok; ++k) ok = (s[k] = slab_stream(dev, k - 1)) != nullptr;
    const int m = side ? K + 1 : K;
    if (side) s[K] = *side;
    ok = ok && cudaEventCreateWithFlags(&fork, cudaEventDisableTiming) == cudaSuccess;
    for (int k = 0; k < m && ok; ++k)
      for (int j = 0; j < 2 && ok; ++j) ok = cudaEventCreateWithFlags(&ev[k][j], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {  // (a failed slab_stream need not leave an error behind)
      const cudaError_t e = cudaGetLastError();
      status = e != cudaSuccess ? (int)e : (int)cudaErrorUnknown;
      return;
    }
    cudaEventRecord(fork, caller);
    for (int k = 1; k < m; ++k) cudaStreamWaitEvent(s[k], fork, 0);
    n = m;
  }
  ~StreamFork() { release(); }

  void release() {
    for (int k = 1; k < n; ++k) {
      cudaEventRecord(fork, s[k]);
      cudaStreamWaitEvent(s[0], fork, 0);
    }
    n = 0;
    for (auto& evk : ev)
      for (cudaEvent_t& e : evk) {
        if (e) cudaEventDestroy(e);
        e = nullptr;
      }
    if (fork) cudaEventDestroy(fork);
    fork = nullptr;
  }

  // status of a call whose launches returned rc, after the join
  int join(int rc) {
    release();
    if (rc != TSU_OK) return rc;
    TSU_RETURN_LAUNCH_STATUS();
  }
};

// the whole-lattice sweeps of tsu_ising2d_sweeps (no halos)
int launch_sweeps(const Lattice& L, uint32_t sweep0, int n_sweeps, cudaStream_t st) {
  const Geom& g = L.g;
  if (n_sweeps == 0) return TSU_OK;
  // many replicas: independent chunks of replicas, one stream each, no dependency between them at all
  const int KR = split_replicas(g.n_replicas, g.rows, g.cols);
  if (KR > 1) {
    StreamFork F(st, KR);
    if (F.status != TSU_OK) return F.status;
    int rc = TSU_OK;
    for (int k = 0; k < KR && rc == TSU_OK; ++k) {
      const int r0 = (int)((long long)g.n_replicas * k / KR), r1 = (int)((long long)g.n_replicas * (k + 1) / KR);
      const Lattice c = L.replicas(r0, r1);
      for (int t = 0; t < 2 * n_sweeps && rc == TSU_OK; ++t)
        rc = launch_half_sweep(c, t & 1, sweep0 + (uint32_t)(t >> 1), nullptr, nullptr, 0, g.rows, KR, F.s[k]);
    }
    return F.join(rc);
  }
  const int K = split_ranges(g.n_replicas, g.rows, g.cols);
  if (K <= 2) {
    for (int t = 0; t < 2 * n_sweeps; ++t) {
      const int rc = launch_half_sweep(L, t & 1, sweep0 + (uint32_t)(t >> 1), nullptr, nullptr, 0, g.rows, 1, st);
      if (rc != TSU_OK) return rc;
    }
    return TSU_OK;
  }
  StreamFork F(st, K);
  if (F.status != TSU_OK) return F.status;
  int bound[kMaxSplit + 1];
  for (int k = 0; k <= K; ++k) bound[k] = (int)((long long)g.rows * k / K);
  int rc = TSU_OK;
  for (int t = 0; t < 2 * n_sweeps && rc == TSU_OK; ++t) {
    const int j = t & 1, jp = j ^ 1;
    // the range launched first changes every half-sweep: with periodic rows range 0 depends on range K - 1, and what
    // the first range of a half-sweep depends on should be what the half-sweep before launched first
    for (int i = 0; i < K && rc == TSU_OK; ++i) {
      const int k = (t + i) % K, above = (k + K - 1) % K, below = (k + 1) % K;
      if (t > 0) {
        if (k > 0 || g.wrap_rows) cudaStreamWaitEvent(F.s[k], F.ev[above][jp], 0);
        if (k + 1 < K || g.wrap_rows) cudaStreamWaitEvent(F.s[k], F.ev[below][jp], 0);
      }
      rc = launch_half_sweep(L, j, sweep0 + (uint32_t)(t >> 1), nullptr, nullptr, bound[k], bound[k + 1], K, F.s[k]);
      cudaEventRecord(F.ev[k][j], F.s[k]);
    }
  }
  return F.join(rc);
}

// true when a replica is small enough that per-half-sweep launches would be pure launch latency
bool resident_eligible(int n_replicas, int rows, int cols) {
  if (tuning().resident == 0) return false;
  const long long per_rep = (long long)rows * words_per_row(cols);
  // <= 16 words per thread and half-sweep, and not enough replicas to fill the GPU with the wide kernels
  return per_rep <= 16LL * kResidentThreads && (long long)n_replicas * per_rep <= 148LL * 2048;
}

int launch_resident_sweeps(const Lattice& L, uint32_t sweep0, int n_sweeps, cudaStream_t st) {
  const SweepParams P = sweep_params(L, 0, sweep0, nullptr, nullptr);
  if (L.B.words)
    sweeps_resident_kernel<true><<<L.g.n_replicas, kResidentThreads, 0, st>>>(P, n_sweeps, L.B);
  else
    sweeps_resident_kernel<false><<<L.g.n_replicas, kResidentThreads, 0, st>>>(P, n_sweeps, kNoBonds);
  TSU_RETURN_LAUNCH_STATUS();
}

// full-word lattices count at HBM speed (observables_fast_kernel); the others word by word
bool obs_fast(int cols) { return cols % 256 == 0 && !tuning().obs_generic; }

// the counts of tsu_ising2d_observables into out[replica][2] (zeroed first)
int launch_observables(const uint32_t* state, const Geom& g, const BondParams& B, const uint32_t* next_rows,
                       unsigned long long* out, cudaStream_t st) {
  const int n_replicas = g.n_replicas, rows = g.rows;
  cudaError_t e = cudaMemsetAsync(out, 0, sizeof(unsigned long long) * 2 * (size_t)n_replicas, st);
  if (e != cudaSuccess) return (int)e;
  if (obs_fast(g.cols)) {
    const int nvec = g.wpr / 4;
    int strip = 64;  // long strips re-read one row in `strip`; short ones fill the GPU for small batches
    while (strip > 1 && (long long)n_replicas * nvec * ((rows + strip - 1) / strip) < 148LL * 2048) strip >>= 1;
    const int n_strips = (rows + strip - 1) / strip;
    const long long per_rep_pad = ((long long)n_strips * nvec + 31) / 32 * 32;
    const unsigned grid = blocks_for((long long)n_replicas * per_rep_pad, 128);
    if (B.words)
      observables_fast_kernel<true><<<grid, 128, 0, st>>>(state, g, next_rows, strip, n_strips, out, B);
    else
      observables_fast_kernel<false><<<grid, 128, 0, st>>>(state, g, next_rows, strip, n_strips, out, kNoBonds);
    TSU_RETURN_LAUNCH_STATUS();
  }
  TSU_CHECK_ARG(n_replicas <= 65535);  // gridDim.y of the word-by-word kernel
  const long long n_words = 2LL * rows * g.wpr;
  long long bx = (n_words + 255) / 256;
  const long long cap = (148LL * 8 + n_replicas - 1) / n_replicas;  // about 8 CTAs per SM in total
  if (bx > cap) bx = cap < 1 ? 1 : cap;
  dim3 grid((unsigned)bx, (unsigned)n_replicas);
  if (B.words)
    observables_kernel<true><<<grid, 256, 0, st>>>(state, g, next_rows, out, B);
  else
    observables_kernel<false><<<grid, 256, 0, st>>>(state, g, next_rows, out, kNoBonds);
  TSU_RETURN_LAUNCH_STATUS();
}

// The anneal of tsu_ising2d_anneal for lattices too large for anneal_resident_kernel, on one stream: the initial state
// is evaluated, then every step is one sweep (L.lut + 32 k is its table), the counts, anneal_select_kernel and, when
// the best states are kept, anneal_copy_kernel.  pieces > 1: L is one of that many replica chunks running concurrently.
int launch_anneal(const Lattice& L, const AnnealOut& A, int n_steps, uint32_t sweep0, unsigned long long* obs, int pieces,
                  cudaStream_t st) {
  const Geom& g = L.g;
  const int n = g.n_replicas;
  const long long rep_vecs = 2LL * g.rows * g.wpr / 4;  // wpr is a multiple of 4
  long long bx = (rep_vecs + 255) / 256;
  const long long cap = (148LL * 8 + n - 1) / n;  // about 8 CTAs per SM when every replica improves
  if (bx > cap) bx = cap < 1 ? 1 : cap;
  const dim3 copy_grid((unsigned)bx, (unsigned)(n < 65535 ? n : 65535));
  for (int k = -1; k < n_steps; ++k) {
    if (k >= 0) {
      Lattice Lk = L;
      Lk.lut = L.lut + 32 * (size_t)k;
      const uint32_t sweep = sweep0 + (uint32_t)k;
      int rc;
      if (pieces > 1) {  // a replica chunk: its half-sweeps back to back, as launch_sweeps runs them
        rc = launch_half_sweep(Lk, 0, sweep, nullptr, nullptr, 0, g.rows, pieces, st);
        if (rc == TSU_OK) rc = launch_half_sweep(Lk, 1, sweep, nullptr, nullptr, 0, g.rows, pieces, st);
      } else {  // row ranges on streams of their own are joined back into st before the counts
        rc = launch_sweeps(Lk, sweep, 1, st);
      }
      if (rc != TSU_OK) return rc;
    }
    const int rc = launch_observables(L.state, g, L.B, nullptr, obs, st);
    if (rc != TSU_OK) return rc;
    anneal_select_kernel<<<blocks_for(n, 128), 128, 0, st>>>(obs, n, A);
    if (A.best_energy)
      anneal_copy_kernel<<<copy_grid, 256, 0, st>>>(reinterpret_cast<const uint4*>(L.state),
                                                    reinterpret_cast<uint4*>(A.best_state), obs, n, rep_vecs);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
  }
  return TSU_OK;
}

// The counts of a population-annealing step into obs[replica][2]: the observables kernels, or one warp per replica where
// the word-by-word kernel's grid would be too tall (more than 65535 replicas of lattices without full words).
int launch_population_counts(const Lattice& L, unsigned long long* obs, cudaStream_t st) {
  const Geom& g = L.g;
  if (obs_fast(g.cols) || g.n_replicas <= 65535) return launch_observables(L.state, g, L.B, nullptr, obs, st);
  const unsigned grid = blocks_for(32LL * g.n_replicas, 256);
  if (L.B.words)
    pa_count_kernel<true><<<grid, 256, 0, st>>>(L.state, g, obs, L.B);
  else
    pa_count_kernel<false><<<grid, 256, 0, st>>>(L.state, g, obs, kNoBonds);
  TSU_RETURN_LAUNCH_STATUS();
}

// E of every replica, and per population the count sums and E_ref, of the state L holds now
int launch_population_reduce(const Lattice& L, const PopParams& Q, const AnnealOut& A, unsigned long long* obs,
                             unsigned long long* sums, cudaStream_t st) {
  const int rc = launch_population_counts(L, obs, st);
  if (rc != TSU_OK) return rc;
  long long bx = (Q.rp + kPaThreads - 1) / kPaThreads;
  const long long cap = (148LL * 8 + Q.n_pop - 1) / Q.n_pop;  // about 8 CTAs per SM in total
  if (bx > cap) bx = cap;
  pa_reduce_kernel<<<dim3((unsigned)bx, (unsigned)Q.n_pop), kPaThreads, 0, st>>>(obs, Q, A, sums);
  TSU_RETURN_LAUNCH_STATUS();
}

// bytes of the Swendsen-Wang work buffer per replica (layout at ClusterParams); 0 for lattices it cannot label
long long cluster_rep_bytes(int rows, int cols) {
  if (rows <= 0 || cols <= 0 || (long long)rows * cols > 2147483647LL) return 0;
  const long long label_bytes = (4LL * rows * cols + 15) / 16 * 16;
  return label_bytes + 24LL * rows * words_per_row(cols);
}

// n_steps Swendsen-Wang steps of the replicas of L, which own C.work: one launch for lattices whose labels fit a
// block's shared memory, otherwise four launches per step (bonds, local labels, merges across tiles, flips)
int launch_swendsen_wang(const Lattice& L, const ClusterParams& C, uint32_t sweep0, int n_steps, cudaStream_t st) {
  const Geom& g = L.g;
  SweepParams P = sweep_params(L, 0, sweep0, nullptr, nullptr);
  const bool bonded = L.B.words != nullptr;
  if (tuning().resident != 0 && (long long)g.rows * g.cols <= kClusterResidentSites) {
    const size_t smem = sizeof(int32_t) * (size_t)g.rows * g.cols;
    if (bonded)
      cluster_resident_kernel<true><<<g.n_replicas, kClusterThreads, smem, st>>>(P, L.B, C, n_steps);
    else
      cluster_resident_kernel<false><<<g.n_replicas, kClusterThreads, smem, st>>>(P, kNoBonds, C, n_steps);
    TSU_RETURN_LAUNCH_STATUS();
  }
  const unsigned word_grid = blocks_for(2LL * g.rows * g.wpr * g.n_replicas, kClusterThreads);
  const int tiles_x = (g.cols + kClusterTileCols - 1) / kClusterTileCols;
  const int tiles_y = (g.rows + kClusterTileRows - 1) / kClusterTileRows;
  const unsigned merge_grid =
      blocks_for(((long long)tiles_y * g.cols + (long long)g.rows * tiles_x) * g.n_replicas, kClusterThreads);
  for (int s = 0; s < n_steps; ++s) {
    P.sweep = sweep0 + (uint32_t)s;
    if (bonded)
      cluster_bonds_kernel<true><<<word_grid, kClusterThreads, 0, st>>>(P, L.B, C);
    else
      cluster_bonds_kernel<false><<<word_grid, kClusterThreads, 0, st>>>(P, kNoBonds, C);
    cluster_local_kernel<<<(unsigned)((long long)tiles_x * tiles_y * g.n_replicas), kClusterThreads, 0, st>>>(
        P, C, tiles_x, tiles_x * tiles_y);
    cluster_merge_kernel<<<merge_grid, kClusterThreads, 0, st>>>(P, C, tiles_y, tiles_x);
    cluster_flip_kernel<<<word_grid, kClusterThreads, 0, st>>>(P, C);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
  }
  return TSU_OK;
}

}  // namespace

extern "C" {

void tsu_ising2d_reload_tuning(void) { g_tuning = Tuning(); }

#ifdef TSU_LATTICE_TRACE
int tsu_debug_lattice_trace(unsigned long long* h_out) {  // 4 x 3 x 8192 words
  return (int)cudaMemcpyFromSymbol(h_out, g_lat_trace, sizeof(unsigned long long) * 4 * 3 * kTraceCtas);
}
#endif

int64_t tsu_ising2d_words_per_row(int cols) { return cols > 0 ? words_per_row(cols) : 0; }

int64_t tsu_ising2d_state_words(int rows, int cols) {
  return (rows > 0 && cols > 0) ? 2LL * rows * words_per_row(cols) : 0;
}

int tsu_ising2d_init_random(uint32_t* d_state, int n_replicas, int rows, int cols, uint64_t seed, uint32_t replica0,
                            int row0, uintptr_t stream) {
  TSU_CHECK_ARG(d_state && geom_ok(n_replicas, rows, cols) && rows_ok(rows, row0));
  Geom g = make_geom(n_replicas, rows, cols, 0, 0, row0);
  const long long total = 2LL * rows * g.wpr * n_replicas;
  init_random_kernel<<<blocks_for(total, 256), 256, 0, tsu_stream(stream)>>>(d_state, g, replica0, (uint32_t)seed,
                                                                            (uint32_t)(seed >> 32));
  TSU_RETURN_LAUNCH_STATUS();
}

int tsu_ising2d_pack(const int8_t* d_spins, uint32_t* d_state, int n_replicas, int rows, int cols, uintptr_t stream) {
  TSU_CHECK_ARG(d_spins && d_state && geom_ok(n_replicas, rows, cols));
  Geom g = make_geom(n_replicas, rows, cols, 0, 0, 0);
  const long long total = 2LL * rows * g.wpr * n_replicas;
  pack_kernel<<<blocks_for(total, 256), 256, 0, tsu_stream(stream)>>>(d_spins, d_state, g);
  TSU_RETURN_LAUNCH_STATUS();
}

int tsu_ising2d_unpack(const uint32_t* d_state, int8_t* d_spins, int n_replicas, int rows, int cols, int as_pm1,
                       uintptr_t stream) {
  TSU_CHECK_ARG(d_spins && d_state && geom_ok(n_replicas, rows, cols));
  Geom g = make_geom(n_replicas, rows, cols, 0, 0, 0);
  const long long total = 2LL * rows * g.wpr * n_replicas;
  unpack_kernel<<<blocks_for(total, 256), 256, 0, tsu_stream(stream)>>>(d_state, d_spins, g, as_pm1);
  TSU_RETURN_LAUNCH_STATUS();
}

int tsu_ising2d_half_sweep(int jit_handle, uint32_t* d_state, int n_replicas, int rows, int cols, int wrap_rows,
                           int wrap_cols, int colour, const uint32_t* d_lut, const int32_t* d_lut_index,
                           const uint32_t* d_bonds, const int32_t* d_bond_index, uint64_t seed, uint32_t sweep,
                           uint32_t replica0, int row0, const uint32_t* d_halo_top, const uint32_t* d_halo_bot,
                           int row_begin, int row_end, uintptr_t stream) {
  const Lattice L = {d_state, make_geom(n_replicas, rows, cols, wrap_rows, wrap_cols, row0), d_lut, d_lut_index,
                     {d_bonds, d_bond_index}, seed, replica0, jit_function(jit_handle, d_lut_index, d_bonds)};
  TSU_CHECK_ARG(d_state && d_lut && args_ok(L.g, L.B, d_halo_top || d_halo_bot, colour, row_begin, row_end));
  return launch_half_sweep(L, colour, sweep, d_halo_top, d_halo_bot, row_begin, row_end, 1, tsu_stream(stream));
}

int tsu_ising2d_slab_sweeps_p2p(int jit_handle, uint32_t* d_state, int n_replicas, int rows, int cols, int wrap_cols,
                                const uint32_t* d_lut, const int32_t* d_lut_index, uint64_t seed, uint32_t sweep0,
                                int n_sweeps, uint32_t replica0, int row0, uint32_t* d_halo, uint32_t* d_flags,
                                uint32_t* d_up_halo, uint32_t* d_up_flags, uint32_t* d_down_halo, uint32_t* d_down_flags,
                                uint32_t msgs_colour0, uint32_t msgs_colour1, uintptr_t main_stream,
                                uintptr_t side_stream) {
  const Lattice L = {d_state, make_geom(n_replicas, rows, cols, 0, wrap_cols, row0), d_lut, d_lut_index, kNoBonds, seed,
                     replica0, jit_function(jit_handle, d_lut_index, nullptr)};
  TSU_CHECK_ARG(d_state && d_lut && d_halo && d_flags && args_ok(L.g, L.B, false, 0, 0, rows));
  TSU_CHECK_ARG(rows >= 4 && n_sweeps >= 0 && main_stream != side_stream);
  TSU_CHECK_ARG((d_up_halo == nullptr) == (d_up_flags == nullptr) && (d_down_halo == nullptr) == (d_down_flags == nullptr));
  cudaStream_t main = tsu_stream(main_stream), side = tsu_stream(side_stream);
  const int wpr = L.g.wpr;
  const size_t side_words = (size_t)n_replicas * wpr;  // one halo row set
  auto halo = [&](uint32_t* base, int colour, int which) { return base ? base + ((size_t)colour * 2 + which) * side_words : nullptr; };
  auto flag = [&](uint32_t* base, int colour, int which) { return base ? base + colour * 2 + which : nullptr; };
  uint32_t msgs[2] = {msgs_colour0, msgs_colour1};
  // The interior rows are cut into row ranges launched on streams of their own: range k of a half-sweep depends only on
  // ranges k - 1, k, k + 1 (and, at the ends, on the boundary rows) of the half-sweep before, so the first ranges of
  // the next half-sweep fill the SMs while the last ranges of this one drain.  A single launch per half-sweep loses
  // ~15 us to its tail (launch gap + the last warps finishing alone), 6 % of a 16384 x 131072 slab.
  const int K = split_ranges(n_replicas, rows - 2, cols);
  int bound[kMaxSplit + 1];  // range k = local rows [bound[k], bound[k + 1])
  for (int k = 0; k <= K; ++k) bound[k] = 1 + (int)((long long)(rows - 2) * k / K);
  // range k runs on F.s[k]; the boundary rows run on the side stream F.s[K] and record F.ev[K].  Everything the caller
  // queued on the main stream (e.g. a changed state) precedes the first rows sent and updated.
  StreamFork F(main, K, &side);
  if (F.status != TSU_OK) return F.status;
  const unsigned send_grid = blocks_for(2LL * n_replicas * (wpr / 4), 256) < 64u ? blocks_for(2LL * n_replicas * (wpr / 4), 256) : 64u;
  // what a half-sweep of `colour` sends afterwards: my first row to the rank above (its "below" halo), my last row
  // to the rank below (its "above" halo), then the message number
  auto send = [&](int colour) {
    ++msgs[colour];
    slab_send_rows_kernel<<<send_grid, 256, 0, side>>>(d_state, n_replicas, rows, wpr, colour, halo(d_up_halo, colour, 1),
                                                      halo(d_down_halo, colour, 0));
    slab_signal_kernel<<<1, 1, 0, side>>>(flag(d_up_flags, colour, 1), flag(d_down_flags, colour, 0), msgs[colour]);
  };
  int rc = TSU_OK;
  send(1);  // colour 0 goes first and reads colour 1
  for (int t = 0; t < 2 * n_sweeps && rc == TSU_OK; ++t) {
    const int colour = t & 1, opp = 1 - colour, j = t & 1, jp = j ^ 1;
    const uint32_t sweep = sweep0 + (uint32_t)(t >> 1);
    // interior ranges: each reads and overwrites rows next to what its neighbours updated in the half-sweep before
    for (int k = 0; k < K && rc == TSU_OK; ++k) {
      if (t > 0) {
        if (k > 0) cudaStreamWaitEvent(F.s[k], F.ev[k - 1][jp], 0);
        if (k + 1 < K) cudaStreamWaitEvent(F.s[k], F.ev[k + 1][jp], 0);
        if (k == 0 || k + 1 == K) cudaStreamWaitEvent(F.s[k], F.ev[K][jp], 0);
      }
      rc = launch_half_sweep(L, colour, sweep, nullptr, nullptr, bound[k], bound[k + 1], K, F.s[k]);
      cudaEventRecord(F.ev[k][j], F.s[k]);
    }
    if (rc != TSU_OK) break;
    // boundary rows on the side stream: after the previous update of the rows next to them and the arrival of the
    // neighbours' rows of the other colour
    if (t > 0) {
      cudaStreamWaitEvent(side, F.ev[0][jp], 0);
      if (K > 1) cudaStreamWaitEvent(side, F.ev[K - 1][jp], 0);
    }
    const uint32_t* top = d_up_halo ? halo(d_halo, opp, 0) : nullptr;
    const uint32_t* bot = d_down_halo ? halo(d_halo, opp, 1) : nullptr;
    if (top || bot)
      slab_wait_kernel<<<1, 1, 0, side>>>(top ? flag(d_flags, opp, 0) : nullptr, bot ? flag(d_flags, opp, 1) : nullptr,
                                          msgs[opp], d_flags + 8);
    rc = launch_half_sweep(L, colour, sweep, top, bot, 0, 1, 1, side);
    if (rc == TSU_OK) rc = launch_half_sweep(L, colour, sweep, top, bot, rows - 1, rows, 1, side);
    cudaEventRecord(F.ev[K][j], side);
    send(colour);
  }
  return F.join(rc);
}

int tsu_ising2d_sweeps(int jit_handle, uint32_t* d_state, int n_replicas, int rows, int cols, int wrap_rows,
                       int wrap_cols, const uint32_t* d_lut, const int32_t* d_lut_index, const uint32_t* d_bonds,
                       const int32_t* d_bond_index, uint64_t seed, uint32_t sweep0, int n_sweeps, uint32_t replica0,
                       uintptr_t stream) {
  const Lattice L = {d_state, make_geom(n_replicas, rows, cols, wrap_rows, wrap_cols, 0), d_lut, d_lut_index,
                     {d_bonds, d_bond_index}, seed, replica0, jit_function(jit_handle, d_lut_index, d_bonds)};
  TSU_CHECK_ARG(d_state && d_lut && n_sweeps >= 0 && args_ok(L.g, L.B, false, 0, 0, rows));
  if (n_sweeps > 0 && resident_eligible(n_replicas, rows, cols))  // launch latency dominates: one launch for everything
    return launch_resident_sweeps(L, sweep0, n_sweeps, tsu_stream(stream));
  return launch_sweeps(L, sweep0, n_sweeps, tsu_stream(stream));
}

int tsu_ising2d_half_sweep_injected(uint32_t* d_state, int n_replicas, int rows, int cols, int wrap_rows,
                                    int wrap_cols, int colour, const uint32_t* d_lut, const int32_t* d_lut_index,
                                    const uint32_t* d_bonds, const int32_t* d_bond_index, const uint32_t* d_uniforms,
                                    int row0, const uint32_t* d_halo_top, const uint32_t* d_halo_bot,
                                    uintptr_t stream) {
  const Lattice L = {d_state, make_geom(n_replicas, rows, cols, wrap_rows, wrap_cols, row0), d_lut, d_lut_index,
                     {d_bonds, d_bond_index}, 0, 0, JitKernel{nullptr, 0, 0}};
  TSU_CHECK_ARG(d_state && d_lut && d_uniforms && args_ok(L.g, L.B, d_halo_top || d_halo_bot, colour, 0, rows));
  const SweepParams P = sweep_params(L, colour, 0, d_halo_top, d_halo_bot);
  const unsigned grid = blocks_for((long long)n_replicas * rows * L.g.wpr, 128);
  cudaStream_t st = tsu_stream(stream);
  if (d_bonds)
    half_sweep_injected_kernel<true><<<grid, 128, 0, st>>>(P, d_uniforms, L.B);
  else
    half_sweep_injected_kernel<false><<<grid, 128, 0, st>>>(P, d_uniforms, kNoBonds);
  TSU_RETURN_LAUNCH_STATUS();
}

int tsu_ising2d_observables(const uint32_t* d_state, int n_replicas, int rows, int cols, int wrap_rows, int wrap_cols,
                            const uint32_t* d_bonds, const int32_t* d_bond_index, int row0, const uint32_t* d_next_rows,
                            unsigned long long* d_out, uintptr_t stream) {
  const Geom g = make_geom(n_replicas, rows, cols, wrap_rows, wrap_cols, row0);
  const BondParams B = {d_bonds, d_bond_index};
  TSU_CHECK_ARG(d_state && d_out && args_ok(g, B, d_next_rows != nullptr, 0, 0, rows));
  return launch_observables(d_state, g, B, d_next_rows, d_out, tsu_stream(stream));
}

int tsu_ising2d_anneal(uint32_t* d_state, int n_replicas, int rows, int cols, int wrap_rows, int wrap_cols,
                       const uint32_t* d_luts, int n_steps, const uint32_t* d_bonds, const int32_t* d_bond_index,
                       uint64_t seed, uint32_t sweep0, uint32_t replica0, double J, double h, long long n_bonds,
                       long long n_sites, unsigned long long* d_obs, double* d_energy, double* d_best_energy,
                       uint32_t* d_best_state, uintptr_t stream) {
  const Lattice L = {d_state, make_geom(n_replicas, rows, cols, wrap_rows, wrap_cols, 0), d_luts, nullptr,
                     {d_bonds, d_bond_index}, seed, replica0, JitKernel{nullptr, 0, 0}};
  TSU_CHECK_ARG(d_state && args_ok(L.g, L.B, false, 0, 0, rows) && n_steps >= 0 && (d_luts || n_steps == 0));
  TSU_CHECK_ARG(d_obs && d_energy && (d_best_energy == nullptr) == (d_best_state == nullptr));
  const AnnealOut A = {J, h, n_bonds, n_sites, d_energy, d_best_energy, d_best_state};
  cudaStream_t st = tsu_stream(stream);
  if (resident_eligible(n_replicas, rows, cols)) {
    const SweepParams P = sweep_params(L, 0, sweep0, nullptr, nullptr);
    if (d_bonds)
      anneal_resident_kernel<true><<<n_replicas, kResidentThreads, 0, st>>>(P, d_luts, n_steps, L.B, A);
    else
      anneal_resident_kernel<false><<<n_replicas, kResidentThreads, 0, st>>>(P, d_luts, n_steps, kNoBonds, A);
    TSU_RETURN_LAUNCH_STATUS();
  }
  TSU_CHECK_ARG(obs_fast(cols) || n_replicas <= 65535);  // as tsu_ising2d_observables
  const int KR = split_replicas(n_replicas, rows, cols);
  if (KR == 1) return launch_anneal(L, A, n_steps, sweep0, d_obs, 1, st);
  // replica chunks do not depend on each other: each runs its whole anneal on its own stream
  StreamFork F(st, KR);
  if (F.status != TSU_OK) return F.status;
  int rc = TSU_OK;
  for (int k = 0; k < KR && rc == TSU_OK; ++k) {
    const int r0 = (int)((long long)n_replicas * k / KR), r1 = (int)((long long)n_replicas * (k + 1) / KR);
    AnnealOut Ak = A;
    Ak.energy += r0;
    if (Ak.best_energy) {
      Ak.best_energy += r0;
      Ak.best_state += (size_t)r0 * 2 * rows * L.g.wpr;
    }
    rc = launch_anneal(L.replicas(r0, r1), Ak, n_steps, sweep0, d_obs + 2 * (size_t)r0, KR, F.s[k]);
  }
  return F.join(rc);
}

int64_t tsu_ising2d_population_work_bytes(int n_replicas, int n_populations) {
  if (n_replicas <= 0 || n_populations <= 0 || n_replicas % n_populations) return 0;
  const long long rp = n_replicas / n_populations, nt = (rp + kPaTile - 1) / kPaTile;
  return 8LL * (n_replicas + (long long)n_populations * (nt + 2));
}

int tsu_ising2d_population_anneal(uint32_t* d_state, uint32_t* d_scratch, int n_replicas, int rows, int cols,
                                  int wrap_rows, int wrap_cols, const uint32_t* d_luts, const double* d_dbeta,
                                  int n_steps, int sweeps_per_step, int n_populations, const uint32_t* d_bonds,
                                  const int32_t* d_bond_index, uint64_t seed, uint32_t sweep0, uint32_t replica0,
                                  double J, double h, long long n_bonds, long long n_sites, int32_t* d_family,
                                  int32_t* d_family_scratch, unsigned long long* d_weight_sum, double* d_energy_ref,
                                  unsigned long long* d_count_sums, unsigned long long* d_obs, double* d_energy,
                                  void* d_work, size_t work_bytes, uintptr_t stream) {
  Lattice L = {d_state, make_geom(n_replicas, rows, cols, wrap_rows, wrap_cols, 0), d_luts, nullptr,
               {d_bonds, d_bond_index}, seed, replica0, JitKernel{nullptr, 0, 0}};
  TSU_CHECK_ARG(d_state && d_scratch && d_state != d_scratch && args_ok(L.g, L.B, false, 0, 0, rows));
  TSU_CHECK_ARG(n_steps >= 0 && sweeps_per_step >= 1 && n_populations >= 1 && n_populations <= 65535 &&
                n_replicas % n_populations == 0);
  TSU_CHECK_ARG(n_steps == 0 || (d_luts && d_dbeta && d_weight_sum && d_energy_ref));
  TSU_CHECK_ARG(d_family && d_family_scratch && d_family != d_family_scratch && d_count_sums && d_obs && d_energy);
  TSU_CHECK_ARG(d_work && work_bytes >= (size_t)tsu_ising2d_population_work_bytes(n_replicas, n_populations));
  PopParams Q;
  Q.rp = n_replicas / n_populations;
  Q.n_pop = n_populations;
  Q.nt = (Q.rp + kPaTile - 1) / kPaTile;
  int lg = 0;
  while ((1LL << lg) < Q.rp) ++lg;
  Q.s = 62 - lg;
  Q.prefix = static_cast<unsigned long long*>(d_work);
  Q.tile_off = Q.prefix + n_replicas;
  Q.min_key = Q.tile_off + (size_t)n_populations * Q.nt;
  Q.draw = Q.min_key + n_populations;
  const AnnealOut A = {J, h, n_bonds, n_sites, d_energy, nullptr, nullptr};
  cudaStream_t st = tsu_stream(stream);
  const size_t sums_per_step = 2 * (size_t)n_populations;
  cudaError_t e = cudaMemsetAsync(d_count_sums, 0, sizeof(unsigned long long) * sums_per_step * (n_steps + 1), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(Q.min_key, 0xff, sizeof(unsigned long long) * n_populations, st);
  if (e != cudaSuccess) return (int)e;
  // the gather: a group of threads per child, at least 4 vectors per thread, or whole blocks for large replicas
  const long long rep_vecs = 2LL * rows * L.g.wpr / 4;  // wpr is a multiple of 4
  int group = 1;
  while (group < 256 && 4LL * group < rep_vecs) group <<= 1;
  dim3 gather_grid;
  if (group < 256) {
    gather_grid = dim3(blocks_for(n_replicas, 256 / group));
  } else {
    long long bx = (rep_vecs + 4 * 256 - 1) / (4 * 256);
    const long long cap = (148LL * 8 + n_replicas - 1) / n_replicas;  // about 8 CTAs per SM in total
    if (bx > cap) bx = cap;
    gather_grid = dim3((unsigned)bx, (unsigned)(n_replicas < 65535 ? n_replicas : 65535));
  }
  const bool resident = resident_eligible(n_replicas, rows, cols);
  uint32_t* other = d_scratch;
  int32_t* fam = d_family;
  int32_t* fam_other = d_family_scratch;
  for (int k = 0; k < n_steps; ++k) {
    int rc = launch_population_reduce(L, Q, A, d_obs, d_count_sums + sums_per_step * k, st);
    if (rc != TSU_OK) return rc;
    const uint32_t sweep = sweep0 + (uint32_t)k * (uint32_t)sweeps_per_step;
    pa_weights_kernel<<<dim3((unsigned)Q.nt, (unsigned)n_populations), kPaThreads, 0, st>>>(d_energy, d_dbeta + k, Q);
    pa_scan_kernel<<<n_populations, kPaScanThreads, 0, st>>>(Q, (uint32_t)seed, (uint32_t)(seed >> 32), sweep, replica0,
                                                             d_weight_sum + (size_t)n_populations * k,
                                                             d_energy_ref + (size_t)n_populations * k);
    pa_gather_kernel<<<gather_grid, 256, 0, st>>>(reinterpret_cast<const uint4*>(L.state), reinterpret_cast<uint4*>(other),
                                                 fam, fam_other, Q, d_weight_sum + (size_t)n_populations * k, rep_vecs,
                                                 group);
    e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    std::swap(L.state, other);
    std::swap(fam, fam_other);
    Lattice Lk = L;
    Lk.lut = d_luts + 32 * (size_t)k;
    rc = resident ? launch_resident_sweeps(Lk, sweep, sweeps_per_step, st) : launch_sweeps(Lk, sweep, sweeps_per_step, st);
    if (rc != TSU_OK) return rc;
  }
  const int rc = launch_population_reduce(L, Q, A, d_obs, d_count_sums + sums_per_step * n_steps, st);
  if (rc != TSU_OK) return rc;
  if (L.state != d_state) {  // an odd number of gathers: the result is in the scratch buffers
    e = cudaMemcpyAsync(d_state, L.state, sizeof(uint32_t) * 2 * (size_t)rows * L.g.wpr * n_replicas,
                        cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(d_family, fam, sizeof(int32_t) * (size_t)n_replicas, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return (int)e;
  }
  TSU_RETURN_LAUNCH_STATUS();
}

int64_t tsu_ising2d_cluster_work_bytes(int n_replicas, int rows, int cols) {
  return n_replicas > 0 ? n_replicas * cluster_rep_bytes(rows, cols) : 0;
}

int tsu_ising2d_swendsen_wang(uint32_t* d_state, int n_replicas, int rows, int cols, int wrap_rows, int wrap_cols,
                              const uint64_t* d_thresholds, const int32_t* d_lut_index, int coupling_sign,
                              const uint32_t* d_bonds, const int32_t* d_bond_index, uint64_t seed, uint32_t sweep0,
                              int n_steps, uint32_t replica0, void* d_work, size_t work_bytes, uintptr_t stream) {
  const Lattice L = {d_state, make_geom(n_replicas, rows, cols, wrap_rows, wrap_cols, 0), nullptr, d_lut_index,
                     {d_bonds, d_bond_index}, seed, replica0, JitKernel{nullptr, 0, 0}};
  TSU_CHECK_ARG(d_state && d_thresholds && d_work && n_steps >= 0 && (coupling_sign == 1 || coupling_sign == -1));
  TSU_CHECK_ARG(args_ok(L.g, L.B, false, 0, 0, rows));
  const long long rep_bytes = cluster_rep_bytes(rows, cols);
  TSU_CHECK_ARG(rep_bytes > 0 && work_bytes >= (size_t)rep_bytes);
  if (n_steps == 0) return TSU_OK;
  const long long fit = (long long)(work_bytes / (size_t)rep_bytes);
  const int chunk = fit < n_replicas ? (int)fit : n_replicas;
  ClusterParams C;
  C.thresholds = reinterpret_cast<const unsigned long long*>(d_thresholds);
  C.sign = coupling_sign;
  C.work = static_cast<char*>(d_work);
  C.rep_bytes = (size_t)rep_bytes;
  C.act_offset = (4 * (size_t)rows * cols + 15) / 16 * 16;
  C.flip_offset = C.act_offset + 16 * (size_t)rows * L.g.wpr;
  cudaStream_t st = tsu_stream(stream);
  // chunks one after the other, each through all its steps: the bits depend on no chunk size
  for (int r0 = 0; r0 < n_replicas; r0 += chunk) {
    const int rc = launch_swendsen_wang(L.replicas(r0, r0 + chunk < n_replicas ? r0 + chunk : n_replicas), C, sweep0,
                                        n_steps, st);
    if (rc != TSU_OK) return rc;
  }
  return TSU_OK;
}

int tsu_ising2d_energy_from_observables(const unsigned long long* d_obs, int n_replicas, double J, double h,
                                        int64_t n_bonds, int64_t n_sites, double* d_energy, uintptr_t stream) {
  TSU_CHECK_ARG(d_obs && d_energy && n_replicas > 0);
  energy_from_obs_kernel<<<blocks_for(n_replicas, 128), 128, 0, tsu_stream(stream)>>>(d_obs, n_replicas, J, h, n_bonds,
                                                                                    n_sites, d_energy);
  TSU_RETURN_LAUNCH_STATUS();
}


int tsu_ising2d_jit_prepare(const uint32_t* h_lut, const char* src_dir, char* log_buf, int log_len) {
  TSU_CHECK_ARG(h_lut && src_dir);
  if (log_buf && log_len > 0) log_buf[0] = 0;
  std::lock_guard<std::mutex> lock(g_jit_mutex);
  if (!tsu_jit::available()) {
    if (log_buf && log_len > 0) snprintf(log_buf, log_len, "libnvrtc.so / libcuda.so.1 not available");
    return 0;
  }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  unsigned tab[8];
  for (int k = 0; k < 8; ++k) {
    unsigned m = 0;
    for (int u = 0; u < 5; ++u) m |= ((h_lut[20 + u] >> (31 - k)) & 1u) << u;
    tab[k] = m;
  }
  unsigned fz = 0;  // classes whose threshold has zero low 24 bits and is not "always accept"
  for (int u = 0; u < 5; ++u)
    if ((h_lut[20 + u] & 0x00ffffffu) == 0u && !((h_lut[25] >> (20 + u)) & 1u)) fz |= 1u << u;
  char key[160];
  snprintf(key, sizeof key, "%d:%u,%u,%u,%u,%u,%u,%u,%u;%u;%u", dev, tab[0], tab[1], tab[2], tab[3], tab[4], tab[5], tab[6],
           tab[7], fz, (h_lut[25] >> 20) & 31u);
  auto it = g_jit_cache.find(key);
  if (it != g_jit_cache.end()) return it->second;
  std::string src;
  for (int k = 0; k < 8; ++k) src += "#define TSU_FT" + std::to_string(k) + " " + std::to_string(tab[k]) + "\n";
  src += "#define TSU_FZ " + std::to_string(fz) + "\n";
  const int jw = tuning().jit_w == 2 ? 2 : (tuning().jit_w == 4 ? 4 : kDefaultJitW);
  const int jt = (tuning().jit_threads == 32 || tuning().jit_threads == 64) ? tuning().jit_threads : kDefaultJitThreads;
  const int minb = tuning().jit_minb > 0 ? tuning().jit_minb : (jw == 2 ? 8 : kDefaultJitMinB) * (128 / jt);
  src += "#define TSU_ALWAYS " + std::to_string((h_lut[25] >> 20) & 31u) + "u\n";
  src += "#define TSU_JIT_MINB " + std::to_string(minb) + "\n";
  src += "#define TSU_JIT_W " + std::to_string(jw) + "\n";
  src += "#define TSU_JIT_THREADS " + std::to_string(jt) + "\n";
  src += "#define TSU_FAST_WARPS " + std::to_string(jt / 32) + "\n";
  if (tuning().jit_unroll > 1) src += "#define TSU_ROW_UNROLL " + std::to_string(tuning().jit_unroll) + "\n";
  src +=
      "#include \"ising2d_fast.cuh\"\n"
      "extern \"C\" __global__ void __launch_bounds__(TSU_JIT_THREADS, TSU_JIT_MINB) tsu_jit_half_sweep(tsu_fast::SweepParams P) {\n"
      "  tsu_fast::half_sweep_fast_body<TSU_JIT_W>(P);\n}\n";
  std::string log;
  void* fn = tsu_jit::compile(src, "tsu_jit.cu", "tsu_jit_half_sweep", src_dir, log);
  if (!fn) {
    if (log_buf && log_len > 0) snprintf(log_buf, log_len, "%s", log.c_str());
    g_jit_cache[key] = 0;
    return 0;
  }
  g_jit_functions.push_back(JitKernel{fn, jw, jt});
  const int handle = (int)g_jit_functions.size();
  g_jit_cache[key] = handle;
  return handle;
}

// ---- Edwards-Anderson +-J lattices: the same update with bond words XOR-ed into the neighbour words ----------
int tsu_ising2d_pack_bonds(const int8_t* d_signs, uint32_t* d_bonds, int n_real, int rows, int cols, int wrap_rows,
                           int wrap_cols, uintptr_t stream) {
  const Geom g = make_geom(n_real, rows, cols, wrap_rows, wrap_cols, 0);
  TSU_CHECK_ARG(d_signs && d_bonds && args_ok(g, kNoBonds, false, 0, 0, rows));
  const long long total = 8LL * n_real * rows * g.wpr;
  pack_bonds_kernel<<<blocks_for(total, 256), 256, 0, tsu_stream(stream)>>>(d_signs, d_bonds, n_real, g);
  TSU_RETURN_LAUNCH_STATUS();
}

int tsu_ising2d_overlap(const uint32_t* d_state, int n_replicas, int rows, int cols, const int32_t* d_pairs, int n_pairs,
                        unsigned long long* d_out, uintptr_t stream) {
  TSU_CHECK_ARG(d_state && d_pairs && d_out && geom_ok(n_replicas, rows, cols));
  TSU_CHECK_ARG(n_pairs > 0 && n_pairs <= 65535);  // gridDim.y
  cudaStream_t st = tsu_stream(stream);
  cudaError_t e = cudaMemsetAsync(d_out, 0, sizeof(unsigned long long) * (size_t)n_pairs, st);
  if (e != cudaSuccess) return (int)e;
  const long long rep_vecs = 2LL * rows * words_per_row(cols) / 4;  // wpr is a multiple of 4
  long long bx = (rep_vecs + 255) / 256;
  const long long cap = (148LL * 8 + n_pairs - 1) / n_pairs;
  if (bx > cap) bx = cap < 1 ? 1 : cap;
  overlap_kernel<<<dim3((unsigned)bx, (unsigned)n_pairs), 256, 0, st>>>(d_state, rep_vecs, d_pairs, d_out);
  TSU_RETURN_LAUNCH_STATUS();
}

}  // extern "C"
