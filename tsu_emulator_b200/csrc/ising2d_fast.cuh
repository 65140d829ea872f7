// Wide path of the bit-packed checkerboard heat-bath update (see ising2d.cu for the algorithm notes).
//
// This header is compiled twice: by nvcc as part of libtsu_b200.so (threshold truth tables read at run
// time, threshold-bit select through a brx.idx jump table) and by NVRTC at run time with the eight 5-bit
// truth tables of one temperature as compile-time constants (TSU_FT0..TSU_FT7, TSU_FZ, TSU_ALWAYS): the
// select becomes one lop3 with a literal immediate and the jump tables disappear.  Keep it free of host headers.
//
// Work split: a thread owns W consecutive words (W = 4: 128 spins, 16-byte accesses; W = 2: 64 spins, 8-byte
// accesses, half the registers and twice the resident warps) of `strip_rows` consecutive rows.
// Per row and word: 7 ALU instructions for the bit-sliced up-neighbour count, 2 Philox calls for the top 8
// bit-planes of the 32 uniforms (tsu_lattice_stream: the call-invariant half of rounds 1-3 lives in five registers),
// 3 per plane for the borrow-chain compare.
// Lanes whose top byte ties with their threshold's (2^-8 each) need the low 24 bits of their uniform, one Philox
// call per lane: a thread that has any such lane in a row parks the row's tie masks and up-counts in a per-warp
// ring in shared memory (one ballot, no per-word bookkeeping); whenever 32 rows are parked the warp makes one
// pass over them, one parked row and one tie lane per lane of the warp, ORs the accepted lanes into the stored
// words and parks the rows that have further tie lanes again.
#pragma once
#ifdef __CUDACC_RTC__
typedef unsigned int uint32_t;
typedef unsigned long long uint64_t;
typedef unsigned char uint8_t;
typedef int int32_t;
typedef unsigned long size_t;
#else
#include <stdint.h>
#include <stddef.h>
#endif
#include "philox.cuh"

#define TSU_PRAGMA_STR(x) _Pragma(#x)
#define TSU_UNROLL(n) TSU_PRAGMA_STR(unroll n)

namespace tsu_fast {

__device__ __forceinline__ uint32_t lop3_maj(uint32_t a, uint32_t b, uint32_t c) { return (a & b) | (a & c) | (b & c); }

struct Geom {
  int rows, cols, wpr;
  int wrap_rows, wrap_cols;
  int row0;
  int n_replicas;
};

__host__ __device__ __forceinline__ int colour_count(int cols, int p) { return (cols - p + 1) >> 1; }

__host__ __device__ __forceinline__ int words_per_row(int cols) {
  int ck = (cols + 1) / 2;
  int w = (ck + 31) / 32;
  return (w + 3) / 4 * 4;
}

struct Planes {
  const uint32_t* opp;       // plane of the colour NOT being updated: [rows][wpr]
  const uint32_t* halo_top;  // opposite-colour row above local row 0, or nullptr
  const uint32_t* halo_bot;  // opposite-colour row below local row rows-1, or nullptr
};

__device__ __forceinline__ const uint32_t* opp_row(const Planes& P, const Geom& g, int i) {
  if (i < 0) return P.halo_top ? P.halo_top : (g.wrap_rows ? P.opp + (size_t)(g.rows - 1) * g.wpr : nullptr);
  if (i >= g.rows) return P.halo_bot ? P.halo_bot : (g.wrap_rows ? P.opp : nullptr);
  return P.opp + (size_t)i * g.wpr;
}

// Philox coordinates of a launch: what the per-word calls share
struct Coords {
  uint32_t colour, sweep, replica, k0, k1;
};

__device__ __forceinline__ tsu_u32x4 lattice_call(const Coords& q, uint32_t w, uint32_t row_g, uint32_t kind) {
  return tsu_lattice_philox(w, q.colour, kind, row_g, q.sweep, q.replica, q.k0, q.k1);
}

struct SweepParams {
  uint32_t* state;
  const uint32_t* lut;
  const int32_t* lut_index;
  const uint32_t* halo_top;
  const uint32_t* halo_bot;
  Geom g;
  int colour;
  uint32_t sweep, replica0, k0, k1;
  tsu_philox_keys keys;  // round keys of (k0, k1): constant-bank operands of the wide path
  int strip_rows;  // rows per thread strip (wide path)
  int n_strips;    // strips per replica (wide path)
  int row_begin, row_end;  // local rows the wide path updates (rows without a north / south neighbour are left to the rim pass)
  int nvec_fast;           // 4-word groups per row the wide path updates (all their lanes exist); the rest is rim
};

// Edwards-Anderson +-J bonds (tsu_ising2d_*_bonded): uint32 words[realisation][colour][4][rows][wpr] aligned with the
// state words, direction order N, S, W, E.  Bit j of a word is 1 iff the bond between own-colour lane j and that
// neighbour is antiferromagnetic; absent neighbours and padding lanes have 0.  XOR-ing a neighbour word with its
// bond word turns the up-count into the count of bond-satisfying neighbours, which the ferromagnet's threshold
// table then serves unchanged: 4J sigma b + 2h - 2J sigma summed over the bonds = 4J u' + 2h - 2J d.
enum { kBondN = 0, kBondS = 1, kBondW = 2, kBondE = 3 };
struct BondParams {
  const uint32_t* words;  // nullptr: ferromagnet (all bonds +1)
  const int32_t* index;   // [n_replicas] realisation of each replica, or nullptr (all use realisation 0)
};

// bond words of (replica rep, colour): direction d of local row i, word w at [d * plane + i * wpr + w]
__device__ __forceinline__ const uint32_t* bond_base(const BondParams& B, const Geom& g, int rep, int colour) {
  const size_t plane = (size_t)g.rows * g.wpr;
  const size_t k = B.index ? (size_t)B.index[rep] : 0;
  return B.words + (k * 2 + (size_t)colour) * 4 * plane;
}

// lop3 with a compile-time truth table: out bit = (LUT >> (4a + 2b + c)) & 1
template <int LUT>
__device__ __forceinline__ uint32_t lop3_imm(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(d) : "r"(a), "r"(b), "r"(c), "n"(LUT));
  return d;
}

// Threshold bit of every lane for one bit-plane: tk = table[up-count], up-count = 4 c2 + 2 c1 + c0.
// The 5-entry truth table T (bit u = threshold bit of class u) is warp-uniform, so instead of four bitwise
// selects per word (ALU pipe) an indexed branch (brx.idx -> SASS BRX) picks the lop3 immediate: one LOP3 per
// word plus one jump per plane shared by the thread's words.
#define TSU_TK_CASE4(I)                                                                   \
  "L" #I ": lop3.b32 %0, %4, %8, %12, " #I "; lop3.b32 %1, %5, %9, %13, " #I ";"          \
  " lop3.b32 %2, %6, %10, %14, " #I "; lop3.b32 %3, %7, %11, %15, " #I "; bra.uni LDONE;\n"
#define TSU_TK_CASE2(I) "L" #I ": lop3.b32 %0, %2, %4, %6, " #I "; lop3.b32 %1, %3, %5, %7, " #I "; bra.uni LDONE;\n"
#define TSU_TK_TARGETS                                                                                            \
  "LTAB: .branchtargets L0, L1, L2, L3, L4, L5, L6, L7, L8, L9, L10, L11, L12, L13, L14, L15, L16, L17, "         \
  "L18, L19, L20, L21, L22, L23, L24, L25, L26, L27, L28, L29, L30, L31;\n"
#define TSU_TK_ALL(C)                                                                                             \
  C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(9) C(10) C(11) C(12) C(13) C(14) C(15) C(16) C(17) C(18) C(19)   \
  C(20) C(21) C(22) C(23) C(24) C(25) C(26) C(27) C(28) C(29) C(30) C(31)

template <int W>
__device__ __forceinline__ void tk_select(uint32_t T, const uint32_t (&c2)[W], const uint32_t (&c1)[W],
                                          const uint32_t (&c0)[W], uint32_t (&tk)[W]) {
  if constexpr (W == 4) {
    asm("{\n" TSU_TK_TARGETS "brx.idx %16, LTAB;\n" TSU_TK_ALL(TSU_TK_CASE4) "LDONE:\n}\n"
        : "=r"(tk[0]), "=r"(tk[1]), "=r"(tk[2]), "=r"(tk[3])
        : "r"(c2[0]), "r"(c2[1]), "r"(c2[2]), "r"(c2[3]), "r"(c1[0]), "r"(c1[1]), "r"(c1[2]), "r"(c1[3]),
          "r"(c0[0]), "r"(c0[1]), "r"(c0[2]), "r"(c0[3]), "r"(T & 31u));
  } else {
    asm("{\n" TSU_TK_TARGETS "brx.idx %8, LTAB;\n" TSU_TK_ALL(TSU_TK_CASE2) "LDONE:\n}\n"
        : "=r"(tk[0]), "=r"(tk[1])
        : "r"(c2[0]), "r"(c2[1]), "r"(c1[0]), "r"(c1[1]), "r"(c0[0]), "r"(c0[1]), "r"(T & 31u));
  }
}

template <int W>
__device__ __forceinline__ void ld_words(const uint32_t* __restrict__ p, uint32_t (&a)[W]) {
  if constexpr (W == 4) {
    const uint4 v = *reinterpret_cast<const uint4*>(p);
    a[0] = v.x; a[1] = v.y; a[2] = v.z; a[3] = v.w;
  } else {
    const uint2 v = *reinterpret_cast<const uint2*>(p);
    a[0] = v.x; a[1] = v.y;
  }
}

template <int W>
__device__ __forceinline__ void st_words(uint32_t* p, const uint32_t (&a)[W]) {
  if constexpr (W == 4) {
    *reinterpret_cast<uint4*>(p) = make_uint4(a[0], a[1], a[2], a[3]);
  } else {
    *reinterpret_cast<uint2*>(p) = make_uint2(a[0], a[1]);
  }
}

// ---- tie lanes ------------------------------------------------------------------------------------------
// One ring per warp: kRingSlots parked rows of (eq[W], c0[W], c1[W], c2[W], local row, first word).  The record
// stride (20 words for W = 4, 10 for W = 2) makes the vector stores of consecutive slots bank-conflict free.
constexpr int kRingSlots = 128;  // <= 63 parked rows before a pass + <= 32 parked again by it
template <int W>
struct TieRec {
  static constexpr int kWords = 4 * W + (W == 4 ? 4 : 2);
};

// low 24 bits of the uniform of lane j of word w: accepted iff below the low 24 bits of the threshold
__device__ __forceinline__ bool tie_lane_accepts(const Coords& q, const tsu_philox_keys& K, uint32_t w, uint32_t row_g,
                                                 int j, uint32_t up, const uint32_t* __restrict__ lut) {
  const tsu_u32x4 lo = tsu_philox4x32_10_keyed(TSU_LATTICE_C0(w, q.colour),
                                               TSU_LATTICE_C1(row_g, w, TSU_KIND_LOW0 + (uint32_t)(j >> 2)), q.sweep,
                                               q.replica, K);
  const int sel = j & 3;
  const uint32_t vv = sel == 0 ? lo.x : (sel == 1 ? lo.y : (sel == 2 ? lo.z : lo.w));
  return (vv >> 8) < (__ldg(lut + 20 + up) & 0x00ffffffu);
}

// One pass over the n <= 32 oldest parked rows: lane l takes row l, resolves its FIRST tie lane and, if the row has
// more, parks it again at the tail (so every pass has one Philox call of useful work per lane instead of as many
// iterations as the unluckiest row has ties).  Returns the number of rows parked again.
template <int W>
__device__ __forceinline__ uint32_t drain_pass(uint32_t* ring, uint32_t head, uint32_t count, uint32_t n, uint32_t lane,
                                               uint32_t lanes_below, uint32_t* own, const Geom& g,
                                               const uint32_t* __restrict__ lut, const Coords& q,
                                               const tsu_philox_keys& K) {
  constexpr int REC = TieRec<W>::kWords;
  const uint32_t* r = ring + ((head + lane) & (kRingSlots - 1)) * REC;
  uint32_t e[W];
  uint32_t rest = 0u;
  if (lane < n) {
    ld_words<W>(r, e);
    const uint2 tag = *reinterpret_cast<const uint2*>(r + 4 * W);  // (local row, first word)
    // first word that has a tie lane
    int k = W - 1;
    uint32_t m = e[W - 1];
#pragma unroll
    for (int kk = W - 2; kk >= 0; --kk) {
      if (e[kk]) {
        k = kk;
        m = e[kk];
      }
    }
    const int j = __ffs(m) - 1;
    const uint32_t bit = 1u << j;
    const uint32_t up = ((r[W + k] >> j) & 1u) | (((r[2 * W + k] >> j) & 1u) << 1) | (((r[3 * W + k] >> j) & 1u) << 2);
    if (tie_lane_accepts(q, K, tag.y + (uint32_t)k, (uint32_t)g.row0 + tag.x, j, up, lut))
      atomicOr(own + (size_t)tag.x * g.wpr + tag.y + k, bit);
#pragma unroll
    for (int kk = 0; kk < W; ++kk) {
      if (kk == k) e[kk] &= ~bit;
      rest |= e[kk];
    }
  }
  const uint32_t again = __ballot_sync(0xffffffffu, rest != 0u);
  if (rest != 0u) {
    uint32_t* d = ring + ((head + count + (uint32_t)__popc(again & lanes_below)) & (kRingSlots - 1)) * REC;
    st_words<W>(d, e);
#pragma unroll
    for (int f = 1; f < 4; ++f) {
      uint32_t t[W];
      ld_words<W>(r + f * W, t);
      st_words<W>(d + f * W, t);
    }
    *reinterpret_cast<uint2*>(d + 4 * W) = *reinterpret_cast<const uint2*>(r + 4 * W);
  }
  return (uint32_t)__popc(again);
}

// Periodic columns at a word boundary, every word full, a neighbour row above and below every local row in
// [row_begin, row_end) (wrap or halo).  Threads of a warp always belong to the same replica (thread index space
// padded to a multiple of 32 per replica), so the threshold tables are warp-uniform.
#ifndef TSU_FAST_WARPS
#define TSU_FAST_WARPS 4  // warps per CTA the kernel is launched with (warps never cooperate: any CTA size works)
#endif
template <int W, bool BONDED = false>
__device__ __forceinline__ void half_sweep_fast_body(const SweepParams& P, const BondParams& B = BondParams{nullptr, nullptr}) {
  constexpr int REC = TieRec<W>::kWords;
  __shared__ __align__(16) uint32_t tie_rings[TSU_FAST_WARPS][kRingSlots * REC];  // one ring per warp of the CTA
  const Geom& g = P.g;
  const int nvec = P.nvec_fast * (4 / W);  // W-word groups per row
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int per_rep = P.n_strips * nvec;
  const int per_rep_pad = (per_rep + 31) & ~31;
  const int rep = (int)(tid / per_rep_pad);
  if (rep >= g.n_replicas) return;  // whole warps only: per_rep_pad is a multiple of 32
  const int rem = (int)(tid - (long long)rep * per_rep_pad);
  const bool active = rem < per_rep;
  const int strip = active ? rem / nvec : 0;
  const int v = active ? rem - strip * nvec : 0;
  const int r_begin = P.row_begin + strip * P.strip_rows;
  const int r_end = active ? min(P.row_end, r_begin + P.strip_rows) : r_begin;
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t lanes_below = (1u << lane) - 1u;
  uint32_t* ring = tie_rings[threadIdx.x >> 5];
  uint32_t q_head = 0u, q_count = 0u;  // warp-uniform

  const size_t plane = (size_t)g.rows * g.wpr;
  uint32_t* own = P.state + ((size_t)rep * 2 + P.colour) * plane;
  Planes pl;
  pl.opp = P.state + ((size_t)rep * 2 + (1 - P.colour)) * plane;
  pl.halo_top = P.halo_top ? P.halo_top + (size_t)rep * g.wpr : nullptr;
  pl.halo_bot = P.halo_bot ? P.halo_bot + (size_t)rep * g.wpr : nullptr;
  const uint32_t* __restrict__ lut = P.lut + (P.lut_index ? (size_t)P.lut_index[rep] * 32 : 0);

#ifndef TSU_FT0
  // per-plane truth tables of the degree-4 classes (5 bits each, planes 0-5 in Tlo, 6-7 in Thi)
  uint32_t Tlo = 0u, Thi = 0u;
  {
    uint32_t t[5];
#pragma unroll
    for (int u = 0; u < 5; ++u) t[u] = __ldg(lut + 20 + u);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      uint32_t m = 0u;
#pragma unroll
      for (int u = 0; u < 5; ++u) m |= ((t[u] >> (31 - k)) & 1u) << u;
      if (k < 6)
        Tlo |= m << (5 * k);
      else
        Thi |= m << (5 * (k - 6));
    }
  }
  const uint32_t always = (__ldg(lut + 25) >> 20) & 31u;
#else
  constexpr uint32_t always = TSU_ALWAYS;
#endif

  Coords q;
  q.colour = (uint32_t)P.colour;
  q.sweep = P.sweep;
  q.replica = P.replica0 + (uint32_t)rep;
  q.k0 = P.k0;
  q.k1 = P.k1;

  const int w0 = v * W;
  const int w_prev = (w0 == 0) ? g.wpr - 1 : w0 - 1;
  const int w_next = (w0 + W == g.wpr) ? 0 : w0 + W;
  // the W words of a thread lie in one 4-word group: one stream serves all their plane calls
  const tsu_lattice_stream rng = tsu_lattice_stream_init(TSU_LATTICE_C0(w0, P.colour), q.sweep, q.replica, P.keys);

  uint32_t n[W], c[W], s[W];
#pragma unroll
  for (int k = 0; k < W; ++k) n[k] = c[k] = s[k] = 0u;
  uint32_t side_c = 0u;  // neighbour word of the centre row needed by the funnel shift
  if (active) {
    ld_words<W>(opp_row(pl, g, r_begin - 1) + w0, n);
    const uint32_t* rc0 = opp_row(pl, g, r_begin);
    ld_words<W>(rc0 + w0, c);
    side_c = rc0[((g.row0 + r_begin + P.colour) & 1) ? w_next : w_prev];
    ld_words<W>(opp_row(pl, g, r_begin + 1) + w0, s);
  }
  // bonded: the N, S, W, E bond words of the current row, and a running pointer to those of the next one
  uint32_t bd[4][W];
  const uint32_t* p_bd = nullptr;
  if constexpr (BONDED) {
#pragma unroll
    for (int d = 0; d < 4; ++d)
#pragma unroll
      for (int k = 0; k < W; ++k) bd[d][k] = 0u;
    p_bd = bond_base(B, g, rep, P.colour) + (size_t)r_begin * g.wpr + w0;
    if (active) {
#pragma unroll
      for (int d = 0; d < 4; ++d) ld_words<W>(p_bd + (size_t)d * plane, bd[d]);
    }
    p_bd += g.wpr;
  }
  // running addresses: row it + 2 of the other colour (prefetch), the row being written; the row below the last
  // local row (halo or wrap) replaces the prefetch address in the one iteration that needs it
  const size_t stride = (size_t)g.wpr;
  const uint32_t* p_s2 = pl.opp + (size_t)(r_begin + 2) * stride + w0;
  const uint32_t* p_bottom = (pl.halo_bot ? pl.halo_bot : pl.opp) + w0;
  uint32_t* p_own = own + (size_t)r_begin * stride + w0;
  const int it_bottom = g.rows - 2 - r_begin;
  const int n_rows = r_end - r_begin;
  // side word of a row relative to its word w0, one row above p_s2: previous word if the row's own columns are
  // even, next word if they are odd
  const int d_even = w_prev - w0 - g.wpr, d_odd = w_next - w0 - g.wpr;
  int p = (g.row0 + r_begin + P.colour) & 1;
  // counter word 1 of the plane calls = (global row | (w0 & 3) << 24) ^ (k << 24 | kind << 26): the row part is
  // xored into the stream once per row
  uint32_t c1_row = (uint32_t)(g.row0 + r_begin) | (((uint32_t)w0 & 3u) << 24);
#ifdef TSU_ROW_UNROLL
  TSU_UNROLL(TSU_ROW_UNROLL)
#endif
  for (int it = 0; it < P.strip_rows; ++it) {
    const bool row_valid = it < n_rows;
    // prefetch the row after next (and the side word of the next row) while this row is computed
    uint32_t s2[W];
#pragma unroll
    for (int k = 0; k < W; ++k) s2[k] = s[k];
    uint32_t side_s = 0u;
    uint32_t bd2[4][W];
    if constexpr (BONDED) {
#pragma unroll
      for (int d = 0; d < 4; ++d)
#pragma unroll
        for (int k = 0; k < W; ++k) bd2[d][k] = bd[d][k];
    }
    if (it + 1 < n_rows) {
      side_s = p_s2[p ? d_even : d_odd];  // the next row has the opposite parity
      ld_words<W>(it == it_bottom ? p_bottom : p_s2, s2);
      if constexpr (BONDED) {
#pragma unroll
        for (int d = 0; d < 4; ++d) ld_words<W>(p_bd + (size_t)d * plane, bd2[d]);
      }
    }
    uint32_t lt[W], eq[W], c0[W], c1[W], c2[W];
    uint32_t any = 0u;
    if (row_valid) {
      uint32_t sd[W];
      if (p) {  // own columns odd: the second horizontal neighbour is the next lane of the other plane
#pragma unroll
        for (int k = 0; k + 1 < W; ++k) sd[k] = __funnelshift_r(c[k], c[k + 1], 1);
        sd[W - 1] = __funnelshift_r(c[W - 1], side_c, 1);
      } else {  // own columns even: the previous lane
        sd[0] = __funnelshift_l(side_c, c[0], 1);
#pragma unroll
        for (int k = 1; k < W; ++k) sd[k] = __funnelshift_l(c[k - 1], c[k], 1);
      }
      // bit-sliced up-neighbour count of the words
#pragma unroll
      for (int k = 0; k < W; ++k) {
        if constexpr (BONDED) {  // bond-corrected neighbour bits; the centre word is the west neighbour iff p
          const uint32_t nn = n[k] ^ bd[kBondN][k], ss = s[k] ^ bd[kBondS][k];
          const uint32_t cc = c[k] ^ (p ? bd[kBondW][k] : bd[kBondE][k]);
          const uint32_t sdd = sd[k] ^ (p ? bd[kBondE][k] : bd[kBondW][k]);
          const uint32_t s1 = nn ^ ss ^ cc;
          const uint32_t m1 = lop3_maj(nn, ss, cc);
          c0[k] = s1 ^ sdd;
          const uint32_t k2 = s1 & sdd;
          c1[k] = m1 ^ k2;
          c2[k] = m1 & k2;
        } else {
          const uint32_t s1 = n[k] ^ s[k] ^ c[k];
          const uint32_t m1 = lop3_maj(n[k], s[k], c[k]);
          c0[k] = s1 ^ sd[k];
          const uint32_t k2 = s1 & sd[k];
          c1[k] = m1 ^ k2;
          c2[k] = m1 & k2;
        }
      }
      // borrow-chain compare of the top 8 bits of the uniforms against the thresholds, least significant
      // plane first; planes 4-7 (second Philox call) are consumed before planes 0-3 are generated
#pragma unroll
      for (int k = 0; k < W; ++k) {
        eq[k] = 0xffffffffu;
        lt[k] = 0u;
      }
      const uint32_t x0_row = rng.A ^ c1_row;
#pragma unroll
      for (int half = 1; half >= 0; --half) {
        uint32_t r[W][4];
#pragma unroll
        for (int k = 0; k < W; ++k) {
          const tsu_u32x4 pp = tsu_lattice_stream_call_x0(
              rng, x0_row ^ (((uint32_t)k << 24) | ((half ? TSU_KIND_PLANE1 : TSU_KIND_PLANE0) << 26)), P.keys);
          r[k][0] = pp.x; r[k][1] = pp.y; r[k][2] = pp.z; r[k][3] = pp.w;
        }
#pragma unroll
        for (int kk = 3; kk >= 0; --kk) {
          const int k = half * 4 + kk;
          uint32_t tk[W];
#ifdef TSU_FT0
          {
            constexpr int kTab[8] = {TSU_FT0, TSU_FT1, TSU_FT2, TSU_FT3, TSU_FT4, TSU_FT5, TSU_FT6, TSU_FT7};
#pragma unroll
            for (int j = 0; j < W; ++j) {
              switch (k) {  // k is a compile-time constant after unrolling
                case 0: tk[j] = lop3_imm<kTab[0]>(c2[j], c1[j], c0[j]); break;
                case 1: tk[j] = lop3_imm<kTab[1]>(c2[j], c1[j], c0[j]); break;
                case 2: tk[j] = lop3_imm<kTab[2]>(c2[j], c1[j], c0[j]); break;
                case 3: tk[j] = lop3_imm<kTab[3]>(c2[j], c1[j], c0[j]); break;
                case 4: tk[j] = lop3_imm<kTab[4]>(c2[j], c1[j], c0[j]); break;
                case 5: tk[j] = lop3_imm<kTab[5]>(c2[j], c1[j], c0[j]); break;
                case 6: tk[j] = lop3_imm<kTab[6]>(c2[j], c1[j], c0[j]); break;
                default: tk[j] = lop3_imm<kTab[7]>(c2[j], c1[j], c0[j]); break;
              }
            }
          }
#else
          tk_select<W>(k < 6 ? (Tlo >> (5 * k)) : (Thi >> (5 * (k - 6))), c2, c1, c0, tk);
#endif
#pragma unroll
          for (int j = 0; j < W; ++j) {
            const uint32_t x = r[j][kk] ^ tk[j];
            lt[j] = (~r[j][kk] & tk[j]) | (~x & lt[j]);
            eq[j] &= ~x;
          }
        }
      }
      if (always) {  // classes with p == 1.0 (threshold 2^32 does not fit 32 bits)
#pragma unroll
        for (int j = 0; j < W; ++j) {
          uint32_t am = 0u;
          if (always & 1u) am |= ~c2[j] & ~c1[j] & ~c0[j];
          if (always & 2u) am |= ~c2[j] & ~c1[j] & c0[j];
          if (always & 4u) am |= ~c2[j] & c1[j] & ~c0[j];
          if (always & 8u) am |= ~c2[j] & c1[j] & c0[j];
          if (always & 16u) am |= c2[j];
          lt[j] |= am;
          eq[j] &= ~am;
        }
      }
#ifdef TSU_FZ
      // classes whose threshold has zero low 24 bits (e.g. p = 1/2 exactly): a tie can never be accepted by the
      // low bits, so those lanes need no second draw
      if (TSU_FZ != 0) {
#pragma unroll
        for (int j = 0; j < W; ++j) eq[j] &= ~lop3_imm<TSU_FZ>(c2[j], c1[j], c0[j]);
      }
#endif
      // the row without its tie lanes; they are ORed in when the parked row is resolved
      st_words<W>(p_own, lt);
      any = eq[0];
#pragma unroll
      for (int k = 1; k < W; ++k) any |= eq[k];
    }
    // ---- park the row if it has tie lanes ----
    const uint32_t parked = __ballot_sync(0xffffffffu, any != 0u);
    if (any != 0u) {
      uint32_t* r = ring + ((q_head + q_count + (uint32_t)__popc(parked & lanes_below)) & (kRingSlots - 1)) * REC;
      st_words<W>(r, eq);
      st_words<W>(r + W, c0);
      st_words<W>(r + 2 * W, c1);
      st_words<W>(r + 3 * W, c2);
      *reinterpret_cast<uint2*>(r + 4 * W) = make_uint2((uint32_t)(r_begin + it), (uint32_t)w0);
    }
    q_count += (uint32_t)__popc(parked);
    if (q_count >= 32u) {
      __syncwarp();  // parked rows and the stored words are visible to the warp
      q_count += drain_pass<W>(ring, q_head, q_count, 32u, lane, lanes_below, own, g, lut, q, P.keys) - 32u;
      q_head = (q_head + 32u) & (kRingSlots - 1);
    }
#pragma unroll
    for (int k = 0; k < W; ++k) {
      n[k] = c[k];
      c[k] = s[k];
      s[k] = s2[k];
    }
    side_c = side_s;
    if constexpr (BONDED) {
#pragma unroll
      for (int d = 0; d < 4; ++d)
#pragma unroll
        for (int k = 0; k < W; ++k) bd[d][k] = bd2[d][k];
      p_bd += stride;
    }
    p_s2 += stride;
    p_own += stride;
    p ^= 1;
    c1_row += 1u;
  }
  while (q_count) {  // what is still parked at the end of the strip
    __syncwarp();
    const uint32_t n = q_count < 32u ? q_count : 32u;
    q_count += drain_pass<W>(ring, q_head, q_count, n, lane, lanes_below, own, g, lut, q, P.keys) - n;
    q_head = (q_head + n) & (kRingSlots - 1);
  }
}

}  // namespace tsu_fast
