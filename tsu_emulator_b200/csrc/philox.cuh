// Counter-based Philox4x32-10 (Salmon et al., SC'11), device + host.
//
// Replaces the reference's global NumPy MT19937 stream (tsu/gibbs.py:126,157,201,270,320,368;
// tsu/core.py:78,143).  Every random number in this library is a pure function of
// (seed, stream coordinates), so results do not depend on launch geometry or on how a
// lattice is split across GPUs.
//
// One call = 10 rounds of { 2 x IMAD.WIDE.U32, 2 x LOP3 } : 20 fma-pipe + 20 alu-pipe
// instructions for 128 random bits, all in registers.
#pragma once
#ifndef __CUDACC_RTC__
#include <stdint.h>
#endif

#define TSU_PHILOX_M0 0xD2511F53u
#define TSU_PHILOX_M1 0xCD9E8D57u
#define TSU_PHILOX_W0 0x9E3779B9u
#define TSU_PHILOX_W1 0xBB67AE85u

struct tsu_u32x4 {
  uint32_t x, y, z, w;
};

__host__ __device__ __forceinline__ void tsu_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#ifdef __CUDA_ARCH__
  // one IMAD.WIDE.U32 (left to itself the compiler sometimes emits IMAD.HI + IMAD: two issue slots)
  uint64_t p;
  asm("mul.wide.u32 %0, %1, %2;" : "=l"(p) : "r"(a), "r"(b));
  lo = (uint32_t)p;
  hi = (uint32_t)(p >> 32);
#else
  uint64_t p = (uint64_t)a * (uint64_t)b;
  lo = (uint32_t)p;
  hi = (uint32_t)(p >> 32);
#endif
}

__host__ __device__ __forceinline__ tsu_u32x4 tsu_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                               uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    tsu_mulhilo(TSU_PHILOX_M0, c0, hi0, lo0);
    tsu_mulhilo(TSU_PHILOX_M1, c2, hi1, lo1);
    uint32_t n0 = hi1 ^ c1 ^ k0;
    uint32_t n2 = hi0 ^ c3 ^ k1;
    c0 = n0;
    c1 = lo1;
    c2 = n2;
    c3 = lo0;
    k0 += TSU_PHILOX_W0;
    k1 += TSU_PHILOX_W1;
  }
  tsu_u32x4 o;
  o.x = c0;
  o.y = c1;
  o.z = c2;
  o.w = c3;
  return o;
}

// The ten round keys of a seed, computed once on the host and handed to kernels inside their parameter struct:
// a round then reads its keys as constant-bank operands of the xors instead of adding the Weyl constants per call.
struct tsu_philox_keys {
  uint32_t k0[10], k1[10];
};

__host__ __device__ __forceinline__ tsu_philox_keys tsu_philox_key_schedule(uint32_t k0, uint32_t k1) {
  tsu_philox_keys K;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    K.k0[r] = k0 + (uint32_t)r * TSU_PHILOX_W0;
    K.k1[r] = k1 + (uint32_t)r * TSU_PHILOX_W1;
  }
  return K;
}

__host__ __device__ __forceinline__ tsu_u32x4 tsu_philox4x32_10_keyed(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                                     const tsu_philox_keys& K) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    tsu_mulhilo(TSU_PHILOX_M0, c0, hi0, lo0);
    tsu_mulhilo(TSU_PHILOX_M1, c2, hi1, lo1);
    const uint32_t n0 = hi1 ^ c1 ^ K.k0[r];
    const uint32_t n2 = hi0 ^ c3 ^ K.k1[r];
    c0 = n0;
    c1 = lo1;
    c2 = n2;
    c3 = lo0;
  }
  tsu_u32x4 o;
  o.x = c0;
  o.y = c1;
  o.z = c2;
  o.w = c3;
  return o;
}

// ---- stream coordinates ---------------------------------------------------------------
// Lattice stream (ising2d.cu):
//   counter = ( (w >> 2) | colour << 24,  global_row | (w & 3) << 24 | kind << 26,  sweep,  replica ),  key = seed
//   kind 0,1  : bit-plane calls (planes 0-3 / 4-7 = top 8 bits of every lane's uniform)
//   kind 2    : initial configuration
//   kind 3    : population annealing, one call per population and step (w = colour = row = 0, replica = the
//               population's first replica, sweep = the step's first sweep; words x | y << 32 are the 64-bit draw)
//   kind 4    : Swendsen-Wang cluster flips: bit b of word x of the call of the cluster root's word (as kind 2)
//   kind 8-15 : low 24 bits, one call per group of 4 lanes (lane b uses word b&3 of call 8+(b>>2))
//   kind 16,17 / 24-31 : Swendsen-Wang east-bond uniforms (bit-planes / low 24 bits, as kinds 0,1 / 8-15)
//   kind 18,19 / 32-39 : Swendsen-Wang south-bond uniforms (bit-planes / low 24 bits, as kinds 0,1 / 8-15)
// Everything that changes between the calls a thread makes while it walks down its rows (row, word within
// the 4-word group, kind) sits in counter word 1; words 0, 2, 3 are fixed per thread.  Philox round 1 then
// multiplies only fixed values, and half of rounds 2 and 3 is fixed as well: tsu_lattice_stream keeps those
// parts in five registers and a call costs 16 wide multiplies + 18 xors instead of 20 + 20.  Same function,
// same bits as tsu_philox4x32_10 on the full counter (tests/test_philox.py).
#define TSU_KIND_PLANE0 0u
#define TSU_KIND_PLANE1 1u
#define TSU_KIND_INIT 2u
#define TSU_KIND_RESAMPLE 3u
#define TSU_KIND_LOW0 8u
#define TSU_KIND_CLUSTER_FLIP 4u
#define TSU_KIND_BOND_E_PLANE0 16u
#define TSU_KIND_BOND_S_PLANE0 18u
#define TSU_KIND_BOND_E_LOW0 24u
#define TSU_KIND_BOND_S_LOW0 32u
#define TSU_LATTICE_MAX_ROWS (1 << 24)
#define TSU_LATTICE_C0(w, colour) (((uint32_t)(w) >> 2) | ((uint32_t)(colour) << 24))
#define TSU_LATTICE_C1(row, w, kind) ((uint32_t)(row) | (((uint32_t)(w) & 3u) << 24) | ((uint32_t)(kind) << 26))

__host__ __device__ __forceinline__ tsu_u32x4 tsu_lattice_philox(uint32_t w, uint32_t colour, uint32_t kind,
                                                                uint32_t row_g, uint32_t sweep, uint32_t replica,
                                                                uint32_t k0, uint32_t k1) {
  return tsu_philox4x32_10(TSU_LATTICE_C0(w, colour), TSU_LATTICE_C1(row_g, w, kind), sweep, replica, k0, k1);
}

struct tsu_lattice_stream {
  uint32_t A;   // hi(M1 * sweep) ^ key0[0]: counter word 0 after round 1 is A ^ c1
  uint32_t D1;  // lo(M0 * c0) ^ key1[1]
  uint32_t F2;  // lo(M1 * C) ^ key0[2],  C = hi(M0 * c0) ^ replica ^ key1[0]
  uint32_t G;   // hi(M0 * E) ^ key1[2],  E = hi(M1 * C) ^ lo(M1 * sweep) ^ key0[1]
  uint32_t H;   // lo(M0 * E)
};

__host__ __device__ __forceinline__ tsu_lattice_stream tsu_lattice_stream_init(uint32_t c0, uint32_t sweep,
                                                                              uint32_t replica,
                                                                              const tsu_philox_keys& K) {
  tsu_lattice_stream s;
  uint32_t hi0, lo0, hi1, lo1;
  tsu_mulhilo(TSU_PHILOX_M1, sweep, hi1, lo1);
  tsu_mulhilo(TSU_PHILOX_M0, c0, hi0, lo0);
  s.A = hi1 ^ K.k0[0];
  const uint32_t B = lo1, C = hi0 ^ replica ^ K.k1[0], D = lo0;
  tsu_mulhilo(TSU_PHILOX_M1, C, hi1, lo1);
  const uint32_t E = hi1 ^ B ^ K.k0[1], F = lo1;
  s.D1 = D ^ K.k1[1];
  tsu_mulhilo(TSU_PHILOX_M0, E, hi0, lo0);
  s.F2 = F ^ K.k0[2];
  s.G = hi0 ^ K.k1[2];
  s.H = lo0;
  return s;
}

// x0 = s.A ^ c1 (counter word 0 after round 1); callers that make many calls per row xor the row part once
__host__ __device__ __forceinline__ tsu_u32x4 tsu_lattice_stream_call_x0(const tsu_lattice_stream& s, uint32_t x0,
                                                                        const tsu_philox_keys& K);

__host__ __device__ __forceinline__ tsu_u32x4 tsu_lattice_stream_call(const tsu_lattice_stream& s, uint32_t c1,
                                                                     const tsu_philox_keys& K) {
  return tsu_lattice_stream_call_x0(s, s.A ^ c1, K);
}

__host__ __device__ __forceinline__ tsu_u32x4 tsu_lattice_stream_call_x0(const tsu_lattice_stream& s, uint32_t x0,
                                                                        const tsu_philox_keys& K) {
  uint32_t hi, lo;
  tsu_mulhilo(TSU_PHILOX_M0, x0, hi, lo);  // round 2, the half that depends on c1
  const uint32_t y2 = hi ^ s.D1, y3 = lo;
  tsu_mulhilo(TSU_PHILOX_M1, y2, hi, lo);        // round 3
  uint32_t c0 = hi ^ s.F2, c1n = lo, c2 = s.G ^ y3, c3 = s.H;
#pragma unroll
  for (int r = 3; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    tsu_mulhilo(TSU_PHILOX_M0, c0, hi0, lo0);
    tsu_mulhilo(TSU_PHILOX_M1, c2, hi1, lo1);
    const uint32_t n0 = hi1 ^ c1n ^ K.k0[r];
    const uint32_t n2 = hi0 ^ c3 ^ K.k1[r];
    c0 = n0;
    c1n = lo1;
    c2 = n2;
    c3 = lo0;
  }
  tsu_u32x4 o;
  o.x = c0;
  o.y = c1n;
  o.z = c2;
  o.w = c3;
  return o;
}

// Generic streams (dense Gibbs / Langevin / fill): counter = (index_lo, index_hi, step, stream_tag)
#define TSU_STREAM_FILL 0x46494C4Cu      // 'FILL'
#define TSU_STREAM_DENSE 0x44454E53u     // 'DENS'
#define TSU_STREAM_DENSE_TC 0x44454E54u  // 'DENT': tensor-core dense path, counter = (site>>2, chain, sweep, tag)
#define TSU_STREAM_DENSE_INIT 0x44494E49u  // 'DINI'
#define TSU_STREAM_LANGEVIN 0x4C414E47u  // 'LANG'
#define TSU_STREAM_LANGEVIN_INIT 0x4C494E49u  // 'LINI'
#define TSU_STREAM_PT_SWAP 0x50545357u   // 'PTSW'
