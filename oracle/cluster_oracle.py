"""
ORACLE (test infrastructure, not product code): the Swendsen-Wang step of tsu_ising2d_swendsen_wang
(csrc/ising2d.cu) restated in NumPy and SciPy.

One step at sweep index s of replica r (coupling J, temperature T_r, bond signs sigma, +1 without bonds):
  1. satisfied  every bond the wiring creates (ising2d_bonds_oracle.bond_list: right and down of every site, wraps of
                periodic dimensions longer than 2) with J sigma_ij s_i s_j > 0
  2. active     a satisfied bond is active iff u < t, t = ceil(p 2^32), p = -expm1(-2|J| / T) (t = 2^32: always);
                u is the 32-bit uniform of the site the bond starts from, built as the Gibbs uniform
                (ising2d_oracle.lattice_uniforms_u32) from kinds 16, 17 / 24-31 (east) or 18, 19 / 32-39 (south)
  3. clusters   connected components of the active bonds; a cluster's root is its smallest site index row * cols + col
  4. flip       a cluster flips iff the root's bit of the kind-4 call (w, colour, 4, row, s, replica) is 1 (the
                init_bits construction with kind 4 and sweep s)
"""

import math

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from . import ising2d_bonds_oracle as B
from . import ising2d_oracle as O
from .philox_ref import philox4x32_10

KIND_FLIP = 4
KIND_EAST_PLANE0, KIND_EAST_LOW0 = 16, 24
KIND_SOUTH_PLANE0, KIND_SOUTH_LOW0 = 18, 32


def threshold(J: float, T: float) -> int:
    """t = ceil(p 2^32) with p = -expm1(-2|J| / T) in float64"""
    return int(math.ceil(-math.expm1(-2.0 * abs(J) / T) * 4294967296.0))


def bond_uniforms_u32(seed: int, replica: int, sweep: int, rows: int, cols: int, plane0: int, low0: int) -> np.ndarray:
    """u32[rows, cols]: the uniform of the bond that starts at every site (bit-plane kinds plane0, plane0 + 1, low-bit
    kinds low0 + (b >> 2)), for both colours"""
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    out = np.zeros((rows, cols), dtype=np.uint64)
    for colour in range(2):
        i, j, mask, w, b = O._site_words(rows, cols, colour)
        i_b, w_b, b_b = np.broadcast_arrays(i, w, b)
        b64 = b_b.astype(np.uint64)
        u = np.zeros((rows, cols), dtype=np.uint64)
        for call in range(2):
            c0, c1 = O.lattice_counter(w_b, colour, plane0 + call, i_b)
            o = philox4x32_10(c0, c1, sweep & 0xFFFFFFFF, replica, k0, k1)
            for q in range(4):
                u |= ((o[q].astype(np.uint64) >> b64) & np.uint64(1)) << np.uint64(31 - (call * 4 + q))
        c0, c1 = O.lattice_counter(w_b, colour, np.uint64(low0) + (b64 >> np.uint64(2)), i_b)
        o = philox4x32_10(c0, c1, sweep & 0xFFFFFFFF, replica, k0, k1)
        u |= np.choose(b_b & 3, [x.astype(np.uint64) for x in o]) >> np.uint64(8)
        out = np.where(mask, u, out)
    return out.astype(np.uint32)


def flip_bits(seed: int, replica: int, sweep: int, rows: int, cols: int) -> np.ndarray:
    """int64[rows, cols]: bit b of output word 0 of the kind-4 call of every site's word"""
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    bits = np.zeros((rows, cols), dtype=np.int64)
    for colour in range(2):
        i, j, mask, w, b = O._site_words(rows, cols, colour)
        i_b, w_b, b_b = np.broadcast_arrays(i, w, b)
        c0, c1 = O.lattice_counter(w_b, colour, KIND_FLIP, i_b)
        o = philox4x32_10(c0, c1, sweep & 0xFFFFFFFF, replica, k0, k1)
        bits = np.where(mask, ((o[0].astype(np.uint64) >> b_b.astype(np.uint64)) & np.uint64(1)).astype(np.int64), bits)
    return bits


def bonds(rows: int, cols: int, periodic: bool, signs=None):
    """(a, b, sigma, east): every bond the wiring creates; a is the site it starts from, east marks right bonds"""
    s = np.ones((2, rows, cols), dtype=np.int64) if signs is None else np.asarray(signs)
    a, b, g = B.bond_list(rows, cols, periodic, s)
    n_east = int(((np.arange(cols) < cols - 1) | (periodic and cols > 2)).sum()) * rows
    east = np.arange(a.size) < n_east
    return a, b, g, east


def satisfied(bits, J: float, periodic: bool, signs=None):
    """bool per bond of bonds(): J sigma_ij s_i s_j > 0"""
    bits = np.asarray(bits)
    a, b, g, _ = bonds(*bits.shape, periodic, signs)
    s = 2 * bits.reshape(-1).astype(np.int64) - 1
    return J * g * s[a] * s[b] > 0


def roots(n_sites: int, a, b, active) -> np.ndarray:
    """root (smallest site index of its cluster) of every site, for the active bonds (a, b); several replicas are one
    block-diagonal graph of n_sites nodes"""
    a, b = np.asarray(a)[active], np.asarray(b)[active]
    graph = coo_matrix((np.ones(a.size, dtype=np.int8), (a, b)), shape=(n_sites, n_sites))
    n, label = connected_components(graph, directed=False)
    low = np.full(n, n_sites, dtype=np.int64)
    np.minimum.at(low, label, np.arange(n_sites))
    return low[label]


def active_bonds(bits, J: float, T: float, periodic: bool, seed: int, replica: int, sweep: int, signs=None):
    """(a, b, active) of one replica at one step"""
    bits = np.asarray(bits)
    R, C = bits.shape
    a, b, g, east = bonds(R, C, periodic, signs)
    ue = bond_uniforms_u32(seed, replica, sweep, R, C, KIND_EAST_PLANE0, KIND_EAST_LOW0).reshape(-1)
    us = bond_uniforms_u32(seed, replica, sweep, R, C, KIND_SOUTH_PLANE0, KIND_SOUTH_LOW0).reshape(-1)
    u = np.where(east, ue[a], us[a]).astype(np.int64)
    return a, b, satisfied(bits, J, periodic, signs) & (u < threshold(J, T))


def sw_steps(states, J: float, temps, periodic: bool, seed: int, replica0: int, sweep0: int, n_steps: int,
             signs=None):
    """n_steps Swendsen-Wang steps of every replica: states [n, rows, cols] in {0, 1}; temps and signs per replica
    (signs: None, one (2, rows, cols) realisation or a list of them)"""
    x = np.array(states, dtype=np.int64, copy=True)
    n, R, C = x.shape
    N = R * C
    temps = np.broadcast_to(np.asarray(temps, dtype=np.float64), (n,))
    sg = signs if isinstance(signs, list) else [signs] * n
    for k in range(n_steps):
        s = sweep0 + k
        aa, bb, act, flips = [], [], [], []
        for r in range(n):
            a, b, on = active_bonds(x[r], J, float(temps[r]), periodic, seed, replica0 + r, s, sg[r])
            aa.append(a + r * N)
            bb.append(b + r * N)
            act.append(on)
            flips.append(flip_bits(seed, replica0 + r, s, R, C).reshape(-1))
        root = roots(n * N, np.concatenate(aa), np.concatenate(bb), np.concatenate(act))
        x ^= np.concatenate(flips)[root].reshape(n, R, C)
    return x
