"""
ORACLE (test infrastructure, not product code): the Houdayer cluster move of tsu_ising2d_houdayer (csrc/ising2d.cu)
restated in NumPy and SciPy.

One step at sweep index s of the pair (a, b) of replicas (states in {0, 1}):
  1. differ     d_i = x^a_i xor x^b_i
  2. active     a bond the wiring creates (cluster_oracle.bonds: right and down of every site, wraps of periodic
                dimensions longer than 2) is active iff d = 1 at both its ends; no randomness, temperature or sign
  3. clusters   connected components of the active bonds over the sites with d = 1; a cluster's root is its smallest
                site index row * cols + col
  4. flip       a cluster flips in both replicas iff the root's bit of the kind-5 call (w, colour, 5, row, s,
                replica0 + a) is 1 (the init_bits construction with kind 5 and sweep s); sites with d = 0 never change
"""

import numpy as np

from . import cluster_oracle as SW
from . import ising2d_oracle as O
from .philox_ref import philox4x32_10

KIND_FLIP = 5


def flip_bits(seed: int, replica: int, sweep: int, rows: int, cols: int) -> np.ndarray:
    """int64[rows, cols]: bit b of output word 0 of the kind-5 call of every site's word"""
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    bits = np.zeros((rows, cols), dtype=np.int64)
    for colour in range(2):
        i, j, mask, w, b = O._site_words(rows, cols, colour)
        i_b, w_b, b_b = np.broadcast_arrays(i, w, b)
        c0, c1 = O.lattice_counter(w_b, colour, KIND_FLIP, i_b)
        o = philox4x32_10(c0, c1, sweep & 0xFFFFFFFF, replica, k0, k1)
        bits = np.where(mask, ((o[0].astype(np.uint64) >> b_b.astype(np.uint64)) & np.uint64(1)).astype(np.int64), bits)
    return bits


def cluster_roots(d, periodic: bool) -> np.ndarray:
    """int64[rows * cols]: root of every site (row-major) for the difference pattern d [rows, cols] in {0, 1}; a site
    with d = 0 is its own root"""
    d = np.asarray(d)
    rows, cols = d.shape
    a, b, _, _ = SW.bonds(rows, cols, periodic)
    flat = d.reshape(-1).astype(bool)
    return SW.roots(rows * cols, a, b, flat[a] & flat[b])


def pair_step(xa, xb, periodic: bool, seed: int, replica: int, sweep: int):
    """one step of the pair (xa, xb) [rows, cols] in {0, 1}; `replica` = replica0 + a.  Returns the new (xa, xb)."""
    xa, xb = np.asarray(xa), np.asarray(xb)
    rows, cols = xa.shape
    d = xa ^ xb
    root = cluster_roots(d, periodic)
    m = (d.reshape(-1) & flip_bits(seed, replica, sweep, rows, cols).reshape(-1)[root].astype(d.dtype)).reshape(rows, cols)
    return xa ^ m, xb ^ m


def houdayer_steps(states, pairs, periodic: bool, seed: int, replica0: int, sweep0: int, n_steps: int):
    """n_steps steps of every pair (a, b) of `pairs` (disjoint) of states [n, rows, cols] in {0, 1}"""
    x = np.array(states, dtype=np.int64, copy=True)
    for k in range(n_steps):
        for a, b in np.asarray(pairs).reshape(-1, 2):
            x[a], x[b] = pair_step(x[a], x[b], periodic, seed, replica0 + int(a), sweep0 + k)
    return x
