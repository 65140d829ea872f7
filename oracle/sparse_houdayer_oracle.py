"""
ORACLE (test infrastructure, not product code): the Houdayer cluster move on sparse couplings of tsu_sparse_houdayer
(csrc/sparse_houdayer.cu) restated in NumPy and SciPy.

One step at index s of the pair (a, b) of chains (states in {0, 1}, couplings in CSR with ascending columns):
  1. differ     d_i = x^a_i xor x^b_i
  2. graph      edge {i, j} for every stored entry J_ij != 0 of row i with j > i (self couplings never join)
  3. clusters   connected components of the graph restricted to the sites with d = 1; a cluster's root is its smallest
                site index
  4. flip       a cluster flips in both chains iff bit 0 of word 0 of Philox(counter = (root, chain0 + a, s, 'HOUD'),
                key = seed) is 1; sites with d = 0 never change
"""

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from .philox_ref import philox4x32_10

STREAM_HOUDAYER = 0x484F5544  # 'HOUD'


def cluster_roots(rowptr, col, d, val=None) -> np.ndarray:
    """int64[N]: root (smallest site index of its cluster) of every site for the difference pattern d [N] in {0, 1};
    a site with d = 0 is its own root.  val: the CSR values (entries equal to 0 make no edge), or None"""
    rowptr, col = np.asarray(rowptr, dtype=np.int64), np.asarray(col, dtype=np.int64)
    d = np.asarray(d).astype(bool)
    N = d.size
    row = np.repeat(np.arange(N), np.diff(rowptr))
    keep = (col > row) & d[row] & d[col]
    if val is not None:
        keep &= np.asarray(val) != 0
    graph = coo_matrix((np.ones(int(keep.sum()), dtype=np.int8), (row[keep], col[keep])), shape=(N, N))
    n, label = connected_components(graph, directed=False)
    low = np.full(n, N, dtype=np.int64)
    np.minimum.at(low, label, np.arange(N))
    return low[label]


def flip_bits(seed: int, chain: int, step: int, N: int) -> np.ndarray:
    """int64[N]: the flip bit a cluster rooted at each site draws"""
    o = philox4x32_10(np.arange(N), chain & 0xFFFFFFFF, step & 0xFFFFFFFF, STREAM_HOUDAYER, seed & 0xFFFFFFFF,
                      (seed >> 32) & 0xFFFFFFFF)
    return (o[0] & 1).astype(np.int64)


def pair_step(xa, xb, csr, seed: int, chain: int, step: int):
    """one step of the pair (xa, xb) [N] in {0, 1}; csr = (rowptr, col, val); `chain` = chain0 + a.  Returns the new
    (xa, xb)."""
    xa, xb = np.asarray(xa, dtype=np.int64), np.asarray(xb, dtype=np.int64)
    rowptr, col, val = csr
    d = xa ^ xb
    root = cluster_roots(rowptr, col, d, val)
    m = d & flip_bits(seed, chain, step, d.size)[root]
    return xa ^ m, xb ^ m


def houdayer_steps(states, pairs, csr, seed: int, chain0: int, step0: int, n_steps: int):
    """n_steps steps of every pair (a, b) of `pairs` (disjoint) of states [n_chains, N] in {0, 1}; pairs with an index
    outside [0, n_chains) or a == b are skipped"""
    x = np.array(states, dtype=np.int64, copy=True)
    n = x.shape[0]
    for k in range(n_steps):
        for a, b in np.asarray(pairs).reshape(-1, 2):
            a, b = int(a), int(b)
            if a < 0 or b < 0 or a >= n or b >= n or a == b:
                continue
            x[a], x[b] = pair_step(x[a], x[b], csr, seed, chain0 + a, step0 + k)
    return x


def energy(state, csr, bias=None) -> float:
    """E = -1/2 s^T J s - b^T s of one state [N] in {0, 1} under CSR couplings"""
    rowptr, col, val = csr
    s = np.asarray(state, dtype=np.float64)
    row = np.repeat(np.arange(s.size), np.diff(rowptr))
    e = -0.5 * float(np.sum(np.asarray(val) * s[row] * s[np.asarray(col)]))
    if bias is not None:
        e -= float(np.dot(bias, s))
    return e
