"""CPU: the Houdayer oracle (oracle/houdayer_oracle.py) is a valid Markov chain step for a pair of replicas.  Its exact
transition matrix over all pair states of small lattices, built from the oracle's own cluster decomposition by
enumerating every subset of clusters, is stochastic and symmetric, keeps E_a + E_b on every nonzero entry and leaves
the product of the two Boltzmann distributions invariant, with and without a field; the oracle's step lands on the
support of that matrix; and pairs that agree everywhere are untouched."""
import numpy as np
import pytest
from scipy.sparse import coo_matrix

from oracle import cluster_oracle as SW
from oracle import houdayer_oracle as H


def energies(rows, cols, J, h, periodic, signs):
    """E = -J sum_bonds sigma s_i s_j - h sum_i s_i of every state (index sum_i bit_i 2^i over row-major sites)"""
    N = rows * cols
    s = 2 * ((np.arange(1 << N)[:, None] >> np.arange(N)) & 1) - 1
    a, b, g, _ = SW.bonds(rows, cols, periodic, signs)
    return -J * (g[None, :] * s[:, a] * s[:, b]).sum(axis=1) - h * s.sum(axis=1)


def transition_matrix(rows, cols, periodic):
    """sparse P[(a, b), (a', b')] of one move, pair states indexed a * 2^N + b: for each difference pattern d, every
    subset of its clusters flips in both replicas with probability 2^-n_clusters"""
    N = rows * cols
    weights = 1 << np.arange(N)
    xa = np.arange(1 << N)
    src, dst, val = [], [], []
    for d in range(1 << N):
        bits = (d >> np.arange(N)) & 1
        root = H.cluster_roots(bits.reshape(rows, cols), periodic)
        clusters = np.unique(root[bits == 1])
        member = (root[None, :] == clusters[:, None]).astype(np.int64)  # [n_clusters, N]
        patterns = ((np.arange(1 << clusters.size)[:, None] >> np.arange(clusters.size)) & 1) @ member @ weights
        xb = xa ^ d
        for f in patterns:
            src.append(xa * (1 << N) + xb)
            dst.append((xa ^ f) * (1 << N) + (xb ^ f))
            val.append(np.full(xa.size, 1.0 / (1 << clusters.size)))
    n = 1 << (2 * N)
    return coo_matrix((np.concatenate(val), (np.concatenate(src), np.concatenate(dst))), shape=(n, n)).tocsr()


CASES = [(2, 3, False), (2, 4, True)]  # open; wrapped columns (a periodic length-2 dimension has no wrap)
MODELS = [("ferro", 0.0), ("ferro", 0.3), ("signs", 0.0), ("signs", 0.3)]


@pytest.mark.parametrize("rows,cols,periodic", CASES)
def test_exact_transition_matrix(rows, cols, periodic):
    P = transition_matrix(rows, cols, periodic)
    assert np.abs(np.asarray(P.sum(axis=1)).ravel() - 1.0).max() < 1e-12
    assert abs(P - P.T).max() < 1e-15
    coo = P.tocoo()
    for model, h in MODELS:
        signs = np.random.default_rng(7).choice(np.array([-1, 1]), size=(2, rows, cols)) if model == "signs" else None
        T = 1.3
        E = energies(rows, cols, 1.0, h, periodic, signs)
        pair_E = (E[:, None] + E[None, :]).reshape(-1)
        assert np.abs(pair_E[coo.row] - pair_E[coo.col]).max() < 1e-12, (model, h)
        pi = np.exp(-(E - E.min()) / T)
        pi /= pi.sum()
        pi2 = np.outer(pi, pi).reshape(-1)
        assert np.abs(P.T @ pi2 - pi2).max() < 1e-12, (model, h)


@pytest.mark.parametrize("rows,cols,periodic", CASES)
def test_oracle_step_lies_on_the_support(rows, cols, periodic):
    P = transition_matrix(rows, cols, periodic)
    N = rows * cols
    weights = 1 << np.arange(N)
    rng = np.random.default_rng(11)
    for k in range(200):
        x = rng.integers(0, 2, (2, rows, cols))
        ya, yb = H.pair_step(x[0], x[1], periodic, 5, 3, k)
        src = int(x[0].reshape(-1) @ weights) * (1 << N) + int(x[1].reshape(-1) @ weights)
        dst = int(ya.reshape(-1) @ weights) * (1 << N) + int(yb.reshape(-1) @ weights)
        assert P[src, dst] > 0


def test_pairs_that_agree_are_untouched():
    rng = np.random.default_rng(5)
    x = rng.integers(0, 2, (3, 20, 30))
    states = np.stack([x[0], x[0], x[1], x[1], x[2], x[2]])
    out = H.houdayer_steps(states, [(0, 1), (3, 2), (4, 5)], True, 9, 0, 0, 3)
    assert (out == states).all()


def test_clusters_flip_whole_in_both_replicas():
    rng = np.random.default_rng(6)
    rows, cols = 24, 40
    xa, xb = rng.integers(0, 2, (2, rows, cols))
    ya, yb = H.pair_step(xa, xb, True, 9, 4, 2)
    d = xa ^ xb
    assert ((ya ^ yb) == d).all()                          # the difference pattern is kept
    assert ((ya ^ xa) == (yb ^ xb)).all() and not ((ya ^ xa) & ~d.astype(bool)).any()
    root = H.cluster_roots(d, True)
    flipped = (ya ^ xa).reshape(-1)
    for r in np.unique(root[d.reshape(-1) == 1]):
        f = flipped[root == r]
        assert (f == f[0]).all()
        assert f[0] == H.flip_bits(9, 4, 2, rows, cols).reshape(-1)[r]
