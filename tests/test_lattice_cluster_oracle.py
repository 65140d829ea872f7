"""CPU: the Swendsen-Wang oracle (oracle/cluster_oracle.py) is a valid Markov chain step.  Its exact transition matrix
on small lattices, built by enumerating every subset of the satisfied bonds with the oracle's own bond and component
functions, is stochastic and leaves the Boltzmann distribution invariant; at p = 1 its clusters are the aligned
domains; and bonds are activated with probability p."""
import itertools

import numpy as np
import pytest
from scipy import ndimage

from oracle import cluster_oracle as SW


def transition_matrix(rows, cols, J, T, periodic, signs):
    """P[x, y] of one SW step, states indexed by sum_i bit_i 2^i over the row-major sites"""
    N = rows * cols
    n_states = 1 << N
    a, b, _, _ = SW.bonds(rows, cols, periodic, signs)
    p = -np.expm1(-2.0 * abs(J) / T)
    P = np.zeros((n_states, n_states))
    weights = 1 << np.arange(N)
    for x in range(n_states):
        bits = (x >> np.arange(N)) & 1
        sat = np.flatnonzero(SW.satisfied(bits.reshape(rows, cols), J, periodic, signs))
        for k in range(sat.size + 1):
            for chosen in itertools.combinations(sat, k):
                active = np.zeros(a.size, dtype=bool)
                active[list(chosen)] = True
                prob = p ** k * (1 - p) ** (sat.size - k)
                root = SW.roots(N, a, b, active)
                clusters = np.unique(root)
                member = (root[None, :] == clusters[:, None]).astype(np.int64)  # [n_clusters, N]
                patterns = ((np.arange(1 << clusters.size)[:, None] >> np.arange(clusters.size)) & 1) @ member
                ys = x ^ (patterns @ weights)
                np.add.at(P[x], ys, prob / (1 << clusters.size))
    return P


def boltzmann(rows, cols, J, T, periodic, signs):
    N = rows * cols
    s = 2 * ((np.arange(1 << N)[:, None] >> np.arange(N)) & 1) - 1
    a, b, g, _ = SW.bonds(rows, cols, periodic, signs)
    E = -J * (g[None, :] * s[:, a] * s[:, b]).sum(axis=1)
    w = np.exp(-(E - E.min()) / T)
    return w / w.sum()


CASES = [
    (2, 3, False, 1.0, 1.5, None),
    (2, 4, True, 1.0, 2.0, None),  # wrapped columns; a periodic length-2 dimension has no wrap
    (2, 3, False, -1.0, 1.2, None),
    (2, 4, True, 1.0, 1.3, "signs"),
]


@pytest.mark.parametrize("rows,cols,periodic,J,T,model", CASES)
def test_exact_transition_matrix_keeps_boltzmann(rows, cols, periodic, J, T, model):
    signs = np.random.default_rng(7).choice(np.array([-1, 1]), size=(2, rows, cols)) if model == "signs" else None
    P = transition_matrix(rows, cols, J, T, periodic, signs)
    assert np.abs(P.sum(axis=1) - 1.0).max() < 1e-12
    pi = boltzmann(rows, cols, J, T, periodic, signs)
    assert np.abs(pi @ P - pi).max() < 1e-12


def test_p_one_clusters_are_aligned_domains():
    rng = np.random.default_rng(3)
    rows, cols = 20, 30
    bits = (rng.random((rows, cols)) < 0.5).astype(np.int64)
    a, b, on = SW.active_bonds(bits, 1.0, 0.02, False, 5, 0, 0)
    assert SW.threshold(1.0, 0.02) == 1 << 32
    assert (on == SW.satisfied(bits, 1.0, False)).all()
    root = SW.roots(rows * cols, a, b, on).reshape(rows, cols)
    for v in (0, 1):
        lab, n = ndimage.label(bits == v)
        for k in range(1, n + 1):
            r = root[lab == k]
            assert (r == r[0]).all()
            assert r[0] == np.flatnonzero((lab == k).reshape(-1))[0]  # the domain's smallest site index


def test_active_fraction_is_p():
    rng = np.random.default_rng(4)
    rows = cols = 512
    J, T = 1.0, 2.269
    bits = (rng.random((rows, cols)) < 0.5).astype(np.int64)
    _, _, on = SW.active_bonds(bits, J, T, True, 99, 3, 17)
    sat = SW.satisfied(bits, J, True)
    p = -np.expm1(-2.0 * J / T)
    n = int(sat.sum())
    assert not (on & ~sat).any()
    assert abs(on.sum() / n - p) < 5 * np.sqrt(p * (1 - p) / n)
