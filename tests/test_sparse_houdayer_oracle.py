"""Houdayer cluster moves on sparse couplings (tsu_sparse_houdayer, SparseProblem.houdayer).

CPU: the oracle (oracle/sparse_houdayer_oracle.py) labels the clusters of a 2-D periodic lattice's CSR as the lattice
oracle does; its move keeps E_a + E_b and the overlap exactly for dyadic symmetric J with bias and self couplings,
leaves d = 0 sites alone, flips clusters whole and is an involution for a fixed step.

GPU: the C-ABI move equals the oracle bit for bit on 3-D +-J glasses, random Gaussian graphs with bias and self
couplings, graphs with isolated sites and 2-D lattices, for 1 and 5 steps, more pairs than SMs, and N on both sides of
the shared-memory cap; split calls, chunked workspaces, skipped pairs and a wrapping chain0 give the same bits; the
energies it writes equal a zero-sweep tsu_sparse_gibbs_run bit for bit."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import cluster_oracle as SW
from oracle import houdayer_oracle as H
from oracle import sparse_houdayer_oracle as SH

gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------------ graphs
def csr_of(J):
    """(rowptr, col, val) of a scipy matrix, columns ascending, no stored zeros"""
    m = sp.csr_matrix(J, dtype=np.float64)
    m.sum_duplicates()
    m.eliminate_zeros()
    m.sort_indices()
    return m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data.astype(np.float64)


def symmetric(a, b, v, N):
    """symmetric scipy matrix with J_ab = J_ba = v"""
    m = sp.coo_matrix((v, (a, b)), shape=(N, N)).tocsr()
    return (m + m.T).tocsr()


def ea3d(L, seed):
    """periodic L^3 +-J Edwards-Anderson glass, site (x, y, z) -> (x L + y) L + z"""
    rng = np.random.default_rng(seed)
    idx = np.arange(L ** 3).reshape(L, L, L)
    a = np.concatenate([idx.ravel()] * 3)
    b = np.concatenate([np.roll(idx, -1, axis=ax).ravel() for ax in range(3)])
    return symmetric(a, b, rng.choice([-1.0, 1.0], a.size), L ** 3)


def gaussian_graph(N, seed, density=0.08, dyadic=False):
    """random sparse symmetric couplings with self couplings (dyadic: multiples of 1/8)"""
    rng = np.random.default_rng(seed)
    A = sp.random(N, N, density=density, random_state=seed, format="coo")
    v = np.round(rng.normal(size=A.nnz) * 8) / 8 if dyadic else rng.normal(size=A.nnz)
    J = symmetric(A.row, A.col, v, N).tolil()
    J.setdiag(np.round(rng.normal(size=N) * 4) / 4)
    return J.tocsr()


def isolated_graph(N, seed):
    """a chain over the even sites; odd sites have no couplings at all"""
    even = np.arange(0, N - 2, 2)
    return symmetric(even, even + 2, np.random.default_rng(seed).normal(size=even.size), N)


def lattice2d(rows, cols, seed):
    """the bonds of a periodic 2-D lattice as sparse couplings, sites numbered row-major"""
    a, b, _, _ = SW.bonds(rows, cols, True)
    return symmetric(a, b, np.random.default_rng(seed).choice([-1.0, 1.0], a.size), rows * cols)


def regular3(N, seed):
    """a ring with one random perfect matching of chords: degree 3 almost everywhere"""
    rng = np.random.default_rng(seed)
    i = np.arange(N)
    p = rng.permutation(N).reshape(-1, 2)
    a, b = np.concatenate([i, p[:, 0]]), np.concatenate([(i + 1) % N, p[:, 1]])
    keep = a != b
    return symmetric(a[keep], b[keep], rng.choice([-1.0, 1.0], int(keep.sum())), N)


def pair_states(rng, n_chains, N, pairs, density=0.5):
    """random states; the second chain of each pair differs from the first on a random pattern of the given density"""
    x = rng.integers(0, 2, (n_chains, N))
    for a, b in pairs:
        x[b] = x[a] ^ (rng.random(N) < density)
    return x


# ------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("rows,cols", [(4, 4), (6, 10), (16, 16)])
def test_roots_equal_lattice_oracle(rows, cols):
    rowptr, col, val = csr_of(lattice2d(rows, cols, 1))
    rng = np.random.default_rng(rows * cols)
    for p in (0.3, 0.6, 0.9):
        d = (rng.random((rows, cols)) < p).astype(np.int64)
        assert np.array_equal(SH.cluster_roots(rowptr, col, d.ravel(), val), H.cluster_roots(d, True))


def test_move_invariants():
    N = 120
    J = gaussian_graph(N, 5, density=0.05, dyadic=True)
    csr = csr_of(J)
    bias = np.random.default_rng(1).normal(size=N)   # any bias: its terms are only permuted between the chains
    rng = np.random.default_rng(2)
    flipped_some = False
    for trial in range(20):
        xa = rng.integers(0, 2, N)
        xb = xa ^ (rng.random(N) < rng.uniform(0.1, 0.9))
        ya, yb = SH.pair_step(xa, xb, csr, seed=9, chain=trial, step=trial)
        d = xa ^ xb
        assert np.array_equal(ya ^ yb, d)                                  # the overlap pattern is kept
        assert np.array_equal(ya[d == 0], xa[d == 0]) and np.array_equal(yb[d == 0], xb[d == 0])
        ea = SH.energy(xa, csr) + SH.energy(xb, csr)
        assert SH.energy(ya, csr) + SH.energy(yb, csr) == ea               # exact for dyadic J
        eb = SH.energy(xa, csr, bias) + SH.energy(xb, csr, bias)
        assert abs(SH.energy(ya, csr, bias) + SH.energy(yb, csr, bias) - eb) < 1e-9
        root = SH.cluster_roots(csr[0], csr[1], d, csr[2])
        f = ya ^ xa
        for r in np.unique(root[d == 1]):                                  # clusters flip whole
            assert len(set(f[root == r])) == 1
        flipped_some |= bool(f.any())
        za, zb = SH.pair_step(ya, yb, csr, seed=9, chain=trial, step=trial)
        assert np.array_equal(za, xa) and np.array_equal(zb, xb)            # involution for a fixed step
    assert flipped_some


def test_zero_entries_make_no_edge():
    rowptr = np.array([0, 1, 2], dtype=np.int32)
    col = np.array([1, 0], dtype=np.int32)
    d = np.array([1, 1])
    assert SH.cluster_roots(rowptr, col, d, np.array([0.0, 0.0])).tolist() == [0, 1]
    assert SH.cluster_roots(rowptr, col, d, np.array([1.0, 1.0])).tolist() == [0, 0]


# ------------------------------------------------------------------------------------------------------- GPU
def problem(J, bias=None):
    import torch

    from tsu_emulator_b200.sparse import SparseProblem

    return SparseProblem(J, bias, torch.device("cuda", 0))


def run_move(prob, x, pairs, seed, step0, n_steps, chain0, energy=False):
    """SparseProblem.houdayer on the host states x; returns (states, energies or None)"""
    import torch

    st = torch.from_numpy(np.ascontiguousarray(x.astype(np.uint8))).cuda()
    pr = torch.from_numpy(np.ascontiguousarray(np.asarray(pairs, dtype=np.int32).reshape(-1, 2))).cuda()
    e = torch.full((x.shape[0],), np.nan, dtype=torch.float64, device="cuda") if energy else None
    prob.houdayer(st, pr, pr.shape[0], seed=seed, step0=step0, n_steps=n_steps, chain0=chain0, energy=e)
    return st.cpu().numpy().astype(np.int64), (None if e is None else e.cpu().numpy())


def sweep_energies(prob, x):
    """energies tsu_sparse_gibbs_run reports for the states x after zero sweeps"""
    import torch

    st = torch.from_numpy(np.ascontiguousarray(x.astype(np.uint8))).cuda()
    _, e, _, _ = prob.run(st, T=1.0, seed=0, sweep0=0, chain0=0, n_burnin=0, n_samples=0, sweeps_per_sample=0,
                          want_energy=True)
    return e.cpu().numpy()


GRAPHS = {
    "ea3d_L4": lambda: ea3d(4, 1),
    "ea3d_L6": lambda: ea3d(6, 2),
    "ea3d_L8": lambda: ea3d(8, 3),
    "gaussian_bias_self": lambda: gaussian_graph(300, 4),
    "isolated_sites": lambda: isolated_graph(90, 5),
    "lattice2d_12x20": lambda: lattice2d(12, 20, 6),
}


@gpu
@pytest.mark.parametrize("name", list(GRAPHS))
@pytest.mark.parametrize("n_steps", [1, 5])
def test_move_equals_oracle(name, n_steps):
    J = GRAPHS[name]()
    N = J.shape[0]
    bias = np.random.default_rng(N).normal(size=N) if name == "gaussian_bias_self" else None
    prob = problem(J, bias)
    rng = np.random.default_rng(N + n_steps)
    pairs = [(3, 0), (1, 2), (5, 4), (6, 9)]          # any order; chains 7 and 8 are in no pair
    x = pair_states(rng, 10, N, pairs, density=0.3)   # sparse enough for several clusters per pair
    seed, step0, chain0 = 1234 + n_steps, 17, 40
    got, e = run_move(prob, x, pairs, seed, step0, n_steps, chain0, energy=True)
    want = SH.houdayer_steps(x, pairs, csr_of(J), seed, chain0, step0, n_steps)
    assert np.array_equal(got, want)
    assert not np.array_equal(got, x)
    done = np.array(pairs).ravel()
    assert np.array_equal(e[done], sweep_energies(prob, got)[done])        # bit for bit
    assert np.isnan(e[[7, 8]]).all()                                       # chains of no pair are not written


@gpu
def test_many_pairs_several_waves():
    """300 pairs (more than the 148 SMs take at once), dyadic couplings: oracle bits, and E_a + E_b kept exactly"""
    J = gaussian_graph(64, 8, density=0.1, dyadic=True)
    prob = problem(J, np.round(np.random.default_rng(0).normal(size=64) * 4) / 4)
    rng = np.random.default_rng(3)
    n = 600
    pairs = rng.permutation(n).reshape(-1, 2)
    x = pair_states(rng, n, 64, pairs)
    got, e = run_move(prob, x, pairs, 77, 0, 2, 5, energy=True)
    assert np.array_equal(got, SH.houdayer_steps(x, pairs, csr_of(J), 77, 5, 0, 2))
    e0 = sweep_energies(prob, x)
    assert np.array_equal(e[pairs[:, 0]] + e[pairs[:, 1]], e0[pairs[:, 0]] + e0[pairs[:, 1]])
    assert np.array_equal(e, sweep_energies(prob, got))


BIG = {"regular3_32768": lambda: regular3(32768, 13), "ea3d_L40": lambda: ea3d(40, 9),
       "regular3_1e5": lambda: regular3(100000, 10)}


@gpu
@pytest.mark.parametrize("name", list(BIG))
def test_large_n_equals_oracle(name):
    """N at the shared-memory cap (32768: rows and labels in 192 KB of shared memory) and above it (labels in the
    workspace); there a one-pair workspace (chunks) gives the same bits"""
    import torch

    from tsu_emulator_b200 import _lib

    J = BIG[name]()
    N = J.shape[0]
    prob = problem(J)
    rng = np.random.default_rng(N)
    pairs = [(0, 3), (2, 1), (4, 5)]
    x = pair_states(rng, 7, N, pairs, density=0.5)
    got, e = run_move(prob, x, pairs, 5, 3, 2, 11, energy=True)
    want = SH.houdayer_steps(x, pairs, csr_of(J), 5, 11, 3, 2)
    assert np.array_equal(got, want)
    assert np.array_equal(e[:6], sweep_energies(prob, got)[:6])
    lib = _lib.load()
    per = int(lib.tsu_sparse_houdayer_work_bytes(1, N))
    if per == 0:   # labels in shared memory: no workspace
        return
    # one pair's workspace: three chunks
    work = torch.empty(per // 8 + 1, dtype=torch.int64, device="cuda")
    st = torch.from_numpy(x.astype(np.uint8)).cuda()
    pr = torch.tensor(pairs, dtype=torch.int32, device="cuda")
    _lib.call("tsu_sparse_houdayer", prob.rowptr.data_ptr(), prob.col.data_ptr(), prob.val.data_ptr(), None,
              st.data_ptr(), 7, N, pr.data_ptr(), 3, 5, 3, 2, 11, None, work.data_ptr(), per + 7,
              _lib.current_stream())
    assert np.array_equal(st.cpu().numpy(), want)


@gpu
def test_split_calls_skips_and_wrapping_chain0():
    J = ea3d(6, 12)
    N = J.shape[0]
    prob = problem(J)
    rng = np.random.default_rng(4)
    pairs = [(0, 1), (2, 3), (4, 5)]
    x = pair_states(rng, 8, N, pairs)
    chain0 = 2 ** 32 - 3                                   # chain0 + a wraps for a >= 3
    one, _ = run_move(prob, x, pairs, 8, 100, 3, chain0)
    split, _ = run_move(prob, x, pairs, 8, 100, 1, chain0)
    split, _ = run_move(prob, split, pairs, 8, 101, 2, chain0)
    assert np.array_equal(one, split)
    assert np.array_equal(one, SH.houdayer_steps(x, pairs, csr_of(J), 8, chain0, 100, 3))
    # skipped pairs (out of range, a == b) leave every row byte-identical, the good pair still moves; the rows of the
    # skipped chains hold bytes other than 0 / 1, which a processed row would get back as 0 / 1
    y = x.copy()
    y[6] = rng.choice([0, 1, 2, 255], N)
    y[7] = rng.choice([0, 2, 3, 255], N)
    bad = [(6, 6), (7, 8), (-1, 7), (0, 1)]
    got, _ = run_move(prob, y, bad, 8, 100, 3, chain0)
    assert np.array_equal(got[2:], y[2:])
    assert np.array_equal(got[:2], one[:2])
