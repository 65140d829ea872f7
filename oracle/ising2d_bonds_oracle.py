"""
ORACLE (test infrastructure, not product code): the heat-bath update of oracle/ising2d_oracle.py on an
Edwards-Anderson +-J lattice, J_ij = J * sigma_ij with sigma_ij = +-1 per nearest-neighbour bond.

Reference semantics: the dense bit model of tsu/models/ising.py:127-148 (J_bit = 4 J_ij, bias 2h - 2 rowsum(J),
bias_mode "physical") with the coupling matrix holding J * sigma_ij on the bonds IsingGrid wires
(tsu/models/ising.py:343-361), swept by tsu/gibbs.py:128-162.  `dense_bit_model_bonds` builds that model and
tests/test_lattice_bonds_oracle.py checks `checkerboard_sweeps_bonds` against `gibbs_sweep_port` on it.

Sign layout (Ising2DEngine): signs[0, i, j] is the bond (i, j)-(i, (j+1) % C), signs[1, i, j] the bond
(i, j)-((i+1) % R, j).  Entries of bonds the wiring does not create are ignored: open edges, and the wrap of a
periodic dimension of length <= 2 (set_coupling assigns, so that wrap adds no bond).

The local field of the bit model is 4J u' + 2h - 2J d with u' = sum_j (b_j XOR [sigma_ij = -1]): the
ferromagnet's threshold table indexed by the bond-corrected up-count (what the CUDA kernels compute).
"""

import numpy as np

from . import ising2d_oracle as O


def bond_list(rows: int, cols: int, periodic: bool, signs):
    """(a, b, sigma) int arrays over the bonds the wiring creates; a, b are row-major site indices"""
    s = np.asarray(signs)
    assert s.shape == (2, rows, cols)
    wrap_r = periodic and rows > 2
    wrap_c = periodic and cols > 2
    i, j = np.meshgrid(np.arange(rows), np.arange(cols), indexing="ij")
    a, b, g = [], [], []
    h_ok = (j < cols - 1) | wrap_c
    a.append((i * cols + j)[h_ok])
    b.append((i * cols + (j + 1) % cols)[h_ok])
    g.append(s[0][h_ok])
    v_ok = (i < rows - 1) | wrap_r
    a.append((i * cols + j)[v_ok])
    b.append((((i + 1) % rows) * cols + j)[v_ok])
    g.append(s[1][v_ok])
    return np.concatenate(a), np.concatenate(b), np.concatenate(g).astype(np.int64)


def neighbour_up_and_degree_bonds(bits, periodic: bool, signs):
    """bond-corrected up-count u' (neighbour bit XOR [sigma = -1]) and degree of every site"""
    bits = np.asarray(bits, dtype=np.int64)
    R, C = bits.shape
    a, b, g = bond_list(R, C, periodic, signs)
    flat = bits.reshape(-1)
    anti = (g < 0).astype(np.int64)
    up = np.zeros(R * C, dtype=np.int64)
    deg = np.zeros(R * C, dtype=np.int64)
    np.add.at(up, a, flat[b] ^ anti)
    np.add.at(up, b, flat[a] ^ anti)
    np.add.at(deg, a, 1)
    np.add.at(deg, b, 1)
    return up.reshape(R, C), deg.reshape(R, C)


def half_sweep_bonds(bits, colour, u32, J, h, T, periodic, signs):
    """update every site of `colour` (they do not interact) - in place"""
    R, C = bits.shape
    i = np.arange(R)[:, None]
    j = np.arange(C)[None, :]
    mask = ((i + j) & 1) == colour
    up, deg = neighbour_up_and_degree_bonds(bits, periodic, signs)
    p = O.acceptance_probability(J, h, T, up, deg, "physical")
    new = ((u32.astype(np.float64) / 4294967296.0) < p).astype(bits.dtype)
    bits[mask] = new[mask]
    return bits


def checkerboard_sweeps_bonds(bits0, u32_per_sweep, J, h, T, periodic, signs):
    """n sweeps (black then white) with injected uniforms u32_per_sweep[t, i, j]"""
    bits = np.array(bits0, dtype=np.int64, copy=True)
    for t in range(len(u32_per_sweep)):
        for colour in (0, 1):
            half_sweep_bonds(bits, colour, u32_per_sweep[t], J, h, T, periodic, signs)
    return bits


def checkerboard_sweeps_philox_bonds(bits0, seed, replica, sweep0, n_sweeps, J, h, T, periodic, signs):
    """what the bonded CUDA kernels must reproduce bit for bit in Philox mode"""
    R, C = np.asarray(bits0).shape
    u = np.stack([O.philox_uniform_field(seed, replica, sweep0 + t, R, C) for t in range(n_sweeps)]) if n_sweeps else []
    return checkerboard_sweeps_bonds(bits0, u, J, h, T, periodic, signs)


def unsatisfied_bonds(bits, periodic, signs) -> int:
    """number of bonds with sigma s_i s_j = -1"""
    s = 2 * np.asarray(bits, dtype=np.int64).reshape(-1) - 1
    R, C = np.asarray(bits).shape
    a, b, g = bond_list(R, C, periodic, signs)
    return int((g * s[a] * s[b] < 0).sum())


def energy_bonds(bits, J, h, periodic, signs) -> float:
    """E = -J sum_<ij> sigma_ij s_i s_j - h sum_i s_i"""
    s = 2 * np.asarray(bits, dtype=np.int64) - 1
    R, C = s.shape
    a, b, g = bond_list(R, C, periodic, signs)
    flat = s.reshape(-1)
    return float(-J * (g * flat[a] * flat[b]).sum() - h * s.sum())


def dense_bit_model_bonds(rows, cols, J, h, periodic, signs):
    """dense (J_bit, h_bit) of the +-J lattice as IsingGrid + _get_bit_coupling/_get_bit_bias ("physical") would build
    it with coupling J * sigma on every wired bond"""
    n = rows * cols
    Jm = np.zeros((n, n))
    a, b, g = bond_list(rows, cols, periodic, signs)
    Jm[a, b] = J * g
    Jm[b, a] = J * g
    hb = 2 * np.ones(n) * h - 2 * np.sum(Jm, axis=1)
    return 4 * Jm, hb


def exact_moments(rows, cols, J, h, T, periodic, signs):
    """exact <E>, <E^2> and <q^2> (two independent replicas) by enumerating all 2^(rows cols) states"""
    n = rows * cols
    assert n <= 20
    states = ((np.arange(1 << n)[:, None] >> np.arange(n)[None, :]) & 1).astype(np.int64)
    s = 2 * states - 1
    a, b, g = bond_list(rows, cols, periodic, signs)
    E = -J * (g[None, :] * s[:, a] * s[:, b]).sum(axis=1) - h * s.sum(axis=1)
    w = np.exp(-(E - E.min()) / T)
    w /= w.sum()
    mE = float((w * E).sum())
    mE2 = float((w * E * E).sum())
    # <q^2> = (1/N^2) sum_ij <s_i s_j>^2
    C = (s * w[:, None]).T @ s
    mq2 = float((C * C).sum()) / (n * n)
    return mE, mE2, mq2
