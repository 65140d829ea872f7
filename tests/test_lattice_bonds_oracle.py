"""CPU: the Edwards-Anderson +-J lattice oracle (bond-corrected up-count on the ferromagnet's table) against the
literal port of the reference's sweep on the dense +-J bit model, and the rejection of what the bonded kernels cannot
serve, from Python and from the C-ABI, without a GPU."""
import ctypes

import numpy as np
import pytest

from oracle import ising2d_bonds_oracle as B
from oracle import ising2d_oracle as O

GEOMETRIES = [
    # rows, cols, periodic
    (6, 8, False),   # open
    (6, 8, True),    # periodic
    (5, 7, False),   # ragged (odd sizes)
    (4, 10, True),
    (1, 9, False),   # one row
    (9, 1, False),   # one column
    (2, 6, True),    # periodic, rows of length 2: that wrap adds no bond
    (6, 2, True),    # periodic, columns of length 2
    (2, 2, True),
]


def random_signs(rng, rows, cols):
    return rng.choice(np.array([-1, 1], dtype=np.int8), size=(2, rows, cols))


@pytest.mark.parametrize("rows,cols,periodic", GEOMETRIES)
def test_bonded_oracle_equals_literal_port_on_dense_pm_j(rows, cols, periodic):
    rng = np.random.default_rng(rows * 100 + cols + periodic)
    # dyadic J and h: every field is exact in float64 on both sides
    for J, h, T in [(1.0, 0.0, 2.0), (0.75, 0.125, 1.5), (-0.5, -0.25, 0.7)]:
        signs = random_signs(rng, rows, cols)
        bits0 = rng.integers(0, 2, (rows, cols))
        U = rng.integers(0, 2**32, (3, rows, cols), dtype=np.uint64).astype(np.uint32)
        Jb, hb = B.dense_bit_model_bonds(rows, cols, J, h, periodic, signs)
        order = O.checkerboard_order(rows, cols)
        s = bits0.ravel().copy()
        for t in range(3):
            s = O.gibbs_sweep_port(s, Jb, hb, T, order, U[t].ravel()[order].astype(np.float64) / 2**32)
        got = B.checkerboard_sweeps_bonds(bits0, U, J, h, T, periodic, signs)
        assert (s.reshape(rows, cols) == got).all()
        # energy: the dense spin Hamiltonian, each bond once
        sp = 2 * got.ravel() - 1
        Jm = Jb / 4
        assert B.energy_bonds(got, J, h, periodic, signs) == pytest.approx(-0.5 * sp @ Jm @ sp - h * sp.sum(), abs=1e-12)
        n_bonds = len(B.bond_list(rows, cols, periodic, signs)[2])
        unsat = B.unsatisfied_bonds(got, periodic, signs)
        assert B.energy_bonds(got, J, h, periodic, signs) == pytest.approx(
            -J * (n_bonds - 2 * unsat) - h * (2 * got.sum() - got.size), abs=1e-12)


def test_all_plus_bonds_are_the_ferromagnet():
    rng = np.random.default_rng(5)
    for rows, cols, periodic in GEOMETRIES:
        ones = np.ones((2, rows, cols), dtype=np.int8)
        bits0 = rng.integers(0, 2, (rows, cols))
        U = rng.integers(0, 2**32, (2, rows, cols), dtype=np.uint64).astype(np.uint32)
        assert (B.checkerboard_sweeps_bonds(bits0, U, 1.0, 0.1, 2.0, periodic, ones) ==
                O.checkerboard_sweeps(bits0, U, 1.0, 0.1, 2.0, periodic)).all()
        assert B.energy_bonds(bits0, 1.0, 0.1, periodic, ones) == pytest.approx(O.energy(bits0, 1.0, 0.1, periodic))


def test_ignored_bond_entries_change_nothing():
    """open edges and the wrap of a periodic dimension of length 2 create no bond: their signs are never read"""
    rng = np.random.default_rng(8)
    for rows, cols, periodic in [(5, 7, False), (2, 6, True), (6, 2, True)]:
        signs = random_signs(rng, rows, cols)
        flipped = signs.copy()
        if not periodic or cols <= 2:
            flipped[0, :, cols - 1] *= -1
        if not periodic or rows <= 2:
            flipped[1, rows - 1, :] *= -1
        bits0 = rng.integers(0, 2, (rows, cols))
        U = rng.integers(0, 2**32, (2, rows, cols), dtype=np.uint64).astype(np.uint32)
        assert (B.checkerboard_sweeps_bonds(bits0, U, 1.0, 0.0, 1.0, periodic, signs) ==
                B.checkerboard_sweeps_bonds(bits0, U, 1.0, 0.0, 1.0, periodic, flipped)).all()


def test_exact_moments_of_a_tiny_lattice():
    """enumeration helper against a direct sum on a 2 x 3 open lattice"""
    rng = np.random.default_rng(1)
    signs = random_signs(rng, 2, 3)
    mE, mE2, mq2 = B.exact_moments(2, 3, 1.0, 0.0, 1.3, False, signs)
    Es, ws, ss = [], [], []
    for k in range(64):
        bits = ((k >> np.arange(6)) & 1).reshape(2, 3)
        E = B.energy_bonds(bits, 1.0, 0.0, False, signs)
        Es.append(E)
        ws.append(np.exp(-E / 1.3))
        ss.append(2 * bits.ravel() - 1)
    w = np.array(ws) / sum(ws)
    Es, ss = np.array(Es), np.array(ss)
    assert mE == pytest.approx((w * Es).sum())
    assert mE2 == pytest.approx((w * Es**2).sum())
    q2 = sum(w[a] * w[b] * (ss[a] @ ss[b] / 6) ** 2 for a in range(64) for b in range(64))
    assert mq2 == pytest.approx(q2)


# ---------------------------------------------------------------------------- rejection without a GPU
def engine(**kw):
    from tsu_emulator_b200.lattice import Ising2DEngine

    args = dict(rows=4, cols=6, n_replicas=2, periodic=True)
    args.update(kw)
    return Ising2DEngine(**args)


@pytest.mark.parametrize("bonds,index,match", [
    (np.full((2, 4, 6), 2), None, r"\+1 or -1"),
    (np.zeros((2, 4, 6)), None, r"\+1 or -1"),
    (np.ones((2, 4, 6)) * 0.5, None, r"\+1 or -1"),
    (np.ones((2, 4, 5)), None, "shape"),
    (np.ones((3, 4, 6)), None, "shape"),
    (np.ones((1, 1, 2, 4, 6)), None, "shape"),
    (np.ones((3, 2, 4, 6)), None, "bond_index is required"),
    (np.ones((3, 2, 4, 6)), [0, 3], r"\[0, 3\)"),
    (np.ones((3, 2, 4, 6)), [0, -1], r"\[0, 3\)"),
    (np.ones((3, 2, 4, 6)), [0, 1, 2], "2 integers"),
    (np.ones((3, 2, 4, 6)), [0.0, 1.0], "2 integers"),
])
def test_malformed_bonds_are_rejected(bonds, index, match):
    with pytest.raises(ValueError, match=match):
        engine(bonds=bonds, bond_index=index)


def test_reference_bias_and_slabs_are_rejected():
    ones = np.ones((2, 4, 6), dtype=np.int8)
    with pytest.raises(ValueError, match="physical"):
        engine(bonds=ones, bias_mode="reference")
    with pytest.raises(ValueError, match="row-slab"):
        engine(bonds=ones, global_rows=8, periodic=False)
    with pytest.raises(ValueError, match="row-slab"):
        engine(bonds=ones, row0=4, periodic=False)
    with pytest.raises(ValueError, match="needs bonds"):
        engine(bond_index=[0, 0])


def test_check_bonds_defaults():
    from tsu_emulator_b200.lattice import check_bonds

    b, idx = check_bonds(np.ones((2, 4, 6)), None, 4, 6, 3)
    assert b.shape == (1, 2, 4, 6) and b.dtype == np.int8 and idx is None
    b, idx = check_bonds(-np.ones((3, 2, 4, 6)), None, 4, 6, 3)
    assert (idx == np.arange(3)).all() and (b == -1).all()
    _, idx = check_bonds(np.ones((2, 2, 4, 6)), np.array([1, 0, 1]), 4, 6, 3)
    assert idx.dtype == np.int32 and list(idx) == [1, 0, 1]


def test_merged_lattice_abi_rejects_bonded_arguments_before_any_cuda_call():
    from tsu_emulator_b200 import _lib

    lib = _lib.load()
    bad = _lib.TSU_ERR_INVALID_ARG
    p = ctypes.c_void_p(256)  # never dereferenced: every call below fails its argument check
    # missing pointers (a bond index without bond words)
    assert lib.tsu_ising2d_pack_bonds(None, p, 1, 4, 4, 1, 1, 0) == bad
    assert lib.tsu_ising2d_pack_bonds(p, None, 1, 4, 4, 1, 1, 0) == bad
    assert lib.tsu_ising2d_sweeps(0, p, 1, 4, 4, 1, 1, p, None, None, p, 0, 0, 1, 0, 0) == bad
    assert lib.tsu_ising2d_half_sweep(0, p, 1, 4, 4, 1, 1, 0, p, None, None, p, 0, 0, 0, 0, None, None, 0, 4, 0) == bad
    assert lib.tsu_ising2d_half_sweep_injected(p, 1, 4, 4, 1, 1, 0, p, None, None, p, p, 0, None, None, 0) == bad
    assert lib.tsu_ising2d_observables(p, 1, 4, 4, 1, 1, None, p, 0, None, p, 0) == bad
    assert lib.tsu_ising2d_overlap(p, 2, 4, 4, None, 1, p, 0) == bad
    # geometry, colour, row ranges, wraps, pair counts
    assert lib.tsu_ising2d_pack_bonds(p, p, 0, 4, 4, 0, 0, 0) == bad
    assert lib.tsu_ising2d_pack_bonds(p, p, 1, 4, 2, 0, 1, 0) == bad     # column wrap of length 2
    assert lib.tsu_ising2d_pack_bonds(p, p, 1, 5, 4, 1, 0, 0) == bad     # odd periodic rows
    assert lib.tsu_ising2d_sweeps(0, p, 1, 4, 4, 1, 1, p, None, p, None, 0, 0, -1, 0, 0) == bad
    assert lib.tsu_ising2d_sweeps(0, p, 1, 4, 3, 1, 1, p, None, p, None, 0, 0, 1, 0, 0) == bad
    assert lib.tsu_ising2d_half_sweep(0, p, 1, 4, 4, 1, 1, 2, p, None, p, None, 0, 0, 0, 0, None, None, 0, 4, 0) == bad
    assert lib.tsu_ising2d_half_sweep(0, p, 1, 4, 4, 1, 1, 0, p, None, p, None, 0, 0, 0, 0, None, None, 3, 2, 0) == bad
    assert lib.tsu_ising2d_half_sweep(0, p, 1, 4, 4, 1, 1, 0, p, None, p, None, 0, 0, 0, 0, None, None, 0, 5, 0) == bad
    assert lib.tsu_ising2d_half_sweep_injected(p, 1, 4, 4, 1, 1, 0, p, None, p, None, None, 0, None, None, 0) == bad
    assert lib.tsu_ising2d_observables(p, 0, 4, 4, 1, 1, p, None, 0, None, p, 0) == bad
    assert lib.tsu_ising2d_overlap(p, 2, 4, 4, p, 0, p, 0) == bad
    assert lib.tsu_ising2d_overlap(p, 2, 4, 4, p, 65536, p, 0) == bad
    # bond words are indexed by local row: no halos, row slabs or next rows with bonds
    assert lib.tsu_ising2d_half_sweep(0, p, 1, 4, 4, 0, 1, 0, p, None, p, None, 0, 0, 0, 0, p, None, 0, 4, 0) == bad
    assert lib.tsu_ising2d_half_sweep(0, p, 1, 4, 4, 0, 1, 0, p, None, p, None, 0, 0, 0, 4, None, None, 0, 4, 0) == bad
    assert lib.tsu_ising2d_half_sweep_injected(p, 1, 4, 4, 0, 1, 0, p, None, p, None, p, 0, None, p, 0) == bad
    assert lib.tsu_ising2d_half_sweep_injected(p, 1, 4, 4, 0, 1, 0, p, None, p, None, p, 4, None, None, 0) == bad
    assert lib.tsu_ising2d_observables(p, 1, 4, 4, 0, 1, p, None, 0, p, p, 0) == bad
    assert lib.tsu_ising2d_observables(p, 1, 4, 4, 0, 1, p, None, 4, None, p, 0) == bad
