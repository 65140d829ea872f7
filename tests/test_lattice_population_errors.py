"""Argument rules of lattice population annealing: they are checked before any device work, so these run without a GPU."""
import ctypes
import math

import numpy as np
import pytest
import torch


def bare_engine(is_slab=False, bias_mode="physical", n_replicas=4, bond_index=None):
    """an Ising2DEngine with no device state: anything that got past the checks would fail on a missing attribute"""
    from tsu_emulator_b200.lattice import Ising2DEngine

    eng = object.__new__(Ising2DEngine)
    eng.is_slab = is_slab
    eng.bias_mode = bias_mode
    eng.n_replicas = n_replicas
    eng.rows, eng.cols = 8, 8
    eng.bond_index = None if bond_index is None else torch.tensor(bond_index, dtype=torch.int32)
    return eng


def result(n_populations, r_pop, rows=8, cols=8):
    from tsu_emulator_b200.lattice import PopulationResult

    return PopulationResult(None, torch.zeros(n_populations * r_pop, dtype=torch.int32),
                            torch.zeros((2, n_populations), dtype=torch.int64), None, None, np.array([2.0, 1.0]),
                            math.inf, None, r_pop, 62, rows, cols, 1.0, 0.0, 128, 64)


@pytest.mark.parametrize("temps", [[], [[1.0, 2.0]], 1.5, [2.0, 0.0], [2.0, -1.0], [np.inf, 1.0], [1.0, np.nan]])
def test_bad_schedules_raise(temps):
    with pytest.raises(ValueError, match="temperatures"):
        bare_engine().population_annealing(temps)


def test_increasing_schedule_and_bad_start_raise():
    with pytest.raises(ValueError, match="non-increasing"):
        bare_engine().population_annealing([2.0, 1.0, 1.5])
    with pytest.raises(ValueError, match="T_start"):
        bare_engine().population_annealing([2.0, 1.0], T_start=1.5)
    with pytest.raises(ValueError, match="T_start"):
        bare_engine().population_annealing([2.0, 1.0], T_start=0.0)


def test_engine_and_population_arguments_raise():
    with pytest.raises(ValueError, match="row-slab"):
        bare_engine(is_slab=True).population_annealing([1.0])
    with pytest.raises(ValueError, match="bias_mode"):
        bare_engine(bias_mode="reference").population_annealing([1.0])
    for theta in (0, -3):
        with pytest.raises(ValueError, match="sweeps_per_step"):
            bare_engine().population_annealing([1.0], sweeps_per_step=theta)
    for P in (0, 3, 5, -1):
        with pytest.raises(ValueError, match="n_populations"):
            bare_engine().population_annealing([1.0], n_populations=P)
    with pytest.raises(ValueError, match="bond_index"):
        bare_engine(bond_index=[0, 0, 1, 1]).population_annealing([1.0])  # one population, two realisations
    with pytest.raises(ValueError, match="bond_index"):
        bare_engine(bond_index=[0, 1, 1, 1]).population_annealing([1.0], n_populations=2)


def test_previous_of_another_shape_raises():
    with pytest.raises(ValueError, match="previous"):
        bare_engine().population_annealing([1.0], n_populations=2, previous=result(1, 4))
    with pytest.raises(ValueError, match="previous"):
        bare_engine().population_annealing([1.0], n_populations=2, previous=result(2, 4))
    with pytest.raises(ValueError, match="previous"):
        bare_engine().population_annealing([1.0], n_populations=2, previous=result(2, 2, rows=6))
    # a previous run's last temperature becomes T_start: a schedule that starts above it is rejected
    with pytest.raises(ValueError, match="T_start"):
        bare_engine().population_annealing([1.5], n_populations=2, previous=result(2, 2))


def test_free_energy_needs_an_infinite_start():
    r = result(2, 2)
    r.T_start = 3.0
    with pytest.raises(ValueError, match="T_start = inf"):
        r.free_energy()


def test_work_bytes():
    from tsu_emulator_b200 import _lib

    lib = _lib.load()
    assert lib.tsu_ising2d_population_work_bytes(4096, 4) == 8 * (4096 + 4 * (1 + 2))
    assert lib.tsu_ising2d_population_work_bytes(131072, 1) == 8 * (131072 + 128 + 2)
    assert lib.tsu_ising2d_population_work_bytes(6, 3) == 8 * (6 + 3 * 3)
    assert lib.tsu_ising2d_population_work_bytes(6, 4) == 0
    assert lib.tsu_ising2d_population_work_bytes(0, 1) == 0


def test_abi_rejects_bad_arguments_before_any_cuda_call():
    from tsu_emulator_b200 import _lib

    lib = _lib.load()
    fake, fake2 = ctypes.c_void_p(256), ctypes.c_void_p(512)  # never dereferenced: the arguments are rejected first
    work = int(lib.tsu_ising2d_population_work_bytes(4, 2))
    good = dict(state=fake, scratch=fake2, n_replicas=4, rows=8, cols=8, wrap_rows=1, wrap_cols=1, luts=fake,
                dbeta=fake, n_steps=3, theta=2, n_populations=2, bonds=None, bond_index=None, seed=1, sweep0=0,
                replica0=0, J=1.0, h=0.0, n_bonds=128, n_sites=64, family=fake, family_scratch=fake2, weight_sum=fake,
                energy_ref=fake, count_sums=fake, obs=fake, energy=fake, work=fake, work_bytes=work, stream=0)

    def run(**kw):
        a = dict(good, **kw)
        return lib.tsu_ising2d_population_anneal(*a.values())

    bad = _lib.TSU_ERR_INVALID_ARG
    assert run(n_populations=3) == bad             # does not divide n_replicas
    assert run(n_populations=0) == bad
    assert run(n_replicas=70000 * 2, n_populations=70000) == bad  # populations are a grid dimension
    assert run(theta=0) == bad
    assert run(n_steps=-1) == bad
    assert run(scratch=fake) == bad                # the scratch state must be another buffer
    assert run(family_scratch=fake) == bad
    assert run(work_bytes=work - 8) == bad         # too small a workspace
    for name in ("state", "scratch", "luts", "dbeta", "family", "family_scratch", "weight_sum", "energy_ref",
                 "count_sums", "obs", "energy", "work"):
        assert run(**{name: None}) == bad, name
    assert run(n_replicas=0) == bad
    assert run(rows=7) == bad                      # periodic rows must be even
    assert run(cols=2) == bad                      # a periodic length-2 dimension has no wrap
    assert run(bond_index=fake) == bad             # a bond index needs bond words
