"""Argument rules of lattice annealing: they are checked before any device work, so these run without a GPU."""
import ctypes

import numpy as np
import pytest


def bare_engine(is_slab=False):
    """an Ising2DEngine with no device state: anything that got past the checks would fail on a missing attribute"""
    from tsu_emulator_b200.lattice import Ising2DEngine

    eng = object.__new__(Ising2DEngine)
    eng.is_slab = is_slab
    eng.n_replicas = 2
    return eng


@pytest.mark.parametrize("temps", [[], [[1.0, 2.0]], 1.5, [2.0, 0.0], [2.0, -1.0], [np.inf, 1.0], [1.0, np.nan]])
def test_bad_schedules_raise(temps):
    with pytest.raises(ValueError, match="temperatures"):
        bare_engine().anneal(temps)


def test_row_slabs_and_bad_simulated_annealing_arguments_raise():
    with pytest.raises(ValueError, match="row-slab"):
        bare_engine(is_slab=True).anneal([1.0, 0.5])
    with pytest.raises(ValueError, match="row-slab"):
        bare_engine(is_slab=True).simulated_annealing(2.0, 0.5, 10)
    with pytest.raises(ValueError, match="n_steps"):
        bare_engine().simulated_annealing(2.0, 0.5, -1)
    with pytest.raises(ValueError, match="temperatures"):
        bare_engine().simulated_annealing(2.0, 0.0, 10)  # every step after the first at T = 0
    with pytest.raises(ValueError, match="temperatures"):
        bare_engine().simulated_annealing(np.nan, 0.5, 10)


def test_abi_rejects_bad_arguments_before_any_cuda_call():
    from tsu_emulator_b200 import _lib

    lib = _lib.load()
    fake = ctypes.c_void_p(256)  # never dereferenced: the arguments are rejected first
    good = dict(state=fake, n_replicas=2, rows=8, cols=8, wrap_rows=1, wrap_cols=1, luts=fake, n_steps=3, bonds=None,
                bond_index=None, seed=1, sweep0=0, replica0=0, J=1.0, h=0.0, n_bonds=128, n_sites=64, obs=fake,
                energy=fake, best_energy=fake, best_state=fake, stream=0)

    def run(**kw):
        a = dict(good, **kw)
        return lib.tsu_ising2d_anneal(*a.values())

    bad = _lib.TSU_ERR_INVALID_ARG
    assert run(n_steps=-1) == bad
    assert run(luts=None) == bad                   # tables are needed when there are steps
    assert run(obs=None) == bad
    assert run(energy=None) == bad
    assert run(best_energy=None) == bad            # the best pointers come in pairs
    assert run(best_state=None) == bad
    assert run(state=None) == bad
    assert run(n_replicas=0) == bad
    assert run(rows=7) == bad                      # periodic rows must be even
    assert run(cols=2) == bad                      # a periodic length-2 dimension has no wrap
    assert run(bond_index=fake) == bad             # a bond index needs bond words
    # the word-by-word counts take one grid row per replica (gridDim.y <= 65535)
    assert run(n_replicas=70000, rows=64, cols=100, n_bonds=12800, n_sites=6400) == bad


def test_schedule_is_the_dense_samplers():
    from tsu_emulator_b200.gibbs import annealing_temperatures

    for T0, T1, n in [(10.0, 0.1, 1000), (5.0, 0.5, 7), (3, 1, 4), (2.5, 2.5, 3), (1.0, 4.0, 1)]:
        steps = np.arange(n, dtype=np.float64)
        exp = T0 * (T1 / T0) ** (steps / n)
        lin = T0 + (T1 - T0) * steps / n
        assert annealing_temperatures(T0, T1, n, "exponential").tobytes() == exp.tobytes()
        assert annealing_temperatures(T0, T1, n, "linear").tobytes() == lin.tobytes()
    assert annealing_temperatures(10.0, 0.1, 0).shape == (0,)
