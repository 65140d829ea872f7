"""Argument rules of GibbsSampler.population_annealing and of the C entry points tsu_population_resample /
tsu_population_moments: all are checked before any device work, so these run without a GPU.  Also the tests'
resampling step (tests/population_resample.py) against the lattice oracle's population_anneal."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import population_oracle as PO
from population_resample import resample_populations


def sampler(precision="float64"):
    from tsu_emulator_b200 import GibbsSampler

    return GibbsSampler(seed=3, precision=precision)


J8 = np.zeros((8, 8))


def result(n_populations, r_pop, N=8, backend="float64"):
    """a DensePopulationResult with host tensors: only its shape and back end are read before the device work"""
    from tsu_emulator_b200.gibbs import DensePopulationResult

    C = n_populations * r_pop
    return DensePopulationResult(torch.zeros((C, N), dtype=torch.uint8), None, torch.zeros(C, dtype=torch.int32),
                                 torch.zeros((2, n_populations), dtype=torch.int64), None, None, np.array([2.0, 1.0]),
                                 math.inf, None, r_pop, 62, N, 0, backend)


@pytest.mark.parametrize("temps", [[], [[1.0, 2.0]], 1.5, [2.0, 0.0], [2.0, -1.0], [np.inf, 1.0], [1.0, np.nan]])
def test_bad_schedules_raise(temps):
    with pytest.raises(ValueError, match="temperatures"):
        sampler().population_annealing(J8, temps)


def test_increasing_schedule_and_bad_start_raise():
    with pytest.raises(ValueError, match="non-increasing"):
        sampler().population_annealing(J8, [2.0, 1.0, 1.5])
    with pytest.raises(ValueError, match="T_start"):
        sampler().population_annealing(J8, [2.0, 1.0], T_start=1.5)
    with pytest.raises(ValueError, match="T_start"):
        sampler().population_annealing(J8, [2.0, 1.0], T_start=0.0)


def test_sweeps_chains_and_populations_raise():
    for theta in (0, -3):
        with pytest.raises(ValueError, match="sweeps_per_step"):
            sampler().population_annealing(J8, [1.0], sweeps_per_step=theta)
    for C in (0, -4):
        with pytest.raises(ValueError, match="n_chains"):
            sampler().population_annealing(J8, [1.0], n_chains=C)
    for P, C in ((0, 4), (3, 4), (5, 4), (-1, 4), (65536, 65536 * 2)):
        with pytest.raises(ValueError, match="n_populations must divide n_chains"):
            sampler().population_annealing(J8, [1.0], n_chains=C, n_populations=P)


def test_previous_of_another_run_raises():
    run = lambda prev, **kw: sampler(kw.pop("precision", "float64")).population_annealing(
        kw.pop("J", J8), [1.0], n_chains=4, n_populations=2, previous=prev, **kw)
    with pytest.raises(ValueError, match="previous"):
        run(result(1, 4))                                   # other populations
    with pytest.raises(ValueError, match="previous"):
        run(result(2, 4))                                   # other chain count
    with pytest.raises(ValueError, match="previous"):
        run(result(2, 2, N=9))                              # other model size
    with pytest.raises(ValueError, match="previous"):
        run(result(2, 2, backend="bf16"))                   # other back end
    with pytest.raises(ValueError, match="previous"):
        run(result(2, 2), precision="float32")
    with pytest.raises(ValueError, match="previous"):
        run(result(2, 2), chromatic=True)
    with pytest.raises(ValueError, match="previous"):
        run(object())
    # a previous run's last temperature becomes T_start: a schedule that starts above it is rejected
    with pytest.raises(ValueError, match="T_start"):
        sampler().population_annealing(J8, [1.5], n_chains=4, n_populations=2, previous=result(2, 2))


def test_chromatic_needs_a_float64_sampler():
    for precision in ("float32", "bf16"):
        with pytest.raises(ValueError, match="chromatic=True .* use a 'float64' sampler"):
            sampler(precision).population_annealing(J8, [1.0], n_chains=4, chromatic=True)


def test_specific_heat_and_mean_energy_from_moments():
    r = result(2, 4)
    r.temperatures = np.array([2.0, 0.5])
    E = np.array([[[-1.0, 0.5, 2.0, 0.0], [3.0, 3.0, 3.0, 3.0]], [[-4.0, -4.0, -2.0, 0.0], [1.0, -1.0, 1.0, -1.0]]])
    m = np.zeros((3, 2, 2))
    m[1:, :, 0], m[1:, :, 1] = E.sum(-1), (E * E).sum(-1)
    r.energy_moments = torch.from_numpy(m)
    assert np.allclose(r.mean_energy(), E.mean(-1))
    assert np.allclose(r.specific_heat(), E.var(-1) / r.temperatures[:, None] ** 2 / 8)
    r.T_start = 3.0
    with pytest.raises(ValueError, match="T_start = inf"):
        r.free_energy()


def test_abi_rejects_bad_arguments_before_any_cuda_call():
    from tsu_emulator_b200 import _lib

    lib = _lib.load()
    fake, fake2 = ctypes.c_void_p(256), ctypes.c_void_p(512)  # never dereferenced: the arguments are rejected first
    work = int(lib.tsu_ising2d_population_work_bytes(6, 2))
    good = dict(state=fake, state_out=fake2, family=fake, family_out=fake2, energy=fake, dbeta=fake, n_chains=6,
                n_populations=2, row_bytes=33, seed=1, sweep=0, chain0=0, weight_sum=fake, energy_ref=fake, work=fake,
                work_bytes=work, stream=0)

    def run(**kw):
        a = dict(good, **kw)
        return lib.tsu_population_resample(*a.values())

    bad = _lib.TSU_ERR_INVALID_ARG
    for name in ("state", "state_out", "family", "family_out", "energy", "dbeta", "weight_sum", "energy_ref", "work"):
        assert run(**{name: None}) == bad, name
    assert run(n_chains=0, n_populations=1) == bad
    assert run(n_chains=-6) == bad
    assert run(n_populations=4) == bad             # does not divide n_chains
    assert run(n_populations=0) == bad
    assert run(n_chains=70000 * 2, n_populations=70000) == bad  # populations are a grid dimension
    assert run(row_bytes=0) == bad
    assert run(row_bytes=-16) == bad
    assert run(state_out=fake) == bad              # the output rows must be another buffer
    assert run(family_out=fake) == bad
    assert run(work_bytes=work - 8) == bad         # too small a workspace
    assert run(work=ctypes.c_void_p(260)) == bad   # not 8-byte aligned

    def moments(**kw):
        a = dict(dict(energy=fake, n_chains=6, n_populations=2, moments=fake2, stream=0), **kw)
        return lib.tsu_population_moments(*a.values())

    assert moments(energy=None) == bad
    assert moments(moments=None) == bad
    assert moments(n_chains=0, n_populations=1) == bad
    assert moments(n_populations=4) == bad
    assert moments(n_populations=0) == bad
    assert moments(n_chains=70000, n_populations=70000) == bad


@pytest.mark.parametrize("P,r_pop", [(1, 64), (3, 5), (4, 75), (2, 1)])
def test_resample_populations_equals_the_lattice_oracle_step(P, r_pop):
    """the tests' resampling step equals step 0 of the lattice oracle's population_anneal on its own energies: distinct
    family ids make the family after the step name every child's parent; W and E_ref are compared too"""
    rows, cols, J, h, periodic = 4, 4, 1.0, 0.25, True
    rng = np.random.default_rng(P * 100 + r_pop)
    n = P * r_pop
    nb = PO.n_bonds_of(rows, cols, periodic)
    for dbeta, chain0 in ((0.0, 0), (0.37, 12345), (2.5, 0xFFFFFFF0)):  # the last wraps chain0 + p R_p past 2^32
        states = [rng.integers(0, 2, (rows, cols)) for _ in range(n)]
        family = [int(f) for f in rng.permutation(1000)[:n]]
        energy = [PO.energy_of_counts(*PO.counts(b, periodic), J, h, nb, rows * cols) for b in states]
        parents, fam, W, e_ref = resample_populations(energy, family, dbeta, 99, chain0, 17, P)
        _, want_fam, want_W, want_ref, _, _ = PO.population_anneal(states, family, [1.0], [dbeta], 1, P, 99, chain0, 17,
                                                                   J, h, periodic)
        assert fam == want_fam and fam == [family[i] for i in parents]
        assert W == list(want_W[0]) and np.array_equal(e_ref, want_ref[0])
        if dbeta == 0.0:
            assert list(parents) == list(range(n))  # equal weights: every child is its own parent
            assert W == [r_pop << PO.weight_shift(r_pop)] * P
