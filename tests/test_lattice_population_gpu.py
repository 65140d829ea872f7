"""GPU: population annealing on the bit-packed lattices (Ising2DEngine.population_annealing,
tsu_ising2d_population_anneal).  States, families, weight sums, reference energies, count sums and energies equal the
CPU oracle bit for bit; a constant temperature equals plain sweeps on every launch path; split calls and chunk views of
whole populations equal one call; free energies and mean energies match exact enumeration."""
import math

import numpy as np
import pytest
import torch

from oracle import population_oracle as PA
from test_lattice_anneal_gpu import MODELS, engine_kwargs, twins
from test_lattice_bonds_gpu import LAUNCH_PATHS, make_engine, random_signs, realisation_4x4

pytestmark = pytest.mark.gpu

SCHEDULE = [3.0, 1.5, 0.4]  # from T_start = inf; the last step's dbeta (1.83) duplicates or drops most replicas


def population_engine(rows, cols, periodic, P, r_pop, model, J=1.0, h=0.3, seed=1234, replica0=7):
    n = P * r_pop
    kw = dict(n_replicas=n, coupling=J, field=h, periodic=periodic, seed=seed, replica0=replica0)
    signs = None
    rng = np.random.default_rng(rows * 31 + cols + P)
    if model == "bonds":
        signs = [random_signs(rng, 2, rows, cols)] * P
        kw["bonds"] = signs[0]
    elif model == "bonds_per_population":
        signs = list(random_signs(rng, P, 2, rows, cols))
        kw["bonds"] = np.stack(signs)
        kw["bond_index"] = np.repeat(np.arange(P), r_pop)
    return make_engine(rows, cols, **kw), signs


def assert_equals_oracle(res, eng, start, family0, Ts, T_start, theta, P, sweep0, periodic, signs):
    dbeta = np.diff(np.concatenate([[0.0 if math.isinf(T_start) else 1.0 / T_start], 1.0 / np.asarray(Ts)]))
    states, family, W, e_ref, sums, energy = PA.population_anneal(
        start, family0, Ts, dbeta, theta, P, eng.seed, eng.replica0, sweep0, eng.coupling, eng.field, periodic, signs)
    got = eng.get_spins(pm1=False)
    for r in range(eng.n_replicas):
        assert (got[r] == states[r]).all(), f"replica {r}: {(got[r] != states[r]).sum()} mismatching spins"
    assert res.family.cpu().tolist() == family
    assert res.weight_sum.cpu().tolist() == W.tolist()
    assert res.energy_ref.cpu().tolist() == e_ref.tolist()
    assert res.count_sums.cpu().tolist() == sums.tolist()
    assert res.energy.cpu().tolist() == energy.tolist()
    return family


@pytest.mark.parametrize("P,r_pop", [(3, 1), (2, 3), (1, 64)])
@pytest.mark.parametrize("resident", ["1", "0"])
@pytest.mark.parametrize("model", ["ferro", "bonds", "bonds_per_population"])
@pytest.mark.parametrize("rows,cols,periodic", [(6, 8, True), (7, 5, False), (4, 70, True)])
def test_population_anneal_equals_cpu_oracle(rows, cols, periodic, model, resident, P, r_pop, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    eng, signs = population_engine(rows, cols, periodic, P, r_pop, model)
    eng.init_random()
    eng.sweep_index = 5
    start = list(eng.get_spins(pm1=False))
    theta = 2
    res = eng.population_annealing(SCHEDULE, sweeps_per_step=theta, n_populations=P)
    family = assert_equals_oracle(res, eng, start, [eng.replica0 + r for r in range(eng.n_replicas)], SCHEDULE,
                                  math.inf, theta, P, 5, periodic, signs)
    assert eng.sweep_index == 5 + theta * len(SCHEDULE) and eng.temperatures.tolist() == [SCHEDULE[-1]]
    if r_pop == 64:
        assert len(set(family)) < 32  # most replicas were duplicated or dropped
        assert res.rho_t()[0] > 2.0


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("rows,cols,periodic,n_rep,knobs", LAUNCH_PATHS)
def test_constant_temperature_equals_sweeps(rows, cols, periodic, n_rep, knobs, model, tuning):
    for k, v in knobs.items():
        tuning.setenv(k, v)
    kw = engine_kwargs(rows, cols, periodic, n_rep, model)
    eng, ref = twins(rows, cols, kw)
    eng.sweep_index = ref.sweep_index = 9
    T, n_steps, theta = 2.0, 3, 2
    P = n_rep if model == "bonds_per_replica" else 1
    res = eng.population_annealing([T] * n_steps, sweeps_per_step=theta, n_populations=P, T_start=T)
    ref.set_temperature(T)
    ref.sweep(n_steps * theta)
    assert torch.equal(eng.state, ref.state) and eng.sweep_index == ref.sweep_index
    assert res.family.cpu().tolist() == list(range(kw["replica0"], kw["replica0"] + n_rep))
    assert (res.weight_sum.cpu() == (n_rep // P) << res.shift).all()
    assert torch.equal(res.energy, ref.energy_tensor())


@pytest.mark.parametrize("resident", ["1", "0"])
def test_split_calls_equal_one_call(resident, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    P, r_pop, Ts = 2, 16, [4.0, 2.0, 1.5, 1.0, 0.6]
    one, _ = population_engine(12, 70, True, P, r_pop, "bonds_per_population")
    split, _ = population_engine(12, 70, True, P, r_pop, "bonds_per_population")
    one.init_random()
    split.state.copy_(one.state)
    whole = one.population_annealing(Ts, sweeps_per_step=3, n_populations=P)
    first = split.population_annealing(Ts[:2], sweeps_per_step=3, n_populations=P)
    second = split.population_annealing(Ts[2:], sweeps_per_step=3, n_populations=P, previous=first)
    assert second.family is first.family and second.T_start == Ts[1]
    assert torch.equal(one.state, split.state) and one.sweep_index == split.sweep_index
    assert torch.equal(whole.family, second.family) and torch.equal(whole.energy, second.energy)
    assert torch.equal(whole.weight_sum, torch.cat([first.weight_sum, second.weight_sum]))
    assert torch.equal(whole.energy_ref, torch.cat([first.energy_ref, second.energy_ref]))
    assert torch.equal(whole.count_sums, torch.cat([first.count_sums[:-1], second.count_sums]))
    assert np.allclose(whole.log_z_ratio()[2:], whole.log_z_ratio()[1] + second.log_z_ratio(), rtol=1e-13, atol=0)


@pytest.mark.parametrize("resident", ["1", "0"])
@pytest.mark.parametrize("model", ["ferro", "bonds_per_population"])
def test_chunk_views_of_whole_populations_equal_the_whole_run(model, resident, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    P, r_pop, Ts = 4, 8, [3.0, 1.0, 0.5]
    whole, _ = population_engine(12, 70, True, P, r_pop, model)
    chunked, _ = population_engine(12, 70, True, P, r_pop, model)
    whole.init_random()
    chunked.state.copy_(whole.state)
    res = whole.population_annealing(Ts, sweeps_per_step=2, n_populations=P)
    for p0, count in [(0, 1), (1, 2), (3, 1)]:
        view = chunked.chunk_view(p0 * r_pop, count * r_pop)
        part = view.population_annealing(Ts, sweeps_per_step=2, n_populations=count)
        sl = slice(p0 * r_pop, (p0 + count) * r_pop)
        assert torch.equal(part.family, res.family[sl]) and torch.equal(part.energy, res.energy[sl])
        assert torch.equal(part.weight_sum, res.weight_sum[:, p0:p0 + count])
        assert torch.equal(part.energy_ref, res.energy_ref[:, p0:p0 + count])
        assert torch.equal(part.count_sums, res.count_sums[:, p0:p0 + count])
    assert torch.equal(whole.state, chunked.state)


# ----------------------------------------------------------------------------- statistics
@pytest.mark.parametrize("case", ["pm_j_periodic", "ferro_open_field"])
def test_free_energy_and_mean_energy_match_exact_enumeration(case):
    if case == "pm_j_periodic":
        signs, J, h, periodic = realisation_4x4(), 1.0, 0.0, True
    else:
        signs, J, h, periodic = None, 1.0, 0.25, False
    P, r_pop = 32, 2048
    betas = 2.0 * np.arange(1, 51) / 50  # T from 25 down to 0.5
    Ts = 1.0 / betas
    eng = make_engine(4, 4, n_replicas=P * r_pop, coupling=J, field=h, periodic=periodic, seed=3, bonds=signs)
    eng.init_random()
    res = eng.population_annealing(Ts, sweeps_per_step=10, n_populations=P)
    # 65536 replicas without full words: counted one warp per replica; the observables kernels take halves
    half = P * r_pop // 2
    assert torch.equal(res.energy, torch.cat([eng.chunk_view(0, half).energy_tensor(),
                                              eng.chunk_view(half, half).energy_tensor()]))
    f = res.free_energy()
    for k in (9, 24, 49):
        lz, _ = PA.exact_log_partition(4, 4, J, h, Ts[k], periodic, signs)
        exact = -Ts[k] * lz / 16
        se = f[k].std(ddof=1) / np.sqrt(P)
        assert abs(f[k].mean() - exact) < 5 * se + 1e-12, (k, f[k].mean(), exact, se)
    mE = res.mean_energy()[-1]
    exact_E = PA.exact_log_partition(4, 4, J, h, Ts[-1], periodic, signs)[1]
    se = mE.std(ddof=1) / np.sqrt(P)
    assert abs(mE.mean() - exact_E) < 5 * se + 1e-12, (mE.mean(), exact_E, se)
    assert (res.rho_t() >= 1.0).all()
