"""GPU: simulated annealing on the bit-packed lattices (Ising2DEngine.anneal, tsu_ising2d_anneal).  One call equals, bit
for bit, the host loop set_temperature / sweep(1) / energy_tensor with the strict best update, on every launch path,
for the ferromagnet and +-J bonds; it equals the CPU oracle step for step; split calls and chunk views equal one call;
the best buffers are in/out; and small +-J instances reach their exactly enumerated ground states."""
import numpy as np
import pytest
import torch

from oracle import ising2d_bonds_oracle as B
from oracle import ising2d_oracle as O
from test_lattice_bonds_gpu import LAUNCH_PATHS, make_engine, random_signs

pytestmark = pytest.mark.gpu

SCHEDULE = [3.0, 2.0, 2.0, 1.2, 0.6, 0.3]  # a repeated temperature shares one table


def host_loop(eng, Ts, best_energy=None, best_state=None):
    """the loop anneal() replaces: (energy after each step, best_energy, best_state); the engine is advanced"""
    if best_energy is None:
        best_energy = torch.full((eng.n_replicas,), float("inf"), dtype=torch.float64, device=eng.device)
        best_state = torch.empty_like(eng.state)
    best_energy, best_state = best_energy.clone(), best_state.clone()
    energies = []

    def update():
        e = eng.energy_tensor()
        better = e < best_energy
        best_energy[better] = e[better]
        best_state[better] = eng.state[better]
        energies.append(e)

    update()
    for T in Ts:
        eng.set_temperature(T)
        eng.sweep(1)
        update()
    return energies, best_energy, best_state


MODELS = ["ferro", "bonds", "bonds_per_replica"]


def engine_kwargs(rows, cols, periodic, n_rep, model, bias_mode="physical"):
    kw = dict(n_replicas=n_rep, coupling=1.0, field=0.05, periodic=periodic, seed=31, replica0=3, bias_mode=bias_mode)
    rng = np.random.default_rng(rows * 131 + cols)
    if model == "bonds":
        kw["bonds"] = random_signs(rng, 2, rows, cols)
    elif model == "bonds_per_replica":
        kw["bonds"] = random_signs(rng, n_rep, 2, rows, cols)
    return kw


def twins(rows, cols, kw, n=2):
    engines = [make_engine(rows, cols, **kw) for _ in range(n)]
    engines[0].init_random()
    for e in engines[1:]:
        e.state.copy_(engines[0].state)
    return engines


def assert_same(res, energies, best_energy, best_state, eng, ref):
    assert torch.equal(eng.state, ref.state)
    assert eng.sweep_index == ref.sweep_index
    assert torch.equal(res.energy, energies[-1])
    assert torch.equal(res.best_energy, best_energy)
    assert torch.equal(res.best_state, best_state)


# the launch paths of the bonded tests, plus row ranges and an open chunked lattice with the resident kernel off
ANNEAL_PATHS = LAUNCH_PATHS + [
    (1024, 256, True, 1, {"TSU_LATTICE_SPLIT": "4", "TSU_LATTICE_RESIDENT": "0"}),
    (1024, 256, False, 1, {"TSU_LATTICE_SPLIT": "4", "TSU_LATTICE_RESIDENT": "0"}),
    (33, 300, False, 16, {"TSU_LATTICE_SPLIT": "4", "TSU_LATTICE_RESIDENT": "0"}),
]


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("rows,cols,periodic,n_rep,knobs", ANNEAL_PATHS)
def test_anneal_equals_host_loop(rows, cols, periodic, n_rep, knobs, model, tuning):
    for k, v in knobs.items():
        tuning.setenv(k, v)
    kw = engine_kwargs(rows, cols, periodic, n_rep, model)
    eng, ref, split = twins(rows, cols, kw, 3)
    eng.sweep_index = ref.sweep_index = split.sweep_index = 5
    res = eng.anneal(SCHEDULE)
    energies, best_energy, best_state = host_loop(ref, SCHEDULE)
    assert_same(res, energies, best_energy, best_state, eng, ref)
    assert eng.temperatures.tolist() == [SCHEDULE[-1]] and eng.lut_index is None
    # the same anneal in two calls that share the best buffers; each call's energies are the loop's at that point
    first = split.anneal(SCHEDULE[:2])
    assert torch.equal(first.energy, energies[2])
    again = split.anneal(SCHEDULE[2:], best=first)
    assert again is first
    assert_same(again, energies, best_energy, best_state, split, ref)


@pytest.mark.parametrize("resident", ["1", "0"])
@pytest.mark.parametrize("rows,cols,periodic,n_rep", [(12, 70, True, 3), (64, 512, False, 2)])
def test_reference_bias_equals_host_loop(rows, cols, periodic, n_rep, resident, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    eng, ref = twins(rows, cols, engine_kwargs(rows, cols, periodic, n_rep, "ferro", bias_mode="reference"))
    res = eng.anneal(SCHEDULE)
    assert_same(res, *host_loop(ref, SCHEDULE), eng, ref)


def test_track_best_false_writes_only_energy():
    kw = engine_kwargs(12, 70, True, 3, "bonds")
    eng, ref = twins(12, 70, kw)
    res = eng.anneal(SCHEDULE, track_best=False)
    energies, _, _ = host_loop(ref, SCHEDULE)
    assert res.best_energy is None and res.best_state is None
    assert torch.equal(res.energy, energies[-1]) and torch.equal(eng.state, ref.state)
    with pytest.raises(ValueError):
        res.best_spins()


# ----------------------------------------------------------------------------- CPU oracle
def anneal_philox(bits0, seed, replica, sweep0, Ts, J, h, periodic, signs=None):
    """per step: the oracle's Philox sweep at T_k, then E (energy / energy_bonds), then the strict best update;
    returns (final bits, final E, best E, best bits)"""
    def energy(b):
        return O.energy(b, J, h, periodic) if signs is None else B.energy_bonds(b, J, h, periodic, signs)

    bits = np.array(bits0, dtype=np.int64)
    e = best_e = energy(bits)
    best = bits.copy()
    for k, T in enumerate(Ts):
        if signs is None:
            bits = O.checkerboard_sweeps_philox(bits, seed, replica, sweep0 + k, 1, J, h, T, periodic)
        else:
            bits = B.checkerboard_sweeps_philox_bonds(bits, seed, replica, sweep0 + k, 1, J, h, T, periodic, signs)
        e = energy(bits)
        if e < best_e:
            best_e, best = e, bits.copy()
    return bits, e, best_e, best


@pytest.mark.parametrize("bonded", [False, True])
@pytest.mark.parametrize("resident", ["1", "0"])
@pytest.mark.parametrize("rows,cols,periodic", [(6, 8, True), (7, 5, False), (4, 70, True), (5, 66, False)])
def test_anneal_equals_cpu_oracle(rows, cols, periodic, resident, bonded, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    J, h, seed, n_rep, replica0 = 0.75, 0.25, 1234, 2, 7  # dyadic: every energy is exact
    signs = random_signs(np.random.default_rng(rows * cols), 2, rows, cols) if bonded else None
    eng = make_engine(rows, cols, n_replicas=n_rep, coupling=J, field=h, periodic=periodic, seed=seed,
                      replica0=replica0, bonds=signs)
    eng.init_random()
    eng.sweep_index = 3
    start = eng.get_spins(pm1=False)
    res = eng.anneal(SCHEDULE)
    got = eng.get_spins(pm1=False)
    best_bits = res.best_spins(pm1=False).cpu().numpy()
    for r in range(n_rep):
        bits, e, best_e, best = anneal_philox(start[r], seed, replica0 + r, 3, SCHEDULE, J, h, periodic, signs)
        assert (got[r] == bits).all(), f"replica {r}: {(got[r] != bits).sum()} mismatching spins"
        assert res.energy[r].item() == e
        assert res.best_energy[r].item() == best_e
        assert (best_bits[r] == best).all()


# ----------------------------------------------------------------------------- split calls and chunk views
@pytest.mark.parametrize("resident", ["1", "0"])
@pytest.mark.parametrize("model", MODELS)
def test_chunk_views_equal_the_whole_engine(model, resident, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    rows, cols, n_rep = 12, 70, 6
    whole, chunked = twins(rows, cols, engine_kwargs(rows, cols, True, n_rep, model))
    res = whole.anneal(SCHEDULE)
    for start, count in [(0, 2), (2, 3), (5, 1)]:
        view = chunked.chunk_view(start, count)
        part = view.anneal(SCHEDULE)
        sl = slice(start, start + count)
        assert torch.equal(part.energy, res.energy[sl])
        assert torch.equal(part.best_energy, res.best_energy[sl])
        assert torch.equal(part.best_state, res.best_state[sl])
    assert torch.equal(whole.state, chunked.state)


# ----------------------------------------------------------------------------- best buffers, with sentinels
SENTINEL = 0x5A5A5A5A


@pytest.mark.parametrize("resident", ["1", "0"])
def test_best_buffers_are_in_out(resident, tuning):
    from tsu_emulator_b200.lattice import AnnealResult

    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    rows, cols, n_rep = 12, 70, 3
    eng = make_engine(rows, cols, **engine_kwargs(rows, cols, True, n_rep, "bonds"))
    eng.init_random()

    def sentinels(value):
        return AnnealResult(None, torch.full((n_rep,), value, dtype=torch.float64, device=eng.device),
                            torch.full_like(eng.state, SENTINEL), rows, cols)

    # +inf: the initial state of every replica is copied
    start = eng.state.clone()
    r = eng.simulated_annealing(n_steps=0, best=sentinels(float("inf")))
    assert torch.equal(r.best_state, start) and torch.equal(r.best_energy, eng.energy_tensor())
    assert torch.equal(r.energy, r.best_energy) and eng.sweep_index == 0 and torch.equal(eng.state, start)
    # -inf: nothing is ever better, so best_state keeps its sentinel bytes
    r = eng.anneal(SCHEDULE, best=sentinels(float("-inf")))
    assert (r.best_state == SENTINEL).all() and (r.best_energy == float("-inf")).all()
    # an equal energy copies nothing
    eq = sentinels(0.0)
    eq.best_energy.copy_(eng.energy_tensor())
    r = eng.simulated_annealing(n_steps=0, best=eq)
    assert (r.best_state == SENTINEL).all() and torch.equal(r.best_energy, r.energy)


# ----------------------------------------------------------------------------- exact ground states
def exact_ground_energy(rows, cols, J, periodic, signs):
    """min over all 2^(rows cols) states of E = -J sum sigma s_i s_j (h = 0)"""
    a, b, g = B.bond_list(rows, cols, periodic, signs)
    idx = np.arange(1 << (rows * cols), dtype=np.uint32)
    unsat = np.zeros(idx.size, dtype=np.int16)
    for ai, bi, gi in zip(a, b, g):
        differ = ((idx >> np.uint32(ai)) ^ (idx >> np.uint32(bi))) & np.uint32(1)
        unsat += (differ == (1 if gi > 0 else 0)).astype(np.int16)
    return float(-J * (len(g) - 2 * int(unsat.min())))


@pytest.mark.parametrize("rows,cols,periodic,seed", [(4, 6, False, 11), (4, 4, True, 12)])
def test_anneal_reaches_exact_ground_state(rows, cols, periodic, seed):
    J, n_rep = 1.0, 512
    signs = random_signs(np.random.default_rng(seed), 2, rows, cols)
    eng = make_engine(rows, cols, n_replicas=n_rep, coupling=J, periodic=periodic, seed=seed, bonds=signs)
    eng.init_random()
    res = eng.simulated_annealing(T_initial=3.0, T_final=0.05, n_steps=400)
    best_e = res.best_energy.cpu().numpy()
    assert best_e.min() == exact_ground_energy(rows, cols, J, periodic, signs)
    bits = res.best_spins(pm1=False).cpu().numpy()
    for r in range(n_rep):
        assert B.energy_bonds(bits[r], J, 0.0, periodic, signs) == best_e[r]
