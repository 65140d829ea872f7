"""GPU: Edwards-Anderson +-J lattices on the bit-packed kernels.  All-+1 bonds reproduce the ferromagnet's bits on every
launch path; random bonds reproduce the bonded oracle bit for bit (Philox and injected uniforms); per-replica
realisations, observables, overlaps, equilibrium moments and replica exchange are checked against host computations
and exact enumeration."""
import numpy as np
import pytest

from oracle import ising2d_bonds_oracle as B
from oracle import ising2d_oracle as O

pytestmark = pytest.mark.gpu


def make_engine(rows, cols, **kw):
    from tsu_emulator_b200.lattice import Ising2DEngine

    return Ising2DEngine(rows, cols, **kw)


def random_signs(rng, *shape):
    return rng.choice(np.array([-1, 1], dtype=np.int8), size=shape)


# ----------------------------------------------------------------------------- all bonds +1 == ferromagnet
# (rows, cols, periodic, n_replicas, knobs): every launch path the engine selects
LAUNCH_PATHS = [
    (50, 50, False, 2, {}),                                          # resident kernel
    (50, 50, False, 2, {"TSU_LATTICE_RESIDENT": "0"}),               # generic, one launch per half-sweep
    (12, 70, True, 3, {"TSU_LATTICE_RESIDENT": "0"}),
    (64, 512, True, 2, {"TSU_LATTICE_RESIDENT": "0"}),               # wide, W = 4
    (64, 512, True, 2, {"TSU_LATTICE_RESIDENT": "0", "TSU_LATTICE_W": "2"}),
    (64, 512, False, 2, {"TSU_LATTICE_RESIDENT": "0"}),              # wide + rim (open)
    (10, 300, True, 2, {"TSU_LATTICE_RESIDENT": "0"}),               # wide + rim (ragged)
    (9, 1000, False, 2, {"TSU_LATTICE_RESIDENT": "0", "TSU_LATTICE_W": "2"}),
    (64, 512, False, 2, {"TSU_LATTICE_RESIDENT": "0", "TSU_LATTICE_OPEN_GENERIC": "1"}),
    (1024, 256, True, 1, {"TSU_LATTICE_SPLIT": "4"}),                # row ranges on their own streams
    (1024, 256, False, 1, {"TSU_LATTICE_SPLIT": "4"}),
    (32, 256, True, 16, {"TSU_LATTICE_SPLIT": "4", "TSU_LATTICE_RESIDENT": "0"}),  # replica chunks
]


@pytest.mark.parametrize("rows,cols,periodic,n_rep,knobs", LAUNCH_PATHS)
def test_all_plus_bonds_equal_the_ferromagnet(rows, cols, periodic, n_rep, knobs, tuning):
    for k, v in knobs.items():
        tuning.setenv(k, v)
    kw = dict(n_replicas=n_rep, coupling=1.0, field=0.05, temperature=[2.0 + 0.1 * r for r in range(n_rep)],
              periodic=periodic, seed=31, replica0=3)
    ferro = make_engine(rows, cols, **kw)
    bonded = make_engine(rows, cols, bonds=np.ones((2, rows, cols), dtype=np.int8), **kw)
    ferro.init_random()
    bonded.state.copy_(ferro.state)
    ferro.sweep(3)
    bonded.sweep(3)
    assert (ferro.state == bonded.state).all()
    assert (ferro.observables_tensor() == bonded.observables_tensor()).all()
    # half-sweeps by row ranges, in any order
    for colour in (0, 1):
        for eng in (ferro, bonded):
            eng.half_sweep(colour, rows=(rows // 3, rows))
            eng.half_sweep(colour, rows=(0, rows // 3))
    assert (ferro.state == bonded.state).all()


# ----------------------------------------------------------------------------- random bonds == oracle
PHILOX_CASES = [
    (8, 256, True, 2.269, 1.0, 0.0),
    (6, 512, True, 0.1, 1.0, 0.0),      # p == 1.0 / 0.0 classes
    (10, 256, True, 1.0, 1.0, 0.25),
    (4, 768, True, 5.0, -1.0, 0.0),
    (50, 50, False, 1.5, 1.0, 0.0),
    (50, 50, True, 1.5, 1.0, 0.0),
    (7, 5, False, 1.0, 0.75, -0.25),
    (12, 70, True, 2.0, 1.0, 0.125),
    (2, 6, True, 3.0, 1.0, 0.0),        # periodic length 2: that wrap creates no bond
    (1, 9, False, 1.5, 1.0, 0.0),
    (9, 1, False, 1.5, 1.0, 0.25),
    (3, 130, False, 2.269, 1.0, 0.0),
    (10, 256, False, 2.269, 1.0, 0.0),  # wide + rim
    (64, 512, False, 1.0, 1.0, 0.125),
    (2, 256, False, 1.5, 1.0, 0.0),     # generic kernel
    (10, 300, True, 2.269, 1.0, 0.0),   # ragged
    (9, 1000, False, 2.0, 1.0, 0.1),
    (6, 2050, True, 2.5, -1.0, 0.0),
    (7, 257, False, 1.5, 1.0, 0.0),
    (8, 510, True, 2.0, 1.0, 0.2),
]


@pytest.mark.parametrize("resident", ["1", "0"])
@pytest.mark.parametrize("rows,cols,periodic,T,J,h", PHILOX_CASES)
def test_random_bonds_match_oracle(rows, cols, periodic, T, J, h, resident, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    rng = np.random.default_rng(rows * 7919 + cols)
    n_rep, n_sweeps, seed = 2, 3, 4321
    signs = random_signs(rng, 2, rows, cols)
    eng = make_engine(rows, cols, n_replicas=n_rep, coupling=J, field=h, temperature=T, periodic=periodic, seed=seed,
                      replica0=5, bonds=signs)
    eng.init_random()
    start = eng.get_spins(pm1=False)
    eng.sweep(n_sweeps)
    got = eng.get_spins(pm1=False)
    for r in range(n_rep):
        want = B.checkerboard_sweeps_philox_bonds(start[r], seed, 5 + r, 0, n_sweeps, J, h, T, periodic, signs)
        assert (got[r] == want).all(), f"replica {r}: {(got[r] != want).sum()} mismatching spins"
    obs = eng.observables_tensor().cpu().numpy()
    energy = eng.energy()
    for r in range(n_rep):
        assert obs[r, 0] == got[r].sum()
        assert obs[r, 1] == B.unsatisfied_bonds(got[r], periodic, signs)
        assert energy[r] == pytest.approx(B.energy_bonds(got[r], J, h, periodic, signs), abs=1e-9)


@pytest.mark.parametrize("rows,cols,periodic", [(6, 8, False), (12, 70, True), (5, 7, False), (2, 6, True), (16, 512, True)])
def test_injected_uniforms_match_oracle(rows, cols, periodic):
    rng = np.random.default_rng(rows + 3 * cols)
    J, h, T = 0.75, 0.125, 1.5
    signs = random_signs(rng, 2, rows, cols)
    bits0 = rng.integers(0, 2, (rows, cols))
    U = rng.integers(0, 2**32, (3, rows, cols), dtype=np.uint64).astype(np.uint32)
    eng = make_engine(rows, cols, coupling=J, field=h, temperature=T, periodic=periodic, bonds=signs)
    eng.set_spins(bits0)
    eng.sweep_injected(U)
    assert (eng.get_spins(pm1=False)[0] == B.checkerboard_sweeps_bonds(bits0, U, J, h, T, periodic, signs)).all()


def test_philox_and_injected_bonded_paths_agree():
    """bit-sliced wide kernel vs per-lane injected kernel on the same Philox uniforms"""
    rows, cols, seed = 16, 512, 9
    signs = random_signs(np.random.default_rng(2), 2, rows, cols)
    a = make_engine(rows, cols, temperature=1.2, seed=seed, bonds=signs)
    b = make_engine(rows, cols, temperature=1.2, seed=seed, bonds=signs)
    a.init_random()
    b.state.copy_(a.state)
    a.sweep(4)
    b.sweep_injected(np.stack([O.philox_uniform_field(seed, 0, t, rows, cols) for t in range(4)]))
    assert (a.state == b.state).all()


# ----------------------------------------------------------------------------- realisation per replica
@pytest.mark.parametrize("rows,cols,periodic,resident", [(12, 70, True, "1"), (64, 512, True, "0"), (9, 1000, False, "0")])
def test_per_replica_realisations_equal_single_realisation_engines(rows, cols, periodic, resident, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    rng = np.random.default_rng(rows)
    K, seed = 3, 77
    signs = random_signs(rng, K, 2, rows, cols)
    index = np.array([2, 0, 1, 2])
    temps = [1.0, 1.5, 2.0, 2.5]
    eng = make_engine(rows, cols, n_replicas=4, temperature=temps, periodic=periodic, seed=seed, bonds=signs,
                      bond_index=index)
    eng.init_random()
    start = eng.state.clone()
    eng.sweep(3)
    for r in range(4):
        one = make_engine(rows, cols, temperature=temps[r], periodic=periodic, seed=seed, replica0=r,
                          bonds=signs[index[r]])
        one.state.copy_(start[r:r + 1])
        one.sweep(3)
        assert (one.state[0] == eng.state[r]).all(), f"replica {r}"
    # chunk views keep each replica's realisation
    view = eng.chunk_view(1, 3)
    before = eng.state.clone()
    view.sweep(1)
    one = make_engine(rows, cols, temperature=temps[3], periodic=periodic, seed=seed, replica0=3, bonds=signs[index[3]])
    one.state.copy_(before[3:4])
    one.sweep_index = view.sweep_index - 1
    one.sweep(1)
    assert (one.state[0] == eng.state[3]).all()
    assert (eng.state[0] == before[0]).all()
    # K = n_replicas defaults to one realisation per replica
    per = make_engine(rows, cols, n_replicas=3, temperature=1.5, periodic=periodic, seed=seed, bonds=signs)
    assert per.bond_index.cpu().tolist() == [0, 1, 2]


# ----------------------------------------------------------------------------- observables
@pytest.mark.parametrize("rows,cols,periodic", [(16, 512, True), (16, 512, False), (6, 256, True), (5, 7, False), (2, 6, True)])
def test_observables_energy_and_overlap_are_exact(rows, cols, periodic, tuning):
    rng = np.random.default_rng(cols)
    n_rep, K = 6, 2
    signs = random_signs(rng, K, 2, rows, cols)
    index = np.array([0, 1, 1, 0, 1, 0])
    J, h = 0.75, -0.25
    eng = make_engine(rows, cols, n_replicas=n_rep, coupling=J, field=h, periodic=periodic, seed=3, bonds=signs,
                      bond_index=index)
    spins = rng.integers(0, 2, (n_rep, rows, cols))
    eng.set_spins(spins)
    obs = eng.observables_tensor().cpu().numpy().copy()
    tuning.setenv("TSU_LATTICE_OBS_GENERIC", "1")
    obs_generic = eng.observables_tensor().cpu().numpy().copy()
    assert (obs == obs_generic).all()
    et = eng.energy_tensor().cpu().numpy()
    for r in range(n_rep):
        s = signs[index[r]]
        assert obs[r, 0] == spins[r].sum()
        assert obs[r, 1] == B.unsatisfied_bonds(spins[r], periodic, s)
        assert et[r] == B.energy_bonds(spins[r], J, h, periodic, s)  # dyadic: exact
    pairs = np.array([[0, 1], [2, 2], [5, 3], [4, 0], [1, 5]])
    q = eng.overlap(pairs)
    for (a, b), qq in zip(pairs, q):
        sa, sb = 2 * spins[a] - 1, 2 * spins[b] - 1
        assert qq == pytest.approx((sa * sb).sum() / (rows * cols), abs=1e-15)
    assert (eng.chunk_view(2, 4).overlap(np.array([[3, 1]])) == q[2:3]).all()


# ----------------------------------------------------------------------------- statistics
def realisation_4x4():
    return random_signs(np.random.default_rng(2024), 2, 4, 4)


def test_moments_match_exact_enumeration():
    signs = realisation_4x4()
    J, h, T = 1.0, 0.0, 1.2
    mE, mE2, mq2 = B.exact_moments(4, 4, J, h, T, True, signs)
    n_rep = 8192
    eng = make_engine(4, 4, n_replicas=n_rep, coupling=J, field=h, temperature=T, periodic=True, seed=11, bonds=signs)
    eng.init_random()
    eng.sweep(400)
    E = eng.energy()
    pairs = np.stack([np.arange(0, n_rep, 2), np.arange(1, n_rep, 2)], axis=1)
    q2 = eng.overlap(pairs) ** 2
    for est, exact in [(E, mE), (E * E, mE2), (q2, mq2)]:
        se = est.std(ddof=1) / np.sqrt(len(est))
        assert abs(est.mean() - exact) < 5 * se + 1e-12, (est.mean(), exact, se)


def test_tempering_slot0_energy_matches_exact_enumeration():
    from tsu_emulator_b200.distributed import LatticeTempering

    signs = realisation_4x4()
    temps = [1.0, 1.4, 2.0, 3.0]
    mE = B.exact_moments(4, 4, 1.0, 0.0, temps[0], True, signs)[0]

    def fac(n_local, replica0, temps_local):
        return make_engine(4, 4, n_replicas=n_local, temperature=temps_local, periodic=True, seed=5, replica0=replica0,
                           bonds=signs)

    K = 512
    pt = LatticeTempering(temps, n_ladders=K, engine_factory=fac, n_sweeps=2, swap_interval=1, seed=7,
                          criterion="metropolis")
    for _ in range(100):
        pt.step()
    acc = np.zeros(K)
    n = 100
    for _ in range(n):
        pt.step()
        acc += pt.observables_by_slot()[1][:, 0]
    per_ladder = acc / n
    se = per_ladder.std(ddof=1) / np.sqrt(K)
    assert abs(per_ladder.mean() - mE) < 5 * se, (per_ladder.mean(), mE, se)
    assert int(pt.stats[0]) > 0  # exchanges were attempted
