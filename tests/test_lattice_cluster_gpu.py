"""GPU: Swendsen-Wang cluster updates on the bit-packed lattices (Ising2DEngine.swendsen_wang, tsu_ising2d_swendsen_wang).
States equal the CPU oracle (oracle/cluster_oracle.py) bit for bit on periodic, open and ragged lattices, for J = +-1,
shared and per-replica +-J bonds, on the one-launch and the multi-launch path; per-replica temperatures, split calls,
chunk views and workspace chunks give the same bits; adversarial domains at 4096^2 flip whole; the moments of small
lattices match exact enumeration."""
import numpy as np
import pytest
import torch

from oracle import cluster_oracle as SW
from test_lattice_bonds_gpu import make_engine, random_signs

pytestmark = pytest.mark.gpu

TEMPS = [1.0, 2.269, 5.0, 0.02]  # one per replica; T = 0.02 gives p = 1
SMALL = [(8, 8, True), (16, 64, True), (50, 50, True), (33, 70, False), (17, 31, False), (1, 40, False),
         (40, 1, False), (64, 130, True), (2, 16, True)]
MODELS = ["ferro", "antiferro", "bonds", "bonds_per_replica"]


def cluster_engine(rows, cols, periodic, model, n_rep=len(TEMPS), seed=77, replica0=5, temps=TEMPS):
    kw = dict(n_replicas=n_rep, coupling=-1.0 if model == "antiferro" else 1.0, periodic=periodic, seed=seed,
              replica0=replica0, temperature=temps)
    rng = np.random.default_rng(rows * 97 + cols)
    signs = None
    if model == "bonds":
        signs = random_signs(rng, 2, rows, cols)
        kw["bonds"] = signs
    elif model == "bonds_per_replica":
        signs = list(random_signs(rng, n_rep, 2, rows, cols))
        kw["bonds"] = np.stack(signs)
    eng = make_engine(rows, cols, **kw)
    eng.init_random()
    return eng, signs


def check_against_oracle(eng, periodic, signs, temps, steps):
    """runs the engine through `steps` (cumulative step counts) and compares with the oracle after each"""
    x = eng.get_spins(pm1=False)
    done = 0
    for n in steps:
        sweep0 = eng.sweep_index
        eng.swendsen_wang(n - done)
        x = SW.sw_steps(x, eng.coupling, temps, periodic, eng.seed, eng.replica0, sweep0, n - done, signs)
        got = eng.get_spins(pm1=False)
        for r in range(eng.n_replicas):
            assert (got[r] == x[r]).all(), f"after {n} steps, replica {r}: {(got[r] != x[r]).sum()} sites differ"
        done = n


@pytest.mark.parametrize("resident", ["1", "0"])
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("rows,cols,periodic", SMALL)
def test_small_lattices_equal_oracle(rows, cols, periodic, model, resident, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    eng, signs = cluster_engine(rows, cols, periodic, model)
    eng.sweep_index = 3
    check_against_oracle(eng, periodic, signs, TEMPS, [1, 5])


@pytest.mark.parametrize("rows,cols,periodic,model,steps", [
    (256, 320, True, "ferro", [1, 5]),
    (256, 320, True, "bonds", [1, 5]),
    (300, 1030, False, "ferro", [1, 5]),            # merges across 10 x 5 tiles, open edges
    (300, 1030, False, "bonds_per_replica", [1, 3]),
    (1024, 1024, True, "ferro", [1, 2]),            # T_c: clusters spanning both wraps
])
def test_large_lattices_equal_oracle(rows, cols, periodic, model, steps):
    temps = [2.269, 1.0]
    eng, signs = cluster_engine(rows, cols, periodic, model, n_rep=2, temps=temps)
    check_against_oracle(eng, periodic, signs, temps, steps)


@pytest.mark.parametrize("resident", ["1", "0"])
def test_per_replica_temperatures_equal_single_temperature_engines(resident, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    rows, cols = 48, 64
    eng, _ = cluster_engine(rows, cols, True, "ferro")
    start = eng.state.clone()
    eng.swendsen_wang(4)
    for r, T in enumerate(TEMPS):
        one = make_engine(rows, cols, n_replicas=1, temperature=T, periodic=True, seed=eng.seed,
                          replica0=eng.replica0 + r)
        one.state.copy_(start[r:r + 1])
        one.swendsen_wang(4)
        assert torch.equal(one.state[0], eng.state[r])
    # permuted tables, as replica exchange leaves them
    tab, _ = cluster_engine(rows, cols, True, "ferro")
    tab.state.copy_(start)
    tab.set_temperature_tables([5.0, 0.02, 1.0, 2.269], torch.tensor([2, 3, 0, 1], dtype=torch.int32))
    tab.swendsen_wang(4)
    assert torch.equal(tab.state, eng.state)


@pytest.mark.parametrize("rows,cols", [(50, 50), (100, 300)])
def test_split_calls_chunk_views_and_workspace_chunks_equal_one_call(rows, cols, monkeypatch):
    import tsu_emulator_b200.lattice as lattice

    whole, _ = cluster_engine(rows, cols, True, "bonds_per_replica")
    start = whole.state.clone()
    whole.swendsen_wang(5)
    split, _ = cluster_engine(rows, cols, True, "bonds_per_replica")
    split.swendsen_wang(2).swendsen_wang(3)
    assert torch.equal(split.state, whole.state) and split.sweep_index == 5
    views, _ = cluster_engine(rows, cols, True, "bonds_per_replica")
    views.chunk_view(0, 1).swendsen_wang(5)
    views.chunk_view(1, 3).swendsen_wang(5)
    assert torch.equal(views.state, whole.state)
    monkeypatch.setattr(lattice, "CLUSTER_WORK_BUDGET", 1)  # one replica at a time
    chunked, _ = cluster_engine(rows, cols, True, "bonds_per_replica")
    assert torch.equal(chunked.state, start)
    chunked.swendsen_wang(5)
    assert chunked._cluster_work.numel() * 8 == int(chunked.lib.tsu_ising2d_cluster_work_bytes(1, rows, cols))
    assert torch.equal(chunked.state, whole.state)


def adversarial_domains(L):
    i, j = np.meshgrid(np.arange(L), np.arange(L), indexing="ij")
    serpentine = np.ones((L, L), dtype=np.int64)
    walls = i % 2 == 1
    gap = np.where(i % 4 == 1, j == L - 1, j == 0)
    serpentine[walls & ~gap] = 0
    blocks = ((i // 37 + j // 53) % 2).astype(np.int64)  # not aligned to tiles; merged again across the wraps
    stripes = (((i + j) // 16) % 2).astype(np.int64)     # diagonal stripes spanning both wraps
    return np.stack([serpentine, blocks, stripes])


def test_adversarial_domains_flip_whole_at_p_one():
    L = 4096
    x = adversarial_domains(L)
    eng = make_engine(L, L, n_replicas=3, temperature=0.02, periodic=True, seed=5, replica0=11)
    eng.set_spins(x)
    eng.sweep_index = 8
    eng.swendsen_wang(1)
    got = eng.get_spins(pm1=False)
    a, b, _, _ = SW.bonds(L, L, True)
    for r in range(3):
        root = SW.roots(L * L, a, b, SW.satisfied(x[r], 1.0, True))  # p = 1: the clusters are the domains
        want = x[r] ^ SW.flip_bits(eng.seed, eng.replica0 + r, 8, L, L).reshape(-1)[root].reshape(L, L)
        assert (got[r] == want).all(), f"pattern {r}: {(got[r] != want).sum()} sites differ"
    # J = 0: no bond is active, every site is its own root and flips by its own kind-4 bit
    free = make_engine(L, L, n_replicas=1, coupling=0.0, temperature=1.0, periodic=True, seed=5, replica0=11)
    free.set_spins(x[2])
    free.swendsen_wang(1)
    assert (free.get_spins(pm1=False)[0] == x[2] ^ SW.flip_bits(5, 11, 0, L, L)).all()


def exact_m2(rows, cols, J, T, periodic, signs):
    """exact <E>, <E^2>, <M^2> (M = sum of spins) by enumeration"""
    n = rows * cols
    s = 2 * ((np.arange(1 << n)[:, None] >> np.arange(n)[None, :]) & 1) - 1
    a, b, g, _ = SW.bonds(rows, cols, periodic, signs)
    E = -J * (g[None, :] * s[:, a] * s[:, b]).sum(axis=1)
    w = np.exp(-(E - E.min()) / T)
    w /= w.sum()
    M = s.sum(axis=1)
    return (w * E).sum(), (w * E * E).sum(), (w * M * M).sum()


@pytest.mark.parametrize("with_sweeps", [False, True])
@pytest.mark.parametrize("model", ["ferro", "bonds"])
def test_moments_match_exact_enumeration(model, with_sweeps):
    rows = cols = 4
    J, T, n_rep = 1.0, 2.0 if model == "ferro" else 1.2, 8192
    signs = random_signs(np.random.default_rng(2024), 2, rows, cols) if model == "bonds" else None
    eng = make_engine(rows, cols, n_replicas=n_rep, coupling=J, temperature=T, periodic=True, seed=13, bonds=signs)
    eng.init_random()
    for _ in range(400):  # SW mixes slowly on the frustrated realisation
        eng.swendsen_wang(1)
        if with_sweeps:
            eng.sweep(1)
    E = eng.energy()
    M = eng.magnetization() * rows * cols
    for got, want in zip([E, E * E, M * M], exact_m2(rows, cols, J, T, True, signs)):
        assert abs(got.mean() - want) < 5 * got.std() / np.sqrt(n_rep), (got.mean(), want)


def test_stream_position_after_cluster_steps():
    eng, _ = cluster_engine(64, 130, True, "ferro")
    eng.sweep_index = 10
    eng.swendsen_wang(3)
    assert eng.sweep_index == 13
    fresh = make_engine(64, 130, n_replicas=len(TEMPS), periodic=True, seed=eng.seed, replica0=eng.replica0,
                        temperature=TEMPS)
    fresh.state.copy_(eng.state)
    fresh.sweep_index = 13
    eng.sweep(1)
    fresh.sweep(1)
    assert torch.equal(eng.state, fresh.state)
