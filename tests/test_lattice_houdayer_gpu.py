"""GPU: Houdayer cluster moves on the bit-packed lattices (Ising2DEngine.houdayer, tsu_ising2d_houdayer,
LatticeTempering(houdayer_interval=)).  States equal the CPU oracle (oracle/houdayer_oracle.py) bit for bit on periodic,
open, ragged and single-row/column lattices, for the ferromagnet, shared and per-pair +-J bonds with a field, on the
one-launch and the multi-launch path, with pairs in any order; split calls, chunk views, a one-pair workspace and
interleaving with swendsen_wang give the same bits; skipped pairs leave their replicas alone; E_a + E_b and q_ab are
kept at 4096^2; adversarial difference patterns at 4096^2 flip whole; the moments of 4 x 4 +-J lattices and the slot-0
energy of replica exchange with Houdayer moves match exact enumeration."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import cluster_oracle as SW
from oracle import houdayer_oracle as H
from oracle import ising2d_bonds_oracle as B
from test_lattice_bonds_gpu import make_engine, random_signs, realisation_4x4
from test_lattice_cluster_gpu import adversarial_domains

pytestmark = pytest.mark.gpu

PAIRS = [(3, 0), (1, 2), (5, 4)]       # any order; replica 6 is in no pair
TEMPS = [1.0, 2.0, 2.0, 1.0, 0.5, 0.5, 3.0]
SMALL = [(8, 8, True), (16, 64, True), (50, 50, True), (33, 70, False), (17, 31, False), (1, 40, False),
         (40, 1, False), (64, 130, True), (2, 16, True)]
MODELS = ["ferro", "bonds", "bonds_per_pair"]


def pair_engine(rows, cols, periodic, model, temps=TEMPS, pairs=PAIRS, seed=77, replica0=5, field=0.3):
    """engine with one temperature and one bond realisation per pair; pair 0 starts from independent random states,
    the others from states that differ on a dense random pattern (the differing sites percolate)"""
    n_rep = len(temps)
    kw = dict(n_replicas=n_rep, periodic=periodic, seed=seed, replica0=replica0, temperature=temps, field=field)
    rng = np.random.default_rng(rows * 97 + cols)
    signs = None
    if model == "bonds":
        signs = random_signs(rng, 2, rows, cols)
        kw["bonds"] = signs
    elif model == "bonds_per_pair":
        real = list(random_signs(rng, len(pairs) + 1, 2, rows, cols))
        idx = np.full(n_rep, len(pairs), dtype=np.int32)
        for q, (a, b) in enumerate(pairs):
            idx[a] = idx[b] = q
        kw["bonds"], kw["bond_index"] = np.stack(real), idx
    eng = make_engine(rows, cols, **kw)
    x = rng.integers(0, 2, (n_rep, rows, cols))
    for a, b in pairs[1:]:
        x[b] = x[a] ^ (rng.random((rows, cols)) < 0.7)
    eng.set_spins(x)
    return eng, signs


def check_against_oracle(eng, periodic, pairs, steps):
    """runs the engine through `steps` (cumulative step counts) and compares with the oracle after each"""
    x = eng.get_spins(pm1=False)
    done = 0
    for n in steps:
        sweep0 = eng.sweep_index
        eng.houdayer(pairs, n - done)
        assert eng.sweep_index == sweep0 + n - done
        x = H.houdayer_steps(x, pairs, periodic, eng.seed, eng.replica0, sweep0, n - done)
        got = eng.get_spins(pm1=False)
        for r in range(eng.n_replicas):
            assert (got[r] == x[r]).all(), f"after {n} steps, replica {r}: {(got[r] != x[r]).sum()} sites differ"
        done = n


@pytest.mark.parametrize("resident", ["1", "0"])
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("rows,cols,periodic", SMALL)
def test_small_lattices_equal_oracle(rows, cols, periodic, model, resident, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    eng, _ = pair_engine(rows, cols, periodic, model)
    eng.sweep_index = 3
    start = eng.get_spins(pm1=False)
    check_against_oracle(eng, periodic, PAIRS, [1, 5])
    assert (eng.get_spins(pm1=False)[6] == start[6]).all()


@pytest.mark.parametrize("rows,cols,periodic,model,steps", [
    (256, 320, True, "ferro", [1, 5]),
    (256, 320, True, "bonds", [1, 5]),
    (300, 1030, False, "ferro", [1, 5]),            # merges across 10 x 5 tiles, open edges
    (300, 1030, False, "bonds_per_pair", [1, 3]),
    (1024, 1024, True, "bonds", [1, 2]),            # percolating differences spanning both wraps
])
def test_large_lattices_equal_oracle(rows, cols, periodic, model, steps):
    pairs = [(1, 0), (2, 3)]
    eng, _ = pair_engine(rows, cols, periodic, model, temps=[0.5, 0.5, 1.0, 1.0], pairs=pairs)
    check_against_oracle(eng, periodic, pairs, steps)


PAIRS8 = [(3, 0), (1, 2), (4, 7), (6, 5)]
TEMPS8 = [1.0, 2.0, 2.0, 1.0, 0.7, 0.9, 0.9, 0.7]


@pytest.mark.parametrize("rows,cols", [(50, 50), (100, 300)])
def test_split_calls_chunk_views_and_workspace_chunks_equal_one_call(rows, cols, monkeypatch):
    import tsu_emulator_b200.lattice as lattice

    def fresh():
        return pair_engine(rows, cols, True, "bonds_per_pair", temps=TEMPS8, pairs=PAIRS8)[0]

    whole = fresh()
    start = whole.state.clone()
    whole.houdayer(PAIRS8, 5)
    split = fresh()
    split.houdayer(PAIRS8, 2).houdayer(PAIRS8, 3)
    assert torch.equal(split.state, whole.state) and split.sweep_index == 5
    views = fresh()
    views.chunk_view(0, 4).houdayer([(3, 0), (1, 2)], 5)
    views.chunk_view(4, 4).houdayer([(0, 3), (2, 1)], 5)
    assert torch.equal(views.state, whole.state)
    monkeypatch.setattr(lattice, "CLUSTER_WORK_BUDGET", 1)  # one pair at a time
    chunked = fresh()
    assert torch.equal(chunked.state, start)
    chunked.houdayer(PAIRS8, 5)
    assert chunked._cluster_work.numel() * 8 == int(chunked.lib.tsu_ising2d_cluster_work_bytes(1, rows, cols))
    assert torch.equal(chunked.state, whole.state)


@pytest.mark.parametrize("resident", ["1", "0"])
def test_interleaved_with_swendsen_wang_on_the_shared_workspace(resident, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    rows, cols = 48, 64
    eng, signs = pair_engine(rows, cols, True, "bonds", temps=TEMPS8, pairs=PAIRS8, field=0.0)
    x = eng.get_spins(pm1=False)
    eng.houdayer(PAIRS8, 2)                 # the workspace is sized for 4 pairs ...
    eng.swendsen_wang(1)                    # ... then grown for 8 replicas
    work = eng._cluster_work
    eng.houdayer(PAIRS8, 1)
    assert eng._cluster_work is work        # and shared from then on
    eng.swendsen_wang(2)
    x = H.houdayer_steps(x, PAIRS8, True, eng.seed, eng.replica0, 0, 2)
    x = SW.sw_steps(x, 1.0, TEMPS8, True, eng.seed, eng.replica0, 2, 1, signs)
    x = H.houdayer_steps(x, PAIRS8, True, eng.seed, eng.replica0, 3, 1)
    x = SW.sw_steps(x, 1.0, TEMPS8, True, eng.seed, eng.replica0, 4, 2, signs)
    assert (eng.get_spins(pm1=False) == x).all()
    assert eng.sweep_index == 6


@pytest.mark.parametrize("rows,cols", [(20, 30), (130, 200)])
def test_skipped_pairs_leave_their_replicas_alone(rows, cols):
    """pairs outside [0, n_replicas) or with a == b are skipped by the kernels.  The call sees replicas 1..8 of a
    ten-replica state, so the skipped indices -1 and 8 still name memory of the state (replicas 0 and 9)"""
    from tsu_emulator_b200 import _lib
    from tsu_emulator_b200._lib import ptr

    eng, _ = pair_engine(rows, cols, False, "ferro", temps=[1.0] * 10, pairs=[(1, 2), (3, 4), (0, 9)])
    x = eng.get_spins(pm1=False)
    pairs = [(0, 1), (-1, 2), (3, 3), (4, 8)]   # kept: (0, 1) only
    dev = torch.tensor(pairs, dtype=torch.int32, device=eng.device)
    work = torch.empty(4 * int(eng.lib.tsu_ising2d_cluster_work_bytes(1, rows, cols)) // 8, dtype=torch.int64,
                       device=eng.device)
    rc = eng.lib.tsu_ising2d_houdayer(ctypes.c_void_p(ptr(eng.state[1:9])), 8, rows, cols, 0, 0,
                                      ctypes.c_void_p(ptr(dev)), 4, eng.seed, 7, 2, eng.replica0 + 1,
                                      ctypes.c_void_p(ptr(work)), work.numel() * 8, _lib.current_stream())
    assert rc == _lib.TSU_OK
    want = x.copy()
    want[1:9] = H.houdayer_steps(x[1:9], [(0, 1)], False, eng.seed, eng.replica0 + 1, 7, 2)
    got = eng.get_spins(pm1=False)
    assert not (want[1] == x[1]).all()
    for r in range(10):
        assert (got[r] == want[r]).all(), r


def pair_sums(eng, pairs):
    obs = eng.observables_tensor().cpu().numpy()
    a, b = np.asarray(pairs).T
    return obs[a] + obs[b], eng.overlap(pairs)


def test_energy_sums_and_overlaps_are_kept_at_4096():
    L = 4096
    pairs = [(0, 1), (3, 2)]
    signs = random_signs(np.random.default_rng(8), 2, L, L)
    eng = make_engine(L, L, n_replicas=4, temperature=0.4, field=0.3, periodic=True, seed=3, bonds=signs)
    rng = np.random.default_rng(9)
    x = rng.integers(0, 2, (4, L, L), dtype=np.int8)
    x[2] = x[3] ^ (rng.random((L, L)) < 0.7)   # percolating differences
    eng.set_spins(x)
    sums0, q0 = pair_sums(eng, pairs)
    E0 = eng.energy()
    eng.houdayer(pairs, 1)
    sums1, q1 = pair_sums(eng, pairs)
    assert (sums1 == sums0).all() and (q1 == q0).all()  # integer (up, unsatisfied) counts and q_ab, exactly
    E1 = eng.energy()
    assert not np.array_equal(E0, E1)  # each replica's own energy changes


def test_adversarial_differences_flip_whole_at_4096():
    L = 4096
    d = adversarial_domains(L)  # serpentine, tile-misaligned blocks, diagonal stripes across both wraps
    base = np.random.default_rng(10).integers(0, 2, (3, L, L), dtype=np.int64)
    x = np.empty((6, L, L), dtype=np.int64)
    x[0::2] = base ^ d
    x[1::2] = base
    pairs = [(0, 1), (3, 2), (4, 5)]
    eng = make_engine(L, L, n_replicas=6, temperature=1.0, periodic=True, seed=5, replica0=11)
    eng.set_spins(x)
    eng.sweep_index = 8
    eng.houdayer(pairs, 1)
    got = eng.get_spins(pm1=False)
    for a, b in pairs:
        ya, yb = H.pair_step(x[a], x[b], True, eng.seed, eng.replica0 + a, 8)
        assert (got[a] == ya).all() and (got[b] == yb).all(), f"pair {(a, b)} differs from the oracle"
    assert not (got == x).all()


@pytest.mark.parametrize("h", [0.0, 0.2])
def test_moments_match_exact_enumeration(h):
    signs = realisation_4x4()
    J, T, n_pairs = 1.0, 1.0, 4096
    eng = make_engine(4, 4, n_replicas=2 * n_pairs, coupling=J, field=h, temperature=T, periodic=True, seed=13,
                      bonds=signs)
    eng.init_random()
    pairs = np.arange(2 * n_pairs).reshape(n_pairs, 2)
    for _ in range(500):
        eng.sweep(1)
        eng.houdayer(pairs, 1)
    E = eng.energy()
    q = eng.overlap(pairs)
    for est, exact in zip([E, E * E, q * q], B.exact_moments(4, 4, J, h, T, True, signs)):
        se = est.std(ddof=1) / np.sqrt(len(est))
        assert abs(est.mean() - exact) < 5 * se + 1e-12, (est.mean(), exact, se)


def tempering(K, R_temps, signs, houdayer_interval=None, rows=4, cols=4, n_sweeps=2, swap_interval=1):
    from tsu_emulator_b200.distributed import LatticeTempering

    def fac(n_local, replica0, temps_local):
        eng = make_engine(rows, cols, n_replicas=n_local, temperature=temps_local, periodic=True, seed=5,
                          replica0=replica0, bonds=signs)
        eng.init_random()
        return eng

    kw = {} if houdayer_interval is None else {"houdayer_interval": houdayer_interval}
    return LatticeTempering(R_temps, n_ladders=K, engine_factory=fac, n_sweeps=n_sweeps, swap_interval=swap_interval,
                            seed=7, criterion="metropolis", **kw)


def test_tempering_with_houdayer_reproduces_the_exact_slot_zero_energy():
    signs = realisation_4x4()
    temps = [0.8, 1.2, 1.8, 2.5]
    mE = B.exact_moments(4, 4, 1.0, 0.0, temps[0], True, signs)[0]
    K = 512
    pt = tempering(K, temps, signs, houdayer_interval=1)
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
    assert pt.engine.sweep_index == 200 * (2 + 1)


def test_tempering_houdayer_equals_the_host_loop_and_interval_zero_changes_nothing():
    rows = cols = 8
    signs = random_signs(np.random.default_rng(4), 2, rows, cols)
    temps = [0.5, 0.9, 1.5]
    K, n_it = 4, 12
    plain = tempering(K, temps, signs, rows=rows, cols=cols, swap_interval=3)
    zero = tempering(K, temps, signs, houdayer_interval=0, rows=rows, cols=cols, swap_interval=3)
    for _ in range(n_it):
        plain.step()
        zero.step()
    assert torch.equal(plain.engine.state, zero.engine.state)
    assert torch.equal(plain.slot_replica, zero.slot_replica) and torch.equal(plain.lut_index, zero.lut_index)
    # houdayer_interval = 2 against the same iteration written out with host pairs
    dev = tempering(K, temps, signs, houdayer_interval=2, rows=rows, cols=cols, swap_interval=3)
    host = tempering(K, temps, signs, rows=rows, cols=cols, swap_interval=3)
    for it in range(1, n_it + 1):
        dev.step()
        host.engine.sweep(host.n_sweeps)
        host.iteration += 1
        if it % 2 == 0:
            sr = host.slot_replica.cpu().numpy()
            host.engine.houdayer(np.stack([sr[0::2], sr[1::2]], axis=-1).reshape(-1, 2))
        if it % 3 == 0:
            host.swap_fn(host.gather_energies(), host.T_slot, host.slot_replica, host.lut_index, host.K, host.R, it)
            host.engine.set_lut_index(host.lut_index)
    assert torch.equal(dev.engine.state, host.engine.state)
    assert torch.equal(dev.slot_replica, host.slot_replica)
    assert not torch.equal(dev.engine.state, plain.engine.state)
