"""GPU: parallel tempering on the chromatic CSR back end (GibbsSampler.parallel_tempering(chromatic=True)), alone and
with Houdayer moves between ladders 2m and 2m + 1 (houdayer_interval, houdayer_max_temperature).  The run equals a
host replay built from the C-ABI sweep, exact host energies, the host exchange pass and the oracle move: samples, energy
history, swap counts and final states.  With the detailed-balance criterion and a move every iteration, slot 0 of a
frustrated 16-site +-J graph with bias samples the Boltzmann distribution: mean energy, marginals, pair correlations
and <q^2> between paired ladders equal exact enumeration."""
import itertools

import numpy as np
import pytest
import torch

from oracle import sparse_houdayer_oracle as SH
from oracle_engine import cpu_swap
from test_sparse_houdayer_oracle import csr_of, ea3d, symmetric

pytestmark = pytest.mark.gpu


def dyadic_glass(L, seed):
    """3-D +-J glass with +-1/2 bonds on a random quarter of them and a dyadic bias: exact float64 energies"""
    J = ea3d(L, seed).tocoo()
    rng = np.random.default_rng(seed)
    v = np.where(rng.random(J.nnz) < 0.25, J.data / 2, J.data)
    keep = J.row < J.col
    Js = symmetric(J.row[keep], J.col[keep], v[keep], J.shape[0])
    b = np.round(rng.normal(size=J.shape[0]) * 4) / 4
    return Js, b


def pt_replay(J, b, temps, K, seed, burnin, n_sweeps, n_samples, swap_interval, criterion, hk=0, h_max=np.inf):
    """host replay of parallel_tempering(chromatic=True)"""
    from tsu_emulator_b200 import _lib
    from tsu_emulator_b200.sparse import SparseProblem

    N, R = J.shape[0], len(temps)
    prob = SparseProblem(J, b, torch.device("cuda", 0))
    csr = csr_of(J)
    temps = np.asarray(temps, dtype=np.float64)
    st = torch.empty((K * R, N), dtype=torch.uint8, device="cuda")
    _lib.call("tsu_dense_init_random", st.data_ptr(), K * R, N, seed ^ 0x5DEECE66D, 0, _lib.current_stream())
    sr = np.arange(K * R, dtype=np.int32).reshape(K, R)
    T_chain = np.tile(temps, K)
    swap = cpu_swap(seed, 1 if criterion == "metropolis" else 0)

    def sweeps(n, sweep0):
        prob.run(st, T=1.0, seed=seed, sweep0=sweep0, chain0=0, n_burnin=n, n_samples=0, sweeps_per_sample=0,
                 T_chain=torch.from_numpy(T_chain).cuda())

    sweeps(burnin, 0)
    sweep, step, hstep, attempts, accepts = burnin, 0, 0, 0, 0
    slots = np.nonzero(temps <= h_max)[0]
    samples, hist = np.empty((K, n_samples, N), dtype=np.int64), np.empty((n_samples, K, R))
    for it in range(n_samples):
        sweeps(n_sweeps, sweep)
        sweep += n_sweeps
        x = st.cpu().numpy().astype(np.int64)
        if hk and slots.size and (it + 1) % hk == 0:
            pairs = np.stack((sr[0::2][:, slots], sr[1::2][:, slots]), -1).reshape(-1, 2)
            x = SH.houdayer_steps(x, pairs, csr, seed, 0, hstep, 1)
            hstep += 1
            st.copy_(torch.from_numpy(x.astype(np.uint8)))
        E = np.array([SH.energy(x[r], csr, b) for r in range(K * R)])
        hist[it] = E[sr]
        if (it + 1) % swap_interval == 0:
            step += 1
            before = sr.copy()
            swap(torch.from_numpy(E), torch.from_numpy(temps), torch.from_numpy(sr), np.zeros(K * R, dtype=np.int64),
                 K, R, step)
            attempts += K * (R - 1)
            accepts += swap_accepts(before, sr)
            T_chain[sr.ravel()] = np.tile(temps, K)
        samples[:, it] = x[sr[:, 0]]
    final = st.cpu().numpy().astype(np.int64)
    return samples, hist, attempts, accepts, [[final[sr[k, i]] for i in range(R)] for k in range(K)], hstep


def swap_accepts(before, after):
    """accepted exchanges of one pass: the pass visits the pairs in order, so each accepted pair moves one replica up"""
    n = 0
    for k in range(before.shape[0]):
        row = list(before[k])
        for i in range(len(row) - 1):
            if row[i] != after[k][i]:
                row[i], row[i + 1] = row[i + 1], row[i]
                n += 1
    return n


CASES = [(1, 0, np.inf), (3, 0, np.inf), (2, 1, np.inf), (4, 1, np.inf), (4, 2, 1.0)]


@pytest.mark.parametrize("K,hk,h_max", CASES)
@pytest.mark.parametrize("criterion", ["reference", "metropolis"])
def test_tempering_equals_replay(K, hk, h_max, criterion):
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler

    J, b = dyadic_glass(4, 20 + K)
    temps = [0.5, 0.8, 1.2, 2.0]
    seed, burnin, n_sweeps, n_samples, swap_interval = 31 + K, 3, 2, 8, 2
    smp = GibbsSampler(GibbsConfig(n_burnin=burnin, n_sweeps=n_sweeps), seed=seed)
    samples, info = smp.parallel_tempering(J, temps, b, n_samples=n_samples, swap_interval=swap_interval, n_ladders=K,
                                           criterion=criterion, chromatic=True, houdayer_interval=hk,
                                           houdayer_max_temperature=h_max)
    want, hist, attempts, accepts, final, hsteps = pt_replay(J, b, temps, K, seed, burnin, n_sweeps, n_samples,
                                                        swap_interval, criterion, hk, h_max)
    energies, final_states = info["energies"], info["final_states"]
    if K == 1:
        samples, energies, final_states = samples[None], [energies], [final_states]
    assert samples.shape == (K, n_samples, J.shape[0])
    assert np.array_equal(samples, want)
    for k in range(K):
        assert np.array_equal(np.array(energies[k]).T, hist[:, k]), f"energy history of ladder {k}"
        for i in range(len(temps)):
            assert np.array_equal(final_states[k][i], final[k][i]), f"final state of ladder {k} slot {i}"
    assert info["swap_attempts"] == attempts
    assert info["swap_accepts"] == accepts
    assert smp._houdayer_counter == hsteps == (n_samples // hk if hk else 0)
    assert info["swap_accepts"] > 0


def test_defaults_leave_dense_tempering_alone():
    """chromatic=False, houdayer_interval=0 is the dense run: same samples and energies with and without the
    keywords"""
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler

    J, b = dyadic_glass(3, 7)
    J = J.toarray()
    runs = []
    for kw in ({}, dict(chromatic=False, houdayer_interval=0)):
        smp = GibbsSampler(GibbsConfig(n_burnin=2, n_sweeps=1), seed=4)
        runs.append(smp.parallel_tempering(J, [0.7, 1.5], b, n_samples=5, swap_interval=1, n_ladders=2, **kw))
    assert np.array_equal(runs[0][0], runs[1][0])
    assert runs[0][1]["energies"] == runs[1][1]["energies"]


def test_houdayer_tempering_samples_boltzmann():
    """16 sites, frustrated +-J couplings (a 4 x 4 periodic lattice with random signs and diagonals), dyadic bias,
    zero diagonal; 4 temperatures, 512 ladders, criterion="metropolis", a Houdayer move on every slot at every
    iteration: slot 0 matches exact enumeration within 5 standard errors (batch means over ladders)"""
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler

    N, K, temps = 16, 512, [0.6, 0.9, 1.4, 2.2]
    rng = np.random.default_rng(16)
    idx = np.arange(N).reshape(4, 4)
    a = np.concatenate([idx.ravel(), idx.ravel(), idx[:, :3].ravel()])
    c = np.concatenate([np.roll(idx, -1, 0).ravel(), np.roll(idx, -1, 1).ravel(), np.roll(idx, -1, 0)[:, 1:].ravel()])
    J = symmetric(a, c, rng.choice([-1.0, 1.0], a.size), N)
    b = np.round(rng.normal(size=N) * 2) / 4
    Jd = J.toarray()
    S = np.array(list(itertools.product((0, 1), repeat=N)), dtype=np.float64)
    E_all = -0.5 * np.einsum("si,ij,sj->s", S, Jd, S) - S @ b
    w = np.exp(-(E_all - E_all.min()) / temps[0])
    w /= w.sum()
    exact_e, exact_m = w @ E_all, w @ S
    exact_c = np.einsum("s,si,sj->ij", w, S, S)
    sig = 2 * S - 1
    exact_q2 = float((np.einsum("s,si,sj->ij", w, sig, sig) ** 2).sum() / N ** 2)

    cfg = GibbsConfig(n_burnin=100, n_sweeps=1)
    samples, info = GibbsSampler(cfg, seed=3).parallel_tempering(
        J, temps, b, n_samples=200, swap_interval=1, n_ladders=K, criterion="metropolis", chromatic=True,
        houdayer_interval=1)
    X = samples.astype(np.float64)                                      # [K, n_samples, N]
    E = -0.5 * np.einsum("kti,ij,ktj->kt", X, Jd, X) - X @ b

    def within(per_ladder, exact, what):
        per_ladder = np.asarray(per_ladder)
        m, se = per_ladder.mean(axis=0), per_ladder.std(axis=0, ddof=1) / np.sqrt(per_ladder.shape[0])
        z = np.abs(m - exact) / np.maximum(se, 1e-12)
        assert np.all(z < 5), f"{what}: max z = {z.max():.2f}"

    within(E.mean(axis=1), exact_e, "mean energy")
    within(X.mean(axis=1), exact_m, "marginals")
    within(np.einsum("kti,ktj->kij", X, X) / X.shape[1], exact_c, "pair correlations")
    s = 2 * X - 1
    q = (s[0::2] * s[1::2]).mean(axis=2)                                # [K/2, n_samples]
    within((q * q).mean(axis=1), exact_q2, "<q^2> of paired ladders")
    assert info["swap_accepts"] > 0
