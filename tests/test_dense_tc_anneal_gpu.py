"""Simulated annealing and parallel tempering on the tensor-core dense sampler (GibbsSampler(precision="bf16")), and the
energy pass they rest on (csrc/dense_tc.cu: dense_tc_kernel<M, true>, tsu_dense_tc_energy).

Energy pass.  The fields come from the GEMM that tsu_dense_tc_debug_fields exposes, which is exact for dyadic couplings
(tests/test_dense_tc_kernel_gpu.py); the thread of each chain then sums s_i f_i and s_i b_i in float64 in site order.
So for dyadic J and bias the energy must EQUAL the float64 energy, at every panel count, chain count and tile height;
for Gaussian couplings it must stay within a stated bound of the float64 energy of the bf16 matrix.  Best-state tracking
is checked with sentinel bytes: which rows are written and which are not.

Annealing and tempering.  With dyadic couplings every energy the device computes is exact, so the selection of the best
chain and every swap decision are exact too: a run must equal a host replay built from the C-ABI sweep launch
(tsu_dense_gibbs_tc_run with the same seed and counters), exact host energies and, for tempering, the host swap pass
cpu_swap of tests/oracle_engine.py.  Each replayed sweep is in turn checked against the float64 rule with `replay()`.
A statistical test checks that criterion="metropolis" makes slot 0 of a ladder sample the Boltzmann distribution, and
that the reference's swap expression does not.
"""
import ctypes
import itertools
import math

import numpy as np
import pytest

from test_dense_tc_kernel_gpu import (BIG_C, PANELS, RATE_EXACT_J, SMALL_C, TC_EPS_EXACT_J, _dev, budget,
                                      dyadic_problem, energy_ref, replay, sk_problem, tc_launch, uniforms, upload_j)

gpu = pytest.mark.gpu
M32 = 0xFFFFFFFF
INIT_KEY = 0x5DEECE66D            # GibbsSampler._initial_states: Philox initial states keyed by seed ^ this

# Gaussian SK couplings at N = 4096: |E_tc - E_float64| of the bf16 matrix.  The fields are fp32 sums of 4096 terms of
# size ~1/64 (error ~1e-7 each); the energy sums ~2048 of them.  Measured on a B200 (1000 W): see DESIGN.md section 2.
SK_ENERGY_BOUND = 1e-6 * 4096


# ------------------------------------------------------------------------------------------------ helpers
def tc_energy(Jd, bd, S, energy=None, best_energy=None, best_state=None, n_chains=None):
    """tsu_dense_tc_energy on the device state S ([rows, N] uint8); n_chains defaults to all rows"""
    import torch
    from tsu_emulator_b200 import _lib

    n = int(S.shape[0]) if n_chains is None else n_chains
    if energy is None:
        energy = torch.full((S.shape[0],), float("nan"), dtype=torch.float64, device="cuda")
    _lib.call("tsu_dense_tc_energy", _lib.ptr(Jd), _lib.ptr(bd), _lib.ptr(S), n, int(S.shape[1]), _lib.ptr(energy),
              _lib.ptr(best_energy), _lib.ptr(best_state), _lib.current_stream())
    return energy


def device_energy_ref(S, J64, b64):
    """E = -1/2 s^T J s - b^T s of every row of S in float64 on the device (exact for dyadic J and bias)"""
    Sd = S.double()
    e = -0.5 * (Sd * (Sd @ J64.T)).sum(1)
    return e if b64 is None else e - Sd @ b64


def padded(J, b, Np):
    N = J.shape[0]
    Jp, bp = np.zeros((Np, Np)), np.zeros(Np)
    Jp[:N, :N] = J
    if b is not None:
        bp[:N] = b
    return Jp, (None if b is None else bp)


def schedule(T_initial, T_final, n_steps, kind):
    """the temperatures of GibbsSampler.simulated_annealing, step k of n_steps"""
    steps = np.arange(n_steps, dtype=np.float64)
    if kind == "exponential":
        return T_initial * (T_final / T_initial) ** (steps / n_steps)
    return T_initial + (T_final - T_initial) * steps / n_steps


def init_states(seed, chain0, C, N, Np):
    """the sampler's Philox initial states, padded with zero bits to Np sites"""
    from oracle import dense_oracle as D

    out = np.zeros((C, Np), dtype=np.int64)
    out[:, :N] = [D.philox_init_state(seed ^ INIT_KEY, (chain0 + c) & M32, N) for c in range(C)]
    return out


def swap_accepts(before, after):
    """number of accepted pair swaps of one pass over each ladder, read off the slot -> replica map before and after:
    pair i is the last to touch slot i, so it was swapped iff slot i differs after the pairs below it are applied"""
    n = 0
    for k in range(before.shape[0]):
        cur = list(before[k])
        for i in range(len(cur) - 1):
            if cur[i] != after[k, i]:
                cur[i], cur[i + 1] = cur[i + 1], cur[i]
                n += 1
        assert list(cur) == list(after[k])
    return n


# ------------------------------------------------------------------------------------------------ 1. exact energies
@gpu
@pytest.mark.parametrize("N,counts", [(128 * k, [70]) for k in PANELS] + [(256, SMALL_C), (4096, BIG_C)])
def test_energy_equals_float64_exactly(N, counts, monkeypatch):
    """tsu_dense_tc_energy must EQUAL the float64 energy for dyadic asymmetric J with bias, at every panel count, chain
    count and both tile heights (the same bits from M = 64 and 128)"""
    import torch

    J, b = dyadic_problem(N, N + 5)
    Jd, J64 = upload_j(J)
    bd = _dev(b, np.float32)
    rng = np.random.default_rng(N + 1)
    for C in counts:
        S = _dev(rng.integers(0, 2, (C, N)), np.uint8)
        S[0] = 1
        ref = device_energy_ref(S, J64, bd.double())
        for m in ("64", "128"):
            monkeypatch.setenv("TSU_TC_M", m)
            E = tc_energy(Jd, bd, S)
            bad = int((E != ref).sum())
            assert bad == 0, f"N={N} C={C} M={m}: {bad} energies differ, max {float((E - ref).abs().max()):.3e}"
        monkeypatch.delenv("TSU_TC_M")
        assert torch.equal(tc_energy(Jd, None, S), device_energy_ref(S, J64, None)), f"N={N} C={C} without bias"


@gpu
def test_energy_gaussian_full_wave():
    """Gaussian SK couplings rounded to bf16, N = 4096, one 128-chain tile per SM (18944 chains): the energy is within
    SK_ENERGY_BOUND of the float64 energy of the bf16 matrix"""
    C, N = 18944, 4096
    J = sk_problem(N, 77)
    Jd, J64 = upload_j(J)
    S = _dev(np.random.default_rng(5).integers(0, 2, (C, N)), np.uint8)
    E = tc_energy(Jd, None, S)
    err = float((E - device_energy_ref(S, J64, None)).abs().max())
    print(f"SK N={N} C={C}: max |E_tc - E_float64| = {err:.3e} (bound {SK_ENERGY_BOUND:.1e})")
    assert err < SK_ENERGY_BOUND


# ------------------------------------------------------------------------------------------------ 2. best tracking
@gpu
@pytest.mark.parametrize("tile_m", ["64", "128"])
def test_best_tracking_rows(tile_m, monkeypatch):
    """Best-state tracking on a buffer of 90 rows of which the first 70 are chains (N = 256, dyadic J and bias):
      * best = +inf copies every chain's energy and state;
      * best = the current energy copies nothing (strict <);
      * best one dyadic step above the current energy copies, for every third chain; the others keep sentinels;
      * rows 70 .. 89 of every buffer keep their sentinel bytes throughout.
    At M = 64 the shadow lanes of every tile compute garbage energies: a store from one would change some energy or
    best row, so the exact checks also cover them."""
    import torch

    monkeypatch.setenv("TSU_TC_M", tile_m)
    N, C, rows = 256, 70, 90
    J, b = dyadic_problem(N, 31)
    step = 2.0 ** -int(np.ceil(np.log2(np.sqrt(N))))
    Jd, J64 = upload_j(J)
    bd = _dev(b, np.float32)
    S = _dev(np.random.default_rng(2).integers(0, 2, (rows, N)), np.uint8)
    ref = device_energy_ref(S[:C], J64, bd.double())
    SENT_E, SENT_B = -12345.5, 0xA5

    def buffers(best):
        e = torch.full((rows,), SENT_E, dtype=torch.float64, device="cuda")
        be = torch.full((rows,), SENT_E, dtype=torch.float64, device="cuda")
        be[:C] = best
        bs = torch.full((rows, N), SENT_B, dtype=torch.uint8, device="cuda")
        return e, be, bs

    def untouched_tail(e, be, bs):
        assert (e[C:] == SENT_E).all() and (be[C:] == SENT_E).all() and (bs[C:] == SENT_B).all(), "rows >= n_chains"

    e, be, bs = buffers(float("inf"))
    tc_energy(Jd, bd, S, e, be, bs, n_chains=C)
    assert torch.equal(e[:C], ref) and torch.equal(be[:C], ref) and torch.equal(bs[:C], S[:C])
    untouched_tail(e, be, bs)

    e, be, bs = buffers(ref)
    tc_energy(Jd, bd, S, e, be, bs, n_chains=C)
    assert torch.equal(e[:C], ref) and torch.equal(be[:C], ref), "equal energies must not replace the best"
    assert (bs == SENT_B).all(), "equal energies must not copy a state"
    untouched_tail(e, be, bs)

    up = torch.zeros(C, dtype=torch.bool, device="cuda")
    up[::3] = True
    e, be, bs = buffers(torch.where(up, ref + step, ref))
    tc_energy(Jd, bd, S, e, be, bs, n_chains=C)
    assert torch.equal(be[:C], ref)
    assert torch.equal(bs[:C][up], S[:C][up]), "a best one dyadic step above the energy must be replaced"
    assert (bs[:C][~up] == SENT_B).all(), "rows of chains that did not improve must not be written"
    untouched_tail(e, be, bs)
    assert (S[:C] != SENT_B).all()  # the sentinel is not a bit value: a copied row is always distinguishable


# ------------------------------------------------------------------------------------------------ 3. simulated annealing
@gpu
@pytest.mark.parametrize("N", [100, 384])
@pytest.mark.parametrize("C", [1, 65, 300])
def test_annealing_equals_replay(N, C):
    """simulated_annealing(precision="bf16") with dyadic J and bias, linear and exponential schedules, against a host
    replay: the sampler's Philox initial states, one tsu_dense_gibbs_tc_run per step at float(Ts[k]) (sweep0 = k), exact
    host energies and strict-< best tracking from the initial state on.  The best state, its energy and the chosen chain
    must agree; every replayed sweep must agree with the float64 rule at the fp32-rounded temperature."""
    import torch
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler

    J, b = dyadic_problem(N, 7 * N + C)
    Np = (N + 127) // 128 * 128
    Jp, bp = padded(J, b, Np)
    Jd, J64 = upload_j(Jp)
    bd = _dev(bp, np.float32)
    n_steps = 25
    found, visits = [], 0
    for kind in ("linear", "exponential"):
        seed = 1000 + N + C + len(kind)
        smp = GibbsSampler(GibbsConfig(temperature=0.7), seed=seed, precision="bf16")
        best, e = smp.simulated_annealing(J, b, T_initial=4.0, T_final=0.1, n_steps=n_steps, cooling_schedule=kind,
                                          n_chains=C)
        Ts = schedule(4.0, 0.1, n_steps, kind)
        st = _dev(init_states(seed, 0, C, N, Np), np.uint8)
        best_e = energy_ref(st.cpu().numpy(), Jp, bp)
        best_s = st.cpu().numpy().copy()
        for k in range(n_steps):
            prev = st.clone()
            tc_launch(Jd, bd, st, 1, seed, k, 0, T=float(Ts[k]))
            Tv = torch.full((C,), float(np.float32(Ts[k])), dtype=torch.float64, device="cuda")
            found += replay(prev, st, J64, bd.double(), Tv, torch.from_numpy(uniforms(seed, 0, C, k, Np)).cuda())
            visits += C * Np
            E = energy_ref(st.cpu().numpy(), Jp, bp)
            better = E < best_e
            best_e[better] = E[better]
            best_s[better] = st.cpu().numpy()[better]
        c = int(np.argmin(best_e))
        assert (best == best_s[c, :N]).all(), f"{kind}: best state differs from chain {c} of the replay"
        assert e == best_e[c] == energy_ref(best[None], J, b)[0], (kind, e, best_e[c])
        assert smp.config.temperature == float(Ts[-1])
        assert smp._sweep_counter == n_steps and smp._chain_counter == C
    print(f"annealing N={N} C={C}: {len(found)} disagreeing visits of {visits}, "
          f"max |u - p| = {max([f[-1] for f in found], default=0.0):.2e}")
    assert all(f[-1] < TC_EPS_EXACT_J for f in found)
    assert len(found) <= budget(visits, RATE_EXACT_J)


@gpu
def test_annealing_finds_ground_state():
    """256 anneals of a 16-bit problem (padded to 128 sites) find its ground state, known by enumerating all 2^16"""
    from tsu_emulator_b200 import GibbsSampler

    N = 16
    J, b = dyadic_problem(N, 16, asymmetric=False)
    S = np.array(list(itertools.product((0, 1), repeat=N)), dtype=np.float64)
    E_all = energy_ref(S, J, b)
    best, e = GibbsSampler(seed=5, precision="bf16").simulated_annealing(J, b, T_initial=5.0, T_final=0.05,
                                                                         n_steps=200, n_chains=256)
    print(f"ground state {E_all.min()}, found {e}")
    assert e == E_all.min() and energy_ref(best[None], J, b)[0] == e


# ------------------------------------------------------------------------------------------------ 4. parallel tempering
def pt_replay(J, b, temps, K, seed, burnin, n_sweeps, n_samples, swap_interval, criterion):
    """host replay of parallel_tempering(precision="bf16"): tensor-core sweeps with per-chain T (C-ABI), exact host
    energies, cpu_swap with the sampler's seed and swap counter"""
    import torch
    from oracle_engine import cpu_swap

    N = J.shape[0]
    R = len(temps)
    Np = (N + 127) // 128 * 128
    Jp, bp = padded(J, b, Np)
    Jd, _ = upload_j(Jp)
    bd = _dev(bp, np.float32)
    st = _dev(init_states(seed, 0, K * R, N, Np), np.uint8)
    sr = np.arange(K * R, dtype=np.int32).reshape(K, R)
    T_chain = np.tile(np.asarray(temps, dtype=np.float64), K)
    swap = cpu_swap(seed, 1 if criterion == "metropolis" else 0)
    tc_launch(Jd, bd, st, burnin, seed, 0, 0, _dev(T_chain, np.float64))
    sweep, step, attempts, accepts = burnin, 0, 0, 0
    samples, hist = np.empty((K, n_samples, N), dtype=np.int64), np.empty((n_samples, K, R))
    for it in range(n_samples):
        tc_launch(Jd, bd, st, n_sweeps, seed, sweep, 0, _dev(T_chain, np.float64))
        sweep += n_sweeps
        E = energy_ref(st.cpu().numpy(), Jp, bp)
        hist[it] = E[sr]
        if (it + 1) % swap_interval == 0:
            step += 1
            before = sr.copy()
            srt = torch.from_numpy(sr)
            swap(torch.from_numpy(E), torch.from_numpy(np.asarray(temps, dtype=np.float64)), srt,
                 np.zeros(K * R, dtype=np.int64), K, R, step)
            attempts += K * (R - 1)
            accepts += swap_accepts(before, sr)
            T_chain[sr] = np.asarray(temps)[None, :]
        samples[:, it] = st.cpu().numpy()[sr[:, 0], :N]
    final = st.cpu().numpy()[:, :N].astype(np.int64)
    return samples, hist, attempts, accepts, [[final[sr[k, i]] for i in range(R)] for k in range(K)], sr


@gpu
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("criterion", ["reference", "metropolis"])
def test_tempering_equals_replay(K, criterion):
    """parallel_tempering(precision="bf16", n_ladders=K) with dyadic J and bias at N = 200 (padded to 256) equals the
    host replay: samples, the energy history, swap counts, final states and (through the final state of every slot)
    the slot -> replica map"""
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler

    N, temps = 200, [0.6, 0.9, 1.4, 2.5]
    J, b = dyadic_problem(N, 200 + K)
    seed, burnin, n_sweeps, n_samples, swap_interval = 31 + K, 3, 2, 8, 2
    smp = GibbsSampler(GibbsConfig(n_burnin=burnin, n_sweeps=n_sweeps), seed=seed, precision="bf16")
    samples, info = smp.parallel_tempering(J, temps, b, n_samples=n_samples, swap_interval=swap_interval, n_ladders=K,
                                           criterion=criterion)
    want, hist, attempts, accepts, final, sr = pt_replay(J, b, temps, K, seed, burnin, n_sweeps, n_samples,
                                                         swap_interval, criterion)
    energies, final_states = info["energies"], info["final_states"]
    if K == 1:
        assert samples.shape == (n_samples, N)
        samples, energies, final_states = samples[None], [energies], [final_states]
    assert samples.shape == (K, n_samples, N)
    assert (samples == want).all()
    for k in range(K):
        assert np.array_equal(np.array(energies[k]).T, hist[:, k]), f"energy history of ladder {k}"
        for i in range(len(temps)):
            assert (final_states[k][i] == final[k][i]).all(), f"final state of ladder {k} slot {i}"
    assert info["swap_attempts"] == attempts == K * (len(temps) - 1) * (n_samples // swap_interval)
    assert info["swap_accepts"] == accepts
    print(f"K={K} {criterion}: {accepts} of {attempts} swaps accepted, slot_replica {sr.tolist()}")
    assert accepts > 0
    assert (sr // len(temps) == np.arange(K)[:, None]).all()  # replicas never leave their ladder


@gpu
def test_tempering_metropolis_samples_boltzmann():
    """10 bits, symmetric dyadic couplings with zero diagonal, 4 temperatures, 512 ladders, criterion="metropolis": slot 0's mean energy,
    site marginals and pair correlations equal exact enumeration at temperatures[0] within 5 standard errors (batch
    means over the independent ladders).  The reference's swap expression keeps slot 0 more than 5 standard errors
    above the exact mean energy."""
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler

    N, K, temps = 10, 512, [0.5, 0.8, 1.3, 2.0]
    J, b = dyadic_problem(N, 10, asymmetric=False)
    np.fill_diagonal(J, 0.0)   # the field includes the self term J_ii s_i: only without it is the chain's law Boltzmann
    S = np.array(list(itertools.product((0, 1), repeat=N)), dtype=np.float64)
    E_all = energy_ref(S, J, b)
    w = np.exp(-(E_all - E_all.min()) / temps[0])
    w /= w.sum()
    exact_e, exact_m, exact_c = w @ E_all, w @ S, np.einsum("s,si,sj->ij", w, S, S)

    def run(criterion):
        cfg = GibbsConfig(n_burnin=100, n_sweeps=2)
        samples, info = GibbsSampler(cfg, seed=9, precision="bf16").parallel_tempering(
            J, temps, b, n_samples=100, swap_interval=1, n_ladders=K, criterion=criterion)
        X = samples.astype(np.float64)                                  # [K, n_samples, N]
        per = [(-0.5 * np.einsum("ksi,ij,ksj->ks", X, J, X) - X @ b).mean(1),
               X.mean(1), np.einsum("ksi,ksj->kij", X, X) / X.shape[1]]
        return [(p.mean(0), p.std(0, ddof=1) / math.sqrt(K)) for p in per], info

    (me, se), (mm, sm), (mc, sc) = run("metropolis")[0]
    print(f"metropolis: E = {me:.4f} +- {se:.4f} (exact {exact_e:.4f})")
    assert abs(me - exact_e) < 5 * se
    assert (np.abs(mm - exact_m) < 5 * sm).all(), (mm, exact_m, sm)
    iu = np.triu_indices(N, 1)
    assert (np.abs(mc - exact_c)[iu] < 5 * sc[iu]).all()
    (re, rse), _, _ = run("reference")[0]
    print(f"reference: E = {re:.4f} +- {rse:.4f} (exact {exact_e:.4f})")
    assert re > exact_e + 5 * rse


def f64_launch(Jt, bd, st, n_sweeps, Td, seed, sweep0, chain0):
    """one tsu_dense_gibbs_run (float64 couplings and fields, Philox) with per-chain temperatures, in place"""
    from tsu_emulator_b200 import _lib

    _lib.call("tsu_dense_gibbs_run", _lib.ptr(Jt), 1, _lib.ptr(bd), _lib.ptr(st), int(st.shape[0]), int(st.shape[1]),
              1.0, _lib.ptr(Td), None, int(n_sweeps), 0, 0, None, None, None, None, 0, None, None, seed, sweep0 & M32,
              chain0 & M32, 1, 0, _lib.current_stream())


@gpu
def test_tempering_ladders_float64_equals_replay():
    """n_ladders = 2 with criterion="metropolis" on the float64 path (N = 40) equals a replay through
    tsu_dense_gibbs_run with per-chain temperatures, exact host energies and cpu_swap"""
    import torch
    from oracle_engine import cpu_swap
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler

    N, K, temps, seed = 40, 2, np.array([0.7, 1.1, 1.8]), 12
    R = len(temps)
    J, b = dyadic_problem(N, 40)
    burnin, n_sweeps, n_samples = 4, 3, 6
    samples, info = GibbsSampler(GibbsConfig(n_burnin=burnin, n_sweeps=n_sweeps), seed=seed).parallel_tempering(
        J, list(temps), b, n_samples=n_samples, swap_interval=1, n_ladders=K, criterion="metropolis")
    Jt = _dev(J.T, np.float64)
    bd = _dev(b, np.float64)
    st = _dev(init_states(seed, 0, K * R, N, N), np.uint8)
    sr = np.arange(K * R, dtype=np.int32).reshape(K, R)
    T_chain = np.tile(temps, K)
    f64_launch(Jt, bd, st, burnin, _dev(T_chain, np.float64), seed, 0, 0)
    swap, accepts = cpu_swap(seed, 1), 0
    for it in range(n_samples):
        f64_launch(Jt, bd, st, n_sweeps, _dev(T_chain, np.float64), seed, burnin + it * n_sweeps, 0)
        E = energy_ref(st.cpu().numpy(), J, b)
        for k in range(K):
            assert np.array_equal(np.array(info["energies"][k])[:, it], E[sr[k]])
        before = sr.copy()
        swap(torch.from_numpy(E), torch.from_numpy(temps), torch.from_numpy(sr), np.zeros(K * R, np.int64), K, R, it + 1)
        accepts += swap_accepts(before, sr)
        T_chain[sr] = temps[None, :]
        assert (samples[:, it] == st.cpu().numpy()[sr[:, 0]]).all()
    final = st.cpu().numpy()
    for k in range(K):
        for i in range(R):
            assert (info["final_states"][k][i] == final[sr[k, i]]).all()
    assert info["swap_attempts"] == K * (R - 1) * n_samples and info["swap_accepts"] == accepts > 0


# ------------------------------------------------------------------------------------------------ 5. contracts
@gpu
def test_bf16_anneal_and_tempering_contracts():
    """output shapes, the final config.temperature, the sampler's counters (sweeps, chains, swap passes) advancing so
    that the next call continues the Philox streams, and the rejections"""
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler

    N = 50
    J, b = dyadic_problem(N, 3)
    smp = GibbsSampler(GibbsConfig(n_burnin=2, n_sweeps=3), seed=4, precision="bf16")
    best, e = smp.simulated_annealing(J, b, T_initial=3.0, T_final=0.2, n_steps=7, n_chains=5)
    assert best.shape == (N,) and best.dtype == np.int64 and isinstance(e, float)
    assert smp.config.temperature == float(schedule(3.0, 0.2, 7, "exponential")[-1])
    assert (smp._sweep_counter, smp._chain_counter) == (7, 5)
    best0, e0 = smp.simulated_annealing(J, b, n_steps=0, n_chains=2)
    assert best0.shape == (N,) and (smp._sweep_counter, smp._chain_counter) == (7, 7)
    samples, info = smp.parallel_tempering(J, [0.5, 1.0, 2.0], b, n_samples=4, swap_interval=2, n_ladders=3)
    assert samples.shape == (3, 4, N)
    assert len(info["energies"]) == 3 and all(len(l) == 3 and len(l[0]) == 4 for l in info["energies"])
    assert len(info["final_states"]) == 3 and info["final_states"][2][1].shape == (N,)
    assert info["swap_attempts"] == 3 * 2 * 2
    assert (smp._sweep_counter, smp._chain_counter, smp._swap_counter) == (7 + 2 + 4 * 3, 7 + 9, 2)
    s1, i1 = smp.parallel_tempering(J, [0.5, 1.0], b, n_samples=3)
    assert s1.shape == (3, N) and len(i1["energies"]) == 2 and len(i1["energies"][0]) == 3
    with pytest.raises(ValueError, match="parity mode"):
        smp.simulated_annealing(J, b, n_steps=3, _uniforms=np.zeros((3, N)))
    with pytest.raises(ValueError, match="float64"):
        smp.simulated_annealing(J, b, n_steps=3, chromatic=True)
    with pytest.raises(ValueError, match="parity mode"):
        smp.parallel_tempering(J, [1.0, 2.0], b, n_samples=1, _inject={})
    with pytest.raises(ValueError, match="parity mode"):
        GibbsSampler().parallel_tempering(J, [1.0, 2.0], b, n_samples=1, n_ladders=2, _inject={})
    with pytest.raises(ValueError, match="n_ladders"):
        smp.parallel_tempering(J, [1.0, 2.0], b, n_samples=1, n_ladders=0)
    with pytest.raises(ValueError, match="criterion must be 'metropolis' or 'reference'"):
        smp.parallel_tempering(J, [1.0, 2.0], b, n_samples=1, criterion="glauber")
    big = np.zeros((4097, 4097))
    with pytest.raises(ValueError, match="at most 4096"):
        smp.simulated_annealing(big, n_steps=1)
    with pytest.raises(ValueError, match="at most 4096"):
        smp.parallel_tempering(big, [1.0], n_samples=1)


# ------------------------------------------------------------------------------------------------ CPU
def test_energy_entry_point_rejects_bad_arguments_without_gpu():
    """tsu_dense_tc_energy returns TSU_ERR_INVALID_ARG before any CUDA call: null pointers, N not a multiple of 128 or
    above 4096, no chains, and one best pointer without the other"""
    from tsu_emulator_b200 import _lib

    lib = _lib.load()
    p = ctypes.c_void_p(16)  # never dereferenced: every call below fails the argument check
    cases = [
        (None, None, p, 4, 128, p, None, None),
        (p, None, None, 4, 128, p, None, None),
        (p, None, p, 4, 128, None, None, None),
        (p, None, p, 0, 128, p, None, None),
        (p, None, p, 4, 100, p, None, None),
        (p, None, p, 4, 0, p, None, None),
        (p, None, p, 4, 4224, p, None, None),
        (p, None, p, 4, 128, p, p, None),
        (p, None, p, 4, 128, p, None, p),
    ]
    for args in cases:
        assert lib.tsu_dense_tc_energy(*args, 0) == _lib.TSU_ERR_INVALID_ARG, args


def test_swap_accepts_helper():
    """swap_accepts recovers the accepted pairs of a pass from the maps before and after"""
    before = np.array([[0, 1, 2, 3]])
    assert swap_accepts(before, np.array([[0, 1, 2, 3]])) == 0
    assert swap_accepts(before, np.array([[1, 0, 2, 3]])) == 1
    assert swap_accepts(before, np.array([[1, 2, 3, 0]])) == 3      # replica 0 carried up by all three pairs
    assert swap_accepts(before, np.array([[1, 0, 3, 2]])) == 2
