"""GPU parity of the block-per-chain dense Gibbs kernel (csrc/dense_gibbs.cu: dense_gibbs_kernel, one CTA per chain) at
the sizes it serves - N = 33 up to the shared-memory limit, float64 and float32 fields - and through every GibbsSampler
entry point that runs it, against the site-by-site oracle (oracle/dense_oracle.py).

Two coupling families keep the expected result exact rather than within a loose tolerance:
  * dyadic couplings J = m / 2^k (|m| <= 3, non-zero diagonal, bias in multiples of 2^-k, T in {1/2, 1, 2}): every
    field and every h / T is exact in float64 in any summation order, and in float32 at these sizes, so float64 fields
    must reproduce the oracle bit for bit and float32 fields may differ only through expf;
  * Gaussian SK couplings: the kernel's trajectory is replayed one sweep per launch and every site where its bit differs
    from the reference's float64 rule is counted and reported, with |u - p| there checked against a stated budget.

The host oracle is vectorised over chains (`sweep_vec`, `replay`) so that N = 13657 stays cheap; the CPU tests at the
end of the file check those helpers against the plain per-chain oracle.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import dense_oracle as D

gpu = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

# float64 sizes: 32/33 warp -> block kernel, 64/65 and 512/513 change the fields per thread (1 -> 2 -> 4), 1481/1482 is
# the first N whose shared memory needs the opt-in above 48 KB, 4096/4097 is where the 1024-thread cap starts (5 to 7
# fields per thread above it) and 7035 the last N that fits 227 KB
F64_SIZES = [33, 63, 64, 65, 255, 256, 511, 512, 513, 1024, 1481, 1482, 2048, 4095, 4096, 4097, 5000, 7035]
# float32 fields: 2876 is the first N over 48 KB, 13657 the last that fits
F32_SIZES = [2875, 2876, 8000, 13657]

# |u - p| budgets where the kernel may disagree with the float64 rule on its own trajectory:
#   * float64 fields summed in another order than the reference's dot product: ~1e-16 * sqrt(N) in h -> 1e-12;
#   * float32 fields: every addition rounds at 2^-24 relative (6e-8 for |h| <= 1, SK fields stay below ~3).  A field
#     collects N additions when it is computed and one more per flip of any site (< 3 N over the sweeps run here,
#     before a refresh after 8 sweeps), so the random-walk error is ~6e-8 * 3 * sqrt(4 N) / sqrt(12) ~ 1e-7 sqrt(N);
#     |dp| <= |dh| / (4 T) <= |dh| at T >= 1/4, and expf with the float32 rounding of p adds ~2e-7.  Five standard
#     deviations and the expf term: 1e-6 * (sqrt(N) + 1).
F64_EPS = 1e-12


def f32_eps(N):
    return 1e-6 * (np.sqrt(N) + 1.0)


F32_EXPF_EPS = 1e-6   # exact fields (dyadic J): only expf and the float32 rounding of p differ from the reference


# ------------------------------------------------------------------------------------------------ host oracle helpers
def dyadic_problem(N, seed, *, asymmetric=False, dtype=np.float64):
    """J = m / 2^k with |m| <= 3 and a non-zero diagonal (the self term is part of h, gibbs.py:97), bias in multiples of
    2^-k with |b| <= 1; k = ceil(log2 sqrt(N)) keeps typical fields O(1).  Every partial sum is a multiple of 2^-k below
    3 N / 2^k + 1 < 2^(24 - k): exact in float32 and float64 in any order."""
    rng = np.random.default_rng(seed)
    k = int(np.ceil(np.log2(np.sqrt(N))))
    m = rng.integers(-3, 4, size=(N, N), dtype=np.int8)
    if not asymmetric:
        m = np.triu(m) + np.triu(m, 1).T
    J = m.astype(dtype)
    J *= dtype(2.0 ** -k)
    b = rng.integers(-2**k, 2**k + 1, size=N) * 2.0 ** -k
    return J, b


def sk_problem(N, seed, *, dtype=np.float64):
    """symmetric J ~ N(0, 1/N) with zero diagonal (as `dtype`, so the oracle sees exactly the kernel's couplings)"""
    rng = np.random.default_rng(seed)
    J = rng.standard_normal((N, N), dtype=dtype)
    J = np.triu(J, 1)
    J += J.T
    J *= dtype(1.0 / np.sqrt(N))
    b = rng.normal(size=N) * 0.3
    return J, b


def sigmoid_vec(x):
    """gibbs.py:61-77 elementwise: 1 / (1 + exp(-x)), x > 20 -> 1, x < -20 -> 0"""
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(over="ignore"):
        p = 1.0 / (1.0 + np.exp(-x))
    return np.where(x > 20, 1.0, np.where(x < -20, 0.0, p))


def _field(J, b, i, S):
    """h_i = J[i, :] . s + b_i of every chain (gibbs.py:79-100), float64"""
    h = np.asarray(J[i], dtype=np.float64) @ S.T
    return h if b is None else h + b[i]


def sweep_vec(S, J, b, T, U, order=None):
    """one sweep of the reference (gibbs.py:153-160, D.gibbs_sweeps) for every chain at once: S [C, N] bits, T a scalar or
    [C], U [C, NV] the uniform of each visit, order the NV visited sites (None: 0 .. N-1).  Returns the new bits."""
    S = np.array(S, dtype=np.float64)
    T = np.broadcast_to(np.asarray(T, dtype=np.float64), (S.shape[0],))
    for k, i in enumerate(range(S.shape[1]) if order is None else order):
        S[:, i] = U[:, k] < sigmoid_vec(_field(J, b, i, S) / T)
    return S.astype(np.int64)


def replay(start, after, J, b, T, U, order=None):
    """D.tc_sweep_disagreements for every chain at once and any visiting order: the reference's decision at every visit,
    evaluated on the state the kernel had at that moment, against the kernel's bit (which is then kept).
    Returns [(chain, site, |u - p|)] for every visit where the two differ."""
    cur = np.array(start, dtype=np.float64)
    after = np.asarray(after)
    T = np.broadcast_to(np.asarray(T, dtype=np.float64), (cur.shape[0],))
    out = []
    for k, i in enumerate(range(cur.shape[1]) if order is None else order):
        p = sigmoid_vec(_field(J, b, i, cur) / T)
        for c in np.flatnonzero((U[:, k] < p) != (after[:, i] != 0)):
            out.append((int(c), int(i), abs(float(U[c, k]) - float(p[c]))))
        cur[:, i] = after[:, i]
    return out


def energy_vec(S, J, b):
    """E = -1/2 s^T J s - b^T s (gibbs.py:215-236) of every chain, float64, J converted a block of rows at a time"""
    S = np.asarray(S, dtype=np.float64)
    H = np.empty_like(S)
    for r in range(0, S.shape[1], 1024):
        H[:, r:r + 1024] = S @ np.asarray(J[r:r + 1024], dtype=np.float64).T
    e = -0.5 * np.einsum("cn,cn->c", S, H)
    return e if b is None else e - S @ b


def philox_sweep(seed, chain0, C, sweep, sites):
    """[C, NV] uniforms the kernel draws in Philox mode for one sweep, in visiting order"""
    return np.stack([D.philox_uniforms(seed, chain0 + c, sweep, sites) for c in range(C)])


# ------------------------------------------------------------------------------------------------ device helpers
def upload(J, b, dtype):
    """Jt (the transpose the kernel reads, tsu_b200.h) and bias as `dtype` device tensors"""
    import torch

    td = torch.float64 if dtype == np.float64 else torch.float32
    Jt = torch.from_numpy(np.ascontiguousarray(J)).cuda().to(td).t().contiguous()
    bt = None if b is None else torch.from_numpy(np.asarray(b, dtype=np.float64)).cuda().to(td)
    return Jt, bt


def dense_run(Jt, bt, state, *, T=1.0, T_chain=None, T_sweep=None, n_burnin=0, n_samples=0, sweeps_per_sample=0,
              order=None, uniforms=None, want_samples=False, want_energy=False, track_best=False, seed=0, sweep0=0,
              chain0=0, visits=0):
    """one tsu_dense_gibbs_run; `state` (uint8 [C, N] device tensor) is updated in place.  Precision follows Jt's dtype."""
    import torch
    from tsu_emulator_b200 import _lib

    C, N = state.shape
    code = 1 if Jt.dtype == torch.float64 else 0
    dev = lambda a, dt: None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()  # noqa: E731
    Tc, Ts = dev(T_chain, np.float64), dev(T_sweep, np.float64)
    od, ud = dev(order, np.int32), dev(uniforms, np.float64)
    samples = torch.empty((n_samples, C, N), dtype=torch.uint8, device="cuda") if want_samples else None
    energy = torch.empty(C, dtype=torch.float64, device="cuda") if want_energy else None
    best_state = torch.empty((C, N), dtype=torch.uint8, device="cuda") if track_best else None
    best_energy = torch.empty(C, dtype=torch.float64, device="cuda") if track_best else None
    _lib.call("tsu_dense_gibbs_run", _lib.ptr(Jt), code, _lib.ptr(bt), _lib.ptr(state), C, N, float(T), _lib.ptr(Tc),
              _lib.ptr(Ts), n_burnin, n_samples, sweeps_per_sample, _lib.ptr(od), _lib.ptr(ud), _lib.ptr(samples),
              _lib.ptr(energy), int(track_best), _lib.ptr(best_state), _lib.ptr(best_energy), seed, sweep0, chain0, code,
              visits, _lib.current_stream())
    host = lambda t: None if t is None else t.cpu().numpy()  # noqa: E731
    return {"state": state.cpu().numpy().astype(np.int64), "samples": host(samples), "energy": host(energy),
            "best_state": host(best_state), "best_energy": host(best_energy)}


def run_sweep_by_sweep(J, b, init, dtype, T, seed, sweep0, chain0, n_sweeps, orders=None):
    """one launch per sweep (Philox mode): the bits of every chain after every sweep, [n_sweeps, C, N]"""
    import torch

    Jt, bt = upload(J, b, dtype)
    st = torch.from_numpy(np.asarray(init, dtype=np.uint8)).cuda()
    seq = []
    for s in range(n_sweeps):
        seq.append(dense_run(Jt, bt, st, T=T, n_burnin=1, seed=seed, sweep0=sweep0 + s, chain0=chain0,
                             order=None if orders is None else orders[s:s + 1])["state"])
    return np.stack(seq)


def replay_sweeps(seq, init, J, b, T, seed, sweep0, chain0, orders=None):
    """every (sweep, chain, site, |u - p|) where the kernel's bit differs from the reference's rule on its trajectory"""
    found = []
    for s in range(len(seq)):
        sites = np.arange(seq.shape[2]) if orders is None else orders[s]
        U = philox_sweep(seed, chain0, seq.shape[1], sweep0 + s, sites)
        start = init if s == 0 else seq[s - 1]
        found += [(s, *d) for d in replay(start, seq[s], J, b, T, U, None if orders is None else orders[s])]
    return found


def sampler(T=1.0, **kw):
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler

    cfg = {k: kw.pop(k) for k in list(kw) if k in ("n_burnin", "n_sweeps", "update_order")}
    return GibbsSampler(GibbsConfig(temperature=T, **cfg), **kw)


# ------------------------------------------------------------------------------------------------ sizes, dyadic J
@gpu
@pytest.mark.parametrize("N", F64_SIZES)
def test_dyadic_float64_bit_exact(N):
    """float64 fields at every branch boundary of the block kernel: Philox mode with non-zero sweep0 / chain0, sequential
    or random order (explicit d_order), scalar / per-chain / per-sweep temperature, burn-in + samples schedule, final
    energies and best-state tracking, all against the oracle with zero mismatches"""
    import torch

    idx = F64_SIZES.index(N)
    rng = np.random.default_rng(100 + idx)
    C = 3 + idx % 6
    n_sweeps = 3 if N <= 4097 else 2
    J, b = dyadic_problem(N, idx, asymmetric=idx % 4 == 3)
    temps = np.array([0.5, 1.0, 2.0])
    t_mode = idx % 3
    T_chain = rng.choice(temps, C) if t_mode == 1 else None
    T_sweep = rng.choice(temps, n_sweeps) if t_mode == 2 else None
    T = 1.0 if t_mode else 0.5
    orders = np.stack([rng.permutation(N) for _ in range(n_sweeps)]).astype(np.int32) if idx % 2 else None
    init = rng.integers(0, 2, (C, N))
    seed, sweep0, chain0 = 1000 + N, 7 + idx, 3 * N
    Jt, bt = upload(J, b, np.float64)
    got = dense_run(Jt, bt, torch.from_numpy(init.astype(np.uint8)).cuda(), T=T, T_chain=T_chain, T_sweep=T_sweep,
                    n_burnin=1, n_samples=n_sweeps - 1, sweeps_per_sample=1, order=orders, want_samples=True,
                    want_energy=True, track_best=True, seed=seed, sweep0=sweep0, chain0=chain0)
    S, best_e = init, energy_vec(init, J, b)
    best = init.copy()
    for s in range(n_sweeps):
        Ts = T_chain if T_chain is not None else (T_sweep[s] if T_sweep is not None else T)
        sites = np.arange(N) if orders is None else orders[s]
        S = sweep_vec(S, J, b, Ts, philox_sweep(seed, chain0, C, sweep0 + s, sites), None if orders is None else orders[s])
        e = energy_vec(S, J, b)
        better = e < best_e
        best[better], best_e = S[better], np.where(better, e, best_e)
        if s >= 1:
            assert (got["samples"][s - 1] == S).all(), f"sample {s - 1} differs"
    assert (got["state"] == S).all()
    assert (got["energy"] == energy_vec(S, J, b)).all()        # exact: dyadic sums
    assert (got["best_energy"] == best_e).all() and (got["best_state"] == best).all()


@gpu
@pytest.mark.parametrize("N,C,n_sweeps,order_mode", [(600, 592, 8, "random"), (600, 592, 8, "sequential"),
                                                     (4097, 296, 2, "sequential")])
def test_dyadic_float64_full_wave_of_chains(N, C, n_sweeps, order_mode):
    """several CTAs on every SM: the barrier-per-visit protocol (the self-term and bit writes of the site decided in the
    previous step, deferred to the field's owner thread) under full occupancy, against the oracle bit for bit.  A wrong
    owner there is a shared-memory race that corrupts roughly one chain-sweep in a thousand, hence the many chains."""
    import torch

    rng = np.random.default_rng(N)
    J, b = dyadic_problem(N, N + 1)
    init = rng.integers(0, 2, (C, N))
    orders = np.stack([rng.permutation(N) for _ in range(n_sweeps)]).astype(np.int32) if order_mode == "random" else None
    seed, sweep0, chain0 = 5, 11, 17
    Jt, bt = upload(J, b, np.float64)
    got = dense_run(Jt, bt, torch.from_numpy(init.astype(np.uint8)).cuda(), T=1.0, n_burnin=n_sweeps, order=orders,
                    seed=seed, sweep0=sweep0, chain0=chain0)["state"]
    S = init
    for s in range(n_sweeps):
        sites = np.arange(N) if orders is None else orders[s]
        S = sweep_vec(S, J, b, 1.0, philox_sweep(seed, chain0, C, sweep0 + s, sites), None if orders is None else orders[s])
    bad = np.flatnonzero((got != S).any(1))
    assert bad.size == 0, f"{bad.size} of {C} chains differ: {bad[:10]}"


@gpu
@pytest.mark.parametrize("N,dtype", [(600, np.float64), (4097, np.float64), (3000, np.float32)])
def test_dyadic_partial_sweeps(N, dtype):
    """visits_per_sweep < N: each sweep visits N / 3 sites given by d_order (a different subset every sweep), Philox
    uniforms keyed by the visited site, against the oracle on the same visiting orders"""
    import torch

    rng = np.random.default_rng(N + 1)
    C, n_sweeps, NV, T = 5, 3, N // 3, 1.0
    J, b = dyadic_problem(N, N + 7, dtype=dtype)
    init = rng.integers(0, 2, (C, N))
    orders = np.stack([rng.permutation(N)[:NV] for _ in range(n_sweeps)]).astype(np.int32)
    seed, sweep0, chain0 = 606, 2, 9
    Jt, bt = upload(J, b, dtype)
    got = dense_run(Jt, bt, torch.from_numpy(init.astype(np.uint8)).cuda(), T=T, n_burnin=n_sweeps, order=orders,
                    seed=seed, sweep0=sweep0, chain0=chain0, visits=NV)["state"]
    S = init
    for s in range(n_sweeps):
        S = sweep_vec(S, J, b, T, philox_sweep(seed, chain0, C, sweep0 + s, orders[s]), orders[s])
    assert (got == S).all()


@gpu
@pytest.mark.parametrize("N", F32_SIZES)
def test_dyadic_float32_fields_differ_only_through_expf(N):
    """float32 fields, exact with dyadic J: one launch per sweep replayed against the float64 rule; a disagreement may
    only come from expf / the float32 p, i.e. |u - p| < 1e-6, and a handful at most.  The same sweeps in one launch give
    the same bits and an exact energy."""
    import torch

    idx = F32_SIZES.index(N)
    rng = np.random.default_rng(200 + idx)
    C, n_sweeps, T = 4, 2, (0.5, 1.0, 2.0)[idx % 3]
    J, b = dyadic_problem(N, 300 + idx, asymmetric=idx == 1, dtype=np.float32)
    init = rng.integers(0, 2, (C, N))
    orders = np.stack([rng.permutation(N) for _ in range(n_sweeps)]).astype(np.int32) if idx % 2 else None
    seed, sweep0, chain0 = 77 + N, 5, 2 * N
    seq = run_sweep_by_sweep(J, b, init, np.float32, T, seed, sweep0, chain0, n_sweeps, orders)
    found = replay_sweeps(seq, init, J, b, T, seed, sweep0, chain0, orders)
    print(f"float32 fields, dyadic J, N={N}: {len(found)} disagreeing visits of {C * N * n_sweeps}, "
          f"max |u - p| = {max([f[-1] for f in found], default=0.0):.2e}")
    assert all(f[-1] < F32_EXPF_EPS for f in found), found
    assert len(found) <= 2
    Jt, bt = upload(J, b, np.float32)
    one = dense_run(Jt, bt, torch.from_numpy(init.astype(np.uint8)).cuda(), T=T, n_burnin=n_sweeps, order=orders,
                    want_energy=True, seed=seed, sweep0=sweep0, chain0=chain0)
    assert (one["state"] == seq[-1]).all()
    assert (one["energy"] == energy_vec(seq[-1], J, b)).all()


# ------------------------------------------------------------------------------------------------ Gaussian SK couplings
@gpu
@pytest.mark.parametrize("N", [65, 513, 1482, 4097, 7035])
def test_sk_float64_replay(N):
    """Gaussian couplings, float64 fields: the kernel's fields are summed in another order than the reference's dot
    product, so it may disagree only where a uniform lies within ~1e-16 of p; every disagreement is counted"""
    rng = np.random.default_rng(N)
    C, n_sweeps = 4, 2
    J, b = sk_problem(N, N)
    init = rng.integers(0, 2, (C, N))
    orders = np.stack([rng.permutation(N) for _ in range(n_sweeps)]).astype(np.int32) if N % 2 == 0 else None
    seed, sweep0, chain0 = 31337, 3, 40
    seq = run_sweep_by_sweep(J, b, init, np.float64, 1.0, seed, sweep0, chain0, n_sweeps, orders)
    found = replay_sweeps(seq, init, J, b, 1.0, seed, sweep0, chain0, orders)
    print(f"float64 fields, SK J, N={N}: {len(found)} disagreeing visits of {C * N * n_sweeps}, "
          f"max |u - p| = {max([f[-1] for f in found], default=0.0):.2e}")
    assert all(f[-1] < F64_EPS for f in found), found
    assert len(found) <= 1


@gpu
@pytest.mark.parametrize("N", [2876, 13657])
def test_sk_float32_replay(N):
    """Gaussian couplings, float32 fields: disagreements with the float64 rule only within the float32 field error
    f32_eps(N) of p, counted"""
    rng = np.random.default_rng(N)
    C, n_sweeps = 4, 2
    J, b = sk_problem(N, N, dtype=np.float32)
    b = b.astype(np.float32).astype(np.float64)
    init = rng.integers(0, 2, (C, N))
    seed, sweep0, chain0 = 4242, 9, 1
    seq = run_sweep_by_sweep(J, b, init, np.float32, 1.0, seed, sweep0, chain0, n_sweeps)
    found = replay_sweeps(seq, init, J, b, 1.0, seed, sweep0, chain0)
    print(f"float32 fields, SK J, N={N}: {len(found)} disagreeing visits of {C * N * n_sweeps}, "
          f"max |u - p| = {max([f[-1] for f in found], default=0.0):.2e} (budget {f32_eps(N):.1e})")
    assert all(f[-1] < f32_eps(N) for f in found), found
    assert len(found) <= 3


# ------------------------------------------------------------------------------------------------ entry points, N > 32
@gpu
@pytest.mark.parametrize("N,order_mode", [(40, "random"), (600, "sequential"), (600, "random")])
def test_sample_boltzmann_chains_schedule(N, order_mode):
    """GibbsSampler.sample_boltzmann with several chains: burn-in, then n_samples x n_sweeps sweeps (gibbs.py:198-211),
    injected uniforms and orders, against D.sample_boltzmann per chain"""
    rng = np.random.default_rng(N)
    C, burnin, n_samples, n_sweeps, T = 4, 2, 3, 2, 0.5
    J, b = dyadic_problem(N, N + 2, asymmetric=order_mode == "random")
    total = burnin + n_samples * n_sweeps
    U = rng.random((total, C, N))
    orders = np.stack([rng.permutation(N) for _ in range(total)]) if order_mode == "random" else None
    init = rng.integers(0, 2, (C, N))
    smp = sampler(T, n_burnin=burnin, n_sweeps=n_sweeps, update_order=order_mode, seed=2)
    out = smp.sample_boltzmann(J, b, n_samples=n_samples, initial_state=init, n_chains=C, _uniforms=U, _orders=orders)
    assert out.shape == (C, n_samples, N) and out.dtype == int
    for c in range(C):
        want = D.sample_boltzmann(J, b, T, burnin, n_samples, n_sweeps, init[c], U[:, c, :], orders)
        assert (out[c] == want).all(), f"chain {c}"


@gpu
@pytest.mark.parametrize("N", [100, 1500])
def test_sample_chains_float64_energies(N):
    """sample_chains(return_energy=True) with float64 fields: bits against the oracle on the Philox stream, energies
    (chain_energy: block_sum over several warps) against D.compute_energy - exact with dyadic J"""
    rng = np.random.default_rng(N)
    C, n_sweeps, T = 5, 3, 1.0
    J, b = dyadic_problem(N, N + 3)
    init = rng.integers(0, 2, (C, N))
    smp = sampler(T, seed=21)
    out, e = smp.sample_chains(J, b, n_chains=C, n_sweeps=n_sweeps, initial_state=init, return_energy=True)
    S = init
    for s in range(n_sweeps):
        S = sweep_vec(S, J, b, T, philox_sweep(21, 0, C, s, np.arange(N)))
    assert (out == S).all()
    for c in range(C):
        assert e[c] == pytest.approx(D.compute_energy(out[c], J, b), abs=1e-9)


@gpu
def test_sample_chains_float32_refresh_dyadic_exact():
    """float32 fields over 17 sweeps, so the from-scratch refresh runs at sweeps 8 and 16: with dyadic J the fields are
    exact throughout, so the bits equal the oracle and the energies D.compute_energy"""
    N, C, n_sweeps, T = 300, 4, 17, 1.0
    rng = np.random.default_rng(17)
    J, b = dyadic_problem(N, 17)
    init = rng.integers(0, 2, (C, N))
    out, e = sampler(T, seed=9, precision="float32").sample_chains(J, b, n_chains=C, n_sweeps=n_sweeps,
                                                                   initial_state=init, return_energy=True)
    S = init
    for s in range(n_sweeps):
        S = sweep_vec(S, J, b, T, philox_sweep(9, 0, C, s, np.arange(N)))
    assert (out == S).all()
    assert (e == energy_vec(S, J, b)).all()
    for c in range(C):
        assert e[c] == pytest.approx(D.compute_energy(out[c], J, b), abs=1e-9)


# float32 energy: E = -1/2 sum_i s_i (h_i + b_i) over <= N set bits, each h_i within f32_eps(N) (see above)
def f32_energy_tol(N):
    return 0.5 * N * f32_eps(N)


@gpu
def test_sample_chains_float32_refresh_gaussian():
    """Gaussian J, float32 fields, 17 sweeps in one launch: the fields are recomputed from scratch at sweeps 8 and 16, so
    the launch must give the same bits AND the same energy bits as launches of 8 + 8 + 1 sweeps (each of which starts
    from freshly computed fields); the energy is within f32_energy_tol of the float64 recompute"""
    import torch

    N, C, T = 1024, 6, 1.0
    rng = np.random.default_rng(18)
    J, b = sk_problem(N, 18, dtype=np.float32)
    b = b.astype(np.float32).astype(np.float64)
    init = rng.integers(0, 2, (C, N))
    seed = 123
    smp = sampler(T, seed=seed, precision="float32")
    out, e = smp.sample_chains(J, b, n_chains=C, n_sweeps=17, initial_state=init, return_energy=True)
    Jt, bt = upload(J, b, np.float32)
    st = torch.from_numpy(init.astype(np.uint8)).cuda()
    for sweep0, n in ((0, 8), (8, 8), (16, 1)):
        split = dense_run(Jt, bt, st, T=T, n_burnin=n, want_energy=True, seed=seed, sweep0=sweep0)
    assert (split["state"] == out).all()
    assert (split["energy"] == e).all(), (split["energy"] - e)
    ref = energy_vec(out, J, b)
    print(f"float32 energies after 17 sweeps, N={N}: max |E - E_float64| = {np.abs(e - ref).max():.2e} "
          f"(tolerance {f32_energy_tol(N):.1e})")
    assert np.abs(e - ref).max() < f32_energy_tol(N)


@gpu
@pytest.mark.parametrize("N,schedule", [(100, "exponential"), (600, "linear")])
def test_simulated_annealing_block_kernel(N, schedule):
    """simulated_annealing: per-sweep temperature and on-device best tracking (gibbs.py:340-393), injected uniforms,
    one and three chains, against D.simulated_annealing: same best state and energy"""
    rng = np.random.default_rng(N)
    n_steps = 12
    J, b = dyadic_problem(N, N + 4, asymmetric=N == 600)
    for C in (1, 3):
        U = rng.random((n_steps, C, N))
        init = rng.integers(0, 2, (C, N))
        smp = sampler(seed=3)
        best, e = smp.simulated_annealing(J, b, T_initial=5.0, T_final=0.2, n_steps=n_steps, cooling_schedule=schedule,
                                          n_chains=C, _uniforms=U, _initial_state=init)
        want = [D.simulated_annealing(J, b, 5.0, 0.2, n_steps, schedule, init[c], U[:, c, :]) for c in range(C)]
        k = int(np.argmin([w[1] for w in want]))
        assert (best == want[k][0]).all(), f"{C} chains"
        assert e == pytest.approx(want[k][1], abs=1e-9)


@gpu
def test_parallel_tempering_block_kernel():
    """parallel_tempering at N = 80 (per-chain temperatures, energies from chain_energy), injected draws, against
    D.parallel_tempering: samples, swap counts, energies and final states"""
    N, R, burnin, n_sweeps, n_samples, swap_interval = 80, 4, 2, 2, 6, 1
    rng = np.random.default_rng(80)
    J, b = dyadic_problem(N, 81)
    J *= 4.0                                         # with these temperatures some swaps are rejected (15 of 18)
    temps = [0.1, 0.3, 1.0, 4.0]
    inj = {"inits": rng.integers(0, 2, (R, N)), "burn_uniforms": rng.random((R, burnin, N)),
           "sweep_uniforms": rng.random((n_samples, R, n_sweeps, N)), "swap_uniforms": rng.random((n_samples, R - 1))}
    smp = sampler(1.0, n_burnin=burnin, n_sweeps=n_sweeps, seed=4)
    samples, info = smp.parallel_tempering(J, temps, b, n_samples=n_samples, swap_interval=swap_interval, _inject=inj)
    want, winfo = D.parallel_tempering(J, b, temps, burnin, n_sweeps, n_samples, swap_interval, inj["inits"],
                                       inj["burn_uniforms"], inj["sweep_uniforms"], inj["swap_uniforms"])
    assert (samples == want).all()
    assert info["swap_attempts"] == winfo["swap_attempts"] and info["swap_accepts"] == winfo["swap_accepts"]
    assert 0 < winfo["swap_accepts"] < winfo["swap_attempts"]
    assert np.allclose(np.array(info["energies"]), np.array(winfo["energies"]), rtol=0, atol=1e-9)
    assert (np.array(info["final_states"]) == np.array(winfo["final_states"])).all()


@gpu
@pytest.mark.parametrize("N", [100, 1500])
def test_sample_conditional_block_kernel(N):
    """sample_conditional at N > 32 (one visit, visits_per_sweep = 1): the single-site rule of gibbs.py:102-126 on the
    Philox uniform of (site, chain 0, sweep k) for the k-th call"""
    rng = np.random.default_rng(N)
    J, b = dyadic_problem(N, N + 5)
    T, seed = 0.5, 8
    smp = sampler(T, seed=seed)
    ones = 0
    for k in range(12):
        i = int(rng.integers(N))
        state = rng.integers(0, 2, N)
        got = smp.sample_conditional(i, state, J, b)
        u = D.philox_uniforms(seed, 0, k, [i])[0]
        want = 1 if u < D.sigmoid_ref(float(np.dot(J[i], state) + b[i]) / T) else 0
        assert got == want, (k, i)
        ones += got
    assert 0 < ones < 12


@gpu
@pytest.mark.parametrize("N", [513, 2048, 4097])
def test_dense_energy_kernel_many_warps(N):
    """tsu_dense_energy where block_sum combines many warps (up to 32), float64 and float32 couplings, asymmetric J"""
    import torch
    from tsu_emulator_b200 import _lib

    rng = np.random.default_rng(N)
    C = 6
    J = rng.normal(size=(N, N)) / np.sqrt(N)
    b = rng.normal(size=N)
    S = rng.integers(0, 2, (C, N))
    S[0] = 1                                         # every site set: the largest sum
    st = torch.from_numpy(S.astype(np.uint8)).cuda()
    for dtype, code in ((np.float64, 1), (np.float32, 0)):
        Jd, bd = J.astype(dtype).astype(np.float64), b.astype(dtype).astype(np.float64)
        Jt, bt = upload(Jd, bd, dtype)
        e = torch.empty(C, dtype=torch.float64, device="cuda")
        _lib.call("tsu_dense_energy", _lib.ptr(Jt), code, _lib.ptr(bt), _lib.ptr(st), C, N, _lib.ptr(e),
                  _lib.current_stream())
        got = e.cpu().numpy()
        for c in range(C):
            assert got[c] == pytest.approx(D.compute_energy(S[c], Jd, bd), abs=1e-9), (dtype, c)


# ------------------------------------------------------------------------------------------------ decision edges
@gpu
@pytest.mark.parametrize("N,order_mode", [(24, "sequential"), (24, "random"), (40, "sequential"), (40, "random"),
                                          (600, "sequential"), (600, "random")])
def test_uniforms_on_p_fallback_band_and_clamp(N, order_mode):
    """float64 fields decide by logit(u) < h / T and fall back to the reference's u < sigmoid(h / T) within 1e-4 (in
    logit units) and next to the +-20 clamp.  Uniforms placed on p, one ulp below / above it, with logits just inside
    (0.9e-4) and just outside (1.1e-4) the band on both sides, and fields on both sides of the clamp must give the
    reference's bits - on the warp kernel (N = 24) and the block kernel (N = 40, 600).

    The fallback evaluates p with CUDA's exp, which is not correctly rounded: where it gives another p than numpy's for
    some h / T the reference's bit at u = p is not the kernel's to reproduce, so those visits get a random uniform
    instead (counted and printed)."""
    import torch

    rng = np.random.default_rng(N + (order_mode == "random"))
    n_sweeps, T = 4, 0.5
    k = 2 if N <= 40 else 5                         # fields O(1): h / T mostly inside the clamp
    m = rng.integers(-3, 4, size=(N, N))
    J = (np.triu(m) + np.triu(m, 1).T) * 2.0 ** -k
    J[0, 1] = J[1, 0] = 30.0                         # fields far beyond the clamp once both are up
    J[2, 3] = J[3, 2] = -30.0
    b = rng.integers(-2**k, 2**k + 1, size=N) * 2.0 ** -k
    for site, bias in ((4, 20.0 * T), (5, -20.0 * T), (6, 20.0 * T + 2.0 ** -k), (7, -20.0 * T - 2.0 ** -k)):
        J[site, :] = J[:, site] = 0.0                # h / T exactly +-20 (not clamped, strict >) and just beyond
        b[site] = bias
    # every h / T is a multiple of 2^-k / T: p of the device (same libdevice exp as the kernel) on that whole grid
    step = 2.0 ** -k / T
    top = int(np.ceil((np.abs(J).sum(1).max() + np.abs(b).max()) / T / step)) + 1
    xs = np.arange(-top, top + 1) * step
    xd = torch.from_numpy(xs).cuda()
    p_dev = (1.0 / (1.0 + torch.exp(-xd))).cpu().numpy()
    p_dev = np.where(xs > 20, 1.0, np.where(xs < -20, 0.0, p_dev))
    same_p = {float(x): float(pd) == D.sigmoid_ref(float(x)) for x, pd in zip(xs, p_dev)}
    s0 = rng.integers(0, 2, N)
    orders = np.stack([rng.permutation(N) for _ in range(n_sweeps)]) if order_mode == "random" else None
    state = s0.copy()
    U = np.zeros((n_sweeps, N))
    skipped = 0
    logistic = lambda z: 1.0 / (1.0 + np.exp(-z))  # noqa: E731
    for s in range(n_sweeps):
        for v, i in enumerate(range(N) if orders is None else orders[s]):
            x = float(np.dot(J[i, :], state) + b[i]) / T
            p = D.sigmoid_ref(x)
            choice = (s + v) % 8
            if choice < 3 and not same_p[x]:
                choice, skipped = 7, skipped + 1
            with np.errstate(over="ignore"):
                u = [p, np.nextafter(p, 0.0), np.nextafter(p, 1.0), logistic(x + 0.9e-4), logistic(x - 0.9e-4),
                     logistic(x + 1.1e-4), logistic(x - 1.1e-4), rng.random()][choice]
            u = min(max(u, 0.0), np.nextafter(1.0, 0.0))
            U[s, v] = u
            state[i] = 1 if u < p else 0
    want = D.gibbs_sweeps(s0, J, b, T, n_sweeps, U, orders)
    assert (want == state).all()
    print(f"N={N} {order_mode}: {skipped} of {n_sweeps * N} on-p placements moved (device exp differs from numpy's "
          f"at {sum(not v for v in same_p.values())} of {len(same_p)} grid values of h / T)")
    got = sampler(T, update_order=order_mode, seed=1).gibbs_sweep(s0, J, b, n_sweeps=n_sweeps, _uniforms=U,
                                                                  _orders=orders)
    assert (got == want).all(), np.flatnonzero(got != want)


# ------------------------------------------------------------------------------------------------ launch shapes
def _launch_shape_outputs(kind):
    """outputs of the float64 dense path that must not depend on the launch shape, keyed by name.
    kind 'small': N in {1, 2, 5, 16, 31, 32} (warp kernel by default, block kernel under TSU_DENSE_NO_WARP), Gaussian J,
    Philox mode: sample_boltzmann in random order, simulated_annealing, parallel_tempering, and one C-ABI run with
    per-sweep temperatures, samples, energies and best states.
    kind 'large': N in {700, 4097} (fields per thread set by TSU_DENSE_FPT), dyadic J, the same C-ABI runs."""
    import torch

    out = {}
    sizes = [1, 2, 5, 16, 31, 32] if kind == "small" else [700, 4097]
    for N in sizes:
        rng = np.random.default_rng(N)
        if kind == "small":
            J = rng.normal(size=(N, N))
            J = (J + J.T) / 2
            b = rng.normal(size=N) * 0.5
            smp = sampler(1.3, n_burnin=2, n_sweeps=2, update_order="random", seed=N)
            out[f"n{N}_boltzmann"] = smp.sample_boltzmann(J, b, n_samples=3, n_chains=3)
            best, e = sampler(seed=N + 1).simulated_annealing(J, b, T_initial=4.0, T_final=0.2, n_steps=20, n_chains=3)
            out[f"n{N}_anneal_state"], out[f"n{N}_anneal_energy"] = best, np.array([e])
            samples, info = sampler(1.0, n_burnin=2, n_sweeps=2, seed=N + 2).parallel_tempering(
                J, [0.5, 1.0, 2.0], b, n_samples=4, swap_interval=1)
            out[f"n{N}_pt_samples"] = samples
            out[f"n{N}_pt_energies"] = np.array(info["energies"])
            out[f"n{N}_pt_final"] = np.array(info["final_states"])
            out[f"n{N}_pt_swaps"] = np.array([info["swap_attempts"], info["swap_accepts"]])
        else:
            J, b = dyadic_problem(N, N)
        C, n_sweeps = 5, 4
        init = rng.integers(0, 2, (C, N)).astype(np.uint8)
        orders = np.stack([rng.permutation(N) for _ in range(n_sweeps)]).astype(np.int32)
        Jt, bt = upload(J, b, np.float64)
        r = dense_run(Jt, bt, torch.from_numpy(init).cuda(), T_sweep=np.array([3.0, 1.5, 0.7, 0.3]), n_burnin=1,
                      n_samples=3, sweeps_per_sample=1, order=orders, want_samples=True, want_energy=True,
                      track_best=True, seed=99, sweep0=4, chain0=6)
        for key, val in r.items():
            out[f"n{N}_run_{key}"] = val
        r = dense_run(Jt, bt, torch.from_numpy(init).cuda(), T_chain=np.array([0.4, 0.8, 1.0, 2.0, 5.0]),
                      n_burnin=n_sweeps, want_energy=True, seed=98, sweep0=1, chain0=2)
        out[f"n{N}_tchain_state"], out[f"n{N}_tchain_energy"] = r["state"], r["energy"]
    return out


def _launch_shape_in_subprocess(tmp_path, kind, env):
    """_launch_shape_outputs(kind) in a fresh process (the library reads TSU_DENSE_NO_WARP / TSU_DENSE_FPT once)"""
    path = os.path.join(str(tmp_path), f"{kind}.npz")
    code = ("import sys, numpy as np; sys.path[:0] = [sys.argv[1], sys.argv[2]]; "
            "from test_dense_block_kernel_gpu import _launch_shape_outputs; "
            "np.savez(sys.argv[4], **_launch_shape_outputs(sys.argv[3]))")
    full_env = dict(os.environ, **env)
    res = subprocess.run([sys.executable, "-c", code, ROOT, HERE, kind, path], cwd=ROOT, env=full_env,
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    with np.load(path) as z:
        return {k: z[k] for k in z.files}


def _assert_same_outputs(want, got, label):
    assert set(got) == set(want), label
    for key in want:
        a, g = np.asarray(want[key]), np.asarray(got[key])
        assert a.shape == g.shape and a.dtype == g.dtype, (label, key)
        if a.dtype.kind == "f":
            assert (a.view(np.uint64) == g.view(np.uint64)).all(), (label, key, a, g)
        else:
            assert (a == g).all(), (label, key)


@gpu
def test_no_warp_kernel_same_bits(tmp_path):
    """TSU_DENSE_NO_WARP=1 sends N <= 32 to the block kernel instead of the warp kernel, which is documented to change
    the launch shape only: bits, samples, energies and best states must be identical, N = 32 using bit 31 of the mask"""
    if os.environ.get("TSU_DENSE_NO_WARP") is not None or os.environ.get("TSU_DENSE_FPT") is not None:
        pytest.skip("this process already runs with a dense launch-shape override")
    want = _launch_shape_outputs("small")
    got = _launch_shape_in_subprocess(tmp_path, "small", {"TSU_DENSE_NO_WARP": "1"})
    _assert_same_outputs(want, got, "TSU_DENSE_NO_WARP=1")


@gpu
def test_fields_per_thread_same_bits(tmp_path):
    """TSU_DENSE_FPT sets the fields per thread (the block size): 1, 3 and 8 must give the default's bits, samples, best
    states and (dyadic J: exact) energies at N = 700 and 4097 (where 1 per thread hits the 1024-thread cap)"""
    if os.environ.get("TSU_DENSE_NO_WARP") is not None or os.environ.get("TSU_DENSE_FPT") is not None:
        pytest.skip("this process already runs with a dense launch-shape override")
    want = _launch_shape_outputs("large")
    for fpt in ("1", "3", "8"):
        got = _launch_shape_in_subprocess(tmp_path, "large", {"TSU_DENSE_FPT": fpt})
        _assert_same_outputs(want, got, f"TSU_DENSE_FPT={fpt}")


# ------------------------------------------------------------------------------------------------ the size limit
@gpu
def test_size_limit_raises_and_sampler_still_works():
    """float64 fields at N = 7036 and float32 at 13658 do not fit the kernel's shared memory: a ValueError naming the
    limit before anything runs, the sampler's Philox offsets untouched, and a following valid call correct.  The native
    entry point agrees with the host bound (TSU_ERR_UNSUPPORTED one past it)."""
    import torch
    from tsu_emulator_b200 import _lib
    from tsu_emulator_b200.gibbs import DENSE_MAX_N

    J, b = dyadic_problem(64, 64)
    rng = np.random.default_rng(64)
    init = rng.integers(0, 2, (3, 64))
    for precision, code, n in (("float64", 1, 7036), ("float32", 0, 13658)):
        assert DENSE_MAX_N[precision] == n - 1
        smp = sampler(1.0, seed=12, precision=precision)
        with pytest.raises(ValueError, match=f"at most {n - 1} bits"):
            smp.sample_chains(np.zeros((n, n)), n_chains=2, n_sweeps=1)
        with pytest.raises(ValueError, match=f"at most {n - 1} bits"):
            smp.gibbs_sweep(np.zeros(n, dtype=int), np.zeros((n, n)))
        out = smp.sample_chains(J, b, n_chains=3, n_sweeps=2, initial_state=init)
        S = init
        for s in range(2):
            S = sweep_vec(S, J, b, 1.0, philox_sweep(12, 0, 3, s, np.arange(64)))
        assert (out == S).all(), precision
        Jt = torch.zeros((n, n), dtype=torch.float64 if code else torch.float32, device="cuda")
        st = torch.zeros((1, n), dtype=torch.uint8, device="cuda")
        with pytest.raises(_lib.TsuNativeError) as err:
            dense_run(Jt, None, st, n_burnin=1)
        assert err.value.code == _lib.TSU_ERR_UNSUPPORTED
        del Jt


# ------------------------------------------------------------------------------------------------ CPU: the helpers
def test_vectorised_oracle_matches_gibbs_sweeps():
    """sweep_vec equals D.gibbs_sweeps chain by chain (dyadic and Gaussian J, bias or none, sequential, random and
    partial visiting orders, per-chain temperatures); replay equals D.tc_sweep_disagreements; energy_vec equals
    D.compute_energy"""
    rng = np.random.default_rng(0)
    for N, C, family in ((5, 3, "dyadic"), (33, 4, "dyadic"), (40, 3, "gauss"), (70, 5, "gauss")):
        J, b = dyadic_problem(N, N, asymmetric=N == 33) if family == "dyadic" else sk_problem(N, N)
        if family == "gauss":
            J = J + np.diag(rng.normal(size=N))
        for bias in (b, None):
            T = rng.choice([0.5, 1.0, 2.0], C)
            init = rng.integers(0, 2, (C, N))
            for order in (None, rng.permutation(N), rng.permutation(N)[: N // 2]):
                NV = N if order is None else len(order)
                U = rng.random((C, NV))
                got = sweep_vec(init, J, bias, T, U, order)
                for c in range(C):
                    want = D.gibbs_sweeps(init[c], J, bias, T[c], 1, U[c][None], None if order is None else order[None])
                    assert (got[c] == want).all(), (N, family, c)
            e = energy_vec(init, J, bias)
            assert np.allclose(e, [D.compute_energy(init[c], J, bias) for c in range(C)], rtol=0, atol=1e-12)
            # replay against a trajectory with some bits flipped on purpose
            U = rng.random((C, N))
            after = sweep_vec(init, J, bias, T, U)
            after[:, rng.integers(N, size=3)] ^= 1
            found = replay(init, after, J, bias, T, U)
            for c in range(C):
                ref = D.tc_sweep_disagreements(init[c], after[c], J, bias, T[c], U[c])
                assert [(s, pytest.approx(e)) for s, e in ref] == [(s, e) for cc, s, e in found if cc == c]
    assert sweep_vec(np.zeros((1, 2)), np.zeros((2, 2)), np.array([50.0, -50.0]), 1.0, np.full((1, 2), 0.5)).tolist() \
        == [[1, 0]]                                 # the +-20 clamp


def test_dense_size_limit_is_checked_on_the_host():
    """_DenseProblem names the dense kernel's limit before it touches the device"""
    from tsu_emulator_b200.gibbs import DENSE_MAX_N, _DenseProblem

    for precision, n in DENSE_MAX_N.items():
        with pytest.raises(ValueError, match=f"precision='{precision}'.*at most {n} bits.*got {n + 1}"):
            _DenseProblem(np.zeros((n + 1, n + 1)), None, precision, None)
