"""Population annealing on GibbsSampler (tsu_population_resample, tsu_population_moments and the back ends' sweeps).

With dyadic couplings and bias every energy the device computes is exact, so every resampling decision is exact too: a
run must equal a host replay built from the sampler's Philox initial states, exact host energies, the resampling
step of tests/population_resample.py, a host gather and the same back end's C-ABI sweep at T_k, sweep0 + k theta and
chain0.  The bf16 (tensor-core), float64, float32 and chromatic back ends are each replayed; the C entry points are
checked on their own for row layouts, population blocks and a 2^20-chain population; the estimates are checked against
exact enumeration of a 16-bit model.
"""
import itertools
import math

import numpy as np
import pytest

from oracle import population_oracle as PO
from population_resample import resample_populations
from test_dense_block_kernel_gpu import dyadic_problem
from test_dense_tc_anneal_gpu import SK_ENERGY_BOUND, device_energy_ref, init_states, padded
from test_dense_tc_kernel_gpu import _dev, energy_ref, sk_problem, tc_launch, upload_j

gpu = pytest.mark.gpu
M32 = 0xFFFFFFFF
SENTINEL = 0xA5


# ------------------------------------------------------------------------------------------------ problems
def random_graph(N, seed, density=0.1):
    """symmetric sparse couplings m / 4 (m in +-1..3), zero diagonal, bias in multiples of 1/4: dyadic"""
    rng = np.random.default_rng(seed)
    mask = np.triu(rng.random((N, N)) < density, 1)
    m = np.where(mask, rng.integers(1, 4, (N, N)) * rng.choice([-1, 1], (N, N)), 0)
    J = (m + m.T) * 0.25
    return J, rng.integers(-4, 5, N) * 0.25


def ea_cubic(L, seed):
    """periodic L x L x L Edwards-Anderson +-J couplings, no bias"""
    rng = np.random.default_rng(seed)
    N = L ** 3
    J = np.zeros((N, N))
    for x, y, z in itertools.product(range(L), repeat=3):
        i = (x * L + y) * L + z
        for j in (((x + 1) % L * L + y) * L + z, (x * L + (y + 1) % L) * L + z, (x * L + y) * L + (z + 1) % L):
            J[i, j] = J[j, i] = rng.choice([-1.0, 1.0])
    return J, None


def csr(J):
    from tsu_emulator_b200.sparse import to_csr

    return to_csr(J)


class Backend:
    """a back end of GibbsSampler and its C-ABI sweep, for a dyadic (J, b)"""

    def __init__(self, kind, J, b):
        import torch
        from tsu_emulator_b200.sparse import SparseProblem

        self.kind, self.J, self.b, self.N = kind, J, b, J.shape[0]
        self.precision = "float64" if kind == "chromatic" else kind
        self.coupling = csr(J) if kind == "chromatic" else J
        self.width = (self.N + 127) // 128 * 128 if kind == "bf16" else self.N
        if kind == "bf16":
            Jp, bp = padded(J, b, self.width)
            self.Jd, _ = upload_j(Jp)
            self.bd = _dev(bp, np.float32)
        elif kind == "chromatic":
            self.sp = SparseProblem(self.coupling, b, torch.device("cuda"))
        else:
            dt = np.float64 if kind == "float64" else np.float32
            self.code = 1 if kind == "float64" else 0
            self.Jt, self.bd = _dev(J.T, dt), _dev(b, dt)

    def sampler(self, seed):
        from tsu_emulator_b200 import GibbsSampler

        return GibbsSampler(seed=seed, precision=self.precision)

    def anneal(self, smp, Ts, **kw):
        return smp.population_annealing(self.coupling, Ts, self.b, chromatic=self.kind == "chromatic", **kw)

    def sweep(self, st, n, T, seed, sweep0, chain0):
        """n sweeps at T of the device states st ([C, width] uint8, in place) through the back end's C entry point"""
        from tsu_emulator_b200 import _lib
        from tsu_emulator_b200._lib import ptr

        C = int(st.shape[0])
        if self.kind == "bf16":
            tc_launch(self.Jd, self.bd, st, n, seed, sweep0, chain0, T=T)
        elif self.kind == "chromatic":
            sp = self.sp
            _lib.call("tsu_sparse_gibbs_run", ptr(sp.rowptr), ptr(sp.col), ptr(sp.val), ptr(sp.bias), ptr(sp.cptr),
                      ptr(sp.sites), sp.n_colours, ptr(st), C, self.N, float(T), None, None, int(n), 0, 0, None, None,
                      None, 0, None, None, seed, sweep0 & M32, chain0 & M32, _lib.current_stream())
        else:
            _lib.call("tsu_dense_gibbs_run", ptr(self.Jt), self.code, ptr(self.bd), ptr(st), C, self.N, float(T), None,
                      None, int(n), 0, 0, None, None, None, None, 0, None, None, seed, sweep0 & M32, chain0 & M32,
                      self.code, 0, _lib.current_stream())
        return st

    def energy(self, S):
        """exact float64 energies of host states [C, width]"""
        return energy_ref(np.asarray(S)[:, :self.N], self.J, self.b)


BACKENDS = {
    "bf16-100": ("bf16", lambda: dyadic_problem(100, 1)),
    "bf16-384": ("bf16", lambda: dyadic_problem(384, 2)),
    "float64-33": ("float64", lambda: dyadic_problem(33, 3)),
    "float64-70": ("float64", lambda: dyadic_problem(70, 4)),
    "float32-70": ("float32", lambda: dyadic_problem(70, 5, dtype=np.float32)),
    "chromatic-graph60": ("chromatic", lambda: random_graph(60, 6)),
    "chromatic-ea4": ("chromatic", lambda: ea_cubic(4, 7)),
}
SHAPES = [(1, 64), (3, 5), (4, 75)]
SCHEDULE = [3.0, 1.5, 0.8, 0.4]   # from T_start = inf; the last dbeta duplicates or drops most chains
THETA = 3


def backend(name):
    kind, make = BACKENDS[name]
    J, b = make()
    return Backend(kind, np.asarray(J, dtype=np.float64), b)


def moments_of(E, P):
    E = np.asarray(E).reshape(P, -1)
    return np.stack([E.sum(1), (E * E).sum(1)], axis=1)


def replay(be, S, family, E, Ts, dbeta, P, seed, sweep0, chain0):
    """host replay of population_annealing from host states S [C, width] with energies E; returns the final states,
    family, energies, weight sums, E_ref and moments"""
    n = len(Ts)
    W, eref, mom = [], [], [moments_of(E, P)]
    for k in range(n):
        parents, family, w, e = resample_populations(E, family, dbeta[k], seed, chain0, sweep0 + k * THETA, P)
        W.append(w)
        eref.append(e)
        st = _dev(S[parents], np.uint8)
        S = be.sweep(st, THETA, Ts[k], seed, sweep0 + k * THETA, chain0).cpu().numpy()
        E = be.energy(S)
        mom.append(moments_of(E, P))
    return S, family, E, np.array(W, dtype=np.int64), np.array(eref), np.array(mom)


def assert_equals_replay(res, want, N):
    S, family, E, W, eref, mom = want
    assert np.array_equal(res.states.cpu().numpy(), S[:, :N]), "final states"
    assert np.array_equal(res._state.cpu().numpy(), S), "padding stays zero"
    assert res.family.cpu().numpy().tolist() == [f - (1 << 32) if f >= 1 << 31 else f for f in family], "family"
    assert np.array_equal(res.weight_sum.cpu().numpy(), W), "weight_sum"
    assert np.array_equal(res.energy_ref.cpu().numpy(), eref), "energy_ref"
    assert np.array_equal(res.energy_moments.cpu().numpy(), mom), "energy_moments"
    assert np.array_equal(res.energy.cpu().numpy(), E), "energy"


def dbeta_of(Ts, T_start=math.inf):
    return np.diff(np.concatenate([[0.0 if math.isinf(T_start) else 1.0 / T_start], 1.0 / np.asarray(Ts)]))


# ------------------------------------------------------------------------------------------------ 1. host replay
@gpu
@pytest.mark.parametrize("P,r_pop", SHAPES)
@pytest.mark.parametrize("name", list(BACKENDS))
def test_equals_host_replay(name, P, r_pop):
    """a fresh run (chain0 = 5 after an earlier run of 5 chains) equals the host replay bit for bit, counters included"""
    be = backend(name)
    C, seed = P * r_pop, 4000 + P + r_pop
    if be.kind == "float32":  # the float32 fields and energies of this problem are exact: check before relying on it
        import torch
        from tsu_emulator_b200 import _lib

        S = np.random.default_rng(0).integers(0, 2, (64, be.N))
        e = torch.empty(64, dtype=torch.float64, device="cuda")
        _lib.call("tsu_dense_energy", _lib.ptr(be.Jt), 0, _lib.ptr(be.bd), _lib.ptr(_dev(S, np.uint8)), 64, be.N,
                  _lib.ptr(e), _lib.current_stream())
        assert np.array_equal(e.cpu().numpy(), be.energy(S))
    smp = be.sampler(seed)
    be.anneal(smp, [1.0], n_chains=5, sweeps_per_step=2)          # moves both counters away from 0
    sweep0, chain0 = smp._sweep_counter, smp._chain_counter
    res = be.anneal(smp, SCHEDULE, n_chains=C, n_populations=P, sweeps_per_step=THETA)
    S = init_states(seed, chain0 + sweep0, C, be.N, be.width)     # _initial_states: Philox keyed at the two counters
    want = replay(be, S, list(range(chain0, chain0 + C)), be.energy(S), SCHEDULE, dbeta_of(SCHEDULE), P, seed, sweep0,
                  chain0)
    assert_equals_replay(res, want, be.N)
    assert res.chain0 == chain0 and res.r_pop == r_pop and res.shift == PO.weight_shift(r_pop)
    assert smp._sweep_counter == sweep0 + len(SCHEDULE) * THETA and smp._chain_counter == chain0 + C
    assert smp.config.temperature == SCHEDULE[-1]
    assert (res.rho_t() >= 1).all()


# ------------------------------------------------------------------------------------------------ 2./3. continuation
@gpu
@pytest.mark.parametrize("name", ["bf16-100", "float64-33", "float32-70", "chromatic-graph60"])
def test_zero_dbeta_is_the_identity(name):
    """continuing at the last temperature: every parent is its child, W = R_p 2^s, and the states equal the same number
    of plain sweeps on that back end; the previous result's tensors are left as they were"""
    import torch

    be = backend(name)
    P, r_pop, seed = 3, 5, 11
    smp = be.sampler(seed)
    first = be.anneal(smp, [2.0, 0.5], n_chains=P * r_pop, n_populations=P, sweeps_per_step=THETA)
    kept = [t.clone() for t in (first._state, first.family, first.energy)]
    sweep0 = smp._sweep_counter
    res = be.anneal(smp, [0.5] * 3, n_chains=P * r_pop, n_populations=P, sweeps_per_step=THETA, previous=first)
    assert all(torch.equal(a, b) for a, b in zip(kept, (first._state, first.family, first.energy)))
    assert torch.equal(res.family, first.family)
    assert (res.weight_sum.cpu().numpy() == r_pop << PO.weight_shift(r_pop)).all()
    assert (res.dbeta == 0).all() and res.T_start == 0.5
    plain = be.sweep(first._state.clone(), 3 * THETA, 0.5, seed, sweep0, first.chain0)
    assert torch.equal(res._state, plain)
    assert np.array_equal(res.energy.cpu().numpy(), be.energy(plain.cpu().numpy()))
    assert smp._sweep_counter == sweep0 + 3 * THETA and smp._chain_counter == P * r_pop


@gpu
@pytest.mark.parametrize("name", ["bf16-384", "float64-70", "float32-70", "chromatic-ea4"])
def test_split_runs_equal_one_run(name):
    """steps 2 + 3 with previous= equal 5 steps in one call"""
    import torch

    be = backend(name)
    Ts = [4.0, 2.0, 1.0, 0.7, 0.5]
    kw = dict(n_chains=300, n_populations=4, sweeps_per_step=THETA)
    one = be.anneal(be.sampler(21), Ts, **kw)
    smp = be.sampler(21)
    a = be.anneal(smp, Ts[:2], **kw)
    b = be.anneal(smp, Ts[2:], previous=a, **kw)
    assert torch.equal(b._state, one._state) and torch.equal(b.family, one.family) and torch.equal(b.energy, one.energy)
    assert torch.equal(torch.cat([a.weight_sum, b.weight_sum]), one.weight_sum)
    assert torch.equal(torch.cat([a.energy_ref, b.energy_ref]), one.energy_ref)
    assert torch.equal(torch.cat([a.energy_moments[:2], b.energy_moments]), one.energy_moments)
    assert np.array_equal(np.concatenate([a.dbeta, b.dbeta]), one.dbeta)
    assert np.allclose(np.concatenate([a.log_z_ratio(), a.log_z_ratio()[-1] + b.log_z_ratio()]), one.log_z_ratio())
    assert smp._sweep_counter == 5 * THETA and smp._chain_counter == 300


# ------------------------------------------------------------------------------------------------ 4.-6. C entry points
def abi_resample(src, dst, fam, fam_out, energy, dbeta, C, P, row_bytes, seed, sweep, chain0):
    """tsu_population_resample on raw device addresses; returns (weight_sum, energy_ref)"""
    import torch
    from tsu_emulator_b200 import _lib
    from tsu_emulator_b200._lib import ptr

    work_bytes = int(_lib.load().tsu_ising2d_population_work_bytes(C, P))
    work = torch.empty(work_bytes // 8, dtype=torch.int64, device="cuda")
    ws = torch.empty(P, dtype=torch.int64, device="cuda")
    er = torch.empty(P, dtype=torch.float64, device="cuda")
    d_dbeta = torch.tensor([dbeta], dtype=torch.float64, device="cuda")
    _lib.call("tsu_population_resample", src, dst, ptr(fam), ptr(fam_out), ptr(energy), ptr(d_dbeta), C, P, row_bytes,
              seed, sweep, chain0, ptr(ws), ptr(er), ptr(work), work_bytes, _lib.current_stream())
    return ws, er


def random_energy(C, seed):
    return np.random.default_rng(seed).integers(-200, 200, C) * 0.125


@gpu
def test_populations_are_independent():
    """a block of whole populations run alone (its chain0, its slices) equals its slice of the whole call, for the
    resampling and for the moments"""
    import torch
    from tsu_emulator_b200 import _lib
    from tsu_emulator_b200._lib import ptr

    P, r_pop, row = 4, 75, 33
    C = P * r_pop
    src = _dev(np.random.default_rng(1).integers(0, 256, (C, row)), np.uint8)
    fam = torch.arange(C, dtype=torch.int32, device="cuda") * 7
    E = _dev(random_energy(C, 2), np.float64)
    chain0 = 0xFFFFFF00  # chain0 + p R_p wraps past 2^32
    out, fam_out = torch.empty_like(src), torch.empty_like(fam)
    ws, er = abi_resample(ptr(src), ptr(out), fam, fam_out, E, 0.3, C, P, row, 9, 77, chain0)
    mom = torch.empty((P, 2), dtype=torch.float64, device="cuda")
    _lib.call("tsu_population_moments", ptr(E), C, P, ptr(mom), _lib.current_stream())
    lo, hi = r_pop, 3 * r_pop
    o2, f2 = torch.empty_like(src[lo:hi]), torch.empty_like(fam[lo:hi])
    ws2, er2 = abi_resample(ptr(src[lo:hi]), ptr(o2), fam[lo:hi], f2, E[lo:hi], 0.3, hi - lo, 2, row, 9, 77,
                            (chain0 + lo) & M32)
    assert torch.equal(o2, out[lo:hi]) and torch.equal(f2, fam_out[lo:hi])
    assert torch.equal(ws2, ws[1:3]) and torch.equal(er2, er[1:3])
    mom2 = torch.empty((2, 2), dtype=torch.float64, device="cuda")
    _lib.call("tsu_population_moments", ptr(E[lo:hi]), hi - lo, 2, ptr(mom2), _lib.current_stream())
    assert torch.equal(mom2, mom[1:3])
    parents, fams, W, eref = resample_populations(E.cpu().numpy(), fam.cpu().numpy(), 0.3, 9, chain0, 77, P)
    assert torch.equal(out, src[torch.from_numpy(parents).cuda()]) and fam_out.cpu().tolist() == fams
    assert ws.cpu().tolist() == W and np.array_equal(er.cpu().numpy(), eref)
    assert np.array_equal(mom.cpu().numpy(), moments_of(E.cpu().numpy(), P))


@gpu
def test_gather_layouts():
    """row_bytes 1, 15, 16, 33 and 4096 at 16-byte aligned and odd base addresses (the uint4 and the byte path), chain
    counts on both sides of the gather's grouping (one group of threads per child, whole blocks per child, more
    children than a grid column): the rows equal the oracle's parents' rows and every byte around them keeps its
    sentinel"""
    import torch

    pad = 64
    for row in (1, 15, 16, 33, 4096):
        for C in (5, 300, 66000):
            if row == 4096 and C == 300:
                continue
            P = 3 if C % 3 == 0 else 1
            E = random_energy(C, row + C)
            rows = np.random.default_rng(row * C).integers(0, 256, (C, row)).astype(np.uint8)
            for off in (0, 1):
                src = torch.full((2 * pad + C * row,), SENTINEL, dtype=torch.uint8, device="cuda")
                dst = torch.full_like(src, SENTINEL)
                src[pad + off:pad + off + C * row] = torch.from_numpy(rows.reshape(-1)).cuda()
                fam = torch.arange(C, dtype=torch.int32, device="cuda")
                fam_out = torch.full((C + 2,), -7, dtype=torch.int32, device="cuda")
                base = src.data_ptr() + pad + off
                abi_resample(base, dst.data_ptr() + pad + off, fam, fam_out[1:], _dev(E, np.float64), 0.2, C, P, row,
                             5, 3, 1000)
                parents, _, _, _ = resample_populations(E, range(C), 0.2, 5, 1000, 3, P)
                got = dst.cpu().numpy()
                assert np.array_equal(got[pad + off:pad + off + C * row].reshape(C, row), rows[parents]), (row, C, off)
                assert (got[:pad + off] == SENTINEL).all() and (got[pad + off + C * row:] == SENTINEL).all()
                f = fam_out.cpu().numpy()
                assert np.array_equal(f[1:-1], parents) and f[0] == -7 and f[-1] == -7


@gpu
def test_one_population_of_a_million_chains():
    """2^20 + 3 chains in one population (the scan walks its 1025 tile totals in two chunks) equal the oracle"""
    import torch

    C = (1 << 20) + 3
    E = random_energy(C, 12)
    idx = torch.arange(C, dtype=torch.int32, device="cuda")
    out, fam_out = torch.empty_like(idx), torch.empty_like(idx)
    ws, er = abi_resample(idx.data_ptr(), out.data_ptr(), idx, fam_out, _dev(E, np.float64), 0.05, C, 1, 4, 31, 8, 0)
    parents, _, W, eref = resample_populations(E, range(C), 0.05, 31, 0, 8, 1)
    assert np.array_equal(out.cpu().numpy(), parents) and np.array_equal(fam_out.cpu().numpy(), parents)
    assert ws.cpu().tolist() == W and er.cpu().numpy()[0] == eref[0]


@gpu
def test_full_wave_sk():
    """18944 chains (one 128-chain tile per SM) at N = 4096, Gaussian SK couplings on bf16, 5 steps: W within
    [2^s, 2^62], valid families, and final energies within SK_ENERGY_BOUND of the float64 energies of the bf16 matrix"""
    import torch
    from tsu_emulator_b200 import GibbsSampler

    C, N = 18944, 4096
    J = sk_problem(N, 77)
    res = GibbsSampler(seed=8, precision="bf16").population_annealing(J, [2.0, 1.5, 1.0, 0.7, 0.5], n_chains=C)
    W = res.weight_sum.cpu().numpy()
    assert ((W >= 1 << res.shift) & (W <= 1 << 62)).all()
    fam = res.family.cpu().numpy()
    assert fam.min() >= 0 and fam.max() < C and res.rho_t()[0] >= 1
    J64 = torch.from_numpy(J).cuda()
    err = float((res.energy - device_energy_ref(res.states, J64, None)).abs().max())
    print(f"SK N={N} C={C}: rho_t = {res.rho_t()[0]:.2f}, max |E - E_float64| = {err:.3e}")
    assert err < SK_ENERGY_BOUND


# ------------------------------------------------------------------------------------------------ 7. physics
def small_model():
    """16 bits, symmetric couplings m / 4 (|m| <= 3, zero diagonal: the heat bath then samples exp(-E / T)) and bias in
    multiples of 1/4: exact in bf16"""
    rng = np.random.default_rng(16)
    m = np.triu(rng.integers(-3, 4, (16, 16)), 1)
    return (m + m.T) * 0.25, rng.integers(-4, 5, 16) * 0.25


@gpu
@pytest.mark.parametrize("kind", ["bf16", "float64", "chromatic"])
def test_estimates_match_exact_enumeration(kind):
    """T = inf to 0.5 in 40 steps of theta = 10, 32 populations of 512 chains: at three temperatures the mean over the
    populations of ln Z, <E> and the specific heat lie within 5 standard errors of exact enumeration, and the lowest
    final energy is the ground state"""
    J, b = small_model()
    be = Backend(kind, J, b)
    S = np.array(list(itertools.product((0, 1), repeat=16)), dtype=np.float64)
    E_all = energy_ref(S, J, b)
    Ts = 1.0 / np.linspace(2.0 / 40, 2.0, 40)
    res = be.anneal(be.sampler(123), Ts, n_chains=32 * 512, n_populations=32, sweeps_per_step=10)
    est = {"ln Z": 16 * math.log(2.0) + res.log_z_ratio(), "<E>": res.mean_energy(), "C": res.specific_heat()}
    for k in (9, 24, 39):
        x = -(E_all - E_all.min()) / Ts[k]
        w = np.exp(x)
        mean = (w * E_all).sum() / w.sum()
        exact = {"ln Z": -E_all.min() / Ts[k] + math.log(w.sum()), "<E>": mean,
                 "C": (w * (E_all - mean) ** 2).sum() / w.sum() / Ts[k] ** 2 / 16}
        for key, v in est.items():
            se = v[k].std(ddof=1) / math.sqrt(32)
            print(f"{kind} T={Ts[k]:.3f} {key}: {v[k].mean():.5f} +- {se:.5f}, exact {exact[key]:.5f}")
            assert abs(v[k].mean() - exact[key]) < 5 * se, (kind, k, key)
    assert float(res.energy.min()) == E_all.min()
