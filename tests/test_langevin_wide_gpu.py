"""Langevin sampling above 64 coordinates: the wide kernels (csrc/langevin_wide.cu) behind tsu_langevin_run.

Every coordinate draws the normal of the register kernel (same Philox block and element) and evaluates its gradient and
update through the same device functions, so a coordinate that does not couple to the others has the register
kernel's bits at any dim.  The embedding tests check exactly that; the others check the sampler against the reference
loop, a float64 NumPy replay, chain slicing, its stationary law and the public API."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

QUADRATIC, MIXTURE, DOUBLE_WELL, QUADRATIC_FORM = 0, 1, 2, 3
CAP = {"float64": 131072, "float32": 262144}
QFORM_CAP = 2048
NP_DTYPE = {"float64": np.float64, "float32": np.float32}


def abi_run(dtype, n_chains, dim, kind, params, x_init, *, jitter=0.1, first_exact=1, T=1.0, dt=0.01, gamma=1.0,
            n_burnin=3, n_steps=4, seed=7, chain0=0, normals=None, traj=True):
    """tsu_langevin_run on device copies of the arguments; returns (x, traj) as NumPy arrays of the chain dtype"""
    import torch
    from tsu_emulator_b200 import _lib
    from tsu_emulator_b200._lib import ptr

    tdt = torch.float64 if dtype == "float64" else torch.float32
    dev = torch.device("cuda")
    p = torch.from_numpy(np.ascontiguousarray(params, dtype=np.float64)).to(dev)
    x0 = torch.from_numpy(np.ascontiguousarray(x_init, dtype=np.float64)).to(dev, tdt)
    x = torch.empty((n_chains, dim), dtype=tdt, device=dev)
    tr = torch.empty((n_chains, n_steps, dim), dtype=tdt, device=dev) if traj else None
    nrm = None if normals is None else torch.from_numpy(np.ascontiguousarray(normals)).to(dev, tdt)
    _lib.call("tsu_langevin_run", ptr(x), 1 if dtype == "float64" else 0, int(n_chains), int(dim), int(kind), ptr(p),
              int(p.numel()), ptr(x0), float(jitter), int(first_exact), float(T), float(dt), float(gamma),
              int(n_burnin), int(n_steps), int(seed), int(chain0), ptr(nrm), ptr(tr), _lib.current_stream())
    return x.cpu().numpy(), (tr.cpu().numpy() if traj else None)


def energy_params(kind, dim, rng, k=None):
    """parameters of a `dim`-dimensional energy; with k, also those of its decoupled first k coordinates"""
    if kind == QUADRATIC:
        mu, w = rng.normal(size=dim), rng.uniform(0.5, 2.0, size=dim)
        big = np.concatenate([[0.7], mu, w])
        small = None if k is None else np.concatenate([[0.7], mu[:k], w[:k]])
        return big, small
    if kind == DOUBLE_WELL:
        return np.array([0.6, 1.3]), np.array([0.6, 1.3])
    # QUADRATIC_FORM: A = diag(A1, A2), asymmetric blocks
    def block(n):
        return 1.5 * np.eye(n) + 0.3 * rng.normal(size=(n, n)) / np.sqrt(n)

    k = dim if k is None else k
    A = np.zeros((dim, dim))
    A[:k, :k] = block(k)
    if dim > k:
        A[k:, k:] = block(dim - k)
    b = rng.normal(size=dim)
    big = np.concatenate([A.ravel(), b])
    small = np.concatenate([A[:k, :k].ravel(), b[:k]])
    return big, small


# ------------------------------------------------------------------------------------------------ 1. embedding
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("kind", [QUADRATIC, DOUBLE_WELL, QUADRATIC_FORM])
@pytest.mark.parametrize("injected", [False, True])
def test_first_coordinates_equal_a_register_run(dtype, kind, injected):
    """the first k coordinates of a dim-dimensional run are, bit for bit, the k-dimensional register-kernel run
    (k = 1 and 10 have templated kernels, 64 the generic one); final states and trajectories"""
    cap = QFORM_CAP if kind == QUADRATIC_FORM else CAP[dtype]
    dims = [65, 100, 257, 1024, cap]
    rng = np.random.default_rng(100 + kind)
    n_chains, nb, ns = 5, 3, 4
    for di, dim in enumerate(dims):
        for k in (1, 10, 64):
            big, small = energy_params(kind, dim, rng, k)
            x_init = rng.normal(size=dim)
            first_exact = (di + k) % 2
            normals = None
            if injected:
                normals = rng.normal(size=(n_chains, 1 + nb + ns, dim)).astype(NP_DTYPE[dtype])
            kw = dict(first_exact=first_exact, n_burnin=nb, n_steps=ns, seed=11 + di, chain0=3 * di)
            xb, tb = abi_run(dtype, n_chains, dim, kind, big, x_init, normals=normals, **kw)
            xs, ts = abi_run(dtype, n_chains, k, kind, small, x_init[:k],
                             normals=None if normals is None else normals[:, :, :k], **kw)
            assert np.isfinite(xb).all()
            assert np.array_equal(xb[:, :k], xs), (dim, k, np.abs(xb[:, :k] - xs).max())
            assert np.array_equal(tb[:, :, :k], ts), (dim, k)


# ------------------------------------------------------------------------------------------------ 2. reference loop
@pytest.mark.parametrize("dtype,atol", [("float64", 1e-7), ("float32", 5e-4)])
@pytest.mark.parametrize("dim", [65, 128])
def test_all_kinds_match_the_reference_loop(dtype, atol, dim):
    """injected normals through ThermalSamplingUnit and through the oracle's restatement of core.py:100-162
    (numerical gradient), for the four built-in kinds"""
    from oracle import langevin_oracle as LO
    from tsu_emulator_b200 import (DoubleWellEnergy, MixtureEnergy, QuadraticEnergy, QuadraticFormEnergy,
                                   ThermalSamplingUnit, TSUConfig)

    rng = np.random.default_rng(dim)
    mu, w = rng.normal(size=dim), rng.uniform(0.5, 2.0, size=dim)
    M = rng.normal(size=(dim, dim)) / np.sqrt(dim)
    A = np.eye(dim) + 0.5 * (M + M.T) / 2
    bq = rng.normal(size=dim)
    centres = rng.normal(size=(3, dim)) * 0.3
    wts = np.array([0.2, 0.5, 0.3])
    cases = [
        (QuadraticEnergy(0.8, mu, w), lambda x: float(0.8 * np.sum(w * (x - mu) ** 2))),
        (DoubleWellEnergy(0.5, 1.2), lambda x: float(np.sum(0.5 * (x * x - 1.2) ** 2))),
        (QuadraticFormEnergy(A, bq), lambda x: float(0.5 * x @ A @ x - bq @ x)),
        (MixtureEnergy(centres, wts), LO.mixture_energy(list(centres), wts)),
    ]
    cfg = TSUConfig(temperature=0.7, dt=0.02, friction=1.2, n_burnin=5, n_steps=8)
    n = 3
    x_init = rng.normal(size=dim) * 0.2
    normals = rng.normal(size=(n, 1 + cfg.n_burnin + cfg.n_steps, dim))
    for energy, fn in cases:
        got, traj = ThermalSamplingUnit(cfg, dtype=dtype, seed=1).sample_from_energy(
            energy, x_init, n, return_trajectory=True, _normals=normals)
        want, wtraj = LO.sample_from_energy(fn, x_init, n, normals, temperature=cfg.temperature, dt=cfg.dt,
                                            friction=cfg.friction, n_burnin=cfg.n_burnin, n_steps=cfg.n_steps,
                                            return_trajectory=True)
        assert got.shape == (n, dim)
        assert np.allclose(got, want, rtol=0, atol=atol), (type(energy).__name__, np.abs(got - want).max())
        assert np.allclose(np.array(traj), np.array(wtraj), rtol=0, atol=atol), type(energy).__name__


# ------------------------------------------------------------------------------------------------ 3. NumPy replay
def replay(grad, x_init, normals, *, jitter, first_exact, T, dt, gamma, n_burnin, n_steps):
    """float64 replay of tsu_langevin_run on injected normals with an analytic gradient of all chains at once"""
    x = x_init[None, :] + jitter * normals[:, 0, :]
    if first_exact:
        x[0] = x_init
    noise = np.sqrt(2.0 * T * dt / gamma)
    traj = []
    for s in range(n_burnin + n_steps):
        x = x + (-grad(x) * (dt / gamma)) + noise * normals[:, 1 + s, :]
        if s >= n_burnin:
            traj.append(x.copy())
    return x, np.stack(traj, axis=1)


# Largest |kernel - replay| measured on a B200 (DESIGN.md section 2): 2.2e-15 (QUADRATIC_FORM), 4.4e-16 (MIXTURE)
REPLAY_ATOL = {QUADRATIC_FORM: 1e-13, MIXTURE: 1e-13}


@pytest.mark.parametrize("dim", [512, 2048, "cap"])
@pytest.mark.parametrize("kind", [QUADRATIC_FORM, MIXTURE])
def test_large_dim_replay(kind, dim):
    """dense random asymmetric QUADRATIC_FORM (through the C-ABI) and MIXTURE against a float64 NumPy replay"""
    dim = (QFORM_CAP if kind == QUADRATIC_FORM else CAP["float64"]) if dim == "cap" else dim
    rng = np.random.default_rng(dim + kind)
    n, nb, ns = 11, 4, 5
    T = 1.0
    if kind == QUADRATIC_FORM:
        A = np.eye(dim) + 0.5 * rng.normal(size=(dim, dim)) / np.sqrt(dim)  # asymmetric
        b = rng.normal(size=dim)
        params = np.concatenate([A.ravel(), b])
        grad = lambda x: x @ A.T - b
        x_init, jitter = rng.normal(size=dim), 0.1
    else:
        K = 16
        c0 = rng.normal(size=dim)
        centres = c0[None, :] + rng.normal(size=(K, dim)) / np.sqrt(dim)
        p = rng.uniform(0.5, 1.5, size=K)
        p /= p.sum()
        params = np.concatenate([[K], p, centres.ravel()])
        T = 1.0 / dim  # keeps every d2_k of order 1, so that no weight underflows

        def grad(x):
            d = x[:, None, :] - centres[None, :, :]
            e = p[None, :] * np.exp(-0.5 * (d * d).sum(-1))
            return (e[:, :, None] * d).sum(1) / (e.sum(1) + 1e-10)[:, None]

        x_init, jitter = c0 + 0.2 * rng.normal(size=dim) / np.sqrt(dim), 1.0 / np.sqrt(dim)
    normals = rng.normal(size=(n, 1 + nb + ns, dim))
    kw = dict(jitter=jitter, first_exact=1, T=T, dt=0.02, gamma=1.1, n_burnin=nb, n_steps=ns)
    got, gtraj = abi_run("float64", n, dim, kind, params, x_init, normals=normals, **kw)
    want, wtraj = replay(grad, x_init, normals, **kw)
    err = max(np.abs(got - want).max(), np.abs(gtraj - wtraj).max())
    print(f"replay kind={kind} dim={dim} max|kernel - replay| = {err:.3e}")
    assert err < REPLAY_ATOL[kind], err


# ------------------------------------------------------------------------------------------------ 4. chain slicing
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("kind", [QUADRATIC, DOUBLE_WELL, QUADRATIC_FORM, MIXTURE])
def test_chain_slices_equal_one_launch(dtype, kind):
    """one launch of 77 chains = slices launched with chain0 offsets (the last CTA tile of every kernel is partial)"""
    dim = 150
    rng = np.random.default_rng(5 + kind)
    if kind == MIXTURE:
        centres = rng.normal(size=(5, dim)) * 0.1
        params = np.concatenate([[5], np.full(5, 0.2), centres.ravel()])
    else:
        params, _ = energy_params(kind, dim, rng)
    x_init = rng.normal(size=dim) * 0.1
    kw = dict(first_exact=0, n_burnin=3, n_steps=3, seed=99)
    full, ftraj = abi_run(dtype, 77, dim, kind, params, x_init, chain0=1000, **kw)
    for lo, hi in [(0, 9), (9, 40), (40, 77)]:
        part, ptraj = abi_run(dtype, hi - lo, dim, kind, params, x_init, chain0=1000 + lo, **kw)
        assert np.array_equal(part, full[lo:hi]), (lo, hi)
        assert np.array_equal(ptraj, ftraj[lo:hi]), (lo, hi)


def test_successive_calls_draw_fresh_chains():
    from tsu_emulator_b200 import QuadraticEnergy, ThermalSamplingUnit, TSUConfig

    cfg = TSUConfig(n_burnin=5, n_steps=5)
    x0 = np.linspace(-1, 1, 300)
    tsu = ThermalSamplingUnit(cfg, seed=21)
    a = tsu.sample_from_energy(QuadraticEnergy(), x0, 40)
    b = tsu.sample_from_energy(QuadraticEnergy(), x0, 40)
    both = ThermalSamplingUnit(cfg, seed=21).sample_from_energy(QuadraticEnergy(), x0, 80)
    assert not np.array_equal(a, b)
    assert np.array_equal(a, both[:40])
    # the second call's chains are chains 40.. of the stream; only its first chain starts exactly at x_init
    assert np.array_equal(b[1:], both[41:])
    assert tsu.sample_count == 80


# ------------------------------------------------------------------------------------------------ 5. statistics
def test_quadratic_form_stationary_law_256():
    """E = 1/2 x^T A x - b^T x under Euler-Maruyama: N(A^-1 b, T (A - (h/2) A^2)^-1), h = dt / gamma"""
    from tsu_emulator_b200 import QuadraticFormEnergy, ThermalSamplingUnit, TSUConfig

    d, n = 256, 100000
    rng = np.random.default_rng(3)
    Q, _ = np.linalg.qr(rng.normal(size=(d, d)))
    A = (Q * rng.uniform(1.0, 3.0, size=d)) @ Q.T
    A = 0.5 * (A + A.T)
    b = rng.normal(size=d)
    T, dt = 0.8, 0.05
    cfg = TSUConfig(temperature=T, dt=dt, friction=1.0, n_burnin=400, n_steps=1)
    mean = np.linalg.solve(A, b)
    cov = T * np.linalg.inv(A - 0.5 * dt * A @ A)
    s = ThermalSamplingUnit(cfg, seed=17).sample_from_energy(QuadraticFormEnergy(A, b), mean, n)
    assert s.shape == (n, d)
    se_mean = np.sqrt(np.diag(cov) / n)
    assert np.abs(s.mean(0) - mean).max() < 5 * se_mean.max()
    assert (np.abs(s.mean(0) - mean) < 5 * se_mean).all()
    emp = np.cov(s, rowvar=False)
    sd = np.sqrt(np.diag(cov))
    se_cov = np.sqrt((np.outer(sd, sd) ** 2 + cov ** 2) / n)
    z = np.abs(emp - cov) / se_cov
    assert z.max() < 5, z.max()


def test_isotropic_quadratic_4096_variance():
    from tsu_emulator_b200 import QuadraticEnergy, ThermalSamplingUnit, TSUConfig

    tsu = ThermalSamplingUnit(TSUConfig(temperature=1.0, dt=0.01, friction=1.0, n_burnin=100, n_steps=500), seed=8)
    s = tsu.sample_from_energy(QuadraticEnergy(), np.zeros(4096), 10000)
    assert s.shape == (10000, 4096)
    assert abs(s.var() - 0.505) < 0.001 and abs(s.mean()) < 0.001


def test_double_well_1000_both_wells_in_every_coordinate():
    from tsu_emulator_b200 import ThermalSamplingUnit, TSUConfig

    s = ThermalSamplingUnit(TSUConfig(temperature=0.5, n_burnin=200, n_steps=800), seed=2).sample_from_energy(
        "double_well", np.zeros(1000), 4000)
    frac = (s > 0).mean(0)
    assert frac.min() > 0.35 and frac.max() < 0.65
    assert abs(np.abs(s).mean() - 1.0) < 0.15


def test_bayesian_linear_model_100_features():
    from tsu_emulator_b200 import TSUConfig
    from tsu_emulator_b200.api import BayesianSampler

    rng = np.random.default_rng(0)
    d = 100
    X = rng.normal(size=(200, d))
    y = X @ rng.normal(size=d) + 0.3 * rng.normal(size=200)
    b = BayesianSampler(lambda th, X_, y_: -0.5 * np.sum((y_ - X_ @ th) ** 2), lambda th: -0.5 * np.sum(th ** 2), X, y,
                        dim=d, config=TSUConfig(dt=0.002, n_burnin=1000, n_steps=200), seed=4)
    post = b.sample(4000)
    assert post.shape == (4000, d)
    A = X.T @ X + np.eye(d)
    mean = np.linalg.solve(A, X.T @ y)
    cov = np.linalg.inv(A - 0.5 * 0.002 * A @ A)  # Euler-Maruyama stationary covariance, T = 1
    se = np.sqrt(np.diag(cov) / 4000)
    assert (np.abs(post.mean(0) - mean) < 5 * se).all(), (np.abs(post.mean(0) - mean) / se).max()


# ------------------------------------------------------------------------------------------------ 6. API
def test_api_shapes_above_64():
    from tsu_emulator_b200 import ThermalSamplingUnit, TSUConfig
    from tsu_emulator_b200.api import MultimodalSampler

    tsu = ThermalSamplingUnit(TSUConfig(n_burnin=100, n_steps=500), seed=9)
    out = tsu.sample_boltzmann(lambda x: (x ** 2).sum(), n_samples=5000, dim=200)
    assert out.shape == (5000, 200) and out.dtype == np.float64
    assert abs(out.var() - 0.505) < 0.01 and abs(out.mean()) < 0.01
    assert tsu.sample_count == 5000

    # T = 0.1 keeps |x - c|^2 near 13: at T = 1 it is near 128 in 128 dimensions, every p_k exp(-|x - c_k|^2 / 2) falls
    # far below the energy's + 1e-10 (tsu/api.py:143-149) and the landscape is flat, for the reference as well
    c = np.zeros((2, 128))
    c[0, 0], c[1, 0] = -3.0, 3.0
    m = MultimodalSampler(centers=list(c), weights=[1.0, 1.0], config=TSUConfig(temperature=0.1, n_burnin=200, n_steps=800),
                          seed=3)
    x = m.sample(2000)
    assert x.shape == (2000, 128)
    near = np.minimum(np.abs(x[:, 0] + 3.0), np.abs(x[:, 0] - 3.0))
    assert near.mean() < 0.5 and np.abs(x[:, 1:]).mean() < 0.5

    cfg = TSUConfig(n_burnin=10, n_steps=6)
    t = ThermalSamplingUnit(cfg, seed=5)
    s, traj = t.sample_boltzmann(lambda x: (x ** 2).sum(), n_samples=7, dim=200, return_trajectory=True)
    assert s.shape == (7, 200) and len(traj) == 7 * 6 and traj[0].shape == (200,)
    assert all(np.array_equal(traj[c * 6 + 5], s[c]) for c in range(7))
    xt, tt = ThermalSamplingUnit(cfg, seed=5, dtype="float32").sample_from_energy(
        "quadratic", np.zeros(200), 7, return_trajectory=True, as_tensor=True)
    assert tuple(xt.shape) == (7, 200) and tuple(tt.shape) == (7, 6, 200) and xt.is_cuda
    assert bool((tt[:, -1] == xt).all())
    assert t.sample_count == 7
