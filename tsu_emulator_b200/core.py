"""
Drop-in mirror of the reference's tsu/core.py Langevin engine (TSUConfig, ThermalSamplingUnit and
the exception types) with the sampling loop on the B200 (csrc/langevin.cu, tsu_langevin_run).

The reference differentiates an arbitrary Python `energy_fn` numerically (core.py:82-98) - 2*dim
Python callbacks per step.  A Python callable cannot run on the GPU and there is no CPU fallback, so
`sample_from_energy` resolves the energy in this order:
  1. built-in energy objects (QuadraticEnergy, GaussianEnergy, MixtureEnergy, DoubleWellEnergy) and their names;
  2. a Python callable that is *recognised* as an exact quadratic form: it is probed at 1 + 2d + d(d-1)/2
     points, the fitted quadratic is verified on random points, and the chain runs on the prebuilt kernel with the
     analytic gradient (README's `lambda x: (x**2).sum()`, core.py's Gaussian energy, core.py:227-230);
  3. any other callable is TRACED (tsu_emulator_b200/trace.py): called once on symbolic inputs, differentiated
     analytically, and its gradient compiled by NVRTC into the same chain loop (1-2 s per new function, cached).
     Double wells, mixtures written as Python loops, Rosenbrock-like landscapes, posteriors over data run this way;
  4. what cannot be traced - branches on the value of x, float(...) of an intermediate, calls into compiled code -
     raises SamplingError with the reason.
"""

from dataclasses import dataclass
from typing import Callable, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import ptr


class TSUError(Exception):
    """Base exception for TSU platform (tsu/core.py:12-15)"""

    pass


class ConfigurationError(TSUError):
    """Invalid configuration parameters (tsu/core.py:18-21)"""

    pass


class SamplingError(TSUError):
    """Error during sampling process (tsu/core.py:24-27)"""

    pass


@dataclass
class TSUConfig:
    """tsu/core.py:30-51 (same fields, defaults and validation)"""

    temperature: float = 1.0
    dt: float = 0.01
    friction: float = 1.0
    n_burnin: int = 100
    n_steps: int = 500

    def __post_init__(self):
        if self.temperature <= 0:
            raise ConfigurationError(f"Temperature must be positive, got {self.temperature}")
        if self.dt <= 0 or self.dt > 0.1:
            raise ConfigurationError(f"Time step dt must be in (0, 0.1], got {self.dt}")
        if self.friction <= 0:
            raise ConfigurationError(f"Friction must be positive, got {self.friction}")
        if self.n_burnin < 0:
            raise ConfigurationError(f"Burn-in steps must be non-negative, got {self.n_burnin}")
        if self.n_steps <= 0:
            raise ConfigurationError(f"Number of steps must be positive, got {self.n_steps}")


# ----------------------------------------------------------------------------- built-in energies
ENERGY_QUADRATIC, ENERGY_MIXTURE, ENERGY_DOUBLE_WELL, ENERGY_QUADRATIC_FORM = 0, 1, 2, 3

# Dimension limits (csrc/langevin_wide.cuh).  Up to 64 coordinates every energy runs on the register kernels; above
# that built-in energies and quadratic forms run on the wide kernels, traced energies do not run.
MAX_TRACED_DIM = 64
MAX_DIM = {"float64": 131072, "float32": 262144}  # 16-bit Philox block field x 2 (float64) or 4 (float32) normals
MAX_QUADRATIC_FORM_DIM = 2048                      # shared-memory chain tile of the wide QUADRATIC_FORM kernel
MAX_MIXTURE_CENTRES = 16                           # wide MIXTURE kernel: one thread per (chain, centre)


class BuiltinEnergy:
    """analytic energy evaluated (and differentiated) inside the fused Langevin kernel"""

    kind: int = -1

    def params(self, dim: int) -> np.ndarray:
        raise NotImplementedError

    def __call__(self, x):
        raise NotImplementedError


class QuadraticEnergy(BuiltinEnergy):
    """E(x) = a * sum_i w_i (x_i - mu_i)^2.  README.md:60-61 `(x**2).sum()` is a=1, mu=0, w=1."""

    kind = ENERGY_QUADRATIC

    def __init__(self, a: float = 1.0, mu=0.0, w=1.0):
        self.a, self.mu, self.w = float(a), mu, w

    def params(self, dim):
        mu = np.broadcast_to(np.asarray(self.mu, dtype=np.float64), (dim,))
        w = np.broadcast_to(np.asarray(self.w, dtype=np.float64), (dim,))
        return np.concatenate([[self.a], mu, w])

    def __call__(self, x):
        x = np.atleast_1d(np.asarray(x, dtype=np.float64))
        p = self.params(x.size)
        return float(self.a * np.sum(p[1 + x.size:] * (x - p[1:1 + x.size]) ** 2))


class GaussianEnergy(QuadraticEnergy):
    """E(x) = 1/2 sum ((x - mu)/sigma)^2  (tsu/core.py:227-230; tsu/api.py:124-126 uses the mean: reduce='mean')"""

    def __init__(self, mu=0.0, sigma=1.0, reduce: str = "sum"):
        sigma = np.asarray(sigma, dtype=np.float64)
        if np.any(sigma <= 0):
            raise ConfigurationError(f"Sigma must be positive, got {sigma}")
        self.reduce = reduce
        super().__init__(0.5, mu, 1.0 / sigma**2)

    def params(self, dim):
        p = super().params(dim)
        if self.reduce == "mean":
            p = p.copy()
            p[0] = 0.5 / dim
        return p


class MixtureEnergy(BuiltinEnergy):
    """E(x) = -log(sum_k p_k exp(-|x - c_k|^2 / 2) + 1e-10)  (tsu/api.py:143-149, tsu/demos.py:73-87)"""

    kind = ENERGY_MIXTURE

    def __init__(self, centers, weights):
        self.centers = np.atleast_2d(np.asarray(centers, dtype=np.float64))
        w = np.asarray(weights, dtype=np.float64)
        self.weights = w / w.sum()
        if self.weights.size != self.centers.shape[0]:
            raise ConfigurationError("one weight per centre")

    def params(self, dim):
        if self.centers.shape[1] != dim:
            raise SamplingError(f"mixture centres have dimension {self.centers.shape[1]}, state has {dim}")
        return np.concatenate([[float(len(self.weights))], self.weights, self.centers.ravel()])

    def __call__(self, x):
        x = np.atleast_1d(np.asarray(x, dtype=np.float64))
        d2 = ((x[None, :] - self.centers) ** 2).sum(1)
        return float(-np.log(np.sum(self.weights * np.exp(-0.5 * d2)) + 1e-10))


class DoubleWellEnergy(BuiltinEnergy):
    """E(x) = sum_i a (x_i^2 - b)^2"""

    kind = ENERGY_DOUBLE_WELL

    def __init__(self, a: float = 1.0, b: float = 1.0):
        self.a, self.b = float(a), float(b)

    def params(self, dim):
        return np.array([self.a, self.b])

    def __call__(self, x):
        x = np.atleast_1d(np.asarray(x, dtype=np.float64))
        return float(np.sum(self.a * (x * x - self.b) ** 2))


class QuadraticFormEnergy(BuiltinEnergy):
    """E(x) = 1/2 x^T A x - b^T x + c with symmetric A (what `recognise_quadratic` returns)"""

    kind = ENERGY_QUADRATIC_FORM

    def __init__(self, A, b, c=0.0):
        self.A = np.asarray(A, dtype=np.float64)
        self.b = np.asarray(b, dtype=np.float64)
        self.c = float(c)

    def params(self, dim):
        return np.concatenate([self.A.ravel(), self.b])

    def __call__(self, x):
        x = np.atleast_1d(np.asarray(x, dtype=np.float64))
        return float(0.5 * x @ self.A @ x - self.b @ x + self.c)

    def as_diagonal(self) -> Optional[QuadraticEnergy]:
        """separable form (the common case) runs on the cheaper QUADRATIC kernel path"""
        d = np.diag(self.A).copy()
        scale = max(1.0, float(np.max(np.abs(d)))) if d.size else 1.0
        if np.any(np.abs(self.A - np.diag(d)) > 1e-12 * scale):
            return None
        if np.any(d == 0.0):
            if np.any(self.b[d == 0.0] != 0.0):
                return None
        mu = np.where(d != 0.0, self.b / np.where(d != 0.0, d, 1.0), 0.0)
        return QuadraticEnergy(0.5, mu, d)


def recognise_quadratic(energy_fn: Callable, dim: int, x0: np.ndarray, rtol: float = 1e-8) -> Optional[QuadraticFormEnergy]:
    """fit E(x) = 1/2 x^T A x - b^T x + c from probes of a Python callable; None if it is not quadratic.

    Probes are taken around x0 with unit offsets; the fit is accepted only if it reproduces the callable on
    16 random points (relative 1e-8) - a wrong guess is a SamplingError upstream, never a silent approximation.

    The probes cost 1 + 2d + d(d-1)/2 Python calls: about 5 000 at d = 100 and 525 000 at d = 1024.  For large d
    pass the form itself as QuadraticFormEnergy(A, b) (or a QuadraticEnergy when it is diagonal).
    """
    x0 = np.asarray(x0, dtype=np.float64).reshape(dim)

    def f(v):
        return float(energy_fn(np.array(v, dtype=np.float64)))

    try:
        e0 = f(x0)
        H = np.zeros((dim, dim))
        g = np.zeros(dim)
        ep = np.zeros(dim)
        for i in range(dim):
            d = np.zeros(dim)
            d[i] = 1.0
            ep[i], em = f(x0 + d), f(x0 - d)
            g[i] = 0.5 * (ep[i] - em)
            H[i, i] = ep[i] + em - 2 * e0
        for i in range(dim):
            for j in range(i + 1, dim):
                d = np.zeros(dim)
                d[i] = d[j] = 1.0
                H[i, j] = H[j, i] = f(x0 + d) - ep[i] - ep[j] + e0
        # E(x0 + d) = e0 + g.d + 1/2 d^T H d  ->  A = H, b = H x0 - g, c from e0
        A = H
        b = H @ x0 - g
        c = e0 - (0.5 * x0 @ A @ x0 - b @ x0)
        q = QuadraticFormEnergy(A, b, c)
        rng = np.random.default_rng(12345)
        for _ in range(16):
            v = x0 + rng.normal(size=dim) * 3.0
            a, want = q(v), f(v)
            if not np.isfinite(want) or abs(a - want) > rtol * max(1.0, abs(want)):
                return None
        return q
    except Exception:
        return None


class TracedEnergy(BuiltinEnergy):
    """a Python callable turned into CUDA source for its analytic gradient (trace.py); compiled at first use"""

    kind = 100

    def __init__(self, energy_fn: Callable, dim: int, x0: np.ndarray):
        from .trace import trace_energy

        rng = np.random.default_rng(20240229)
        probes = np.asarray(x0, dtype=np.float64)[None, :] + rng.normal(size=(4, dim))
        tr, _, grads = trace_energy(energy_fn, dim, probes)
        self.fn, self.dim = energy_fn, dim
        self.source = tr.cuda_source(grads)
        self.n_nodes = self.source.count("\n")

    def params(self, dim):
        return np.zeros(1)

    def __call__(self, x):
        return float(self.fn(np.atleast_1d(np.asarray(x, dtype=np.float64))))


def _traced_dim_message(dim: int) -> str:
    return (f"traced Python energies are limited to {MAX_TRACED_DIM} coordinates, got {dim}; built-in energies "
            "(QuadraticEnergy, GaussianEnergy, MixtureEnergy, DoubleWellEnergy) and quadratic forms "
            "(QuadraticFormEnergy, or a callable recognised as one) are not")


# ----------------------------------------------------------------------------- the sampler
class ThermalSamplingUnit:
    """tsu/core.py:54-267 with the Langevin loop fused into one CUDA kernel (one thread per chain)."""

    def __init__(self, config: Optional[TSUConfig] = None, *, seed: Optional[int] = None, dtype: str = "float64",
                 device=None):
        """dtype: arithmetic of the chains.  "float64" (default) is the reference's (numpy float64, core.py:64-80);
        "float32" is the opt-in fast path (MUFU Box-Muller, ~4.6x faster, trajectories within 2e-4 of float64)."""
        self.config = config or TSUConfig()
        self.sample_count = 0
        if dtype not in ("float32", "float64"):
            raise ConfigurationError("dtype must be 'float32' or 'float64'")
        self.dtype = dtype
        self._seed = int(seed) if seed is not None else int(np.random.randint(0, 2**31 - 1))
        self._chain_counter = 0
        self._fill_counter = 0
        self._device = device

    # -- host-side single-step helpers kept for API compatibility (tsu/core.py:64-98) -----------------
    def _langevin_step(self, x: np.ndarray, grad_energy: np.ndarray) -> np.ndarray:
        cfg = self.config
        drift = -grad_energy * cfg.dt / cfg.friction
        noise_scale = np.sqrt(2 * cfg.temperature * cfg.dt / cfg.friction)
        diffusion = noise_scale * np.random.randn(*x.shape)
        return x + drift + diffusion

    def _numerical_gradient(self, energy_fn: Callable, x: np.ndarray, eps: float = 1e-5) -> np.ndarray:
        x = np.atleast_1d(x)
        grad = np.zeros_like(x)
        for i in range(len(x)):
            x_plus = x.copy()
            x_plus[i] += eps
            x_minus = x.copy()
            x_minus[i] -= eps
            grad[i] = (float(energy_fn(x_plus)) - float(energy_fn(x_minus))) / (2 * eps)
        return grad

    # -- energy resolution -----------------------------------------------------------------------
    def _resolve_energy(self, energy_fn, x_init: np.ndarray) -> BuiltinEnergy:
        if isinstance(energy_fn, BuiltinEnergy):
            return energy_fn
        if isinstance(energy_fn, str):
            named = {"quadratic": QuadraticEnergy(), "gaussian": GaussianEnergy(), "double_well": DoubleWellEnergy()}
            if energy_fn in named:
                return named[energy_fn]
            raise SamplingError(f"unknown built-in energy '{energy_fn}'")
        if callable(energy_fn):
            q = recognise_quadratic(energy_fn, x_init.size, x_init)
            if q is not None:
                return q.as_diagonal() or q
            if x_init.size > MAX_TRACED_DIM:
                raise SamplingError(_traced_dim_message(x_init.size))
            from .trace import TraceError

            try:
                return TracedEnergy(energy_fn, x_init.size, x_init)
            except TraceError as exc:
                raise SamplingError(
                    "energy function is neither a built-in energy (QuadraticEnergy, GaussianEnergy, MixtureEnergy, "
                    "DoubleWellEnergy), nor a quadratic form, nor traceable into CUDA: " + str(exc) +
                    ".  Arbitrary Python control flow cannot run on the GPU and this engine has no CPU fallback")
        raise SamplingError("energy must be a built-in energy object, its name, or a Python callable")

    def _check_dim(self, energy: BuiltinEnergy, dim: int):
        """SamplingError for an energy / dim the kernels do not serve (checked before any device work)"""
        if dim <= MAX_TRACED_DIM:
            return
        if isinstance(energy, TracedEnergy):
            raise SamplingError(_traced_dim_message(dim))
        cap = MAX_DIM[self.dtype]
        if dim > cap:
            raise SamplingError(f"{type(energy).__name__} supports at most {cap} coordinates in {self.dtype} "
                                f"(16-bit Philox block index), got {dim}")
        if energy.kind == ENERGY_QUADRATIC_FORM and dim > MAX_QUADRATIC_FORM_DIM:
            raise SamplingError(f"a quadratic form with more than 64 coordinates supports at most "
                                f"{MAX_QUADRATIC_FORM_DIM} coordinates, got {dim} (a diagonal form runs as a "
                                f"QuadraticEnergy, which has no such limit)")
        if energy.kind == ENERGY_MIXTURE and len(energy.weights) > MAX_MIXTURE_CENTRES:
            raise SamplingError(f"a mixture with more than 64 coordinates supports at most {MAX_MIXTURE_CENTRES} "
                                f"centres, got {len(energy.weights)}")

    def _launch(self, energy: BuiltinEnergy, x_init: np.ndarray, n_chains: int, return_trajectory: bool,
                normals=None, as_tensor: bool = False):
        dim = x_init.size
        self._check_dim(energy, dim)
        torch = _lib.require_cuda()
        cfg = self.config
        device = torch.device(self._device) if self._device is not None else torch.device("cuda", torch.cuda.current_device())
        tdt = torch.float32 if self.dtype == "float32" else torch.float64
        code = 0 if self.dtype == "float32" else 1
        params = torch.from_numpy(np.ascontiguousarray(energy.params(dim), dtype=np.float64)).to(device)
        x0 = torch.from_numpy(np.ascontiguousarray(x_init, dtype=np.float64)).to(device=device, dtype=tdt)
        x = torch.empty((n_chains, dim), dtype=tdt, device=device)
        traj = torch.empty((n_chains, cfg.n_steps, dim), dtype=tdt, device=device) if return_trajectory else None
        nrm = None
        if normals is not None:
            nrm = torch.from_numpy(np.ascontiguousarray(normals, dtype=np.float64)).to(device=device, dtype=tdt)
            if tuple(nrm.shape) != (n_chains, 1 + cfg.n_burnin + cfg.n_steps, dim):
                raise SamplingError("injected normals must have shape (n_chains, 1 + n_burnin + n_steps, dim)")
        with torch.cuda.device(device):
            if isinstance(energy, TracedEnergy):
                import ctypes
                import os

                log = ctypes.create_string_buffer(8192)
                src_dir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc").encode()
                handle = int(_lib.load().tsu_langevin_jit_prepare(energy.source.encode(), code, int(dim), src_dir, log, 8192))
                if handle <= 0:
                    raise SamplingError("the traced energy could not be compiled for the GPU: " +
                                        log.value.decode(errors="replace")[:2000])
                _lib.call(
                    "tsu_langevin_run_jit", handle, ptr(x), int(n_chains), ptr(x0), 0.1, 1, float(cfg.temperature),
                    float(cfg.dt), float(cfg.friction), int(cfg.n_burnin), int(cfg.n_steps), self._seed,
                    self._chain_counter, ptr(nrm), ptr(traj), _lib.current_stream(),
                )
            else:
                _lib.call(
                    "tsu_langevin_run", ptr(x), code, int(n_chains), int(dim), int(energy.kind), ptr(params),
                    int(params.numel()), ptr(x0), 0.1, 1, float(cfg.temperature), float(cfg.dt), float(cfg.friction),
                    int(cfg.n_burnin), int(cfg.n_steps), self._seed, self._chain_counter, ptr(nrm), ptr(traj),
                    _lib.current_stream(),
                )
        if normals is None:
            self._chain_counter += n_chains
        self.sample_count += n_chains
        if as_tensor:
            return x, traj
        xs = x.cpu().numpy().astype(np.float64)
        tr = None
        if traj is not None:
            t = traj.cpu().numpy().astype(np.float64)
            tr = [t[c, s] for c in range(n_chains) for s in range(cfg.n_steps)]  # core.py:155-156 order
        return xs, tr

    # -- reference API -----------------------------------------------------------------------------
    def sample_from_energy(self, energy_fn, x_init: np.ndarray, n_samples: int = 1, return_trajectory: bool = False,
                           *, _normals=None, as_tensor: bool = False):
        """tsu/core.py:100-162.  Every sample is an independent chain restarted at x_init
        (+ 0.1 N(0, I) for all but the first, core.py:142-143): n_samples chains run concurrently."""
        if n_samples <= 0:
            raise SamplingError(f"n_samples must be positive, got {n_samples}")
        x_init = np.atleast_1d(np.asarray(x_init, dtype=np.float64))
        try:
            if callable(energy_fn) and not isinstance(energy_fn, BuiltinEnergy):
                test_energy = energy_fn(x_init)
                if not isinstance(test_energy, (int, float, np.number)):
                    raise SamplingError(f"Energy function must return scalar, got {type(test_energy)}")
        except Exception as e:
            raise SamplingError(f"Energy function failed on initial state: {e}")
        energy = self._resolve_energy(energy_fn, x_init)
        samples, traj = self._launch(energy, x_init, int(n_samples), return_trajectory, _normals, as_tensor)
        return (samples, traj) if return_trajectory else samples

    def sample_boltzmann(self, energy, n_samples: int = 1000, dim: int = 1, x_init=None, **kw):
        """README.md:46-64: `tsu.sample_boltzmann(energy, n_samples=1000, dim=10)` -> (n_samples, dim) from exp(-E/T)"""
        x0 = np.zeros(dim) if x_init is None else np.asarray(x_init, dtype=np.float64)
        return self.sample_from_energy(energy, x0, n_samples=n_samples, **kw)

    def sample_gaussian(self, mu: float = 0.0, sigma: float = 1.0, n_samples: int = 1) -> np.ndarray:
        """tsu/core.py:208-241"""
        if sigma <= 0:
            raise ConfigurationError(f"Sigma must be positive, got {sigma}")
        if n_samples <= 0:
            raise ConfigurationError(f"n_samples must be positive, got {n_samples}")
        samples = self.sample_from_energy(GaussianEnergy(mu, sigma), np.array([mu], dtype=np.float64), n_samples)
        return samples.flatten()

    def _dev(self):
        torch = _lib.require_cuda()
        return torch.device(self._device) if self._device is not None else torch.device("cuda", torch.cuda.current_device())

    def _uniform_words(self, n: int):
        """n raw 32-bit Philox words on the device ('FILL' stream; the call counter keeps successive calls apart)"""
        torch = _lib.require_cuda()
        out = torch.empty(int(n), dtype=torch.int32, device=self._dev())
        with torch.cuda.device(out.device):
            _lib.call("tsu_philox_fill_u32", ptr(out), int(n), self._seed, self._fill_counter & 0xFFFFFFFF, _lib.current_stream())
        self._fill_counter += 1
        return out.to(torch.int64) & 0xFFFFFFFF

    def p_bit(self, prob: float, n_samples: int = 1) -> np.ndarray:
        """probabilistic bit: n_samples draws of Bernoulli(prob) as an int array (tsu/core.py:164-206 contract and
        error behaviour).  The reference runs its Langevin loop on a clipped linear energy and thresholds at 0.5: the
        two flat plateaus outside [0, 1] carry Boltzmann weights (1 - prob) and prob, so the walk approximates
        Bernoulli(prob) (0.21 / 0.82 measured for 0.2 / 0.8 with 400 samples).  Here the bit is exact:
        k < ceil(prob * 2^32) on a 32-bit Philox word k."""
        if not 0 <= prob <= 1:
            raise ConfigurationError(f"Probability must be in [0,1], got {prob}")
        if n_samples <= 0:
            raise ConfigurationError(f"n_samples must be positive, got {n_samples}")
        thr = int(np.ceil(float(prob) * 4294967296.0))
        return (self._uniform_words(n_samples) < thr).cpu().numpy().astype(int)

    def sample_categorical(self, probs: np.ndarray, n_samples: int = 1) -> np.ndarray:
        """n_samples category indices with probabilities probs / probs.sum() (tsu/core.py:241-267 contract); exact
        inverse-CDF sampling on 32-bit Philox words instead of the reference's Langevin walk over |x| mod K"""
        p = np.asarray(probs, dtype=np.float64)
        if p.ndim != 1 or p.size == 0 or (p < 0).any() or not p.sum() > 0:
            raise ConfigurationError("probs must be a non-empty 1-D array of non-negative weights with a positive sum")
        if n_samples <= 0:
            raise ConfigurationError(f"n_samples must be positive, got {n_samples}")
        torch = _lib.require_cuda()
        edges = np.ceil(np.cumsum(p / p.sum()) * 4294967296.0)
        edges[-1] = 4294967296.0
        k = self._uniform_words(n_samples)
        idx = torch.searchsorted(torch.from_numpy(edges.astype(np.int64)).to(k.device), k, right=True)
        return idx.cpu().numpy().astype(int)


class ProbabilisticNeuron:
    """single stochastic neuron on a ThermalSamplingUnit (tsu/core.py:270-294): output ~ Bernoulli(sigmoid(w.x + b))"""

    def __init__(self, tsu: ThermalSamplingUnit):
        self.tsu = tsu

    def activate(self, weights: np.ndarray, inputs: np.ndarray, bias: float = 0.0) -> int:
        logit = float(np.dot(weights, inputs) + bias)
        return int(self.tsu.p_bit(1.0 / (1.0 + np.exp(-logit)), n_samples=1)[0])

    def forward_stochastic(self, weights: np.ndarray, inputs: np.ndarray, bias: float = 0.0, n_samples: int = 10) -> float:
        """expected output from n_samples activations (one batched draw instead of the reference's Python loop)"""
        logit = float(np.dot(weights, inputs) + bias)
        return float(np.mean(self.tsu.p_bit(1.0 / (1.0 + np.exp(-logit)), n_samples=n_samples)))


def validate_distribution(samples: np.ndarray, expected_dist: str, params: dict, alpha: float = 0.05) -> dict:
    """host-side check of samples against "gaussian" (KS test) or "bernoulli" (|mean - p| < 0.05): same keys as
    tsu/core.py:298-327"""
    samples = np.asarray(samples)
    results = {"mean": np.mean(samples), "std": np.std(samples), "n_samples": len(samples)}
    if expected_dist == "gaussian":
        from scipy import stats

        mu, sigma = params.get("mu", 0), params.get("sigma", 1)
        ks_stat, p_value = stats.kstest(samples, stats.norm(loc=mu, scale=sigma).cdf)
        results.update(expected_mean=mu, expected_std=sigma, ks_statistic=ks_stat, ks_pvalue=p_value,
                       passes_ks_test=p_value > alpha)
    elif expected_dist == "bernoulli":
        prob = params.get("p", 0.5)
        err = abs(np.mean(samples) - prob)
        results.update(expected_mean=prob, empirical_prob=np.mean(samples), error=err, passes_test=err < 0.05)
    return results


TSU = ThermalSamplingUnit
