"""
Drop-in mirror of the reference's tsu/gibbs.py (GibbsConfig, GibbsSampler, HardwareEmulator) whose
sweeps run on the B200 through libtsu_b200.so.  Same names, arguments, return types and error
messages as the reference (file:line cited per method); there is no CPU fallback - without a CUDA
device every sampling call raises.

Differences that are deliberate and documented:
  * randomness is Philox4x32-10 keyed by a per-sampler seed instead of the global MT19937 stream.
    The seed is drawn from numpy's global stream at construction unless `seed=` is given, so
    `np.random.seed(k)` before constructing a sampler still makes a run reproducible.
  * extra keyword-only arguments (`n_chains`, `precision`, `seed`, `as_tensor`) expose the batch
    dimension the reference only emulates serially (gibbs.py:475-479).
"""

import math
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

from . import _lib
from ._lib import ptr
from .population import PopulationEstimates

M32 = 0xFFFFFFFF


@dataclass
class GibbsConfig:
    """tsu/gibbs.py:19-36 (same fields, defaults and validation messages)"""

    temperature: float = 1.0
    n_burnin: int = 100
    n_sweeps: int = 10
    update_order: str = "sequential"  # 'sequential' or 'random'

    def __post_init__(self):
        if self.temperature <= 0:
            raise ValueError("Temperature must be positive")
        if self.n_burnin < 0:
            raise ValueError("Burn-in steps must be non-negative")
        if self.n_sweeps <= 0:
            raise ValueError("Number of sweeps must be positive")
        if self.update_order not in ["sequential", "random"]:
            raise ValueError("Update order must be 'sequential' or 'random'")


def _host_int64(t) -> np.ndarray:
    """device bits -> the reference's int arrays (gibbs.py:207 `np.zeros(..., dtype=int)`)"""
    return t.cpu().numpy().astype(np.int64)


def _as_square(coupling) -> np.ndarray:
    J = np.asarray(coupling, dtype=np.float64)
    n_bits = J.shape[0]
    if J.shape != (n_bits, n_bits):
        raise ValueError("Coupling matrix must be square")
    return J


def _host_energy(state: np.ndarray, coupling, bias=None) -> float:
    """E = -1/2 s^T J s - b^T s (host arithmetic on one configuration)"""
    energy = -0.5 * state.dot(coupling).dot(state)
    if bias is not None:
        energy -= np.asarray(bias).dot(state)
    return float(energy)


# csrc/dense_gibbs.cu keeps a chain's uniforms (and their logits with float64 fields), fields, self couplings and bits
# in at most 227 KB of shared memory: 33 N + 272 bytes with float64 fields, 17 N + 272 with float32
DENSE_MAX_N = {"float64": 7035, "float32": 13657}

CHROMATIC_NEEDS_FLOAT64 = "chromatic=True (sparse couplings) computes float64 fields: use a 'float64' sampler"


class _DenseProblem:
    """coupling matrix + bias resident on the device (transposed, see tsu_b200.h)"""

    def __init__(self, coupling, bias, precision: str, device, update_order: str = "sequential"):
        J = _as_square(coupling)
        self.N = J.shape[0]
        if precision == "bf16":
            raise ValueError("precision='bf16' (tensor cores) serves sample_boltzmann / sample / sample_chains / "
                             "simulated_annealing / parallel_tempering; this entry point needs a 'float64' or "
                             "'float32' sampler")
        if precision not in ("float64", "float32"):
            raise ValueError("precision must be 'float64', 'float32' or 'bf16'")
        if self.N > DENSE_MAX_N[precision]:
            raise ValueError(f"precision='{precision}' (dense kernel) supports at most {DENSE_MAX_N[precision]} bits "
                             f"(float64: {DENSE_MAX_N['float64']}, float32: {DENSE_MAX_N['float32']}); got {self.N}")
        torch = _lib.require_cuda()
        self.np_dtype = np.float64 if precision == "float64" else np.float32
        self.code = 1 if precision == "float64" else 0
        self.device = device
        self.update_order = update_order
        self.host_J, self.host_bias = J, None
        self.Jt = torch.from_numpy(np.ascontiguousarray(J.T.astype(self.np_dtype))).to(device)
        if bias is not None:
            b = np.asarray(bias, dtype=np.float64)
            if b.shape != (self.N,):
                raise ValueError("bias must have one entry per bit")
            self.bias = torch.from_numpy(np.ascontiguousarray(b.astype(self.np_dtype))).to(device)
            self.host_bias = b
        else:
            self.bias = None

    def _orders(self, n_sweeps: int, seed: int, sweep0: int):
        """visiting order per sweep: None for 'sequential', fresh permutations for 'random' (gibbs.py:153-157)"""
        if self.update_order == "sequential" or n_sweeps == 0:
            return None
        torch = _lib.require_cuda()
        rng = np.random.Generator(np.random.Philox(key=[seed, sweep0]))
        perms = np.stack([rng.permutation(self.N) for _ in range(n_sweeps)]).astype(np.int32)
        return torch.from_numpy(perms).to(self.device)

    def run(self, state, *, T: float, seed: int, sweep0: int, chain0: int, n_burnin: int, n_samples: int,
            sweeps_per_sample: int, T_chain=None, T_sweep=None, uniforms=None, want_samples=False, want_energy=False,
            track_best=False, order=None, visits_per_sweep: int = 0):
        """one launch of tsu_dense_gibbs_run on `state` (uint8 tensor [n_chains, N], updated in place); T_sweep is the
        host float64 temperature of every sweep; without `order` the sweeps follow the problem's update order"""
        torch = _lib.require_cuda()
        device = self.device
        n_chains, N = state.shape
        if order is None and visits_per_sweep == 0:
            order = self._orders(n_burnin + n_samples * sweeps_per_sample, seed, sweep0)
        if T_sweep is not None:
            T_sweep = torch.from_numpy(T_sweep).to(device)
        samples = torch.empty((n_samples, n_chains, N), dtype=torch.uint8, device=device) if want_samples else None
        energy = torch.empty(n_chains, dtype=torch.float64, device=device) if (want_energy or track_best) else None
        best_state = torch.empty((n_chains, N), dtype=torch.uint8, device=device) if track_best else None
        best_energy = torch.empty(n_chains, dtype=torch.float64, device=device) if track_best else None
        with torch.cuda.device(device):
            _lib.call(
                "tsu_dense_gibbs_run", ptr(self.Jt), self.code, ptr(self.bias), ptr(state), n_chains, N, float(T),
                ptr(T_chain), ptr(T_sweep), int(n_burnin), int(n_samples), int(sweeps_per_sample), ptr(order),
                ptr(uniforms), ptr(samples), ptr(energy), int(track_best), ptr(best_state), ptr(best_energy), seed,
                sweep0 & 0xFFFFFFFF, chain0 & 0xFFFFFFFF, self.code, int(visits_per_sweep), _lib.current_stream(),
            )
        return samples, energy, best_state, best_energy

    def energy(self, state: np.ndarray) -> float:
        """energy of a host state under the float64 couplings and bias"""
        return _host_energy(state, self.host_J, self.host_bias)


TC_MAX_N = 4096   # csrc/dense_tc.cu keeps the chain bits of a CTA in shared memory
TC_PANEL = 128


class _TcProblem:
    """couplings of the tensor-core path (csrc/dense_tc.cu): bf16, row-major, N padded with uncoupled sites to a
    multiple of the 128-site panel (their bits are dropped again; a site's uniform depends only on
    (seed, chain, sweep, site), so the padding does not change what the real sites draw)."""

    def __init__(self, coupling, bias, device, update_order):
        torch = _lib.require_cuda()
        J = _as_square(coupling)
        self.N = J.shape[0]
        self.Np = (self.N + TC_PANEL - 1) // TC_PANEL * TC_PANEL
        if self.Np > TC_MAX_N:
            raise ValueError(f"precision='bf16' (tensor-core path) supports at most {TC_MAX_N} bits; got {self.N}")
        if update_order != "sequential":
            raise ValueError("precision='bf16' (tensor-core path) implements the sequential update order only")
        self.device = device
        self.host_J, self.host_bias = J, None
        # upload as given and round on the device (float64 -> float32 -> bf16, the rounding the oracle applies): the
        # host-side conversion of a 4096 x 4096 matrix used to cost several times the 10 sweeps it was uploaded for
        Jd = torch.from_numpy(np.ascontiguousarray(J)).to(device).to(torch.float32).to(torch.bfloat16)
        if self.Np != self.N:
            Jp = torch.zeros((self.Np, self.Np), dtype=torch.bfloat16, device=device)
            Jp[:self.N, :self.N] = Jd
            Jd = Jp
        self.J = Jd.contiguous()
        self.bias = None
        if bias is not None:
            b = np.asarray(bias, dtype=np.float64)
            if b.shape != (self.N,):
                raise ValueError("bias must have one entry per bit")
            bp = np.zeros(self.Np, dtype=np.float32)
            bp[:self.N] = b
            self.bias = torch.from_numpy(bp).to(device)
            self.host_bias = b

    def run(self, state, *, T: float, seed: int, sweep0: int, chain0: int, n_burnin: int, n_samples: int,
            sweeps_per_sample: int, T_chain=None, T_sweep=None, uniforms=None, want_samples=False, want_energy=False,
            track_best=False):
        """the launches of a run on `state` ([n_chains, Np] uint8, updated in place), bf16 couplings, fp32 fields in
        TMEM.  With T_sweep (host float64): an energy pass on the initial state, then per step one sweep at T_sweep[k]
        and an energy pass that keeps every chain's best state.  Otherwise n_burnin sweeps, then sweeps_per_sample
        sweeps before each sample.  With want_energy, one energy pass at the end.  Injected uniforms are a float64 /
        float32 parity mode: the callers reject them."""
        torch = _lib.require_cuda()
        n_chains, N, device = int(state.shape[0]), self.N, self.device
        samples = torch.empty((n_samples, n_chains, N), dtype=torch.uint8, device=device) if want_samples else None
        energy = torch.empty(n_chains, dtype=torch.float64, device=device) if (want_energy or track_best) else None
        best_state = torch.empty_like(state) if track_best else None
        best_energy = torch.full((n_chains,), float("inf"), dtype=torch.float64, device=device) if track_best else None

        def sweeps(n, T, sweep):
            """n sweeps at T, or at the per-chain T_chain; a count <= 0 launches nothing.  Returns the next offset"""
            if n <= 0:
                return sweep
            _lib.call("tsu_dense_gibbs_tc_run", ptr(self.J), ptr(self.bias), ptr(state), n_chains, self.Np,
                      1.0 if T_chain is not None else float(T), ptr(T_chain), int(n), seed, sweep & 0xFFFFFFFF,
                      chain0 & 0xFFFFFFFF, None, _lib.current_stream())
            return sweep + n

        def energy_pass(best: bool):
            _lib.call("tsu_dense_tc_energy", ptr(self.J), ptr(self.bias), ptr(state), n_chains, self.Np, ptr(energy),
                      ptr(best_energy if best else None), ptr(best_state if best else None), _lib.current_stream())

        with torch.cuda.device(device):
            sweep = sweep0
            if T_sweep is not None:
                energy_pass(track_best)   # the initial state is the first best
                for k in range(n_burnin):
                    sweep = sweeps(1, T_sweep[k], sweep)
                    energy_pass(track_best)
            else:
                sweep = sweeps(n_burnin, T, sweep)
                for k in range(n_samples):
                    sweep = sweeps(sweeps_per_sample, T, sweep)
                    samples[k] = state[:, :N]
            if want_energy:
                energy_pass(False)
        return samples, energy, None if best_state is None else best_state[:, :N], best_energy

    def energy(self, state: np.ndarray) -> float:
        """energy of a host state under the float64 couplings and bias (not their bf16 rounding)"""
        return _host_energy(state, self.host_J, self.host_bias)


def annealing_temperatures(T_initial: float, T_final: float, n_steps: int, cooling_schedule: str = "exponential"):
    """float64 [n_steps]: the temperature of every annealing step (tsu/gibbs.py:340-393): T_initial at step 0 towards
    T_final, which is not reached; "exponential" or, for anything else, "linear" cooling"""
    steps = np.arange(n_steps, dtype=np.float64)
    if cooling_schedule == "exponential":
        return T_initial * (T_final / T_initial) ** (steps / n_steps)
    return T_initial + (T_final - T_initial) * steps / n_steps  # linear


class DensePopulationResult(PopulationEstimates):
    """What GibbsSampler.population_annealing returns; pass it back as `previous=` to continue the run.

    Device tensors (P = n_populations, n = len(temperatures)):
      energy          float64 [n_chains], E of every chain's final state (on bf16: under the bf16-rounded couplings)
      family          int32 [n_chains], the initial chain (chain0 + j, mod 2^32) each chain descends from
      weight_sum      int64 [n, P], W of step k; energy_ref float64 [n, P], E_ref of the population entering step k
      energy_moments  float64 [n + 1, P, 2], (sum E, sum E^2) over the population entering step k; entry n: the final
                      states
      states          uint8 [n_chains, N], the final states
    Host: temperatures, T_start, dbeta, r_pop (R_p), shift (s), n_sites (N), chain0, backend ("float64", "float32",
    "bf16" or "chromatic").  ln Z ratios, free energies and rho_t: PopulationEstimates.
    """

    def __init__(self, state, energy, family, weight_sum, energy_ref, energy_moments, temperatures, T_start, dbeta,
                 r_pop, shift, N, chain0, backend):
        self._state = state  # rows padded to the tensor-core panel width: what previous= continues from
        self.energy, self.family = energy, family
        self.weight_sum, self.energy_ref, self.energy_moments = weight_sum, energy_ref, energy_moments
        self.temperatures, self.T_start, self.dbeta = temperatures, float(T_start), dbeta
        self.r_pop, self.shift, self.n_sites = int(r_pop), int(shift), int(N)
        self.chain0, self.backend = int(chain0), backend

    @property
    def states(self):
        return self._state[:, :self.n_sites]

    def mean_energy(self) -> np.ndarray:
        """[n, P]: population mean of E at temperatures[k] (after step k's sweeps), from energy_moments[1:]"""
        return self.energy_moments[1:, :, 0].cpu().numpy() / self.r_pop

    def specific_heat(self) -> np.ndarray:
        """[n, P]: specific heat per spin at temperatures[k], (<E^2> - <E>^2) / (T_k^2 N) over each population"""
        m = self.energy_moments[1:].cpu().numpy() / self.r_pop
        beta = 1.0 / self.temperatures[:, None]
        return beta * beta * (m[..., 1] - m[..., 0] * m[..., 0]) / self.n_sites


class GibbsSampler:
    """tsu/gibbs.py:39-393 on the GPU.

    Every chain is one CTA keeping its N local fields in shared memory (csrc/dense_gibbs.cu); the
    update rule is the reference's: new bit = 1 iff u < sigmoid(h_i / T), h_i = J[i,:].s + b_i
    including the self term, sigmoid clamped at |x| > 20.
    """

    def __init__(self, config: Optional[GibbsConfig] = None, *, seed: Optional[int] = None,
                 precision: str = "float64", device=None):
        self.config = config or GibbsConfig()
        self.sample_count = 0
        if precision not in ("float64", "float32", "bf16"):
            raise ValueError("precision must be 'float64', 'float32' or 'bf16'")
        self.precision = precision
        self._seed = int(seed) if seed is not None else int(np.random.randint(0, 2**31 - 1))
        self._sweep_counter = 0  # Philox offset: advances with every sweep executed
        self._chain_counter = 0
        self._swap_counter = 0   # Philox offset of the replica-exchange draws: advances with every swap pass
        self._houdayer_counter = 0  # step index of the Houdayer moves of parallel_tempering: advances with every move
        self._device = device

    # ------------------------------------------------------------------ scalar helpers
    def _sigmoid(self, x: float) -> float:
        """tsu/gibbs.py:61-77"""
        if x > 20:
            return 1.0
        elif x < -20:
            return 0.0
        return 1.0 / (1.0 + np.exp(-x))

    def _compute_local_field(self, i: int, state: np.ndarray, coupling: np.ndarray,
                             bias: Optional[np.ndarray] = None) -> float:
        """tsu/gibbs.py:79-100: h_i = J[i,:].s + b_i (includes the self term)"""
        h = np.dot(coupling[i, :], state)
        if bias is not None:
            h += bias[i]
        return float(h)

    def compute_energy(self, state: np.ndarray, coupling: np.ndarray, bias: Optional[np.ndarray] = None) -> float:
        """tsu/gibbs.py:215-236: E = -1/2 s^T J s - b^T s (host arithmetic on one configuration)"""
        return _host_energy(np.asarray(state), coupling, bias)

    # ------------------------------------------------------------------ device plumbing
    def _dev(self):
        torch = _lib.require_cuda()
        return torch.device(self._device) if self._device is not None else torch.device("cuda", torch.cuda.current_device())

    def _problem(self, coupling, bias, *, chromatic: bool, tensor_ok: bool):
        """the couplings on the device for the sampler's back end: chromatic CSR (float64 fields), tensor cores (bf16,
        for the entry points that serve them) or the float64 / float32 dense kernel"""
        if chromatic:
            from .sparse import SparseProblem

            if self.precision != "float64":
                raise ValueError(CHROMATIC_NEEDS_FLOAT64)
            return SparseProblem(coupling, bias, self._dev())
        if self.precision == "bf16" and tensor_ok:
            return _TcProblem(coupling, bias, self._dev(), self.config.update_order)
        return _DenseProblem(coupling, bias, self.precision, self._dev(), self.config.update_order)

    def _run(self, prob, state, *, n_burnin: int, n_samples: int, sweeps_per_sample: int, T: Optional[float] = None,
             chain0: Optional[int] = None, **kw):
        """prob.run on `state` at the sampler's temperature (or T), seed and Philox offsets (the chain offset, or
        chain0), which then advance past the sweeps run.  A negative count is an error on the dense and sparse kernels
        and runs nothing on the tensor cores."""
        out = prob.run(state, T=float(self.config.temperature if T is None else T), seed=self._seed,
                       sweep0=self._sweep_counter, chain0=self._chain_counter if chain0 is None else chain0,
                       n_burnin=n_burnin, n_samples=n_samples, sweeps_per_sample=sweeps_per_sample, **kw)
        self._sweep_counter += max(n_burnin, 0) + n_samples * max(sweeps_per_sample, 0)
        return out

    def _initial_states(self, prob, n_chains: int, initial_state=None):
        """uint8 [n_chains, N] states on the device (given, or Philox draws), padded with zero bits to the tensor-core
        problem's panel width"""
        torch = _lib.require_cuda()
        if initial_state is not None:
            a = np.asarray(initial_state)
            if a.ndim == 1:
                if a.shape != (prob.N,):
                    raise ValueError(f"initial_state must have {prob.N} entries, got shape {a.shape}")
                a = np.broadcast_to(a, (n_chains, prob.N))
            elif a.shape != (n_chains, prob.N):
                raise ValueError(f"initial_state must have shape ({prob.N},) or ({n_chains}, {prob.N}), got {a.shape}")
            state = torch.from_numpy(np.ascontiguousarray((a != 0).astype(np.uint8))).to(prob.device)
        else:
            state = torch.empty((n_chains, prob.N), dtype=torch.uint8, device=prob.device)
            with torch.cuda.device(prob.device):
                _lib.call("tsu_dense_init_random", ptr(state), n_chains, prob.N, self._seed ^ 0x5DEECE66D,
                          (self._chain_counter + self._sweep_counter) & 0xFFFFFFFF, _lib.current_stream())
        width = getattr(prob, "Np", prob.N)
        if width == prob.N:
            return state
        padded = torch.zeros((n_chains, width), dtype=torch.uint8, device=prob.device)
        padded[:, :prob.N] = state
        return padded

    @staticmethod
    def _injected(prob, uniforms, orders=None) -> dict:
        """parity mode, as run() arguments on the device: float64 uniforms [sweeps, N] (one chain) or [sweeps, chains,
        N], in visiting order, and visiting orders [sweeps, N] of the dense kernel"""
        torch = _lib.require_cuda()
        kw = {}
        if uniforms is not None:
            a = np.asarray(uniforms, dtype=np.float64)
            if a.ndim == 2:
                a = a[:, None, :]
            kw["uniforms"] = torch.from_numpy(np.ascontiguousarray(a)).to(prob.device)
        if orders is not None:
            kw["order"] = torch.from_numpy(np.ascontiguousarray(np.asarray(orders, dtype=np.int32))).to(prob.device)
        return kw

    @staticmethod
    def _samples_out(samples, n_chains: int, as_tensor: bool):
        """samples [n_samples, n_chains, N] -> (n_samples, N) for one chain, (n_chains, n_samples, N) host int64 for
        more; as_tensor keeps them on the device, chain axis second"""
        if as_tensor:
            return samples if n_chains > 1 else samples[:, 0]
        out = _host_int64(samples)
        return out[:, 0, :] if n_chains == 1 else np.ascontiguousarray(out.transpose(1, 0, 2))

    # ------------------------------------------------------------------ reference API
    def sample_conditional(self, i: int, state: np.ndarray, coupling: np.ndarray,
                           bias: Optional[np.ndarray] = None) -> int:
        """tsu/gibbs.py:102-126: resample bit i given the others (one single-site visit on the device)"""
        torch = _lib.require_cuda()
        prob = self._problem(coupling, bias, chromatic=False, tensor_ok=False)
        st = self._initial_states(prob, 1, np.asarray(state))
        order = torch.tensor([[int(i)]], dtype=torch.int32, device=prob.device)
        self._run(prob, st, n_burnin=1, n_samples=0, sweeps_per_sample=0, order=order, visits_per_sweep=1)
        return int(st[0, int(i)].item())

    def gibbs_sweep(self, state: np.ndarray, coupling: np.ndarray, bias: Optional[np.ndarray] = None,
                    n_sweeps: int = 1, *, chromatic: bool = False, _uniforms=None, _orders=None) -> np.ndarray:
        """tsu/gibbs.py:128-162: n_sweeps sweeps over all bits; the input is not modified (gibbs.py:150).
        chromatic=True: sparse couplings, sites visited colour class by colour class (csrc/sparse_gibbs.cu)"""
        prob = self._problem(coupling, bias, chromatic=chromatic, tensor_ok=False)
        st = self._initial_states(prob, 1, np.asarray(state))
        # a chromatic sweep visits the colour classes: injected orders do not apply
        self._run(prob, st, n_burnin=int(n_sweeps), n_samples=0, sweeps_per_sample=0,
                  **self._injected(prob, _uniforms, None if chromatic else _orders))
        a = np.asarray(state)
        return st[0].cpu().numpy().astype(a.dtype if a.dtype.kind in "iu" else np.int64)

    def sample_boltzmann(self, coupling: np.ndarray, bias: Optional[np.ndarray] = None, n_samples: int = 1000,
                         burnin: Optional[int] = None, initial_state: Optional[np.ndarray] = None, *,
                         n_chains: int = 1, as_tensor: bool = False, chromatic: bool = False, _uniforms=None,
                         _orders=None):
        """tsu/gibbs.py:164-213: burn-in, then n_samples x config.n_sweeps sweeps; one launch (one per group of sweeps
        on the tensor cores).

        n_chains == 1 (default): int array (n_samples, n_bits) like the reference.
        n_chains > 1: (n_chains, n_samples, n_bits) - independent chains run concurrently.
        chromatic=True: sparse couplings (dense array, scipy.sparse matrix or CSR tuple) on the chromatic CSR kernel;
        a sweep visits the sites colour class by colour class instead of in index order.
        """
        burnin = burnin if burnin is not None else self.config.n_burnin
        if self.precision == "bf16" and not chromatic and (_uniforms is not None or _orders is not None):
            raise ValueError("injected draws are a float64 / float32 parity mode; precision='bf16' draws Philox")
        prob = self._problem(coupling, bias, chromatic=chromatic, tensor_ok=True)
        st = self._initial_states(prob, int(n_chains), initial_state)
        samples, _, _, _ = self._run(prob, st, n_burnin=int(burnin), n_samples=int(n_samples),
                                     sweeps_per_sample=self.config.n_sweeps, want_samples=True,
                                     **self._injected(prob, _uniforms, None if chromatic else _orders))
        self._chain_counter += int(n_chains)
        self.sample_count += int(n_samples)
        return self._samples_out(samples, int(n_chains), as_tensor)

    def sample(self, J: np.ndarray, n_samples: int = 1000, **kwargs) -> np.ndarray:
        """README.md:69-80: `sampler.sample(J, n_samples=1000)` -> (n_samples, n_bits) binary configurations"""
        return self.sample_boltzmann(J, n_samples=n_samples, **kwargs)

    def sample_chains(self, coupling, bias=None, n_chains: int = 1024, n_sweeps: Optional[int] = None,
                      initial_state=None, as_tensor: bool = False, return_energy: bool = False):
        """batched entry point: n_chains independent chains, n_sweeps sweeps each, final states returned.

        This is the shape of BASELINE config 3 (dense J, N=4096, 2048 chains, 10 sweeps).  With
        precision="bf16" the fields are evaluated on the tensor cores (tcgen05, csrc/dense_tc.cu) and the energy
        E = -1/2 s^T J s - b^T s is one more tensor-core field evaluation, summed on the device."""
        n_sweeps = self.config.n_sweeps if n_sweeps is None else int(n_sweeps)
        prob = self._problem(coupling, bias, chromatic=False, tensor_ok=True)
        st = self._initial_states(prob, int(n_chains), initial_state)
        _, energy, _, _ = self._run(prob, st, n_burnin=n_sweeps, n_samples=0, sweeps_per_sample=0,
                                    want_energy=return_energy)
        self._chain_counter += int(n_chains)
        st = st[:, :prob.N]
        out = st if as_tensor else _host_int64(st)
        if return_energy:
            return out, (energy if as_tensor else energy.cpu().numpy())
        return out

    def parallel_tempering(self, coupling: np.ndarray, temperatures: List[float], bias: Optional[np.ndarray] = None,
                           n_samples: int = 1000, swap_interval: int = 10, *, n_ladders: int = 1,
                           criterion: str = "reference", chromatic: bool = False, houdayer_interval: int = 0,
                           houdayer_max_temperature: float = math.inf, _inject=None) -> Tuple[np.ndarray, dict]:
        """tsu/gibbs.py:238-338: replicas at `temperatures`, n_sweeps sweeps per iteration, adjacent-pair
        Metropolis swaps every swap_interval iterations, samples from temperature slot 0.

        All replicas advance concurrently (one CTA each on the float64 / float32 kernel, one tensor-core tile row
        each with precision="bf16"); configurations stay in place and the slot -> replica map is permuted by
        tsu_pt_swap, which reproduces the sequential pair order and the draw-only-if-delta<0 rule of
        gibbs.py:308-323.  One device->host copy at the end.

        n_ladders = K independent ladders run in one batch: replica k R + j starts in slot j of ladder k.  With K > 1
        the samples are (K, n_samples, n_bits) (slot 0 of each ladder), the swap counts are totals over the ladders,
        and info["energies"] / info["final_states"] hold one entry per ladder, each shaped as for one ladder.

        criterion="reference" keeps the swap expression of gibbs.py:317, which favours moving high-energy
        configurations to cold slots; "metropolis" is the detailed-balance rule, under which slot 0 samples the
        Boltzmann distribution at temperatures[0].

        chromatic=True: sparse couplings (dense array, scipy.sparse matrix or CSR tuple) on the chromatic CSR kernel
        (float64 sampler); a sweep visits the sites colour class by colour class.

        houdayer_interval = k > 0 (chromatic=True, even n_ladders, symmetric couplings): every k iterations, after the
        sweeps and before the energy record and the exchange pass, one Houdayer move (ICM, Zhu, Ochoa & Katzgraber
        2015; tsu_sparse_houdayer states the exact rule) acts on the replicas of ladders 2m and 2m + 1 at every slot
        whose temperature is at most houdayer_max_temperature.  Hot slots, where difference clusters percolate and the
        move only exchanges configurations, can be left out that way.  The pairs are built on the device; the move
        keeps E_a + E_b and the product of the two Boltzmann distributions, and its step index is the sampler's
        Houdayer counter, which advances by one per move.
        """
        K = int(n_ladders)
        hk = houdayer_interval
        if isinstance(hk, bool) or not isinstance(hk, (int, np.integer)) or hk < 0:
            raise ValueError("houdayer_interval must be a non-negative integer")
        if chromatic and self.precision != "float64":
            raise ValueError(CHROMATIC_NEEDS_FLOAT64)
        if chromatic and _inject is not None:
            raise ValueError("injected draws are a float64 / float32 parity mode of one ladder on the dense kernel")
        if hk > 0:
            from .sparse import is_symmetric_csr, to_csr

            if not chromatic:
                raise ValueError("Houdayer moves run on the chromatic back end: pass chromatic=True")
            if K % 2:
                raise ValueError("Houdayer moves pair ladders 2m and 2m + 1: n_ladders must be even")
            if not float(houdayer_max_temperature) > 0:
                raise ValueError("houdayer_max_temperature must be positive")
            if not is_symmetric_csr(*to_csr(coupling)):
                raise ValueError("Houdayer moves need symmetric couplings (J equal to its transpose)")
        torch = _lib.require_cuda()
        if K < 1:
            raise ValueError("n_ladders must be at least 1")
        if criterion not in ("metropolis", "reference"):
            raise ValueError("criterion must be 'metropolis' or 'reference'")
        if _inject is not None and (self.precision == "bf16" or K > 1):
            raise ValueError("injected draws are a float64 / float32 parity mode of one ladder")
        prob = self._problem(coupling, bias, chromatic=chromatic, tensor_ok=True)
        device = prob.device
        temps = np.asarray(list(temperatures), dtype=np.float64)
        R = temps.size
        if R == 0 or np.any(temps <= 0):
            raise ValueError("Temperature must be positive")
        n_sweeps = self.config.n_sweeps
        T_slot = torch.from_numpy(temps).to(device)
        slot_replica = torch.arange(K * R, dtype=torch.int32, device=device).view(K, R)
        T_chain = T_slot.repeat(K)                         # replica k R + j starts at slot j of ladder k
        stats = torch.zeros(2, dtype=torch.int64, device=device)
        inj = _inject
        states = self._initial_states(prob, K * R, None if inj is None else np.asarray(inj["inits"]))
        bu = None
        if inj is not None:  # parity mode: draws are given per temperature slot; slot i starts on replica i
            bu = torch.from_numpy(np.ascontiguousarray(np.asarray(inj["burn_uniforms"]).transpose(1, 0, 2))).to(device)
        self._run(prob, states, n_burnin=self.config.n_burnin, n_samples=0, sweeps_per_sample=0, T_chain=T_chain,
                  uniforms=bu)
        chain0, h_slots, n_pairs = self._chain_counter, None, 0
        if hk > 0:
            h_slots = torch.from_numpy(np.nonzero(temps <= float(houdayer_max_temperature))[0]).to(device)
            n_pairs = (K // 2) * int(h_slots.numel())
        samples = torch.empty((n_samples, K, prob.N), dtype=torch.uint8, device=device)
        energies = torch.empty((n_samples, K, R), dtype=torch.float64, device=device)
        for it in range(n_samples):
            su = None
            if inj is not None:
                sr_host = slot_replica[0].cpu().numpy()
                u_slot = np.asarray(inj["sweep_uniforms"][it])            # [slot, sweep, N]
                u_rep = np.empty_like(u_slot)
                u_rep[sr_host] = u_slot                                    # replica sr_host[i] sits at slot i
                su = torch.from_numpy(np.ascontiguousarray(u_rep.transpose(1, 0, 2))).to(device)
            _, e, _, _ = self._run(prob, states, n_burnin=n_sweeps, n_samples=0, sweeps_per_sample=0, T_chain=T_chain,
                                   want_energy=True, uniforms=su)
            if n_pairs and (it + 1) % hk == 0:  # ladders 2m and 2m + 1 at the selected slots
                sel = slot_replica[:, h_slots]
                pairs = torch.stack((sel[0::2], sel[1::2]), -1).reshape(-1, 2).contiguous()
                prob.houdayer(states, pairs, n_pairs, seed=self._seed, step0=self._houdayer_counter, n_steps=1,
                              chain0=chain0, energy=e)
                self._houdayer_counter += 1
            energies[it] = e[slot_replica.long()]          # history is kept per temperature slot (gibbs.py:302-303)
            if (it + 1) % swap_interval == 0:
                wu = None
                if inj is not None:
                    wu = torch.from_numpy(np.ascontiguousarray(np.asarray(inj["swap_uniforms"][it], dtype=np.float64))).to(device)
                self._swap_counter += 1
                with torch.cuda.device(device):
                    _lib.call("tsu_pt_swap", ptr(e), ptr(T_slot), ptr(slot_replica), None, K, R, self._seed,
                              self._swap_counter & 0xFFFFFFFF, ptr(stats), ptr(wu), 1 if criterion == "metropolis" else 0,
                              _lib.current_stream())
                T_chain[slot_replica.long()] = T_slot      # every replica takes the temperature of its new slot
            samples[it] = states[slot_replica[:, 0].long(), :prob.N]
        self._chain_counter += K * R
        st = stats.cpu().numpy()
        sr = slot_replica.cpu().numpy()
        states_np = _host_int64(states[:, :prob.N])
        en = energies.cpu().numpy()
        energy_lists = [[list(en[:, k, i]) for i in range(R)] for k in range(K)]
        final_states = [[states_np[sr[k, i]] for i in range(R)] for k in range(K)]
        info = {
            "swap_acceptance_rate": (st[1] / st[0]) if st[0] > 0 else 0,
            "swap_attempts": int(st[0]),
            "swap_accepts": int(st[1]),
            "energies": energy_lists[0] if K == 1 else energy_lists,
            "final_states": final_states[0] if K == 1 else final_states,
        }
        return self._samples_out(samples, K, False), info

    def simulated_annealing(self, coupling: np.ndarray, bias: Optional[np.ndarray] = None, T_initial: float = 10.0,
                            T_final: float = 0.1, n_steps: int = 1000, cooling_schedule: str = "exponential", *,
                            n_chains: int = 1, chromatic: bool = False, _uniforms=None,
                            _initial_state=None) -> Tuple[np.ndarray, float]:
        """tsu/gibbs.py:340-393: one sweep per step at the scheduled temperature, lowest energy tracked.

        The whole anneal is one kernel launch (per-sweep temperature array, on-device best tracking).
        With n_chains > 1 that many independent anneals run concurrently and the best is returned.

        precision="bf16": every step is one tensor-core sweep launch at Ts[k] and one tensor-core energy pass that
        keeps each chain's best state on the device.  The best chain is chosen by the energies of the bf16 model
        (the model this path samples); the returned energy is that state's energy under the caller's float64
        couplings and bias.  The two coincide when the couplings are exact in bf16.
        """
        _lib.require_cuda()
        if self.precision == "bf16" and not chromatic and _uniforms is not None:
            raise ValueError("injected draws are a float64 / float32 parity mode; precision='bf16' draws Philox")
        prob = self._problem(coupling, bias, chromatic=chromatic, tensor_ok=True)
        Ts = annealing_temperatures(T_initial, T_final, n_steps, cooling_schedule)
        st = self._initial_states(prob, int(n_chains), _initial_state)
        if n_steps > 0:
            self.config.temperature = float(Ts[-1])  # the reference leaves the last T in the config (gibbs.py:382)
            _, _, best_state, best_energy = self._run(prob, st, n_burnin=int(n_steps), n_samples=0, sweeps_per_sample=0,
                                                      T_sweep=Ts, track_best=True, **self._injected(prob, _uniforms))
            k = int(np.argmin(best_energy.cpu().numpy()))
            state = _host_int64(best_state[k])
        else:
            state = _host_int64(st[0, :prob.N])
        self._chain_counter += int(n_chains)
        return state, prob.energy(state)

    def population_annealing(self, coupling, temperatures, bias=None, *, n_chains: int = 1024, n_populations: int = 1,
                             sweeps_per_step: int = 10, T_start: float = math.inf, chromatic: bool = False,
                             previous: Optional[DensePopulationResult] = None) -> DensePopulationResult:
        """Population annealing (Hukushima-Iba, Machta) of n_chains chains in one call, with no host sync.

        The chains form n_populations equal contiguous populations of R_p chains, each resampled on its own.  A fresh
        run starts from the sampler's random initial states, which are equilibrium states at T_start = inf.  Step k:
        the energies of the current states, their moments (energy_moments[k]), a resampling of every population in
        proportion to exp(-dbeta_k E) with dbeta_k = 1/T_k - 1/T_{k-1} (T_{-1} = T_start), keeping R_p fixed
        (tsu_population_resample states the exact rule), then sweeps_per_step sweeps at T_k.  The chain at position j
        draws the Philox stream of chain0 + j, and the sweep indices continue from the sampler's counter.  The result
        gives ln Z ratios, free energies, mean energies, specific heats and the family statistic rho_t; see
        DensePopulationResult.

        The back end is the sampler's: precision="bf16" runs the tensor-core sweeps and energy pass, "float64" /
        "float32" the dense kernel, chromatic=True the chromatic CSR kernel (float64 sampler).  On bf16 the energies,
        and so the weights, are those of the bf16-rounded couplings: the model this path samples.

        temperatures must be non-increasing and at most T_start.  previous: the result of an earlier run with the same
        couplings, back end, chain count and populations; its last temperature becomes T_start and its states, family
        and chain0 are continued, so a run split into calls equals one call.  Afterwards the sweep counter has advanced
        by len(temperatures) * sweeps_per_step, the chain counter by n_chains (fresh runs only), and config.temperature
        is temperatures[-1].

        The call holds two state buffers of n_chains rows while it runs (a third when it continues `previous`, whose
        tensors it leaves as they were).
        """
        Ts = np.asarray(temperatures, dtype=np.float64)
        if Ts.ndim != 1 or Ts.size == 0:
            raise ValueError("temperatures must be a non-empty 1-D schedule")
        if not np.all(np.isfinite(Ts)) or np.any(Ts <= 0):
            raise ValueError("temperatures must be positive and finite")
        if np.any(np.diff(Ts) > 0):
            raise ValueError("temperatures must be non-increasing")
        theta, P, C = int(sweeps_per_step), int(n_populations), int(n_chains)
        if theta < 1:
            raise ValueError("sweeps_per_step must be >= 1")
        if C < 1:
            raise ValueError("n_chains must be at least 1")
        if P < 1 or P > 65535 or C % P:
            raise ValueError(f"n_populations must divide n_chains = {C} (and lie in [1, 65535])")
        r_pop = C // P
        N = int(coupling[3]) if isinstance(coupling, tuple) and len(coupling) == 4 else int(np.shape(coupling)[0])
        backend = "chromatic" if chromatic else self.precision
        if previous is not None:
            if (not isinstance(previous, DensePopulationResult) or previous.n_sites != N or previous.backend != backend
                    or tuple(previous.family.shape) != (C,) or previous.n_populations != P or previous.r_pop != r_pop):
                raise ValueError(f"previous must come from a run of {P} populations of {r_pop} chains of {N} bits on "
                                 f"the {backend} back end")
            T_start = float(previous.temperatures[-1])
        T_start = float(T_start)
        if not T_start > 0 or Ts[0] > T_start:
            raise ValueError("T_start must be positive and at least temperatures[0]")
        beta = 1.0 / Ts
        dbeta = np.diff(np.concatenate([[0.0 if math.isinf(T_start) else 1.0 / T_start], beta]))
        prob = self._problem(coupling, bias, chromatic=chromatic, tensor_ok=True)
        torch = _lib.require_cuda()
        dev, n = prob.device, int(Ts.size)
        with torch.cuda.device(dev):
            if previous is None:
                chain0 = self._chain_counter
                state = self._initial_states(prob, C)
                family = (torch.arange(C, dtype=torch.int64, device=dev) + (chain0 & M32)).to(torch.int32)
                _, energy, _, _ = self._run(prob, state, n_burnin=0, n_samples=0, sweeps_per_sample=0, T=Ts[0],
                                            chain0=chain0, want_energy=True)
            else:
                chain0, state, family, energy = previous.chain0, previous._state, previous.family, previous.energy
            other, family_other = torch.empty_like(state), torch.empty_like(family)
            work_bytes = int(_lib.load().tsu_ising2d_population_work_bytes(C, P))
            work = torch.empty(work_bytes // 8, dtype=torch.int64, device=dev)
            d_dbeta = torch.from_numpy(dbeta).to(dev)
            weight_sum = torch.empty((n, P), dtype=torch.int64, device=dev)
            energy_ref = torch.empty((n, P), dtype=torch.float64, device=dev)
            moments = torch.empty((n + 1, P, 2), dtype=torch.float64, device=dev)
            for k in range(n):
                _lib.call("tsu_population_moments", ptr(energy), C, P, ptr(moments[k]), _lib.current_stream())
                _lib.call("tsu_population_resample", ptr(state), ptr(other), ptr(family), ptr(family_other),
                          ptr(energy), ptr(d_dbeta[k]), C, P, int(state.shape[1]), self._seed,
                          self._sweep_counter & M32, chain0 & M32, ptr(weight_sum[k]), ptr(energy_ref[k]), ptr(work),
                          work_bytes, _lib.current_stream())
                state, other, family, family_other = other, state, family_other, family
                if k == 0 and previous is not None:  # previous's tensors stay as they were
                    other, family_other = torch.empty_like(state), torch.empty_like(family)
                _, energy, _, _ = self._run(prob, state, n_burnin=theta, n_samples=0, sweeps_per_sample=0, T=Ts[k],
                                            chain0=chain0, want_energy=True)
            _lib.call("tsu_population_moments", ptr(energy), C, P, ptr(moments[n]), _lib.current_stream())
        if previous is None:
            self._chain_counter += C
        self.config.temperature = float(Ts[-1])
        return DensePopulationResult(state, energy, family, weight_sum, energy_ref, moments, Ts.copy(), T_start, dbeta,
                                     r_pop, 62 - (r_pop - 1).bit_length(), N, chain0, backend)


def _bf16_exact(coupling) -> bool:
    """every coupling survives rounding to bf16 (8 significant bits) and the matrix fits the tensor-core kernel"""
    J = np.asarray(coupling, dtype=np.float64)
    if J.ndim != 2 or J.shape[0] != J.shape[1] or J.shape[0] > TC_MAX_N:
        return False
    u = J.astype(np.float32).view(np.uint32)
    rounded = ((u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000).view(np.float32)
    return bool(np.array_equal(rounded.astype(np.float64), J))


class HardwareEmulator:
    """tsu/gibbs.py:396-487.  The timing model is the reference's arithmetic; sample_parallel finally runs
    its `parallel_chains` chains in parallel (the reference loops over them, gibbs.py:475-479)."""

    def __init__(self, n_bits: int = 100, clock_speed_ghz: float = 1.0, parallel_chains: int = 1000, *,
                 precision: str = "auto"):
        self.n_bits = n_bits
        self.clock_speed_ghz = clock_speed_ghz
        self.parallel_chains = parallel_chains
        self.ns_per_cycle = 1.0 / clock_speed_ghz
        # "auto": the tensor-core path when the couplings are exactly representable in bf16 (e.g. +-1 / integer
        # graphs) and there are enough chains to fill a 64-chain tile; otherwise float64 fields
        self.precision = precision

    def estimate_hardware_time(self, n_samples: int, n_sweeps_per_sample: int) -> dict:
        """tsu/gibbs.py:421-448"""
        time_per_sweep_ns = self.n_bits * self.ns_per_cycle
        time_per_sample_ns = n_sweeps_per_sample * time_per_sweep_ns
        batches_needed = int(np.ceil(n_samples / self.parallel_chains))
        total_time_ns = batches_needed * time_per_sample_ns
        return {
            "time_per_sweep_ns": time_per_sweep_ns,
            "time_per_sample_ns": time_per_sample_ns,
            "batches_needed": batches_needed,
            "total_time_ns": total_time_ns,
            "total_time_us": total_time_ns / 1000,
            "total_time_ms": total_time_ns / 1e6,
            "total_time_s": total_time_ns / 1e9,
            "speedup_vs_classical": None,
        }

    def sample_parallel(self, coupling: np.ndarray, n_samples: int, temperature: float = 1.0) -> Tuple[np.ndarray, dict]:
        """tsu/gibbs.py:450-487: min(parallel_chains, n_samples) chains x ceil(n_samples/parallel_chains)
        samples each (burn-in 100), stacked chain after chain and truncated to n_samples."""
        config = GibbsConfig(temperature=temperature)
        samples_per_chain = int(np.ceil(n_samples / self.parallel_chains))
        n_chains = min(self.parallel_chains, n_samples)
        precision = self.precision
        if precision == "auto":
            precision = "bf16" if (n_chains >= 64 and _bf16_exact(coupling)) else "float64"
        sampler = GibbsSampler(config, precision=precision)
        out = sampler.sample_boltzmann(coupling, n_samples=samples_per_chain, burnin=100, n_chains=n_chains)
        if n_chains == 1:
            out = out[None]
        samples = out.reshape(n_chains * samples_per_chain, -1)[:n_samples]
        timing = self.estimate_hardware_time(n_samples, config.n_sweeps)
        return samples, timing
