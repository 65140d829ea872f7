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

from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

from . import _lib
from ._lib import ptr


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


# csrc/dense_gibbs.cu keeps a chain's uniforms (and their logits with float64 fields), fields, self couplings and bits
# in at most 227 KB of shared memory: 33 N + 272 bytes with float64 fields, 17 N + 272 with float32
DENSE_MAX_N = {"float64": 7035, "float32": 13657}


class _DenseProblem:
    """coupling matrix + bias resident on the device (transposed, see tsu_b200.h)"""

    def __init__(self, coupling, bias, precision: str, device):
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
        self.Jt = torch.from_numpy(np.ascontiguousarray(J.T.astype(self.np_dtype))).to(device)
        if bias is not None:
            b = np.asarray(bias, dtype=np.float64)
            if b.shape != (self.N,):
                raise ValueError("bias must have one entry per bit")
            self.bias = torch.from_numpy(np.ascontiguousarray(b.astype(self.np_dtype))).to(device)
        else:
            self.bias = None


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

    def pad_state(self, st):
        if self.Np == self.N:
            return st
        torch = _lib.require_cuda()
        out = torch.zeros((st.shape[0], self.Np), dtype=torch.uint8, device=st.device)
        out[:, :self.N] = st
        return out


def annealing_temperatures(T_initial: float, T_final: float, n_steps: int, cooling_schedule: str = "exponential"):
    """float64 [n_steps]: the temperature of every annealing step (tsu/gibbs.py:340-393): T_initial at step 0 towards
    T_final, which is not reached; "exponential" or, for anything else, "linear" cooling"""
    steps = np.arange(n_steps, dtype=np.float64)
    if cooling_schedule == "exponential":
        return T_initial * (T_final / T_initial) ** (steps / n_steps)
    return T_initial + (T_final - T_initial) * steps / n_steps  # linear


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
        state = np.asarray(state)
        energy = -0.5 * state.dot(coupling).dot(state)
        if bias is not None:
            energy -= np.asarray(bias).dot(state)
        return float(energy)

    # ------------------------------------------------------------------ device plumbing
    def _dev(self):
        torch = _lib.require_cuda()
        return torch.device(self._device) if self._device is not None else torch.device("cuda", torch.cuda.current_device())

    def _orders(self, n_sweeps: int, N: int, device):
        """visiting order per sweep: None for 'sequential', fresh permutations for 'random' (gibbs.py:153-157)"""
        if self.config.update_order == "sequential" or n_sweeps == 0:
            return None
        torch = _lib.require_cuda()
        rng = np.random.Generator(np.random.Philox(key=[self._seed, self._sweep_counter]))
        perms = np.stack([rng.permutation(N) for _ in range(n_sweeps)]).astype(np.int32)
        return torch.from_numpy(perms).to(device)

    def _run(self, prob: _DenseProblem, state, *, n_burnin: int, n_samples: int, sweeps_per_sample: int,
             T_chain=None, T_sweep=None, want_samples=False, want_energy=False, track_best=False,
             order=None, uniforms=None, visits_per_sweep: int = 0):
        """one launch of tsu_dense_gibbs_run on `state` (uint8 tensor [n_chains, N], updated in place)"""
        torch = _lib.require_cuda()
        device = prob.device
        n_chains, N = state.shape
        total = n_burnin + n_samples * sweeps_per_sample
        if order is None and visits_per_sweep == 0:
            order = self._orders(total, N, device)
        samples = torch.empty((n_samples, n_chains, N), dtype=torch.uint8, device=device) if want_samples else None
        energy = torch.empty(n_chains, dtype=torch.float64, device=device) if (want_energy or track_best) else None
        best_state = torch.empty((n_chains, N), dtype=torch.uint8, device=device) if track_best else None
        best_energy = torch.empty(n_chains, dtype=torch.float64, device=device) if track_best else None
        with torch.cuda.device(device):
            _lib.call(
                "tsu_dense_gibbs_run", ptr(prob.Jt), prob.code, ptr(prob.bias), ptr(state), n_chains, N,
                float(self.config.temperature), ptr(T_chain), ptr(T_sweep), int(n_burnin), int(n_samples),
                int(sweeps_per_sample), ptr(order), ptr(uniforms), ptr(samples), ptr(energy), int(track_best),
                ptr(best_state), ptr(best_energy), self._seed, self._sweep_counter & 0xFFFFFFFF,
                self._chain_counter & 0xFFFFFFFF, prob.code, int(visits_per_sweep), _lib.current_stream(),
            )
        self._sweep_counter += total
        return samples, energy, best_state, best_energy

    def _initial_states(self, prob, n_chains: int, initial_state=None):
        torch = _lib.require_cuda()
        if initial_state is not None:
            a = np.asarray(initial_state)
            if a.ndim == 1:
                if a.shape != (prob.N,):
                    raise ValueError(f"initial_state must have {prob.N} entries, got shape {a.shape}")
                a = np.broadcast_to(a, (n_chains, prob.N))
            elif a.shape != (n_chains, prob.N):
                raise ValueError(f"initial_state must have shape ({prob.N},) or ({n_chains}, {prob.N}), got {a.shape}")
            return torch.from_numpy(np.ascontiguousarray((a != 0).astype(np.uint8))).to(prob.device)
        state = torch.empty((n_chains, prob.N), dtype=torch.uint8, device=prob.device)
        with torch.cuda.device(prob.device):
            _lib.call("tsu_dense_init_random", ptr(state), n_chains, prob.N, self._seed ^ 0x5DEECE66D,
                      (self._chain_counter + self._sweep_counter) & 0xFFFFFFFF, _lib.current_stream())
        return state

    # ------------------------------------------------------------------ reference API
    def sample_conditional(self, i: int, state: np.ndarray, coupling: np.ndarray,
                           bias: Optional[np.ndarray] = None) -> int:
        """tsu/gibbs.py:102-126: resample bit i given the others (one single-site visit on the device)"""
        torch = _lib.require_cuda()
        prob = _DenseProblem(coupling, bias, self.precision, self._dev())
        st = self._initial_states(prob, 1, np.asarray(state))
        order = torch.tensor([[int(i)]], dtype=torch.int32, device=prob.device)
        self._run(prob, st, n_burnin=1, n_samples=0, sweeps_per_sample=0, order=order, visits_per_sweep=1)
        return int(st[0, int(i)].item())

    def _inject(self, prob, uniforms, orders):
        """parity mode: float64 uniforms [sweeps, N] (single chain) / [sweeps, chains, N] and orders [sweeps, N]"""
        torch = _lib.require_cuda()
        u = o = None
        if uniforms is not None:
            a = np.asarray(uniforms, dtype=np.float64)
            if a.ndim == 2:
                a = a[:, None, :]
            u = torch.from_numpy(np.ascontiguousarray(a)).to(prob.device)
        if orders is not None:
            o = torch.from_numpy(np.ascontiguousarray(np.asarray(orders, dtype=np.int32))).to(prob.device)
        return u, o

    def _sparse(self, coupling, bias):
        """couplings in CSR form + colour classes on the device (csrc/sparse_gibbs.cu); float64 fields"""
        from .sparse import SparseProblem

        if self.precision != "float64":
            raise ValueError("chromatic=True (sparse couplings) computes float64 fields: use a 'float64' sampler")
        return SparseProblem(coupling, bias, self._dev())

    def _sparse_run(self, prob, state, uniforms=None, **kw):
        from . import sparse

        torch = _lib.require_cuda()
        u = None
        if uniforms is not None:  # parity mode: [sweeps, N] or [sweeps, chains, N] float64 in VISITING order
            a = np.asarray(uniforms, dtype=np.float64)
            if a.ndim == 2:
                a = a[:, None, :]
            u = torch.from_numpy(np.ascontiguousarray(a)).to(prob.device)
        total = kw["n_burnin"] + kw["n_samples"] * kw["sweeps_per_sample"]
        out = sparse.run(prob, state, T=float(self.config.temperature), seed=self._seed, sweep0=self._sweep_counter,
                         chain0=self._chain_counter, uniforms=u, **kw)
        self._sweep_counter += total
        return out

    def gibbs_sweep(self, state: np.ndarray, coupling: np.ndarray, bias: Optional[np.ndarray] = None,
                    n_sweeps: int = 1, *, chromatic: bool = False, _uniforms=None, _orders=None) -> np.ndarray:
        """tsu/gibbs.py:128-162: n_sweeps sweeps over all bits; the input is not modified (gibbs.py:150).
        chromatic=True: sparse couplings, sites visited colour class by colour class (csrc/sparse_gibbs.cu)"""
        if chromatic:
            prob = self._sparse(coupling, bias)
            st = self._initial_states(prob, 1, np.asarray(state))
            self._sparse_run(prob, st, uniforms=_uniforms, n_burnin=int(n_sweeps), n_samples=0, sweeps_per_sample=0)
            a = np.asarray(state)
            return st[0].cpu().numpy().astype(a.dtype if a.dtype.kind in "iu" else np.int64)
        prob = _DenseProblem(coupling, bias, self.precision, self._dev())
        st = self._initial_states(prob, 1, np.asarray(state))
        u, o = self._inject(prob, _uniforms, _orders)
        self._run(prob, st, n_burnin=int(n_sweeps), n_samples=0, sweeps_per_sample=0, uniforms=u, order=o)
        out = st[0].cpu().numpy().astype(np.asarray(state).dtype if np.asarray(state).dtype.kind in "iu" else np.int64)
        return out

    def sample_boltzmann(self, coupling: np.ndarray, bias: Optional[np.ndarray] = None, n_samples: int = 1000,
                         burnin: Optional[int] = None, initial_state: Optional[np.ndarray] = None, *,
                         n_chains: int = 1, as_tensor: bool = False, chromatic: bool = False, _uniforms=None,
                         _orders=None):
        """tsu/gibbs.py:164-213: burn-in, then n_samples x config.n_sweeps sweeps; one launch.

        n_chains == 1 (default): int array (n_samples, n_bits) like the reference.
        n_chains > 1: (n_chains, n_samples, n_bits) - independent chains run concurrently.
        chromatic=True: sparse couplings (dense array, scipy.sparse matrix or CSR tuple) on the chromatic CSR kernel;
        a sweep visits the sites colour class by colour class instead of in index order.
        """
        burnin = burnin if burnin is not None else self.config.n_burnin
        if chromatic:
            prob = self._sparse(coupling, bias)
            st = self._initial_states(prob, int(n_chains), initial_state)
            samples, _, _, _ = self._sparse_run(prob, st, uniforms=_uniforms, n_burnin=int(burnin),
                                                n_samples=int(n_samples), sweeps_per_sample=self.config.n_sweeps,
                                                want_samples=True)
            self._chain_counter += int(n_chains)
            self.sample_count += int(n_samples)
            if as_tensor:
                return samples if n_chains > 1 else samples[:, 0]
            out = _host_int64(samples)
            return out[:, 0, :] if n_chains == 1 else np.ascontiguousarray(out.transpose(1, 0, 2))
        if self.precision == "bf16":
            if _uniforms is not None or _orders is not None:
                raise ValueError("injected draws are a float64 / float32 parity mode; precision='bf16' draws Philox")
            return self._sample_boltzmann_tensor(coupling, bias, int(n_samples), int(burnin), initial_state,
                                                 int(n_chains), as_tensor)
        prob = _DenseProblem(coupling, bias, self.precision, self._dev())
        st = self._initial_states(prob, int(n_chains), initial_state)
        u, o = self._inject(prob, _uniforms, _orders)
        samples, _, _, _ = self._run(prob, st, n_burnin=int(burnin), n_samples=int(n_samples),
                                     sweeps_per_sample=self.config.n_sweeps, want_samples=True, uniforms=u, order=o)
        self._chain_counter += int(n_chains)
        self.sample_count += int(n_samples)
        if as_tensor:
            return samples if n_chains > 1 else samples[:, 0]
        out = _host_int64(samples)  # (n_samples, n_chains, N)
        if n_chains == 1:
            return out[:, 0, :]
        return np.ascontiguousarray(out.transpose(1, 0, 2))

    def sample(self, J: np.ndarray, n_samples: int = 1000, **kwargs) -> np.ndarray:
        """README.md:69-80: `sampler.sample(J, n_samples=1000)` -> (n_samples, n_bits) binary configurations"""
        return self.sample_boltzmann(J, n_samples=n_samples, **kwargs)

    def _tc_sweeps(self, prob: "_TcProblem", st, n_sweeps: int, T, fields=None):
        """n_sweeps sequential sweeps of all chains of `st` ([n_chains, Np] uint8, in place) on the tensor cores at
        temperature T: a scalar, or a float64 device tensor [n_chains] of per-chain temperatures"""
        torch = _lib.require_cuda()
        if n_sweeps <= 0:
            return
        T_chain = T if isinstance(T, torch.Tensor) else None
        with torch.cuda.device(prob.device):
            _lib.call("tsu_dense_gibbs_tc_run", ptr(prob.J), ptr(prob.bias), ptr(st), int(st.shape[0]), prob.Np,
                      1.0 if T_chain is not None else float(T), ptr(T_chain), int(n_sweeps), self._seed,
                      self._sweep_counter & 0xFFFFFFFF, self._chain_counter & 0xFFFFFFFF, ptr(fields),
                      _lib.current_stream())
        self._sweep_counter += int(n_sweeps)

    @staticmethod
    def _tc_energy(prob: "_TcProblem", st, energy, best_energy=None, best_state=None):
        """energy[c] = -1/2 s^T J s - b^T s of every chain of `st` on the tensor cores (bf16 J, float64 sums); with
        best_energy / best_state, chains whose energy is strictly lower than best_energy take it and their state"""
        torch = _lib.require_cuda()
        with torch.cuda.device(prob.device):
            _lib.call("tsu_dense_tc_energy", ptr(prob.J), ptr(prob.bias), ptr(st), int(st.shape[0]), prob.Np,
                      ptr(energy), ptr(best_energy), ptr(best_state), _lib.current_stream())

    def _sample_boltzmann_tensor(self, coupling, bias, n_samples, burnin, initial_state, n_chains, as_tensor):
        """tsu/gibbs.py:198-211 on csrc/dense_tc.cu: burn-in sweeps, then n_samples x config.n_sweeps sweeps with the
        state of every chain recorded after each group; bf16 couplings, fp32 fields accumulated in TMEM"""
        torch = _lib.require_cuda()
        prob = _TcProblem(coupling, bias, self._dev(), self.config.update_order)
        st = prob.pad_state(self._initial_states(prob, n_chains, initial_state))
        samples = torch.empty((n_samples, n_chains, prob.N), dtype=torch.uint8, device=prob.device)
        T = self.config.temperature
        self._tc_sweeps(prob, st, burnin, T)
        for k in range(n_samples):
            self._tc_sweeps(prob, st, self.config.n_sweeps, T)
            samples[k] = st[:, :prob.N]
        self._chain_counter += n_chains
        self.sample_count += n_samples
        if as_tensor:
            return samples if n_chains > 1 else samples[:, 0]
        out = _host_int64(samples)
        if n_chains == 1:
            return out[:, 0, :]
        return np.ascontiguousarray(out.transpose(1, 0, 2))

    def _sample_chains_tensor(self, coupling, bias, n_chains, n_sweeps, initial_state, as_tensor, return_energy):
        """tensor-core path (csrc/dense_tc.cu): bf16 couplings, fp32 fields accumulated in TMEM"""
        torch = _lib.require_cuda()
        prob = _TcProblem(coupling, bias, self._dev(), self.config.update_order)
        device, N = prob.device, prob.N
        st = prob.pad_state(self._initial_states(prob, int(n_chains), initial_state))
        self._tc_sweeps(prob, st, int(n_sweeps), self.config.temperature)
        self._chain_counter += int(n_chains)
        energy = None
        if return_energy:  # E = -1/2 s^T J s - b^T s: one more tensor-core field evaluation, summed on the device
            energy = torch.empty(int(n_chains), dtype=torch.float64, device=device)
            self._tc_energy(prob, st, energy)
        st = st[:, :N]
        out = st if as_tensor else _host_int64(st)
        if return_energy:
            return out, (energy if as_tensor else energy.cpu().numpy())
        return out

    def sample_chains(self, coupling, bias=None, n_chains: int = 1024, n_sweeps: Optional[int] = None,
                      initial_state=None, as_tensor: bool = False, return_energy: bool = False):
        """batched entry point: n_chains independent chains, n_sweeps sweeps each, final states returned.

        This is the shape of BASELINE config 3 (dense J, N=4096, 2048 chains, 10 sweeps).  With
        precision="bf16" the fields are evaluated on the tensor cores (tcgen05, csrc/dense_tc.cu)."""
        if self.precision == "bf16":
            n_sw = self.config.n_sweeps if n_sweeps is None else int(n_sweeps)
            return self._sample_chains_tensor(coupling, bias, n_chains, n_sw, initial_state, as_tensor, return_energy)
        prob = _DenseProblem(coupling, bias, self.precision, self._dev())
        n_sweeps = self.config.n_sweeps if n_sweeps is None else int(n_sweeps)
        st = self._initial_states(prob, int(n_chains), initial_state)
        _, energy, _, _ = self._run(prob, st, n_burnin=n_sweeps, n_samples=0, sweeps_per_sample=0,
                                    want_energy=return_energy)
        self._chain_counter += int(n_chains)
        out = st if as_tensor else _host_int64(st)
        if return_energy:
            return out, (energy if as_tensor else energy.cpu().numpy())
        return out

    def parallel_tempering(self, coupling: np.ndarray, temperatures: List[float], bias: Optional[np.ndarray] = None,
                           n_samples: int = 1000, swap_interval: int = 10, *, n_ladders: int = 1,
                           criterion: str = "reference", _inject=None) -> Tuple[np.ndarray, dict]:
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
        """
        torch = _lib.require_cuda()
        K = int(n_ladders)
        if K < 1:
            raise ValueError("n_ladders must be at least 1")
        if criterion not in ("metropolis", "reference"):
            raise ValueError("criterion must be 'metropolis' or 'reference'")
        tc = self.precision == "bf16"
        if _inject is not None and (tc or K > 1):
            raise ValueError("injected draws are a float64 / float32 parity mode of one ladder")
        if tc:
            prob = _TcProblem(coupling, bias, self._dev(), self.config.update_order)
        else:
            prob = _DenseProblem(coupling, bias, self.precision, self._dev())
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
        if tc:
            states = prob.pad_state(states)
            e = torch.empty(K * R, dtype=torch.float64, device=device)
            self._tc_sweeps(prob, states, self.config.n_burnin, T_chain)
        else:
            bu = None
            if inj is not None:  # parity mode: draws are given per temperature slot; slot i starts on replica i
                bu = torch.from_numpy(np.ascontiguousarray(np.asarray(inj["burn_uniforms"]).transpose(1, 0, 2))).to(device)
            self._run(prob, states, n_burnin=self.config.n_burnin, n_samples=0, sweeps_per_sample=0, T_chain=T_chain,
                      uniforms=bu)
        samples = torch.empty((n_samples, K, prob.N), dtype=torch.uint8, device=device)
        energies = torch.empty((n_samples, K, R), dtype=torch.float64, device=device)
        for it in range(n_samples):
            if tc:
                self._tc_sweeps(prob, states, n_sweeps, T_chain)
                self._tc_energy(prob, states, e)
            else:
                su = None
                if inj is not None:
                    sr_host = slot_replica[0].cpu().numpy()
                    u_slot = np.asarray(inj["sweep_uniforms"][it])            # [slot, sweep, N]
                    u_rep = np.empty_like(u_slot)
                    u_rep[sr_host] = u_slot                                    # replica sr_host[i] sits at slot i
                    su = torch.from_numpy(np.ascontiguousarray(u_rep.transpose(1, 0, 2))).to(device)
                _, e, _, _ = self._run(prob, states, n_burnin=n_sweeps, n_samples=0, sweeps_per_sample=0,
                                       T_chain=T_chain, want_energy=True, uniforms=su)
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
        out = _host_int64(samples)                         # (n_samples, K, N)
        return (out[:, 0, :], info) if K == 1 else (np.ascontiguousarray(out.transpose(1, 0, 2)), info)

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
        torch = _lib.require_cuda()
        tc = self.precision == "bf16" and not chromatic
        if tc:
            if _uniforms is not None:
                raise ValueError("injected draws are a float64 / float32 parity mode; precision='bf16' draws Philox")
            prob = _TcProblem(coupling, bias, self._dev(), self.config.update_order)
        elif chromatic:
            prob = self._sparse(coupling, bias)
        else:
            prob = _DenseProblem(coupling, bias, self.precision, self._dev())
        Ts = annealing_temperatures(T_initial, T_final, n_steps, cooling_schedule)
        st = self._initial_states(prob, int(n_chains), _initial_state)
        if tc and n_steps > 0:
            st = prob.pad_state(st)
            energy = torch.empty(int(n_chains), dtype=torch.float64, device=prob.device)
            best_energy = torch.full((int(n_chains),), float("inf"), dtype=torch.float64, device=prob.device)
            best_state = torch.empty_like(st)
            self._tc_energy(prob, st, energy, best_energy, best_state)   # the initial state is the first best
            for k in range(int(n_steps)):
                self._tc_sweeps(prob, st, 1, float(Ts[k]))
                self._tc_energy(prob, st, energy, best_energy, best_state)
            self.config.temperature = float(Ts[-1])
            k = int(np.argmin(best_energy.cpu().numpy()))
            state = _host_int64(best_state[k, :prob.N])
        elif n_steps > 0:
            T_sweep = torch.from_numpy(Ts).to(prob.device)
            self.config.temperature = float(Ts[-1])  # the reference leaves the last T in the config (gibbs.py:382)
            if chromatic:
                _, _, best_state, best_energy = self._sparse_run(prob, st, uniforms=_uniforms, n_burnin=int(n_steps),
                                                                 n_samples=0, sweeps_per_sample=0, T_sweep=T_sweep,
                                                                 track_best=True)
            else:
                u, _ = self._inject(prob, _uniforms, None)
                _, _, best_state, best_energy = self._run(prob, st, n_burnin=int(n_steps), n_samples=0,
                                                          sweeps_per_sample=0, T_sweep=T_sweep, track_best=True,
                                                          uniforms=u)
            be = best_energy.cpu().numpy()
            k = int(np.argmin(be))
            state = _host_int64(best_state[k])
        else:
            state = _host_int64(st[0])
        self._chain_counter += int(n_chains)
        if chromatic:
            from .sparse import to_csr

            rowptr, col, val, _ = to_csr(coupling)
            sb = state.astype(np.float64)
            row = np.repeat(np.arange(len(sb)), np.diff(rowptr))
            e = -0.5 * float(np.sum(val * sb[row] * sb[col]))
            if bias is not None:
                e -= float(np.dot(np.asarray(bias, dtype=np.float64), sb))
            return state, e
        J = np.asarray(coupling, dtype=np.float64)
        return state, self.compute_energy(state, J, None if bias is None else np.asarray(bias, dtype=np.float64))


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
