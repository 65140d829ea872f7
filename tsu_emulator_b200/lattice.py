"""
Batched 2-D Ising lattice engine on one B200: host side of the bit-packed checkerboard kernels
(csrc/ising2d.cu, C-ABI tsu_ising2d_* in include/tsu_b200.h).

It replaces, for nearest-neighbour lattices, the reference path
    IsingGrid.__init__ (dense N x N J)            tsu/models/ising.py:320-361
    IsingModel.sample -> GibbsSampler.gibbs_sweep  tsu/models/ising.py:150-181, tsu/gibbs.py:128-162
without ever materialising J: the acceptance probabilities sigmoid(h_bit/T) of the (at most 15)
distinct local environments are tabulated on the host in float64 with the reference's own
formula and handed to the kernel as integer thresholds.
"""

import math
from typing import Optional, Sequence, Union

import numpy as np

from . import _lib
from ._lib import c_void_p, ptr
from .population import PopulationEstimates

LUT_WORDS = 32


def sigmoid_clamped(x: float) -> float:
    """tsu/gibbs.py:61-77: sigma(x) with x > 20 -> 1.0, x < -20 -> 0.0 (strict), float64."""
    if x > 20:
        return 1.0
    elif x < -20:
        return 0.0
    return 1.0 / (1.0 + np.exp(-x))


def build_lut(J: float, h: float, T: float, bias_mode: str = "physical") -> np.ndarray:
    """threshold table uint32[32] for one (J, h, T).

    Entry d*5+u: site with d neighbours, u of them up.  Bit model of tsu/models/ising.py:127-148:
    J_bit = 4J, local field = 4J*u + h_bit (tsu/gibbs.py:96-99), with
      bias_mode "physical":  h_bit =  2h - 2*rowsum(J)   (correct spin->bit transformation)
      bias_mode "reference": h_bit = -2h + 2*rowsum(J)   (what ising.py:148 returns)
    p = sigmoid_clamped(field / T); threshold = ceil(p * 2^32) so that for an integer uniform k,
    (k / 2^32 < p) == (k < threshold).  Entry 25: bit mask of classes with p == 1.0.
    """
    if T <= 0:
        raise ValueError("Temperature must be positive")
    lut = np.zeros(LUT_WORDS, dtype=np.uint32)
    always = 0
    for d in range(5):
        rowsum = J * d
        if bias_mode == "physical":
            bias = 2 * h - 2 * rowsum
        elif bias_mode == "reference":
            bias = -2 * h + 2 * rowsum
        else:
            raise ValueError("bias_mode must be 'physical' or 'reference'")
        for u in range(5):
            field = float(4 * J * u) + float(bias)
            p = sigmoid_clamped(field / T)
            t = int(math.ceil(p * 4294967296.0))
            if t >= 4294967296:
                always |= 1 << (d * 5 + u)
                t = 4294967295
            lut[d * 5 + u] = t
    lut[25] = always
    return lut


def cluster_threshold(J: float, T: float) -> int:
    """Swendsen-Wang bond activation threshold t = ceil(p 2^32), p = 1 - exp(-2|J|/T) in float64, as a Python int: a
    satisfied bond with 32-bit uniform u is active iff u < t; t = 2^32 (p rounds to 1) activates every one."""
    if T <= 0:
        raise ValueError("Temperature must be positive")
    p = -math.expm1(-2.0 * abs(float(J)) / float(T))
    return int(math.ceil(p * 4294967296.0))


# Swendsen-Wang workspace per engine: replicas beyond what fits run in chunks (same bits); tests may lower it
CLUSTER_WORK_BUDGET = 4 << 30


def lattice_bond_count(rows: int, cols: int, wrap_rows: bool, wrap_cols: bool) -> int:
    """number of distinct bonds wired by tsu/models/ising.py:343-361"""
    return rows * (cols - 1) + (rows if wrap_cols else 0) + (rows - 1) * cols + (cols if wrap_rows else 0)


def check_bonds(bonds, bond_index, rows: int, cols: int, n_replicas: int, bias_mode: str = "physical",
                is_slab: bool = False):
    """validated +-1 signs int8 [K, 2, rows, cols] and int32 bond_index [n_replicas] (None: all realisation 0) of an
    Edwards-Anderson engine (see Ising2DEngine); ValueError for anything the bonded kernels cannot serve"""
    if bias_mode != "physical":
        raise ValueError("bonds need bias_mode='physical': the reference bias depends on each site's signed row sum, "
                         "which the threshold table cannot express")
    if is_slab:
        raise ValueError("bonds are not available on row-slab engines")
    b = np.asarray(bonds)
    if b.ndim == 3:
        b = b[None]
    if b.ndim != 4 or b.shape[1:] != (2, rows, cols) or b.shape[0] < 1:
        raise ValueError(f"bonds must have shape (2, {rows}, {cols}) or (K, 2, {rows}, {cols}), got {np.shape(bonds)}")
    if b.dtype == np.bool_ or not np.all((b == 1) | (b == -1)):
        raise ValueError("bonds must hold +1 or -1 only")
    K = b.shape[0]
    if bond_index is None:
        if K == 1:
            idx = None
        elif K == n_replicas:
            idx = np.arange(K, dtype=np.int32)
        else:
            raise ValueError("bond_index is required when the number of realisations is neither 1 nor n_replicas")
    else:
        idx = np.asarray(bond_index)
        if idx.shape != (n_replicas,) or not np.issubdtype(idx.dtype, np.integer):
            raise ValueError(f"bond_index must hold {n_replicas} integers")
        if np.any(idx < 0) or np.any(idx >= K):
            raise ValueError(f"bond_index entries must lie in [0, {K})")
        idx = idx.astype(np.int32)
    return b.astype(np.int8), idx


class AnnealResult:
    """What Ising2DEngine.anneal returns; pass it back as `best=` to continue an anneal.

    energy:      float64 device tensor [n_replicas], E of every replica's final state
    best_energy: float64 device tensor [n_replicas], lowest E seen by each replica (None with track_best=False)
    best_state:  int32 device tensor [n_replicas, 2, rows, wpr], the packed state that had best_energy (same layout as
                 Ising2DEngine.state; None with track_best=False)
    """

    def __init__(self, energy, best_energy, best_state, rows: int, cols: int):
        self.energy, self.best_energy, self.best_state = energy, best_energy, best_state
        self.rows, self.cols = int(rows), int(cols)

    def best_spins(self, pm1: bool = True):
        """int8 device tensor [n_replicas, rows, cols] of the best states ({-1, +1}, or {0, 1} with pm1=False)"""
        if self.best_state is None:
            raise ValueError("this anneal kept no best states (track_best=False)")
        torch = _lib.require_cuda()
        dev = self.best_state.device
        with torch.cuda.device(dev):
            out = torch.empty((self.best_state.shape[0], self.rows, self.cols), dtype=torch.int8, device=dev)
            _lib.call("tsu_ising2d_unpack", ptr(self.best_state), ptr(out), int(self.best_state.shape[0]), self.rows,
                      self.cols, 1 if pm1 else 0, _lib.current_stream())
        return out


class PopulationResult(PopulationEstimates):
    """What Ising2DEngine.population_annealing returns; pass it back as `previous=` to continue the run.

    Device tensors (P = n_populations, n = len(temperatures)):
      energy      float64 [n_replicas], E of every replica's final state
      family      int32 [n_replicas], the initial replica (replica0 + r) each replica descends from
      weight_sum  int64 [n, P], W = sum of the quantised weights floor(exp(-dbeta (E_i - E_ref)) 2^s) of step k
      energy_ref  float64 [n, P], E_ref = lowest E of the population entering step k
      count_sums  int64 [n + 1, P, 2], (sum of up spins, sum of anti-aligned / unsatisfied bonds) of the states
                  entering step k; entry n: the final states
    Host: temperatures, T_start, dbeta, r_pop (R_p), shift (s), rows, cols, J, h, n_bonds, n_sites.
    ln Z ratios, free energies and rho_t: PopulationEstimates.
    """

    def __init__(self, energy, family, weight_sum, energy_ref, count_sums, temperatures, T_start, dbeta, r_pop, shift,
                 rows, cols, J, h, n_bonds, n_sites):
        self.energy, self.family = energy, family
        self.weight_sum, self.energy_ref, self.count_sums = weight_sum, energy_ref, count_sums
        self.temperatures, self.T_start, self.dbeta = temperatures, float(T_start), dbeta
        self.r_pop, self.shift = int(r_pop), int(shift)
        self.rows, self.cols, self.J, self.h = int(rows), int(cols), float(J), float(h)
        self.n_bonds, self.n_sites = int(n_bonds), int(n_sites)

    def mean_energy(self) -> np.ndarray:
        """[n, P]: population mean of E at temperatures[k] (after step k's sweeps), from count_sums[1:]"""
        c = self.count_sums[1:].cpu().numpy().astype(np.float64) / self.r_pop
        return -self.J * (self.n_bonds - 2.0 * c[..., 1]) - self.h * (2.0 * c[..., 0] - self.n_sites)


class Ising2DEngine:
    """n_replicas independent rows x cols lattices (or one row-slab of each) resident in HBM.

    State: torch int32 tensor [n_replicas, 2, rows, wpr] (bit-packed, layout in include/tsu_b200.h).
    Replica r uses temperature temperatures[r] (scalar = shared).  All randomness is
    Philox(seed; replica0+r, sweep index, global row, word), so a lattice split into row slabs
    (row0/halos) or a replica batch split across GPUs (replica0) reproduces the single-GPU bits.

    Edwards-Anderson +-J spin glasses: `bonds` holds +-1 of shape (2, rows, cols) or (K, 2, rows, cols);
    [k, 0, i, j] is the bond (i, j)-(i, (j+1) % cols), [k, 1, i, j] the bond (i, j)-((i+1) % rows, j), and the
    coupling of a bond is coupling * sign.  Entries of bonds the wiring does not create (open edges, the wrap of a
    periodic dimension of length 2) are ignored.  `bond_index` maps each replica to one of the K realisations
    (default: all 0 when K = 1, arange when K = n_replicas).  Whole lattices with bias_mode "physical" only.
    """

    def __init__(
        self,
        rows: int,
        cols: int,
        n_replicas: int = 1,
        coupling: float = 1.0,
        field: float = 0.0,
        temperature: Union[float, Sequence[float]] = 1.0,
        periodic: bool = True,
        seed: int = 0,
        device=None,
        bias_mode: str = "physical",
        replica0: int = 0,
        row0: int = 0,
        global_rows: Optional[int] = None,
        bonds=None,
        bond_index=None,
    ):
        if bonds is not None:  # checked before anything touches the device
            bonds, bond_index = check_bonds(bonds, bond_index, rows, cols, n_replicas, bias_mode,
                                            global_rows is not None and int(global_rows) != int(rows) or int(row0) != 0)
        elif bond_index is not None:
            raise ValueError("bond_index needs bonds")
        torch = _lib.require_cuda()
        self._torch = torch
        self.lib = _lib.load()
        if rows <= 0 or cols <= 0 or n_replicas <= 0:
            raise ValueError("rows, cols and n_replicas must be positive")
        self.rows, self.cols, self.n_replicas = int(rows), int(cols), int(n_replicas)
        self.global_rows = int(global_rows) if global_rows is not None else self.rows
        self.row0 = int(row0)
        self.is_slab = self.global_rows != self.rows
        if periodic and (self.global_rows % 2 or cols % 2):
            raise ValueError("periodic checkerboard lattices need even rows and cols")
        self.periodic = bool(periodic)
        # a periodic dimension of size 2 adds no new bond in the reference (set_coupling assigns)
        self.wrap_rows = self.periodic and self.global_rows > 2
        self.wrap_cols = self.periodic and cols > 2
        self.coupling, self.field = float(coupling), float(field)
        self.bias_mode = bias_mode
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.replica0 = int(replica0)
        self.sweep_index = 0
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.wpr = int(self.lib.tsu_ising2d_words_per_row(self.cols))
        with torch.cuda.device(self.device):
            self.state = torch.zeros((self.n_replicas, 2, self.rows, self.wpr), dtype=torch.int32, device=self.device)
            self._obs = torch.zeros((self.n_replicas, 2), dtype=torch.int64, device=self.device)
        self.lut = None
        self.lut_index = None
        self.bonds = None
        self.bond_index = None
        if bonds is not None:
            self._set_bonds(bonds, bond_index)
        self.set_temperature(temperature)

    def _set_bonds(self, b: np.ndarray, idx: Optional[np.ndarray]):
        """pack validated signs (check_bonds) into the kernels' bond words [K, 2, 4, rows, wpr]"""
        torch = self._torch
        K = b.shape[0]
        self.n_realisations = K
        with torch.cuda.device(self.device):
            signs = torch.from_numpy(np.ascontiguousarray(b.astype(np.int8))).to(self.device)
            self.bonds = torch.empty((K, 2, 4, self.rows, self.wpr), dtype=torch.int32, device=self.device)
            _lib.call("tsu_ising2d_pack_bonds", ptr(signs), ptr(self.bonds), K, self.rows, self.cols, int(self.wrap_rows),
                      int(self.wrap_cols), _lib.current_stream())
            self.bond_index = None if idx is None else torch.from_numpy(idx).to(self.device)

    # ------------------------------------------------------------------ parameters
    def set_temperature(self, temperature):
        torch = self._torch
        temps = np.atleast_1d(np.asarray(temperature, dtype=np.float64))
        if temps.size not in (1, self.n_replicas):
            raise ValueError("temperature must be a scalar or one value per replica")
        if np.any(temps <= 0):
            raise ValueError("Temperature must be positive")
        self.temperatures = temps.copy()
        uniq, inv = np.unique(temps, return_inverse=True)
        luts = np.stack([build_lut(self.coupling, self.field, float(t), self.bias_mode) for t in uniq])
        self.lut = torch.from_numpy(luts.view(np.int32)).to(self.device)
        if temps.size == 1:
            self.lut_index = None
        else:
            self.lut_index = torch.from_numpy(inv.astype(np.int32)).to(self.device)
        self._lut_temps = uniq
        self._jit = self._jit_prepare(luts[0]) if temps.size == 1 and self._jit_worthwhile() else 0

    # NVRTC needs 1-2 s per new temperature and the specialised kernel is ~17 % faster, so it is compiled
    # automatically only where it can pay back within seconds: the wide full-word kernel on >= 2^28 sites.
    JIT_MIN_SITES = 1 << 28

    def _jit_worthwhile(self, force: bool = False) -> bool:
        import os

        if os.environ.get("TSU_B200_NO_JIT") or self.bonds is not None:
            return False  # (the specialised kernel has no bonded form)
        wide = (self.cols // 2) // 32 >= 4 and self.rows >= 3   # at least one 4-word group of full words per row
        if not wide:
            return False  # only the wide full-word kernel has a specialised form (open rims run the generic kernel)
        if force or os.environ.get("TSU_B200_JIT"):
            return True
        return self.n_replicas * self.rows * self.cols >= self.JIT_MIN_SITES

    def specialise(self) -> bool:
        """compile (or fetch from the per-process cache) the half-sweep kernel specialised for the current temperature
        now, whatever the lattice size; returns whether the specialised kernel is in use.  Results are bit-identical."""
        if self.lut_index is None and self._jit_worthwhile(force=True):
            lut_host = self.lut[0].cpu().numpy().view(np.uint32)
            self._jit = self._jit_prepare(lut_host)
        return self._jit > 0

    def _jit_prepare(self, lut_host: np.ndarray) -> int:
        """table-specialised build of the fast kernel (0 = unavailable: the prebuilt kernels are used)"""
        import ctypes
        import os

        if os.environ.get("TSU_B200_NO_JIT"):
            return 0
        src_dir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc").encode()
        log = ctypes.create_string_buffer(4096)
        arr = (ctypes.c_uint32 * LUT_WORDS)(*[int(x) for x in lut_host])
        with self._torch.cuda.device(self.device):
            handle = int(self.lib.tsu_ising2d_jit_prepare(arr, src_dir, log, 4096))
        self._jit_log = log.value.decode(errors="replace")
        return max(handle, 0)

    def set_temperature_tables(self, temperatures, lut_index):
        """one threshold table per entry of `temperatures` (kept in that order) and an explicit
        replica -> table map (int32 tensor [n_replicas]); used by replica exchange, which permutes the map"""
        torch = self._torch
        temps = np.asarray(temperatures, dtype=np.float64)
        if np.any(temps <= 0):
            raise ValueError("Temperature must be positive")
        luts = np.stack([build_lut(self.coupling, self.field, float(t), self.bias_mode) for t in temps])
        self.lut = torch.from_numpy(luts.view(np.int32)).to(self.device)
        self._lut_temps = temps
        self._jit = 0
        self.set_lut_index(lut_index)

    def set_lut_index(self, lut_index):
        torch = self._torch
        idx = torch.as_tensor(lut_index, dtype=torch.int32, device=self.device).contiguous()
        if idx.numel() != self.n_replicas:
            raise ValueError("one table index per replica")
        self.lut_index = idx.clone()
        self.temperatures = self._lut_temps[self.lut_index.cpu().numpy()] if hasattr(self, "_lut_temps") else self.temperatures

    def chunk_view(self, start: int, count: int):
        """engine over replicas [start, start+count) sharing this engine's HBM state (no copy)"""
        cache = self.__dict__.setdefault("_views", {})
        key = (int(start), int(count))
        v = cache.get(key)
        if v is None:
            if start < 0 or count <= 0 or start + count > self.n_replicas:
                raise ValueError("chunk out of range")
            v = object.__new__(Ising2DEngine)
            # (a view gets a Swendsen-Wang workspace of its own: views may run concurrently on different streams)
            v.__dict__.update({k: val for k, val in self.__dict__.items() if k not in ("_views", "_cluster_work")})
            v.n_replicas = int(count)
            v.replica0 = self.replica0 + int(start)
            v.state = self.state[start:start + count]
            v._obs = self._obs[start:start + count]
            v.temperatures = self.temperatures if self.temperatures.size == 1 else self.temperatures[start:start + count]
            cache[key] = v
        v.lut = self.lut
        if hasattr(self, "_lut_temps"):
            v._lut_temps = self._lut_temps
        v.lut_index = None if self.lut_index is None else self.lut_index[start:start + count]
        v.bond_index = None if self.bond_index is None else self.bond_index[start:start + count]
        return v

    # ------------------------------------------------------------------ state i/o
    def init_random(self):
        """iid Bernoulli(1/2) spins from the Philox init stream (np.random.randint of gibbs.py:201)."""
        with self._torch.cuda.device(self.device):
            _lib.call(
                "tsu_ising2d_init_random", ptr(self.state), self.n_replicas, self.rows, self.cols, self.seed,
                self.replica0, self.row0, _lib.current_stream(),
            )
        return self

    def set_spins(self, spins):
        """spins: array [n_replicas, rows, cols] (or [rows, cols]) in {-1,+1} or {0,1}; > 0 means up."""
        torch = self._torch
        a = np.asarray(spins)
        if a.ndim == 2:
            a = a[None]
        if a.shape != (self.n_replicas, self.rows, self.cols):
            raise ValueError(f"expected spins of shape {(self.n_replicas, self.rows, self.cols)}, got {a.shape}")
        host = torch.from_numpy(np.ascontiguousarray((a > 0).astype(np.int8)))
        with torch.cuda.device(self.device):
            dev = host.to(self.device)
            _lib.call("tsu_ising2d_pack", ptr(dev), ptr(self.state), self.n_replicas, self.rows, self.cols,
                      _lib.current_stream())
        return self

    def spins_tensor(self, pm1: bool = True):
        """int8 tensor [n_replicas, rows, cols] on the device"""
        torch = self._torch
        with torch.cuda.device(self.device):
            out = torch.empty((self.n_replicas, self.rows, self.cols), dtype=torch.int8, device=self.device)
            _lib.call("tsu_ising2d_unpack", ptr(self.state), ptr(out), self.n_replicas, self.rows, self.cols,
                      1 if pm1 else 0, _lib.current_stream())
        return out

    def get_spins(self, pm1: bool = True) -> np.ndarray:
        return self.spins_tensor(pm1).cpu().numpy().astype(np.int64)

    # ------------------------------------------------------------------ updates
    def half_sweep(self, colour: int, halo_top=None, halo_bot=None, uniforms=None, rows=None):
        """resample every site of `colour`; halos are [n_replicas, wpr] int32 rows of the other colour.
        rows=(begin, end) restricts the update to those local rows (same bits for any split of the rows)."""
        if self.bonds is not None and (halo_top is not None or halo_bot is not None):
            raise ValueError("bonded engines have no halos")
        if uniforms is not None and rows is not None:
            raise ValueError("row ranges are not available in injected-uniform mode")
        lat = (ptr(self.state), self.n_replicas, self.rows, self.cols, int(self.wrap_rows and not self.is_slab),
                   int(self.wrap_cols), int(colour), ptr(self.lut), ptr(self.lut_index), ptr(self.bonds),
                   ptr(self.bond_index))
        with self._torch.cuda.device(self.device):
            if uniforms is not None:
                _lib.call("tsu_ising2d_half_sweep_injected", *lat, ptr(uniforms), self.row0, ptr(halo_top),
                          ptr(halo_bot), _lib.current_stream())
            else:
                begin, end = (0, self.rows) if rows is None else (int(rows[0]), int(rows[1]))
                _lib.call("tsu_ising2d_half_sweep", self._jit if self.lut_index is None else 0, *lat, self.seed,
                          self.sweep_index & 0xFFFFFFFF, self.replica0, self.row0, ptr(halo_top), ptr(halo_bot), begin,
                          end, _lib.current_stream())

    def sweep(self, n_sweeps: int = 1):
        """n full sweeps: black half-sweep then white half-sweep (one gibbs_update each)."""
        if self.is_slab:
            raise RuntimeError("row-slab engines are driven by ShardedIsing2D (halo exchange between half-sweeps)")
        with self._torch.cuda.device(self.device):
            _lib.call(
                "tsu_ising2d_sweeps", self._jit if self.lut_index is None else 0, ptr(self.state), self.n_replicas,
                self.rows, self.cols, int(self.wrap_rows), int(self.wrap_cols), ptr(self.lut), ptr(self.lut_index),
                ptr(self.bonds), ptr(self.bond_index), self.seed, self.sweep_index & 0xFFFFFFFF, int(n_sweeps),
                self.replica0, _lib.current_stream(),
            )
        self.sweep_index += int(n_sweeps)
        return self

    def sweep_injected(self, uniforms_u32):
        """parity mode: uniforms_u32 [n_sweeps, n_replicas, rows, cols] integers k (meaning k / 2^32)."""
        torch = self._torch
        u = np.asarray(uniforms_u32)
        if u.ndim == 3:
            u = u[:, None]
        dev = torch.from_numpy(np.ascontiguousarray(u.astype(np.uint32)).view(np.int32)).to(self.device)
        for t in range(dev.shape[0]):
            for colour in (0, 1):
                self.half_sweep(colour, uniforms=dev[t])
            self.sweep_index += 1
        return self

    # ------------------------------------------------------------------ annealing
    def anneal(self, temperatures, *, track_best: bool = True, best: Optional[AnnealResult] = None) -> AnnealResult:
        """Simulated annealing (tsu/gibbs.py:340-393) of every replica in one call, with no host sync.

        Step k sweeps once at temperatures[k].  The initial state and the state after every step are evaluated, and a
        replica whose energy is strictly below its best so far takes that energy and a copy of its state.  The result
        equals, bit for bit, the loop

            E = energy_tensor()                      # initial state: the first best
            for T in temperatures:
                set_temperature(T); sweep(1); E = energy_tensor()
                # replicas with E < best_energy take E and copy their state

        Afterwards sweep_index has advanced by len(temperatures) and the engine is at the scalar temperature
        temperatures[-1].  Lattices that sweep() runs in one launch anneal in one launch.

        track_best=True keeps a packed copy of every replica's state on the device, which doubles the state memory
        (34 GB more for 4096 replicas of 8192 x 8192).  best: the AnnealResult of an earlier anneal of this engine; its
        buffers are compared against and updated in place (and decide whether best states are kept), so an anneal
        split into calls equals one call.
        """
        Ts = np.asarray(temperatures, dtype=np.float64)
        if Ts.ndim != 1 or Ts.size == 0:
            raise ValueError("temperatures must be a non-empty 1-D schedule")
        return self._anneal(Ts, track_best, best)

    def simulated_annealing(self, T_initial: float = 10.0, T_final: float = 0.1, n_steps: int = 1000,
                            cooling_schedule: str = "exponential", *, track_best: bool = True,
                            best: Optional[AnnealResult] = None) -> AnnealResult:
        """anneal() along the schedule of GibbsSampler.simulated_annealing: the same float64 temperatures, from
        T_initial towards T_final, "exponential" or "linear".  n_steps = 0 evaluates the initial state only."""
        from .gibbs import annealing_temperatures

        if int(n_steps) < 0:
            raise ValueError("n_steps must be >= 0")
        return self._anneal(annealing_temperatures(T_initial, T_final, int(n_steps), cooling_schedule), track_best, best)

    def _anneal(self, Ts: np.ndarray, track_best: bool, best: Optional[AnnealResult]) -> AnnealResult:
        if self.is_slab:
            raise ValueError("annealing needs whole lattices; row-slab engines cannot anneal")
        if not np.all(np.isfinite(Ts)) or np.any(Ts <= 0):
            raise ValueError("temperatures must be positive and finite")
        torch = self._torch
        n = self.n_replicas
        if best is not None:
            be, bs = best.best_energy, best.best_state
            if (be is None) != (bs is None):
                raise ValueError("best needs both best_energy and best_state, or neither")
            if be is not None and not (be.dtype == torch.float64 and tuple(be.shape) == (n,) and be.is_contiguous()
                                       and be.device == self.device and bs.dtype == torch.int32
                                       and bs.shape == self.state.shape and bs.is_contiguous() and bs.device == self.device):
                raise ValueError(f"best buffers must be float64 [{n}] and int32 {tuple(self.state.shape)}, contiguous, "
                                 f"on {self.device}")
        with torch.cuda.device(self.device):
            energy = torch.empty(n, dtype=torch.float64, device=self.device)
            if best is not None:
                best_energy, best_state = best.best_energy, best.best_state
            elif track_best:
                best_energy = torch.full((n,), float("inf"), dtype=torch.float64, device=self.device)
                best_state = torch.empty_like(self.state)
            else:
                best_energy = best_state = None
            luts = self._schedule_tables(Ts) if Ts.size else None
            _lib.call(
                "tsu_ising2d_anneal", ptr(self.state), n, self.rows, self.cols, int(self.wrap_rows), int(self.wrap_cols),
                ptr(luts), int(Ts.size), ptr(self.bonds), ptr(self.bond_index), self.seed, self.sweep_index & 0xFFFFFFFF,
                self.replica0, self.coupling, self.field, self.n_bonds, self.n_sites, ptr(self._obs), ptr(energy),
                ptr(best_energy), ptr(best_state), _lib.current_stream(),
            )
        self.sweep_index += int(Ts.size)
        if Ts.size:
            self.set_temperature(float(Ts[-1]))  # (host work that overlaps the anneal on the device)
        if best is not None:
            best.energy = energy
            return best
        return AnnealResult(energy, best_energy, best_state, self.rows, self.cols)

    def _schedule_tables(self, Ts: np.ndarray):
        """int32 device tensor [len(Ts), 32]: the threshold table of every step; the last schedule's tables are kept,
        so that repeated anneals along one schedule build and upload nothing"""
        key = (self.coupling, self.field, self.bias_mode, Ts.tobytes())
        cached = self.__dict__.get("_anneal_tables")
        if cached is not None and cached[0] == key:
            return cached[1]
        uniq, inv = np.unique(Ts, return_inverse=True)
        luts = np.stack([build_lut(self.coupling, self.field, float(t), self.bias_mode) for t in uniq])[inv.reshape(-1)]
        tables = self._torch.from_numpy(np.ascontiguousarray(luts).view(np.int32)).to(self.device)
        self._anneal_tables = (key, tables)
        return tables

    # ------------------------------------------------------------------ population annealing
    def population_annealing(self, temperatures, *, sweeps_per_step: int = 10, n_populations: int = 1,
                             T_start: float = math.inf, previous: Optional[PopulationResult] = None) -> PopulationResult:
        """Population annealing (Hukushima-Iba, Machta) of every replica in one call, with no host sync.

        The replicas form n_populations equal contiguous populations of R_p replicas, each resampled on its own (one
        population per disorder realisation: bond_index must be constant within each).  The current state is taken
        to be an equilibrium sample at T_start (inf: beta = 0, e.g. the states of init_random()).  Step k resamples
        every population in proportion to exp(-dbeta_k E) with dbeta_k = 1/T_k - 1/T_{k-1} (T_{-1} = T_start), keeping
        R_p fixed (systematic resampling with integer weights; tsu_ising2d_population_anneal states the exact rule),
        then sweeps sweeps_per_step times at T_k.  The result gives ln Z ratios, free energies, mean energies and the
        family statistic rho_t; see PopulationResult.

        temperatures must be non-increasing and at most T_start.  previous: the result of an earlier run of this
        engine; its last temperature becomes T_start and its family buffer is continued in place, so a run split into
        calls equals one call.  Afterwards sweep_index has advanced by len(temperatures) * sweeps_per_step and the
        engine is at the scalar temperature temperatures[-1].

        The call allocates a second state buffer and a small workspace for its duration, so the state memory doubles
        while it runs.  Always the prebuilt kernels.
        """
        if self.is_slab:
            raise ValueError("population annealing needs whole lattices; row-slab engines cannot run it")
        if self.bias_mode != "physical":
            raise ValueError("population annealing needs bias_mode='physical': the sweeps of the reference bias do not "
                             "sample exp(-E/T), so the resampling weights would be wrong")
        Ts = np.asarray(temperatures, dtype=np.float64)
        if Ts.ndim != 1 or Ts.size == 0:
            raise ValueError("temperatures must be a non-empty 1-D schedule")
        if not np.all(np.isfinite(Ts)) or np.any(Ts <= 0):
            raise ValueError("temperatures must be positive and finite")
        if np.any(np.diff(Ts) > 0):
            raise ValueError("temperatures must be non-increasing")
        theta, P, n = int(sweeps_per_step), int(n_populations), self.n_replicas
        if theta < 1:
            raise ValueError("sweeps_per_step must be >= 1")
        if P < 1 or P > 65535 or n % P:
            raise ValueError(f"n_populations must divide n_replicas = {n} (and lie in [1, 65535])")
        r_pop = n // P
        if previous is not None:
            if (previous.n_populations != P or previous.r_pop != r_pop or tuple(previous.family.shape) != (n,)
                    or (previous.rows, previous.cols) != (self.rows, self.cols)):
                raise ValueError(f"previous must come from a run of {P} populations of {r_pop} replicas of "
                                 f"{self.rows} x {self.cols}")
            T_start = float(previous.temperatures[-1])
        T_start = float(T_start)
        if not T_start > 0 or Ts[0] > T_start:
            raise ValueError("T_start must be positive and at least temperatures[0]")
        if self.bond_index is not None:
            idx = np.asarray(self.bond_index.cpu()).reshape(P, r_pop)
            if np.any(idx != idx[:, :1]):
                raise ValueError("bond_index must be constant within each population (one realisation per population)")
        beta = 1.0 / Ts
        dbeta = np.diff(np.concatenate([[0.0 if math.isinf(T_start) else 1.0 / T_start], beta]))
        torch = self._torch
        dev = self.device
        with torch.cuda.device(dev):
            if previous is not None:
                family = previous.family
            else:
                family = torch.arange(self.replica0, self.replica0 + n, dtype=torch.int32, device=dev)
            scratch = torch.empty_like(self.state)
            family_scratch = torch.empty_like(family)
            work_bytes = int(self.lib.tsu_ising2d_population_work_bytes(n, P))
            work = torch.empty(work_bytes // 8, dtype=torch.int64, device=dev)
            weight_sum = torch.empty((Ts.size, P), dtype=torch.int64, device=dev)
            energy_ref = torch.empty((Ts.size, P), dtype=torch.float64, device=dev)
            count_sums = torch.empty((Ts.size + 1, P, 2), dtype=torch.int64, device=dev)
            energy = torch.empty(n, dtype=torch.float64, device=dev)
            d_dbeta = torch.from_numpy(dbeta).to(dev)
            luts = self._schedule_tables(Ts)
            _lib.call(
                "tsu_ising2d_population_anneal", ptr(self.state), ptr(scratch), n, self.rows, self.cols,
                int(self.wrap_rows), int(self.wrap_cols), ptr(luts), ptr(d_dbeta), int(Ts.size), theta, P,
                ptr(self.bonds), ptr(self.bond_index), self.seed, self.sweep_index & 0xFFFFFFFF, self.replica0,
                self.coupling, self.field, self.n_bonds, self.n_sites, ptr(family), ptr(family_scratch),
                ptr(weight_sum), ptr(energy_ref), ptr(count_sums), ptr(self._obs), ptr(energy), ptr(work), work_bytes,
                _lib.current_stream(),
            )
        self.sweep_index += int(Ts.size) * theta
        self.set_temperature(float(Ts[-1]))
        shift = 62 - (r_pop - 1).bit_length()
        return PopulationResult(energy, family, weight_sum, energy_ref, count_sums, Ts.copy(), T_start, dbeta, r_pop,
                                shift, self.rows, self.cols, self.coupling, self.field, self.n_bonds, self.n_sites)

    # ------------------------------------------------------------------ cluster updates
    def swendsen_wang(self, n_steps: int = 1):
        """n_steps Swendsen-Wang multi-cluster steps of every replica in one call, with no host sync.

        Each replica runs at its current temperature (per-replica temperatures and set_temperature_tables maps
        included, so replica exchange can alternate with it).  A step activates every satisfied bond
        (J sigma_ij s_i s_j > 0) with probability p = 1 - exp(-2|J|/T), labels the clusters of active bonds and flips
        each with probability 1/2; tsu_ising2d_swendsen_wang states the exact random stream.  Near T_c its
        autocorrelation time grows far more slowly with the lattice size than that of sweep().  Afterwards
        sweep_index has advanced by n_steps.

        Field 0, bias_mode "physical" and whole lattices only.  The first call allocates a workspace of about 4.4
        bytes per site for min(n_replicas, CLUSTER_WORK_BUDGET // bytes per replica) replicas, kept with the engine;
        more replicas run in chunks of that many, with the same bits.
        """
        if self.field != 0:
            raise ValueError("Swendsen-Wang updates need field = 0 (a field needs a ghost spin or a cluster heat bath)")
        if self.bias_mode != "physical":
            raise ValueError("Swendsen-Wang updates need bias_mode='physical': the reference bias does not sample "
                             "exp(-E/T)")
        if self.is_slab:
            raise ValueError("Swendsen-Wang updates need whole lattices; row-slab engines cannot run them")
        if isinstance(n_steps, bool) or not isinstance(n_steps, (int, np.integer)) or n_steps < 0:
            raise ValueError("n_steps must be a non-negative integer")
        if self.rows * self.cols >= 1 << 31:
            raise ValueError("Swendsen-Wang labels are int32: rows * cols must stay below 2^31")
        n_steps = int(n_steps)
        if n_steps == 0:
            return self
        torch = self._torch
        with torch.cuda.device(self.device):
            work = self._cluster_workspace(self.n_replicas)
            key = (self.coupling, np.asarray(self._lut_temps).tobytes())
            cached = self.__dict__.get("_cluster_tables")
            if cached is None or cached[0] != key:
                t = np.array([cluster_threshold(self.coupling, float(T)) for T in self._lut_temps], dtype=np.int64)
                cached = (key, torch.from_numpy(t).to(self.device))
                self._cluster_tables = cached
            _lib.call(
                "tsu_ising2d_swendsen_wang", ptr(self.state), self.n_replicas, self.rows, self.cols,
                int(self.wrap_rows), int(self.wrap_cols), ptr(cached[1]), ptr(self.lut_index),
                -1 if self.coupling < 0 else 1, ptr(self.bonds), ptr(self.bond_index), self.seed,
                self.sweep_index & 0xFFFFFFFF, n_steps, self.replica0, ptr(work), work.numel() * 8,
                _lib.current_stream(),
            )
        self.sweep_index += n_steps
        return self

    def _cluster_workspace(self, n_shares: int):
        """the cluster workspace shared by swendsen_wang and houdayer: room for min(n_shares, CLUSTER_WORK_BUDGET //
        bytes per share) replicas or pairs (at least one); reallocated only when a call needs more shares"""
        per_rep = int(self.lib.tsu_ising2d_cluster_work_bytes(1, self.rows, self.cols))
        need = min(n_shares, max(1, CLUSTER_WORK_BUDGET // per_rep)) * per_rep
        work = self.__dict__.get("_cluster_work")
        if work is None or work.numel() * 8 < need:
            work = self._torch.empty(need // 8, dtype=self._torch.int64, device=self.device)
            self._cluster_work = work
        return work

    def houdayer(self, pairs, n_steps: int = 1):
        """n_steps Houdayer cluster moves of every replica pair in `pairs` in one call.

        `pairs` is an integer array [n_pairs, 2] of disjoint pairs (a, b) of this engine's replicas; the two replicas
        of a pair must share the temperature and the bond realisation.  A step takes the sites where the two differ,
        labels the clusters that bonds between such sites form and flips each cluster in both replicas with
        probability 1/2 (tsu_ising2d_houdayer states the exact random stream).  E_a + E_b and q_ab are unchanged and
        the product of the two Boltzmann distributions is kept, for any bonds and any field; each replica's own
        energy changes, which at low temperature moves a 2-D spin glass between valleys far faster than sweep().
        The move keeps the set of differing sites, so it is not ergodic alone: alternate it with sweep().  Afterwards
        sweep_index has advanced by n_steps.

        bias_mode "physical" and whole lattices only; a field is allowed.  Shares the Swendsen-Wang workspace (one
        replica's share per pair, CLUSTER_WORK_BUDGET at most); more pairs run in chunks, with the same bits.  Every
        argument is checked on the host before any device work (with bonds, bond_index is read back for that);
        LatticeTempering(houdayer_interval=k) runs the move with pairs built on the device and no host sync.
        """
        self._houdayer_supported()
        if isinstance(n_steps, bool) or not isinstance(n_steps, (int, np.integer)) or n_steps < 0:
            raise ValueError("n_steps must be a non-negative integer")
        pr = np.asarray(pairs)
        if pr.ndim != 2 or pr.shape[1] != 2 or pr.shape[0] < 1 or not np.issubdtype(pr.dtype, np.integer):
            raise ValueError("pairs must be integers of shape [n_pairs, 2]")
        if np.any(pr < 0) or np.any(pr >= self.n_replicas):
            raise ValueError(f"pair indices must lie in [0, {self.n_replicas})")
        if np.any(pr[:, 0] == pr[:, 1]):
            raise ValueError("a pair needs two different replicas")
        if np.unique(pr).size != pr.size:
            raise ValueError("pairs must be disjoint: a replica appears twice")
        temps = np.broadcast_to(np.asarray(self.temperatures, dtype=np.float64), (self.n_replicas,))
        if np.any(temps[pr[:, 0]] != temps[pr[:, 1]]):
            raise ValueError("the replicas of a pair need the same temperature")
        if self.bond_index is not None:
            bi = np.asarray(self.bond_index.cpu())
            if np.any(bi[pr[:, 0]] != bi[pr[:, 1]]):
                raise ValueError("the replicas of a pair need the same bond realisation (bond_index)")
        if n_steps == 0:
            return self
        with self._torch.cuda.device(self.device):
            dev = self._torch.from_numpy(np.ascontiguousarray(pr.astype(np.int32))).to(self.device)
        return self._houdayer(dev, int(pr.shape[0]), int(n_steps))

    def _houdayer_supported(self):
        """the engine rules of houdayer(), also checked once by LatticeTempering(houdayer_interval > 0)"""
        if self.bias_mode != "physical":
            raise ValueError("Houdayer moves need bias_mode='physical': the reference bias does not sample exp(-E/T)")
        if self.is_slab:
            raise ValueError("Houdayer moves need whole lattices; row-slab engines cannot run them")
        if self.rows * self.cols >= 1 << 31:
            raise ValueError("Houdayer cluster labels are int32: rows * cols must stay below 2^31")

    def _houdayer(self, pairs, n_pairs: int, n_steps: int):
        """houdayer() on validated device pairs (int32 [n_pairs, 2]); no check, no host sync"""
        with self._torch.cuda.device(self.device):
            work = self._cluster_workspace(n_pairs)
            _lib.call(
                "tsu_ising2d_houdayer", ptr(self.state), self.n_replicas, self.rows, self.cols, int(self.wrap_rows),
                int(self.wrap_cols), ptr(pairs), n_pairs, self.seed, self.sweep_index & 0xFFFFFFFF, n_steps,
                self.replica0, ptr(work), work.numel() * 8, _lib.current_stream(),
            )
        self.sweep_index += n_steps
        return self

    # ------------------------------------------------------------------ observables
    def observables_tensor(self, next_rows=None):
        """int64 tensor [n_replicas, 2]: (# up spins, # anti-aligned right+down bonds) of the local rows;
        with bonds the second column counts unsatisfied bonds (sign * s_i * s_j = -1)"""
        if self.bonds is not None and next_rows is not None:
            raise ValueError("bonded engines have no halos")
        with self._torch.cuda.device(self.device):
            _lib.call(
                "tsu_ising2d_observables", ptr(self.state), self.n_replicas, self.rows, self.cols,
                int(self.wrap_rows and not self.is_slab), int(self.wrap_cols), ptr(self.bonds), ptr(self.bond_index),
                self.row0, ptr(next_rows), ptr(self._obs), _lib.current_stream(),
            )
        return self._obs

    @property
    def n_sites(self) -> int:
        return self.rows * self.cols

    @property
    def n_bonds(self) -> int:
        return lattice_bond_count(self.rows, self.cols, self.wrap_rows, self.wrap_cols)

    def overlap_tensor(self, pairs):
        """float64 device tensor [n_pairs]: spin overlap q_ab = (1/N) sum_i s_i^a s_i^b = 1 - 2 diff_ab / N of every
        replica pair (a, b) in `pairs` (shape [n_pairs, 2], indices of this engine's replicas)"""
        torch = self._torch
        pr = np.asarray(pairs)
        if pr.ndim != 2 or pr.shape[1] != 2 or pr.shape[0] < 1 or not np.issubdtype(pr.dtype, np.integer):
            raise ValueError("pairs must be integers of shape [n_pairs, 2]")
        if np.any(pr < 0) or np.any(pr >= self.n_replicas):
            raise ValueError(f"pair indices must lie in [0, {self.n_replicas})")
        with torch.cuda.device(self.device):
            dev = torch.from_numpy(np.ascontiguousarray(pr.astype(np.int32))).to(self.device)
            diff = torch.empty(pr.shape[0], dtype=torch.int64, device=self.device)
            _lib.call("tsu_ising2d_overlap", ptr(self.state), self.n_replicas, self.rows, self.cols, ptr(dev),
                      int(pr.shape[0]), ptr(diff), _lib.current_stream())
            return 1.0 - 2.0 * diff.to(torch.float64) / self.n_sites

    def overlap(self, pairs) -> np.ndarray:
        """spin overlap q_ab of every replica pair (host numpy, see overlap_tensor)"""
        return self.overlap_tensor(pairs).cpu().numpy()

    def magnetization(self) -> np.ndarray:
        """signed magnetisation per spin of every replica (tsu/models/ising.py:183-193 on the current state)"""
        obs = self.observables_tensor().cpu().numpy()
        return (2.0 * obs[:, 0] - self.n_sites) / self.n_sites

    def energy(self) -> np.ndarray:
        """E = -J sum_<ij> s_i s_j - h sum_i s_i of every replica (tsu/models/ising.py:98-117)"""
        obs = self.observables_tensor().cpu().numpy().astype(np.float64)
        return -self.coupling * (self.n_bonds - 2.0 * obs[:, 1]) - self.field * (2.0 * obs[:, 0] - self.n_sites)

    def energy_tensor(self):
        """float64 device tensor of energies (no host sync) - feeds the replica-exchange kernel"""
        torch = self._torch
        obs = self.observables_tensor()
        with torch.cuda.device(self.device):
            e = torch.empty(self.n_replicas, dtype=torch.float64, device=self.device)
            _lib.call(
                "tsu_ising2d_energy_from_observables", ptr(obs), self.n_replicas, self.coupling, self.field,
                self.n_bonds, self.n_sites, ptr(e), _lib.current_stream(),
            )
        return e
