"""
Host side of the chromatic sparse-coupling Gibbs sampler (csrc/sparse_gibbs.cu, tsu_sparse_gibbs_run).

The reference stores every model as a dense N x N matrix and spends one length-N dot product per spin visit
(tsu/gibbs.py:79-100), also for a chain whose rows hold two numbers (tsu/models/ising.py:265-304).  Here the
couplings go to the device in CSR form and a sweep costs the number of non-zeros.  The visiting order of a sweep is
"colour class after colour class" (greedy colouring, no two coupled sites share a colour): a valid sequential sweep of
the reference - the one it performs with update_order="random" when the permutation is that order.
"""

from typing import Optional, Tuple

import numpy as np

from . import _lib
from ._lib import ptr

HOUDAYER_WORK_BUDGET = 1 << 30  # bytes of Houdayer labels a SparseProblem keeps (N > 32768: 4 N bytes per pair)


def is_symmetric_csr(rowptr: np.ndarray, col: np.ndarray, val: np.ndarray, N: int) -> bool:
    """the CSR matrix (columns ascending within a row) equals its transpose in structure and values"""
    from scipy.sparse import csr_matrix

    A = csr_matrix((val, col, rowptr), shape=(N, N))
    T = A.T.tocsr()
    T.sort_indices()
    return (np.array_equal(A.indptr, T.indptr) and np.array_equal(A.indices, T.indices)
            and np.array_equal(A.data, T.data))


def to_csr(coupling) -> Tuple[np.ndarray, np.ndarray, np.ndarray, int]:
    """(rowptr int32[N+1], col int32[nnz], val float64[nnz], N) of a square coupling matrix given as a dense array,
    a scipy.sparse matrix, or an (indptr, indices, data, N) tuple; columns ascending within a row"""
    if isinstance(coupling, tuple) and len(coupling) == 4:
        rowptr, col, val, N = coupling
        return (np.ascontiguousarray(rowptr, dtype=np.int32), np.ascontiguousarray(col, dtype=np.int32),
                np.ascontiguousarray(val, dtype=np.float64), int(N))
    if hasattr(coupling, "tocsr"):
        m = coupling.tocsr().astype(np.float64)
        if m.shape[0] != m.shape[1]:
            raise ValueError("Coupling matrix must be square")
        m.sort_indices()
        m.eliminate_zeros()
        return m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data.astype(np.float64), m.shape[0]
    J = np.asarray(coupling, dtype=np.float64)
    if J.ndim != 2 or J.shape[0] != J.shape[1]:
        raise ValueError("Coupling matrix must be square")
    rows, cols = np.nonzero(J)  # row-major: columns ascending within a row
    rowptr = np.zeros(J.shape[0] + 1, dtype=np.int64)
    np.add.at(rowptr, rows + 1, 1)
    return np.cumsum(rowptr).astype(np.int32), cols.astype(np.int32), J[rows, cols], J.shape[0]


def greedy_colouring(rowptr: np.ndarray, col: np.ndarray, N: int) -> np.ndarray:
    """colour of every site: sites in index order take the smallest colour none of their already coloured neighbours
    (in either direction of a possibly asymmetric matrix) has.  A chain gets colours i & 1."""
    # neighbours in both directions: i needs a colour different from every j with J_ij != 0 or J_ji != 0
    src = np.repeat(np.arange(N), np.diff(rowptr))
    a = np.concatenate([src, col])
    b = np.concatenate([col, src])
    keep = a != b
    a, b = a[keep], b[keep]
    order = np.argsort(a, kind="stable")
    a, b = a[order], b[order]
    ptr_ = np.searchsorted(a, np.arange(N + 1))
    colour = np.full(N, -1, dtype=np.int32)
    for i in range(N):
        nb = colour[b[ptr_[i]:ptr_[i + 1]]]
        used = set(int(c) for c in nb if c >= 0)
        c = 0
        while c in used:
            c += 1
        colour[i] = c
    return colour


def colour_classes(colour: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """(colour_ptr int32[n_colours + 1], colour_sites int32[N]): sites grouped by colour, ascending index within a colour
    - the visiting order of a sweep"""
    n_col = int(colour.max()) + 1 if colour.size else 0
    sites = np.argsort(colour, kind="stable").astype(np.int32)
    counts = np.bincount(colour, minlength=n_col)
    return np.concatenate([[0], np.cumsum(counts)]).astype(np.int32), sites


class SparseProblem:
    """CSR couplings, bias and colour classes resident on the device"""

    def __init__(self, coupling, bias, device):
        torch = _lib.require_cuda()
        rowptr, col, val, N = to_csr(coupling)
        self.N, self.nnz = N, int(val.size)
        self.device = device
        self.csr = (rowptr, col, val)  # host copy of the couplings (energy of a returned state)
        colour = greedy_colouring(rowptr, col, N)
        cptr, sites = colour_classes(colour)
        self.n_colours = len(cptr) - 1
        self.order = sites.copy()  # host copy of the visiting order (parity tests)
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)
        self.rowptr, self.col, self.val = t(rowptr), t(col if col.size else np.zeros(1, np.int32)), t(val if val.size else np.zeros(1))
        self.cptr, self.sites = t(cptr), t(sites)
        self.bias = self.host_bias = None
        self._houdayer_work = None  # Houdayer label workspace (N > 32768), allocated by the first call that needs it
        if bias is not None:
            b = np.asarray(bias, dtype=np.float64)
            if b.shape != (N,):
                raise ValueError("bias must have one entry per bit")
            self.bias, self.host_bias = t(b), b

    def run(self, state, *, T: float, seed: int, sweep0: int, chain0: int, n_burnin: int, n_samples: int,
            sweeps_per_sample: int, T_chain=None, T_sweep=None, uniforms=None, want_samples=False, want_energy=False,
            track_best=False):
        """one launch of tsu_sparse_gibbs_run on `state` (uint8 tensor [n_chains, N], updated in place); T_sweep is
        the host float64 temperature of every sweep"""
        torch = _lib.require_cuda()
        n_chains, N = state.shape
        dev = self.device
        if T_sweep is not None:
            T_sweep = torch.from_numpy(T_sweep).to(dev)
        samples = torch.empty((n_samples, n_chains, N), dtype=torch.uint8, device=dev) if want_samples else None
        energy = torch.empty(n_chains, dtype=torch.float64, device=dev) if (want_energy or track_best) else None
        best_state = torch.empty((n_chains, N), dtype=torch.uint8, device=dev) if track_best else None
        best_energy = torch.empty(n_chains, dtype=torch.float64, device=dev) if track_best else None
        with torch.cuda.device(dev):
            _lib.call("tsu_sparse_gibbs_run", ptr(self.rowptr), ptr(self.col), ptr(self.val), ptr(self.bias),
                      ptr(self.cptr), ptr(self.sites), self.n_colours, ptr(state), int(n_chains), int(N), float(T),
                      ptr(T_chain), ptr(T_sweep), int(n_burnin), int(n_samples), int(sweeps_per_sample), ptr(uniforms),
                      ptr(samples), ptr(energy), int(track_best), ptr(best_state), ptr(best_energy), int(seed),
                      sweep0 & 0xFFFFFFFF, chain0 & 0xFFFFFFFF, _lib.current_stream())
        return samples, energy, best_state, best_energy

    def houdayer(self, state, pairs, n_pairs: int, *, seed: int, step0: int, n_steps: int, chain0: int, energy=None):
        """one launch of tsu_sparse_houdayer on `state` (uint8 tensor [n_chains, N], updated in place): n_steps
        Houdayer moves, step indices step0 .. step0 + n_steps - 1, of the disjoint chain pairs `pairs` (int32 device
        tensor [n_pairs, 2]); with `energy` (float64 [n_chains]) every processed chain's energy is written there.  The
        label workspace of N > 32768 is owned here and grows to what a call needs, at most HOUDAYER_WORK_BUDGET (then
        the pairs run in chunks, with the same bits)."""
        torch = _lib.require_cuda()
        lib = _lib.load()
        n_pairs = int(n_pairs)
        per_pair = int(lib.tsu_sparse_houdayer_work_bytes(1, self.N))
        need = min(n_pairs, max(1, HOUDAYER_WORK_BUDGET // per_pair)) * per_pair if per_pair else 0
        work = self._houdayer_work
        if need and (work is None or work.numel() * 8 < need):
            work = torch.empty(need // 8, dtype=torch.int64, device=self.device)
            self._houdayer_work = work
        with torch.cuda.device(self.device):
            _lib.call("tsu_sparse_houdayer", ptr(self.rowptr), ptr(self.col), ptr(self.val), ptr(self.bias), ptr(state),
                      int(state.shape[0]), self.N, ptr(pairs), n_pairs, int(seed), step0 & 0xFFFFFFFF, int(n_steps),
                      chain0 & 0xFFFFFFFF, ptr(energy), ptr(work if need else None), work.numel() * 8 if need else 0,
                      _lib.current_stream())

    def energy(self, state: np.ndarray) -> float:
        """E = -1/2 s^T J s - b^T s of a host state under the float64 CSR couplings and bias"""
        rowptr, col, val = self.csr
        sb = state.astype(np.float64)
        row = np.repeat(np.arange(len(sb)), np.diff(rowptr))
        e = -0.5 * float(np.sum(val * sb[row] * sb[col]))
        if self.host_bias is not None:
            e -= float(np.dot(self.host_bias, sb))
        return e


def is_sparse_enough(coupling, max_density: float = 0.05, min_n: int = 64) -> bool:
    """heuristic of IsingModel.sample: large and mostly empty matrices take the chromatic CSR kernel"""
    if hasattr(coupling, "tocsr"):
        return True
    J = np.asarray(coupling)
    n = J.shape[0]
    return n >= min_n and np.count_nonzero(J) <= max_density * n * n
