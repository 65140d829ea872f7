"""
Multi-GPU drivers (one process per GPU, torch.distributed; NCCL over NVLink on the box, gloo in CPU tests).

  * SlabShardedIsing2D - ONE large lattice (or a batch of them) split into contiguous row slabs.  Per
    half-sweep every rank needs the opposite-colour row just above and just below its slab: the rows that
    were updated in the previous half-sweep are sent to the ring neighbours (wpr words per replica and
    side: 8 KiB for 131072 columns).  The two boundary rows are updated first on a side stream and sent while
    the interior rows are updated on the main stream.  Philox counters use global row indices, so the bits
    are identical to the single-GPU run for any number of ranks.
  * replica_shard - independent replicas / chains / ladders: contiguous index ranges, no collective.
  * LatticeTempering - K temperature ladders x R temperatures of one lattice size with replica exchange
    (tsu/gibbs.py:238-338 semantics on the lattice kernels).  Lattices never move: the swap permutes the
    replica -> temperature-table index.  With a process group the replicas are sharded across ranks, the
    per-replica energies are all-gathered (K*R float64) and every rank evaluates the same deterministic
    swap pass.

The drivers only talk to an "engine" object (Ising2DEngine on GPUs); the CPU tests plug in an
oracle-backed stand-in to exercise the partitioning and exchange logic under gloo with world_size 2.
"""

from typing import Optional, Sequence

import numpy as np


def replica_shard(n_total: int, rank: int, world: int):
    """contiguous [start, stop) of `n_total` independent units owned by `rank`"""
    base, extra = divmod(n_total, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def _dist():
    import torch.distributed as dist

    return dist


class SlabShardedIsing2D:
    """row-slab decomposition of a rows x cols lattice over the ranks of `group`.

    engine_factory(local_rows, row0) must return an engine exposing
        .state                      tensor [n_replicas, 2, local_rows, wpr] (int32 words)
        .half_sweep(colour, halo_top=..., halo_bot=..., rows=(begin, end))   halos: [n_replicas, wpr] or None
        .sweep_index                incremented by the driver
        .observables_tensor(next_rows=...) -> int64 [n_replicas, 2]

    Overlap (default on CUDA engines with at least 4 local rows): a half-sweep of colour c is issued as
      side stream : rows 0 and L-1 (they need the halos of colour 1-c), then the exchange of the new rows 0 / L-1
      main stream : rows 1 .. L-2 (no halo needed)
    so the 2 x wpr-word messages (8 KiB per side at 131072 columns) and the two one-row launches hide behind the
    interior update.  Dependencies between consecutive half-sweeps are two events: the interior waits for the
    previous boundary update (it reads and overwrites the rows next to it), the boundary update waits for the
    previous interior update.  Same launches, same Philox coordinates, same bits as the serial order.
    """

    def __init__(self, rows: int, cols: int, engine_factory, periodic: bool = True, group=None, overlap=None,
                 transport: str = "auto"):
        dist = _dist()
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        if rows % self.world:
            raise ValueError("rows must be divisible by the number of ranks")
        self.rows, self.cols, self.periodic = rows, cols, periodic
        self.local_rows = rows // self.world
        self.row0 = self.rank * self.local_rows
        self.engine = engine_factory(self.local_rows, self.row0)
        import torch

        st = self.engine.state
        self.n_replicas, self.wpr = st.shape[0], st.shape[3]
        # halo[colour][0 = above row0, 1 = below the last local row]
        self.halo = torch.zeros((2, 2, self.n_replicas, self.wpr), dtype=st.dtype, device=st.device)
        self._next_rows = torch.zeros((self.n_replicas, 2, self.wpr), dtype=st.dtype, device=st.device)
        self.up = (self.rank - 1) % self.world     # owns the rows above mine
        self.down = (self.rank + 1) % self.world   # owns the rows below mine
        self.has_up = self.periodic or self.rank > 0
        self.has_down = self.periodic or self.rank < self.world - 1
        self.overlap = (self.local_rows >= 4) if overlap is None else bool(overlap)
        self._side = None
        if self.overlap and st.is_cuda:
            self._side = torch.cuda.Stream(device=st.device, priority=-1)
        # transport of the halo rows between ranks: "nccl" = send/recv of torch.distributed on the side stream;
        # "p2p" = the ranks map each other's halo buffers (CUDA IPC over NVLink) and the whole pipeline of a sweep()
        # call is issued by ONE C-ABI call (tsu_ising2d_slab_sweeps_p2p): no collective library and no Python in the
        # per-half-sweep path.  "auto" = p2p on CUDA engines with more than one rank, falling back to nccl if the
        # buffers cannot be mapped.
        if transport not in ("auto", "nccl", "p2p"):
            raise ValueError("transport must be 'auto', 'nccl' or 'p2p'")
        self._p2p = None
        if transport != "nccl" and self.overlap and st.is_cuda and self.world > 1 and hasattr(self.engine, "lib"):
            try:
                self._p2p = _PeerHalos(self)
            except Exception:
                if transport == "p2p":
                    raise
                self._p2p = None
        elif transport == "p2p":
            raise ValueError("transport='p2p' needs a CUDA engine, more than one rank and at least 4 local rows")

    @property
    def halo_top(self):  # halos of the colour exchanged last (kept for callers of exchange())
        return self.halo[self._last_colour, 0]

    @property
    def halo_bot(self):
        return self.halo[self._last_colour, 1]

    _last_colour = 0

    # -- halo exchange ---------------------------------------------------------------------------
    def exchange(self, colour: int):
        """make rows (row0-1) and (row0+local_rows) of `colour` available as halo[colour][0] / halo[colour][1]"""
        st = self.engine.state
        self._last_colour = colour
        top, bot = self.halo[colour, 0], self.halo[colour, 1]
        if self.world == 1:
            if self.periodic:
                top.copy_(st[:, colour, -1, :])
                bot.copy_(st[:, colour, 0, :])
            return
        dist = _dist()
        first = st[:, colour, 0, :].contiguous()
        last = st[:, colour, -1, :].contiguous()
        ops = []
        if self.world == 2 and self.periodic:
            # both neighbours are the same peer: messages to one peer match in posting order, so both ranks post
            # (first, last) and receive (the peer's first row = below me, the peer's last row = above me)
            peer = self._peer(self.up)
            ops = [dist.P2POp(dist.isend, first, peer, self.group), dist.P2POp(dist.isend, last, peer, self.group),
                   dist.P2POp(dist.irecv, bot, peer, self.group), dist.P2POp(dist.irecv, top, peer, self.group)]
        else:
            if self.has_up:
                ops.append(dist.P2POp(dist.isend, first, self._peer(self.up), self.group))
                ops.append(dist.P2POp(dist.irecv, top, self._peer(self.up), self.group))
            if self.has_down:
                ops.append(dist.P2POp(dist.isend, last, self._peer(self.down), self.group))
                ops.append(dist.P2POp(dist.irecv, bot, self._peer(self.down), self.group))
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()  # CUDA: the current stream waits for the transfer; gloo: the host does

    def _peer(self, group_rank: int) -> int:
        dist = _dist()
        if self.group is None:
            return group_rank
        return dist.get_global_rank(self.group, group_rank)

    def _halos(self, colour: int):
        """halo rows a half-sweep of `colour` reads (the other colour)"""
        opp = 1 - colour
        return (self.halo[opp, 0] if self.has_up else None), (self.halo[opp, 1] if self.has_down else None)

    # -- updates -----------------------------------------------------------------------------------
    def half_sweep(self, colour: int):
        """serial form: exchange, then one launch for all local rows"""
        self.exchange(1 - colour)
        top, bot = self._halos(colour)
        self.engine.half_sweep(colour, halo_top=top, halo_bot=bot)

    def sweep(self, n_sweeps: int = 1):
        if self._p2p is not None:
            self._p2p.sweeps(int(n_sweeps))
            return self
        if self.world == 1 and getattr(self.engine, "is_slab", True) is False and hasattr(self.engine, "sweep"):
            self.engine.sweep(int(n_sweeps))  # the one slab is the whole lattice: no halos, the engine's own sweeps
            return self
        if not self.overlap:
            for _ in range(n_sweeps):
                self.half_sweep(0)
                self.half_sweep(1)
                self.engine.sweep_index += 1
            return self
        import contextlib

        import torch

        cuda = self._side is not None
        main = torch.cuda.current_stream(self.engine.state.device) if cuda else None
        on_side = (lambda: torch.cuda.stream(self._side)) if cuda else contextlib.nullcontext
        L = self.local_rows
        ev_interior = ev_boundary = None
        with on_side():
            if cuda:
                self._side.wait_stream(main)
            self.exchange(1)  # colour 0 goes first and reads colour 1
        for _ in range(n_sweeps):
            for colour in (0, 1):
                top, bot = self._halos(colour)
                # interior on the main stream
                if cuda and ev_boundary is not None:
                    main.wait_event(ev_boundary)
                self.engine.half_sweep(colour, rows=(1, L - 1))
                ev_prev_interior = ev_interior
                if cuda:
                    ev_interior = torch.cuda.Event()
                    ev_interior.record(main)
                # boundary rows and the exchange of what they produce on the side stream
                with on_side():
                    if cuda and ev_prev_interior is not None:
                        self._side.wait_event(ev_prev_interior)
                    self.engine.half_sweep(colour, halo_top=top, halo_bot=bot, rows=(0, 1))
                    self.engine.half_sweep(colour, halo_top=top, halo_bot=bot, rows=(L - 1, L))
                    if cuda:
                        ev_boundary = torch.cuda.Event()
                        ev_boundary.record(self._side)
                    self.exchange(colour)
            self.engine.sweep_index += 1
        if cuda:
            main.wait_stream(self._side)
        return self

    def transport(self) -> str:
        return "p2p" if self._p2p is not None else ("nccl" if self.world > 1 else "local")

    def close(self):
        """release the peer-mapped halo buffers (collective: every rank calls it)"""
        if self._p2p is not None:
            if self._p2p.status():
                raise RuntimeError("a neighbour's halo rows did not arrive in time during a slab sweep")
            self._p2p.close()
            self._p2p = None

    # -- observables -------------------------------------------------------------------------------
    def observables(self):
        """global (# up spins, # anti-aligned bonds) per replica, summed over the slabs"""
        nxt = None
        if self.periodic or self.world > 1:
            for colour in (0, 1):          # collective: every rank takes part even if it has no lower neighbour
                self.exchange(colour)
                self._next_rows[:, colour, :] = self.halo[colour, 1]
            if self.has_down:
                nxt = self._next_rows
        obs = self.engine.observables_tensor(next_rows=nxt).clone()
        if self.world > 1:
            _dist().all_reduce(obs, group=self.group)
        return obs


class _PeerHalos:
    """halo buffers of a row slab that the ring neighbours map through CUDA IPC, and the one-call sweep pipeline on
    top of them (include/tsu_b200.h: tsu_ising2d_slab_sweeps_p2p)"""

    FLAG_WORDS = 16

    def __init__(self, drv: "SlabShardedIsing2D"):
        """collective over drv.group.  Every phase that can fail locally is followed by an agreement (all-reduce of a
        success flag), so that either every rank ends up with mapped neighbours or every rank raises - no rank is left
        waiting in a collective for one that gave up."""
        import ctypes

        import torch

        from . import _lib

        dist = _dist()
        self.drv = drv
        eng = drv.engine
        self.lib = _lib.load()
        self.device = eng.state.device
        self.halo_words = 4 * drv.n_replicas * drv.wpr
        self.base, self._opened, self.up, self.down = None, {}, None, None
        self.msgs = [0, 0]
        nbytes = 4 * (self.halo_words + self.FLAG_WORDS)

        def agree(ok: bool, what: str):
            flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=self.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=drv.group)
            if int(flag.item()) == 0:
                self._release()
                raise RuntimeError(f"peer-mapped halo buffers are not available on every rank ({what})")

        handle = ctypes.create_string_buffer(64)
        ok = True
        try:
            with torch.cuda.device(self.device):
                base = ctypes.c_void_p()
                _lib.call("tsu_peer_alloc", ctypes.byref(base), nbytes)
                self.base = base.value
                _lib.call("tsu_peer_get_handle", ctypes.c_void_p(self.base), handle)
        except Exception:
            ok = False
        agree(ok, "allocation / IPC export")
        mine = torch.tensor(list(handle.raw), dtype=torch.uint8, device=self.device)
        everyone = [torch.empty_like(mine) for _ in range(drv.world)]
        dist.all_gather(everyone, mine, group=drv.group)

        def open_rank(r):
            if r not in self._opened:
                raw = bytes(everyone[r].cpu().tolist())
                p = ctypes.c_void_p()
                with torch.cuda.device(self.device):
                    _lib.call("tsu_peer_open_handle", ctypes.create_string_buffer(raw, 64), ctypes.byref(p))
                self._opened[r] = p.value
            return self._opened[r]

        try:
            self.up = open_rank(drv.up) if drv.has_up else None
            self.down = open_rank(drv.down) if drv.has_down else None
        except Exception:
            ok = False
        agree(ok, "IPC import of a neighbour's buffer")  # doubles as the barrier before the first rows are written

    def _release(self):
        """local part of close(): unmap the neighbours, free the own buffer"""
        import ctypes

        import torch

        from . import _lib

        with torch.cuda.device(self.device):
            for p in self._opened.values():
                try:
                    _lib.call("tsu_peer_close_handle", ctypes.c_void_p(p))
                except Exception:
                    pass
            self._opened = {}
            if self.base is not None:
                try:
                    _lib.call("tsu_peer_free", ctypes.c_void_p(self.base))
                except Exception:
                    pass
                self.base = None

    def _flags(self, base):
        return None if base is None else base + 4 * self.halo_words

    def sweeps(self, n_sweeps: int):
        import ctypes

        import torch

        from . import _lib

        drv, eng = self.drv, self.drv.engine
        vp = lambda x: None if x is None else ctypes.c_void_p(x)
        with torch.cuda.device(self.device):
            main = torch.cuda.current_stream(self.device)
            _lib.call(
                "tsu_ising2d_slab_sweeps_p2p", int(getattr(eng, "_jit", 0)) if eng.lut_index is None else 0,
                _lib.ptr(eng.state), eng.n_replicas, eng.rows, eng.cols, int(eng.wrap_cols), _lib.ptr(eng.lut),
                _lib.ptr(eng.lut_index), eng.seed, eng.sweep_index & 0xFFFFFFFF, int(n_sweeps), eng.replica0, eng.row0,
                vp(self.base), vp(self._flags(self.base)), vp(self.up), vp(self._flags(self.up)), vp(self.down),
                vp(self._flags(self.down)), self.msgs[0] & 0xFFFFFFFF, self.msgs[1] & 0xFFFFFFFF,
                int(main.cuda_stream), int(drv._side.cuda_stream),
            )
        self.msgs[0] += n_sweeps
        self.msgs[1] += n_sweeps + 1
        eng.sweep_index += n_sweeps

    def status(self) -> int:
        """0, or 1 if a neighbour's rows did not arrive in time (synchronises the device)"""
        import ctypes

        import torch

        from . import _lib

        out = ctypes.c_uint32(0)
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            _lib.call("tsu_peer_read_u32", ctypes.c_void_p(self.base + 4 * (self.halo_words + 8)), ctypes.byref(out))
        return int(out.value)

    def close(self):
        import ctypes

        import torch

        from . import _lib

        if self.base is None:
            return
        torch.cuda.synchronize(self.device)
        _dist().barrier(group=self.drv.group)  # nobody writes into a buffer that is about to go away
        with torch.cuda.device(self.device):
            for p in self._opened.values():
                _lib.call("tsu_peer_close_handle", ctypes.c_void_p(p))
            self._opened = {}
        _dist().barrier(group=self.drv.group)  # every mapping is closed before the owners free
        self._release()


class LatticeTempering:
    """K ladders x R temperatures of rows x cols lattices with replica exchange on the lattice kernels.

    Replica g = ladder * R + j starts at temperature slot j.  Every iteration = n_sweeps sweeps of all
    replicas; every `swap_interval` iterations one exchange pass per ladder (pairs i = 0..R-2 in order,
    Metropolis rule of tsu/gibbs.py:308-323).  `engine_factory(n_local, replica0, temperatures_local)` builds
    the engine of this rank's replica range; swap_fn(energy, T_slot, slot_replica, lut_index, K, R, step)
    performs the pass in place (tsu_pt_swap on GPUs).  criterion="metropolis" (default) is the detailed-balance
    rule; "reference" reproduces the expression of gibbs.py:317 (see include/tsu_b200.h).

    houdayer_interval = k > 0: every k iterations one Houdayer cluster move (Ising2DEngine.houdayer) runs after the
    sweeps and before the exchange pass, pairing ladders 2m and 2m+1 at every temperature slot (pairs built on the
    device from slot_replica, no host sync).  It needs an even n_ladders, one process, and the same bond realisation
    for every replica of ladders 2m and 2m+1.  0 (default): no cluster moves.
    """

    def __init__(self, temperatures: Sequence[float], n_ladders: int, engine_factory, swap_fn=None, group=None,
                 n_sweeps: int = 10, swap_interval: int = 10, seed: int = 0, criterion: str = "metropolis",
                 houdayer_interval: int = 0):
        import torch

        dist = _dist()
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        if (isinstance(houdayer_interval, bool) or not isinstance(houdayer_interval, (int, np.integer))
                or houdayer_interval < 0):
            raise ValueError("houdayer_interval must be a non-negative integer")
        self.houdayer_interval = int(houdayer_interval)
        if self.houdayer_interval:
            if int(n_ladders) % 2:
                raise ValueError("houdayer_interval needs an even n_ladders: ladders 2m and 2m+1 are paired")
            if self.world != 1:
                raise ValueError("houdayer_interval needs one process: ladder pairs are not split across ranks")
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.temps = np.asarray(list(temperatures), dtype=np.float64)
        self.R, self.K = len(self.temps), int(n_ladders)
        self.n_total = self.R * self.K
        self.start, self.stop = replica_shard(self.n_total, self.rank, self.world)
        self.n_sweeps, self.swap_interval, self.seed = int(n_sweeps), int(swap_interval), int(seed)
        slot0 = np.arange(self.n_total) % self.R
        self.engine = engine_factory(self.stop - self.start, self.start, self.temps[slot0[self.start:self.stop]])
        dev = self.engine.state.device
        self.T_slot = torch.from_numpy(self.temps).to(dev)
        self.slot_replica = torch.arange(self.n_total, dtype=torch.int32, device=dev).reshape(self.K, self.R).contiguous()
        self.lut_index = torch.from_numpy(slot0.astype(np.int32)).to(dev)   # replica -> temperature slot
        self.stats = torch.zeros(2, dtype=torch.int64, device=dev)
        self.iteration = 0
        if criterion not in ("metropolis", "reference"):
            raise ValueError("criterion must be 'metropolis' or 'reference'")
        self.criterion = 1 if criterion == "metropolis" else 0
        self.swap_fn = swap_fn or self._swap_cuda
        # the engine's LUT tables must be ordered by slot: one table per temperature of the ladder
        self.engine.set_temperature_tables(self.temps, self.lut_index[self.start:self.stop])
        if self.houdayer_interval:
            self.engine._houdayer_supported()
            if self.engine.bond_index is not None:
                bi = np.asarray(self.engine.bond_index.cpu()).reshape(self.K // 2, 2 * self.R)
                if np.any(bi != bi[:, :1]):
                    raise ValueError("houdayer_interval needs one bond realisation for all replicas of ladders 2m "
                                     "and 2m+1")

    def _swap_cuda(self, energy, T_slot, slot_replica, lut_index, K, R, step):
        from . import _lib
        from ._lib import ptr

        _lib.call("tsu_pt_swap", ptr(energy), ptr(T_slot), ptr(slot_replica), ptr(lut_index), K, R, self.seed,
                  step & 0xFFFFFFFF, ptr(self.stats), None, self.criterion, _lib.current_stream())

    def gather_energies(self):
        import torch

        e_local = self.engine.energy_tensor()
        if self.world == 1:
            return e_local
        dist = _dist()
        sizes = [replica_shard(self.n_total, r, self.world) for r in range(self.world)]
        parts = [torch.empty(b - a, dtype=e_local.dtype, device=e_local.device) for a, b in sizes]
        dist.all_gather(parts, e_local.contiguous(), group=self.group)
        return torch.cat(parts)

    def step(self):
        """one iteration: n_sweeps sweeps, then (every houdayer_interval iterations) one Houdayer move, then (every
        swap_interval iterations) the exchange pass"""
        self.engine.sweep(self.n_sweeps)
        self.iteration += 1
        if self.houdayer_interval and self.iteration % self.houdayer_interval == 0:
            import torch

            sr = self.slot_replica
            pairs = torch.stack((sr[0::2], sr[1::2]), dim=-1).reshape(-1, 2)  # (ladder 2m, ladder 2m+1) per slot
            self.engine._houdayer(pairs, pairs.shape[0], 1)
        if self.iteration % self.swap_interval == 0:
            energy = self.gather_energies()
            self.swap_fn(energy, self.T_slot, self.slot_replica, self.lut_index, self.K, self.R, self.iteration)
            self.engine.set_lut_index(self.lut_index[self.start:self.stop])
        return self

    def observables_by_slot(self):
        """(magnetisation, energy) arrays of shape [K, R] ordered by temperature slot (host numpy)"""
        import torch

        obs = self.engine.observables_tensor().to(torch.float64)
        full = obs
        if self.world > 1:
            dist = _dist()
            sizes = [replica_shard(self.n_total, r, self.world) for r in range(self.world)]
            parts = [torch.empty((b - a, 2), dtype=obs.dtype, device=obs.device) for a, b in sizes]
            dist.all_gather(parts, obs.contiguous(), group=self.group)
            full = torch.cat(parts)
        sr = self.slot_replica.long()
        per_slot = full[sr.reshape(-1)].reshape(self.K, self.R, 2).cpu().numpy()
        n = self.engine.n_sites
        m = (2.0 * per_slot[..., 0] - n) / n
        e = -self.engine.coupling * (self.engine.n_bonds - 2.0 * per_slot[..., 1]) - self.engine.field * (2.0 * per_slot[..., 0] - n)
        return m, e
