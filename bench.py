#!/usr/bin/env python
"""
bench.py - spin-updates/s of the bit-packed 2-D checkerboard Gibbs path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): 2-D Ising 8192 x 8192, T = 2.269, periodic, 4096 independent
replicas per GPU, heat-bath checkerboard sweeps.  One "step" = SWEEPS_PER_STEP full sweeps of all
replicas.  With N > 1 the replica index range is sharded (4096 replicas per rank, no data-path
collective): weak scaling.

value  : updates/s with the lattices resident in HBM (CUDA events, max over ranks).
e2e    : the same through the host API with HOST buffers: every step uploads the packed initial
         lattices from pinned host memory (chunked, overlapped with the sweeps of the previous
         chunk), runs the sweeps and reads magnetisation/energy back.  `h2d_only` is the upload
         alone (same chunks, all ranks at once): the host-side ceiling of the end-to-end number.
roofline: HBM bound; algorithmic bytes = 0.25 B per spin update (read 1 neighbour-colour bit,
         write 1 bit), per half-sweep launch, against the measured copy bandwidth.  `math_issue`
         is the limiter this kernel actually runs into (see DESIGN.md section 5).
cpu_baseline / --impl reference: the UNMODIFIED reference (GibbsSampler.gibbs_sweep of tsu/gibbs.py,
         from oracle/_ref or /root/reference) on the host cores, one process per core, on a bounded
         sample of the workload; the oracle's literal port only if the reference tree is not there.
--dump-outputs DIR: after the timed steps, rank 0 writes what they computed as DIR/<name>.npy (see dump_outputs()).
         Inputs come from fixed seeds, so two builds run with the same arguments can be compared file by file.
secondary: the other BASELINE configurations, timed with CUDA events inside this run:
         C1 (IsingModel2D 50 x 50, 1000 gibbs_update + M + E), C3 (dense SK N = 4096, 2048 chains,
         10 sweeps on tcgen05; tensor roofline), C5 (50-temperature ladders of 1024^2 lattices with
         replica exchange; Langevin 1e6 chains x dim 10, float64 and float32) and C4 (131072^2 as row
         slabs).  Under --gpus N > 1 the row slabs (strong and weak) and the ladders are sharded over
         the N ranks, so the scaling run times the halo exchange and the energy all-gather.
"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (it may be read-only)

L = 8192
N_REPLICAS = 4096
TEMPERATURE = 2.269
SWEEPS_PER_STEP = 10
SEED = 1234
BYTES_PER_UPDATE = 0.25
WORKLOAD = "ising2d_8192x8192_T2.269_periodic_4096replicas_checkerboard_gibbs"
METRIC = "spin_updates_per_s"
UNIT = "spin-updates/s"
CPU_SIZE, CPU_SWEEPS = 64, 30   # bounded sample of the workload for the host-core arm


# ----------------------------------------------------------------------------- CPU arm
def _cpu_worker(args):
    """one process = one host core: the reference's own sweep (or its literal port) on a small periodic lattice"""
    rank, size, n_sweeps, use_ref = args
    import numpy as np

    n = size * size
    if use_ref:
        from oracle import ref_loader

        gibbs, _, ising = ref_loader.load_reference()
        grid = ising.IsingGrid((size, size), J=1.0, config=ising.IsingConfig(temperature=TEMPERATURE), periodic=True)
        Jb = 4.0 * grid.J
        hb = 2.0 * grid.h - 2.0 * grid.J.sum(axis=1)      # spin -> bit transformation of the lattice couplings
        sampler = gibbs.GibbsSampler(gibbs.GibbsConfig(temperature=TEMPERATURE))
        np.random.seed(1000 + rank)
        state = np.random.randint(0, 2, size=n)
        t0 = time.perf_counter()
        state = sampler.gibbs_sweep(state, Jb, hb, n_sweeps=n_sweeps)   # tsu/gibbs.py:128-162, unmodified
        return time.perf_counter() - t0, int(state.sum())
    from oracle import ising2d_oracle as O

    rng = np.random.default_rng(1000 + rank)
    Jb, hb = O.dense_bit_model(size, size, 1.0, 0.0, True)
    order = O.checkerboard_order(size, size)
    state = rng.integers(0, 2, n)
    t0 = time.perf_counter()
    for _ in range(n_sweeps):
        state = O.gibbs_sweep_port(state, Jb, hb, TEMPERATURE, order, rng.random(n))
    return time.perf_counter() - t0, int(state.sum())


def reference_tree_available():
    try:
        from oracle import make_ref

        return make_ref.ref_root() is not None
    except Exception:
        return False


def cpu_baseline(size=CPU_SIZE, n_sweeps=300, cores=None):
    """aggregate updates/s of `cores` independent replicas of a size x size lattice (bounded sample)"""
    import multiprocessing as mp

    if not cores:
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    use_ref = reference_tree_available()
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(r, size, n_sweeps, use_ref) for r in range(cores)])
    wall = time.perf_counter() - t0
    inner = max(r[0] for r in res)
    updates = cores * size * size * n_sweeps
    what = ("the reference's own GibbsSampler.gibbs_sweep (tsu/gibbs.py:128-162, unmodified, oracle/_ref), "
            "IsingGrid dense couplings" if use_ref else
            "literal per-spin NumPy port of tsu/gibbs.py:128-162 (reference tree not available)")
    return {
        "value": updates / inner,
        "unit": UNIT,
        "cores": cores,
        "kind": "reference" if use_ref else "port",
        "sample": f"{cores} independent {size}x{size} periodic lattices x {n_sweeps} sweeps at T={TEMPERATURE}: {what} "
                  f"(dense {size*size}x{size*size} J), one process per core; same update rule as the workload at reduced size",
        "seconds": wall,
    }


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    vals = []
    last = None
    for i in range(warmup + steps):
        last = cpu_baseline(size=CPU_SIZE, n_sweeps=CPU_SWEEPS)
        if i >= warmup:
            vals.append(last["value"])
    v = sum(vals) / len(vals)
    upd_per_step = last["cores"] * CPU_SIZE * CPU_SIZE * CPU_SWEEPS
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": v,
        "unit": UNIT,
        "n_gpus": args.gpus,
        "steps": steps,
        "warmup": warmup,
        "ms_per_step": upd_per_step / v * 1e3,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": "reference CPU path timed on a bounded sample of the workload "
                   f"({last['cores']} lattices of {CPU_SIZE}x{CPU_SIZE} x {CPU_SWEEPS} sweeps per step)"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index, period_ms=200):
        self.device_index = device_index
        self.period_ms = period_ms
        self.proc = None
        self.path = os.path.join(tempfile.gettempdir(), f"tsu_bench_clocks_{os.getpid()}_{id(self)}.csv")

    def start(self):
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", str(self.period_ms),
                 "-i", str(self.device_index)],
                stdout=self.fh, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for n, v in zip(names, f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out["samples"] = len(sm)
            sm.sort()
            out["sm_mhz"] = sm[len(sm) // 2]
            out["sm_max_mhz"] = max(mx)
        out["reasons"] = sorted(reasons)
        return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        d = json.load(open(p))
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                "bf16_tflops_sustained": float(d["bf16_tflops_sustained"]), "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
                "source": "fallback (B200_PROFILING.md)"}


def profiled_kernel():
    """numbers of the committed ncu capture of the half-sweep kernel at this workload (profiles/lattice_kernel.json):
    DRAM bytes per launch, executed instructions per 32-spin word and how many of them go through the integer
    ALU / wide-multiply dispatch, which is what bounds the kernel"""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "lattice_kernel.json")))
        return d if d.get("workload") == WORKLOAD else None
    except Exception:
        return None


# ----------------------------------------------------------------------------- output dump
# what --dump-outputs writes stays under 64 MB for any shape: at most 40 MB of sampled spins (argument check in main()),
# 16 B of observables for each of at most 2^20 replicas, and the sample's indices
DUMP_REPLICAS = 8
DUMP_SPIN_BYTES = 40 << 20
DUMP_OBS_REPLICAS = 1 << 20


def dump_outputs(eng, out_dir):
    """write what the timed sweeps left in `eng`, in the form a caller of Ising2DEngine receives it:
    magnetization.npy, energy.npy        float64 [M]           magnetisation per spin and energy of the first
                                                               M = min(n_replicas, 2^20) replicas
    spins.npy                            float32 [R, K, cols]  +-1 spins of R replicas x K rows, all columns
    spins_replicas.npy, spins_rows.npy   float64 [R], [K]      the replicas and rows spins.npy holds (seeded sample)"""
    import numpy as np
    import torch

    rng = np.random.default_rng(SEED)
    row_bytes = 4 * eng.cols
    n_rep = min(DUMP_REPLICAS, eng.n_replicas, DUMP_SPIN_BYTES // row_bytes)
    n_rows = min(eng.rows, DUMP_SPIN_BYTES // (row_bytes * n_rep))
    replicas = np.sort(rng.choice(eng.n_replicas, n_rep, replace=False))
    rows = np.sort(rng.choice(eng.rows, n_rows, replace=False))
    rows_dev = torch.from_numpy(rows).to(eng.device)
    spins = np.stack([eng.chunk_view(int(r), 1).spins_tensor(pm1=True)[0].index_select(0, rows_dev).cpu().numpy()
                      for r in replicas])
    n_obs = min(eng.n_replicas, DUMP_OBS_REPLICAS)
    arrays = {"magnetization": eng.magnetization()[:n_obs], "energy": eng.energy()[:n_obs],
              "spins": spins.astype(np.float32), "spins_replicas": replicas.astype(np.float64),
              "spins_rows": rows.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------- secondary configurations
def _ev(torch):
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def _max_over_ranks(torch, dist, world, ms):
    if world == 1:
        return ms
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def tc_parity_probe(torch, Jd, T, seed, n_chains=8):
    """the tensor-core sweep against a float64 torch evaluation of the reference's rule on the kernel's own trajectory
    (h_i = J[i,:].s + b_i, accept iff u < sigmoid(h/T), gibbs.py:61-126): number of disagreeing sites and the
    largest |u - p| among them.  One sweep of n_chains chains at the benchmark's matrix."""
    from tsu_emulator_b200 import _lib

    N = Jd.shape[0]
    J64 = Jd.to(torch.float64)
    st0 = (torch.rand(n_chains, N, device="cuda") < 0.5).to(torch.uint8)
    st = st0.clone()
    sweep0, chain0 = 77, 5
    _lib.call("tsu_dense_gibbs_tc_run", _lib.ptr(Jd), None, _lib.ptr(st), n_chains, N, float(T), None, 1, seed, sweep0,
              chain0, None, _lib.current_stream())
    # the kernel's uniforms: 24 bits of word (site & 3) of Philox(counter = (site >> 2, chain, sweep, 'DENT'))
    words = torch.empty((n_chains, N), dtype=torch.int64, device="cuda")
    host = _lib.load()
    import ctypes

    for c in range(n_chains):
        row = []
        for g in range(N // 4):
            ctr = (ctypes.c_uint32 * 4)(g, chain0 + c, sweep0, 0x44454E54)
            key = (ctypes.c_uint32 * 2)(seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
            out = (ctypes.c_uint32 * 4)()
            host.tsu_philox4x32_10_host(ctr, key, out)
            row.extend(int(x) for x in out)
        words[c] = torch.tensor(row, dtype=torch.int64)
    u = (words >> 8).to(torch.float64) / 16777216.0
    cur = st0.to(torch.float64)
    after = st.to(torch.float64)
    n_bad, max_eps = 0, 0.0
    for i in range(N):
        h = cur @ J64[i]
        x = h / T
        p = torch.where(x > 20, torch.ones_like(x), torch.where(x < -20, torch.zeros_like(x), 1.0 / (1.0 + torch.exp(-x))))
        want = (u[:, i] < p).to(torch.float64)
        bad = want != after[:, i]
        if bool(bad.any()):
            n_bad += int(bad.sum())
            max_eps = max(max_eps, float((u[:, i] - p).abs()[bad].max()))
        cur[:, i] = after[:, i]
    return {"sites_checked": n_chains * N, "mismatches": n_bad, "max_eps": max_eps}


def run_secondary(torch, dist, world, rank, local_rank, peaks):
    import numpy as np

    from tsu_emulator_b200 import (GibbsConfig, GibbsSampler, Ising2DEngine, IsingModel2D, QuadraticEnergy,
                                   ThermalSamplingUnit, TSUConfig, _lib)
    from tsu_emulator_b200.distributed import LatticeTempering, SlabShardedIsing2D

    out = {}
    sampler = ClockSampler(local_rank, period_ms=50)
    if rank == 0:
        sampler.start()

    def guarded(name, fn):
        try:
            res = fn()
            if res is not None:
                out[name] = res
        except Exception as exc:  # a secondary configuration must never take the primary line down
            out[name] = {"error": repr(exc)}
        torch.cuda.empty_cache()

    # ---- C4: one 131072 x 131072 lattice as row slabs (strong), and 131072 rows per GPU (weak) -------------------
    def c4(rows, cols, tag, transport="auto"):
        fac = lambda lr, r0: Ising2DEngine(lr, cols, temperature=TEMPERATURE, periodic=True, seed=1, row0=r0,
                                           global_rows=rows).init_random()
        drv = SlabShardedIsing2D(rows, cols, fac, periodic=True, transport=transport)
        drv.sweep(3)
        n_sw = 20
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = _ev(torch)
        a.record()
        drv.sweep(n_sw)
        b.record()
        torch.cuda.synchronize()
        ms = _max_over_ranks(torch, dist, world, a.elapsed_time(b))
        obs = drv.observables()
        kind = drv.transport()
        how = {"p2p": "boundary rows written into the neighbours' peer-mapped halo buffers over NVLink, one C-ABI call per "
                      "sweep batch, overlapped with the interior update",
               "nccl": "NCCL send/recv on a side stream, overlapped with the interior update",
               "local": "local copy"}[kind]
        drv.close()
        upd = float(rows) * cols * n_sw
        ups = upd / ms * 1e3
        return {"workload": f"2D Ising {rows}x{cols}, T=2.269, periodic, {world} row slab(s) of {rows // world} rows, "
                            f"halo exchange per half-sweep ({how}), {n_sw} sweeps", "transport": kind,
                "scaling": tag, "ms_per_sweep": ms / n_sw, "spin_updates_per_s": ups,
                "hbm_frac_per_gpu": ups * BYTES_PER_UPDATE / world / (peaks["hbm_gbs"] * 1e9),
                "energy_per_site": float(-(2.0 * rows * cols - 2.0 * obs[0, 1].item()) / (float(rows) * cols))}

    guarded("C4_strong", lambda: c4(131072, 131072, "strong"))
    if world > 1:
        guarded("C4_weak", lambda: c4(131072 * world, 131072, "weak"))
        guarded("C4_strong_nccl", lambda: c4(131072, 131072, "strong", transport="nccl"))

    # ---- C5a: 50 temperatures x K ladders x 1024^2 with replica exchange, ladders sharded over the ranks ----------
    def c5_ladder():
        temps = np.linspace(0.1, 5.0, 50)
        K = 16 * world
        fac = lambda n, r0, T: Ising2DEngine(1024, 1024, n_replicas=n, temperature=T, periodic=True, seed=5,
                                             replica0=r0).init_random()
        pt = LatticeTempering(temps, n_ladders=K, engine_factory=fac, n_sweeps=10, swap_interval=10, seed=9)
        for _ in range(10):
            pt.step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = _ev(torch)
        a.record()
        for _ in range(20):
            pt.step()
        b.record()
        torch.cuda.synchronize()
        ms = _max_over_ranks(torch, dist, world, a.elapsed_time(b))
        stats = pt.stats.cpu().numpy()
        return {"workload": f"50 temperatures linspace(0.1, 5.0) x {K} ladders x 1024^2 periodic, 20 iterations x 10 sweeps, "
                            f"exchange pass every 10 iterations ({'energies all-gathered over ' + str(world) + ' ranks' if world > 1 else 'one rank'})",
                "scaling": "weak", "ms": ms, "spin_updates_per_s": 20.0 * 10 * K * 50 * 1024 * 1024 / ms * 1e3,
                "swap_accept_rate": float(stats[1] / max(1, stats[0]))}

    guarded("C5_ladder", c5_ladder)

    if world == 1:
        # ---- C1: IsingModel2D size=50, 1000 gibbs_update sweeps + magnetization + energy ---------------------------
        def c1():
            res = {}
            for periodic in (True, False):
                m = IsingModel2D(size=50, coupling=1.0, temperature=2.5, periodic=periodic, seed=0)
                m.gibbs_update(10)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(1000):
                    m.gibbs_update()
                mag, en = m.magnetization(), m.energy()
                dt = time.perf_counter() - t0
                m2 = IsingModel2D(size=50, coupling=1.0, temperature=2.5, periodic=periodic, seed=0)
                m2.gibbs_update(10)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                m2.gibbs_update(1000)
                mag2, en2 = m2.magnetization(), m2.energy()
                dt2 = time.perf_counter() - t0
                res["periodic" if periodic else "open"] = {
                    "wall_ms_1000_calls": dt * 1e3, "spin_updates_per_s": 2.5e6 / dt,
                    "wall_ms_one_call_of_1000": dt2 * 1e3, "spin_updates_per_s_one_call": 2.5e6 / dt2,
                    "same_state": bool(mag == mag2 and en == en2), "magnetization": float(mag), "energy": float(en)}
            res["workload"] = ("IsingModel2D(size=50, coupling=1.0, temperature=2.5): 1000 gibbs_update() + magnetization() "
                               "+ energy(), host wall clock (launch-latency bound: 2500 spins per sweep)")
            return res

        guarded("C1", c1)

        # ---- C3: dense SK N=4096, 2048 chains, 10 sweeps on the tensor cores ------------------------------------------
        def c3():
            N, SW, seed = 4096, 10, 3
            rng = np.random.default_rng(7)
            J = rng.normal(size=(N, N)) / np.sqrt(N)
            J = (J + J.T) / np.sqrt(2)
            np.fill_diagonal(J, 0)
            smp = GibbsSampler(GibbsConfig(temperature=1.0, n_sweeps=SW), seed=seed, precision="bf16")
            api = []
            for _ in range(2):  # the first call also pays lazy kernel loading, allocator growth, the tensor map
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                st = smp.sample_chains(J, None, n_chains=2048, n_sweeps=SW, as_tensor=True)
                torch.cuda.synchronize()
                api.append((time.perf_counter() - t0) * 1e3)
            api_ms = api[1]
            Jd = torch.from_numpy(J).cuda().to(torch.bfloat16).contiguous()
            n_sm = torch.cuda.get_device_properties(0).multi_processor_count
            res = {"workload": f"GibbsSampler(precision='bf16') dense SK couplings (bf16) N={N}, sequential sweeps, tcgen05 + TMEM",
                   "api_ms_2048_chains_10_sweeps_incl_J_upload": api_ms, "api_ms_first_call": api[0],
                   "mean_bit": float(st.float().mean())}
            for C, tag in ((2048, "2048_chains"), (128 * n_sm, "full_wave_%d_chains" % (128 * n_sm))):
                s_ = (torch.rand(C, N, device="cuda") < 0.5).to(torch.uint8)
                _lib.call("tsu_dense_gibbs_tc_run", _lib.ptr(Jd), None, _lib.ptr(s_), C, N, 1.0, None, 1, seed, 0, 0, None,
                          _lib.current_stream())
                best = 1e30
                for _ in range(3):
                    a, b = _ev(torch)
                    a.record()
                    _lib.call("tsu_dense_gibbs_tc_run", _lib.ptr(Jd), None, _lib.ptr(s_), C, N, 1.0, None, SW, seed, 1, 0,
                              None, _lib.current_stream())
                    b.record()
                    torch.cuda.synchronize()
                    best = min(best, a.elapsed_time(b))
                flops = 2.0 * N * N * C * SW
                res[tag] = {"ms": best, "spin_updates_per_s": C * N * SW / best * 1e3, "tflops": flops / best * 1e3 / 1e12,
                            "roofline": {"bound": "tensor", "achieved": flops / best * 1e3 / 1e12,
                                         "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                                         "frac": flops / best * 1e3 / 1e12 / peaks["bf16_tflops_sustained"],
                                         "peak_source": peaks["source"] + " bf16_tflops_sustained (kernel timed alone, but "
                                                        "seconds of tensor work would settle there)"}}
                del s_
            res["parity"] = tc_parity_probe(torch, Jd, 1.0, seed)
            return res

        guarded("C3", c3)

        # ---- C5b: Langevin 1e6 chains, dim 10 Gaussian, float64 (the reference's arithmetic) and float32 ----------------
        def c5_langevin():
            res = {"workload": "ThermalSamplingUnit.sample_from_energy(E = sum x^2, dim 10), 1e6 chains, 100 + 500 steps, dt 0.01"}
            for dtype in ("float64", "float32"):
                tsu = ThermalSamplingUnit(TSUConfig(temperature=1.0, dt=0.01, friction=1.0, n_burnin=100, n_steps=500),
                                          seed=1, dtype=dtype)
                tsu.sample_from_energy(QuadraticEnergy(), np.zeros(10), 1000, as_tensor=True)
                torch.cuda.synchronize()
                ms = 1e30
                for _ in range(2):
                    a, b = _ev(torch)
                    a.record()
                    x = tsu.sample_from_energy(QuadraticEnergy(), np.zeros(10), 1_000_000, as_tensor=True)
                    b.record()
                    torch.cuda.synchronize()
                    ms = min(ms, a.elapsed_time(b))
                res[dtype] = {"ms": ms, "chain_steps_per_s": 1e6 * 600 / ms * 1e3, "coordinate_updates_per_s": 1e6 * 6000 / ms * 1e3,
                              "variance": float(x.var()), "euler_maruyama_theory": 0.5 / (1 - 0.01)}
            return res

        guarded("C5_langevin", c5_langevin)

    if rank == 0:
        out["clocks"] = sampler.stop()
        out["clocks"]["note"] = "nvidia-smi sampled every 50 ms over all secondary configurations of this run"
    return out


# ----------------------------------------------------------------------------- B200 arm
def run_b200_arm(args):
    import torch
    import torch.distributed as dist

    from tsu_emulator_b200.lattice import Ising2DEngine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the B200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    # Host side of the end-to-end leg: run this rank (and first-touch its pinned staging buffer) on the CPU cores that
    # are local to its GPU, so that the N ranks of one box do not pull their uploads across the socket interconnect.
    cpu_mask0 = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa_note = None
    if world > 1 and cpu_mask0 is not None:
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            n_words = (os.cpu_count() + 63) // 64
            words = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
            cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1} & cpu_mask0
            if cpus and cpus != cpu_mask0:
                os.sched_setaffinity(0, cpus)
                numa_note = f"rank pinned to the {len(cpus)} CPU cores NVML reports as local to its GPU"
            else:
                numa_note = (f"NVML reports the same {len(cpu_mask0)} CPU cores as local to every GPU (one NUMA node visible): "
                             "nothing to bind")
        except Exception as exc:  # no NVML / no permission: keep the inherited mask
            numa_note = f"cpu affinity unchanged ({type(exc).__name__})"
    json_fd = None
    if world > 1:
        # NCCL prints its version / debug lines on fd 1 (the image sets NCCL_DEBUG=VERSION).  stdout must carry only
        # the JSON line: park the real stdout and let everything else go to stderr until the line is written.
        sys.stdout.flush()
        json_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n_rep = args.replicas
    size = args.size
    peaks = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng = Ising2DEngine(size, size, n_replicas=n_rep, temperature=TEMPERATURE, periodic=True, seed=SEED,
                        replica0=rank * n_rep)
    eng.init_random()
    updates_per_step = n_rep * size * size * SWEEPS_PER_STEP

    # ---- device-resident timing -------------------------------------------------------
    for _ in range(args.warmup):
        eng.sweep(SWEEPS_PER_STEP)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        eng.sweep(SWEEPS_PER_STEP)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    ms = _max_over_ranks(torch, dist, world, ms)
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs)   # before the end-to-end leg overwrites the lattices
    n_launches = args.steps * SWEEPS_PER_STEP * 2
    value = world * updates_per_step * args.steps / (ms * 1e-3)
    launch_s = ms * 1e-3 / n_launches
    alg_bytes_per_launch = BYTES_PER_UPDATE * n_rep * size * size / 2
    achieved = alg_bytes_per_launch / launch_s / 1e9

    # ---- end to end through the host API: pinned host lattices -> sweeps -> observables -----
    state_bytes = eng.state.numel() * 4
    n_chunks = 32   # upload / sweep pipeline granularity: the exposed ends are one chunk's upload and one chunk's sweeps
    chunk = max(1, n_rep // n_chunks)
    e2e = None
    try:
        # pinned host source: the full 34.4 GB state at N = 1; with N ranks sharing one host the buffer is capped
        # (host RAM / N) and its chunks are re-used round-robin as the source of the per-step uploads - every
        # step still copies state_bytes from pinned host memory to the device
        host_chunks = n_chunks if world == 1 else max(1, n_chunks // world)
        host = torch.empty((host_chunks * chunk,) + tuple(eng.state.shape[1:]), dtype=torch.int32, pin_memory=True)
        host.copy_(eng.state[: host_chunks * chunk])  # synthetic input lattices (any valid packed configuration)
        obs_host = torch.empty((n_rep, 2), dtype=torch.int64, pin_memory=True)
        copy_stream = torch.cuda.Stream()
        main = torch.cuda.current_stream()

        def upload(record_events):
            evs = []
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_stream(main)
                for k, c0 in enumerate(range(0, n_rep, chunk)):
                    n_c = min(chunk, n_rep - c0)
                    h0 = (k % host_chunks) * chunk
                    eng.state[c0:c0 + n_c].copy_(host[h0:h0 + n_c], non_blocking=True)
                    if record_events:
                        ev = torch.cuda.Event()
                        ev.record(copy_stream)
                        evs.append(ev)
            return evs

        def e2e_step():
            evs = upload(True)
            # sweeps of chunk k overlap the upload of chunk k+1
            for k, c0 in enumerate(range(0, n_rep, chunk)):
                main.wait_event(evs[k])
                sub = eng.chunk_view(c0, min(chunk, n_rep - c0))
                sub.sweep(SWEEPS_PER_STEP)
            obs = eng.observables_tensor()
            obs_host.copy_(obs, non_blocking=True)
            main.synchronize()
            return obs_host

        for _ in range(max(1, args.warmup - 1)):
            e2e_step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            e2e_step()
        e1.record()
        barrier()
        e2e_ms = _max_over_ranks(torch, dist, world, e0.elapsed_time(e1))
        # the upload alone, all ranks at the same time: what the host (DRAM + PCIe) can deliver to N GPUs at once
        barrier()
        c0_, c1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0_.record()
        for _ in range(2):
            upload(False)
            main.wait_stream(copy_stream)
        c1_.record()
        barrier()
        h2d_ms = _max_over_ranks(torch, dist, world, c0_.elapsed_time(c1_)) / 2
        e2e = {
            "value": world * updates_per_step * args.steps / (e2e_ms * 1e-3),
            "unit": UNIT,
            "h2d_bytes_per_step": int(state_bytes) * world,
            "d2h_bytes_per_step": int(n_rep * 16) * world,
            "ms_per_step": e2e_ms / args.steps,
            "api": f"Ising2DEngine: pinned host state -> H2D ({n_chunks} chunks, overlapped) -> sweep(10) -> observables -> D2H",
            "pinned_host_bytes": int(host.numel() * 4),
            "host_affinity": numa_note,
            "h2d_only": {"ms_per_step": h2d_ms, "gbs_per_gpu": state_bytes / h2d_ms / 1e6,
                         "gbs_all_gpus": state_bytes * world / h2d_ms / 1e6,
                         "note": "the same uploads without the sweeps, all ranks at once: an end-to-end step cannot be "
                                 "shorter than max(this, the device-resident step)"},
        }
        del host
    except Exception as exc:  # e.g. pinned allocation refused
        e2e = {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "error": repr(exc)}

    jit_on = getattr(eng, "_jit", 0) > 0
    del eng
    torch.cuda.empty_cache()
    secondary = None
    if not args.no_secondary:
        secondary = run_secondary(torch, dist, world, rank, local_rank, peaks)

    cpu = None
    if cpu_mask0 is not None:
        os.sched_setaffinity(0, cpu_mask0)  # the CPU baseline may use every host core again
    if rank == 0 and not args.no_cpu:
        cpu = cpu_baseline()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    prof = profiled_kernel()
    math_issue = None
    if prof and clocks and clocks.get("sm_mhz"):
        # B200 issues LOP3 / SHF / IADD3 and IMAD.WIDE at one warp instruction per 2 cycles per SM sub-partition, and the
        # two do NOT overlap (tools/microbench/pipes.cu): a word costs 2 cycles per such instruction at best
        slots = prof["alu_instr_per_word"] + prof["wide_mul_instr_per_word"]
        words_per_s = value / world / 32.0
        cap_words = 148 * 4 * clocks["sm_mhz"] * 1e6 / (2.0 * slots) * 32
        math_issue = {"alu_instr_per_word": prof["alu_instr_per_word"], "wide_mul_instr_per_word": prof["wide_mul_instr_per_word"],
                      "instr_per_word": prof["instr_per_word"], "cycles_per_slot": 2.0,
                      "frac": words_per_s / cap_words,
                      "note": "fraction of the integer-ALU + wide-multiply dispatch slots (148 SMs x 4 sub-partitions x "
                              "1 warp instruction per 2 cycles at the sampled SM clock) this kernel's executed instruction "
                              "mix occupies; counts from the committed ncu capture (" + prof.get("source", "profiles/") + ")"}
    line = {
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": ms / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "u32",
        "data": "synthetic",
        "config": {
            "workload": WORKLOAD if (size == L and n_rep == N_REPLICAS) else f"ising2d_{size}x{size}_T2.269_periodic_{n_rep}replicas",
            "lattice": [size, size],
            "replicas_per_gpu": n_rep,
            "sweeps_per_step": SWEEPS_PER_STEP,
            "temperature": TEMPERATURE,
            "rng": "philox4x32-10, in-register",
            "cache": "inputs_larger_than_L2 (34.4 GB of packed state per GPU)",
            "sharding": "replica index range per rank, no data-path collective",
        },
        "roofline": {
            "bound": "hbm",
            "achieved": achieved,
            "peak": peaks["hbm_gbs"],
            "unit": "GB/s",
            "frac": achieved / peaks["hbm_gbs"],
            "traffic": prof.get("dram_bytes_per_launch") if prof else None,
            "traffic_source": (prof.get("source") if prof else None),
            "peak_source": peaks["source"] + " hbm_gbs",
            "kernel": ("tsu_jit_half_sweep (NVRTC specialisation of half_sweep_fast_body for this temperature)"
                       if jit_on else "half_sweep_fast_kernel"),
            "algorithmic_bytes_per_launch": alg_bytes_per_launch,
            "launch_ms": launch_s * 1e3,
            "math_issue": math_issue,
        },
        "cpu_baseline": cpu,
        "e2e": e2e,
        "gpu_launches": n_launches,
        "clocks": clocks,
        "secondary": secondary,
    }
    if json_fd is not None:
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
        os.close(json_fd)
    else:
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--replicas", type=int, default=N_REPLICAS, help="replicas per GPU (default = the named workload)")
    ap.add_argument("--size", type=int, default=L)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary configurations")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the state the timed steps computed as DIR/<name>.npy (rank 0's replicas)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 arm")
    if args.dump_outputs and 4 * args.size > DUMP_SPIN_BYTES:
        ap.error(f"--dump-outputs: one row of {args.size} spins exceeds the {DUMP_SPIN_BYTES >> 20} MB spin sample")
    if args.warmup < 3:
        args.warmup = 3 if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
