"""Simulated annealing on the lattice kernels (Ising2DEngine.anneal) against plain sweeps, same process, one JSON line per
workload.

    python tools/lattice_anneal_bench.py [--quick]

Workloads:
  ferro        1024 replicas of 8192^2: an anneal step against one sweep at a fixed temperature
  per_replica  256 replicas of 8192^2 with one +-J realisation per replica: the same comparison
  c1           148 replicas of 50 x 50 (open), 1000 steps: one anneal call against the host loop it replaces
               (set_temperature, sweep(1), energy() with its host sync, the best state kept by hand)
The big workloads anneal from T = 3 down to T = 0.5: the state starts random and cools all the way, so nearly every
replica improves at every step and every step copies nearly every replica (the most the best-state bookkeeping can
cost).  Annealing always runs the prebuilt kernels, so the sweeps it is compared with run with TSU_B200_NO_JIT too.
Each line also gives what the byte model expects on top of the sweep: one pass over the state (and, with a realisation
per replica, over the east and south bond words) for the counts, and one read plus one write of the state for the copy,
at 7.7 TB/s.  Times are CUDA-event medians of alternated runs (the c1 loop
syncs with the host on every step, so both c1 arms are host clocks around a device synchronise).  The first line
carries the GPU name and power limit read in the same run.
"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ["TSU_B200_NO_JIT"] = "1"  # the kernels an anneal runs, for the sweeps it is compared with
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tsu_emulator_b200 import _lib  # noqa: E402
from tsu_emulator_b200._lib import ptr  # noqa: E402
from tsu_emulator_b200.lattice import Ising2DEngine  # noqa: E402

HBM = 7.7e12


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, check=True).stdout.splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unknown ({e})"}


def event_time(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3


def host_time(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t


def per_replica_bonds(e, n, L):
    """one realisation per replica, drawn and packed on the device in chunks (n x 2 L^2 int8 signs would not fit)"""
    with torch.cuda.device(e.device):
        words = torch.empty((n, 2, 4, L, e.wpr), dtype=torch.int32, device=e.device)
        gen = torch.Generator(device=e.device).manual_seed(5)
        for k0 in range(0, n, 16):
            k1 = min(n, k0 + 16)
            signs = (2 * torch.randint(0, 2, (k1 - k0, 2, L, L), generator=gen, device=e.device) - 1).to(torch.int8)
            _lib.call("tsu_ising2d_pack_bonds", ptr(signs), ptr(words[k0:k1]), k1 - k0, L, L, int(e.wrap_rows),
                      int(e.wrap_cols), _lib.current_stream())
            del signs
        e.bonds = words
        e.bond_index = torch.arange(n, dtype=torch.int32, device=e.device)
    return e


def step_vs_sweep(name, eng, steps, reps, info):
    """eng anneals `steps` steps per call; the same engine sweeps `steps` times at a fixed temperature in between"""
    Ts = list(np.geomspace(3.0, 0.5, steps))
    state_bytes = eng.state.numel() * 4
    bond_bytes = 0 if eng.bond_index is None else eng.bonds.numel() * 4 // 2  # the counts read E and S of 4 directions
    res = eng.anneal(Ts)  # warm-up: tables, modules
    eng.set_temperature(1.0)
    eng.sweep(1)
    obs_t = []
    t_anneal, t_sweep = [], []
    for _ in range(reps):
        eng.init_random()  # every anneal starts random and cools: nearly every replica improves at every step
        res.best_energy.fill_(float("inf"))
        t_anneal.append(event_time(lambda: eng.anneal(Ts, best=res)) / steps)
        eng.set_temperature(1.0)
        t_sweep.append(event_time(lambda: eng.sweep(steps)) / steps)
        obs_t.append(event_time(eng.observables_tensor))
    a, s, o = (float(np.median(x)) for x in (t_anneal, t_sweep, obs_t))
    model_obs, model_copy = (state_bytes + bond_bytes) / HBM, 2 * state_bytes / HBM
    print(json.dumps({
        **info, "workload": name, "replicas": eng.n_replicas, "L": eng.rows, "steps_per_call": steps,
        "anneal_step_s": a, "sweep_s": s, "overhead_s": a - s, "overhead_share": a / s - 1,
        "observables_pass_s": o, "model_overhead_s": model_obs + model_copy,
        "model_observables_s": model_obs, "model_copy_s": model_copy,
        "spread_anneal": [min(t_anneal), max(t_anneal)], "spread_sweep": [min(t_sweep), max(t_sweep)],
    }), flush=True)


def c1(reps, info, n_steps=1000):
    Ts = list(np.geomspace(3.0, 0.1, n_steps))
    kw = dict(n_replicas=148, temperature=3.0, periodic=False, seed=7)
    one, loop = Ising2DEngine(50, 50, **kw), Ising2DEngine(50, 50, **kw)

    def host_loop():
        best_e = np.full(loop.n_replicas, np.inf)
        best_s = torch.empty_like(loop.state)
        for T in Ts:
            loop.set_temperature(T)
            loop.sweep(1)
            E = loop.energy()
            better = E < best_e
            best_e[better] = E[better]
            idx = torch.from_numpy(np.flatnonzero(better)).to(loop.device)
            best_s[idx] = loop.state[idx]
        return best_e

    t_first = None
    t_one, t_loop = [], []
    for r in range(reps + 1):
        one.init_random()
        loop.state.copy_(one.state)
        one.sweep_index = loop.sweep_index = 0
        if r == 0:
            one.__dict__.pop("_anneal_tables", None)
        t = host_time(lambda: one.anneal(Ts))
        tl = host_time(host_loop)
        assert torch.equal(one.state, loop.state), "one call and the host loop differ"
        if r == 0:
            t_first = t  # builds and uploads the 1000 tables
        else:
            t_one.append(t)
            t_loop.append(tl)
    print(json.dumps({
        **info, "workload": "c1", "replicas": 148, "rows": 50, "cols": 50, "steps": n_steps,
        "one_call_s": float(np.median(t_one)), "one_call_first_s": t_first, "host_loop_s": float(np.median(t_loop)),
        "speedup": float(np.median(t_loop) / np.median(t_one)),
        "spread_one_call": [min(t_one), max(t_one)], "spread_host_loop": [min(t_loop), max(t_loop)],
    }), flush=True)


def main():
    quick = "--quick" in sys.argv
    info = gpu_info()
    print(json.dumps(info), flush=True)
    L = 1024 if quick else 8192
    n_ferro, n_per = (16, 4) if quick else (1024, 256)
    reps = 3 if quick else 5
    eng = Ising2DEngine(L, L, n_replicas=n_ferro, temperature=1.0, seed=1)
    step_vs_sweep("ferro", eng, 10, reps, info)
    del eng
    torch.cuda.empty_cache()
    eng = per_replica_bonds(Ising2DEngine(L, L, n_replicas=n_per, temperature=1.0, seed=2), n_per, L)
    step_vs_sweep("per_replica", eng, 10, reps, info)
    del eng
    torch.cuda.empty_cache()
    c1(reps, info, 100 if quick else 1000)


if __name__ == "__main__":
    main()
