"""Population annealing on the lattice kernels (Ising2DEngine.population_annealing) against plain sweeps with the same
threshold tables, same process, one JSON line per workload.

    python tools/lattice_population_bench.py [--quick]

Workloads (theta = 10 sweeps per step, 10 steps per call, from T = 3 down to T = 1):
  a  131072 replicas of 32 x 32, one +-J realisation, one population; also the torch loop a user writes today
     (energy_tensor on chunks of 32768 replicas, exp, cumsum, searchsorted, index_select on the state, sweep)
  b  64 realisations x 2048 replicas of 64 x 64, n_populations = 64 (one realisation per population)
  c  16 populations x 1024 replicas of 256 x 256, ferromagnet
Each line gives the PA step time and the time of theta sweeps with the step's table (CUDA-event medians of alternated
runs), their difference (counts, resampling and gather), the byte model of that part at 7.7 TB/s (one read of the
state words, padding included, for the counts; one read and one write for the gather; 16 B per replica for the weights
and the scan) and the summed time of every kernel of one PA call from torch.profiler, by name.  Population annealing
runs the prebuilt kernels, so the sweeps run with TSU_B200_NO_JIT too.  The GPU name and power limit are read in the
same run.
"""
import json
import os
import subprocess
import sys
from collections import defaultdict

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ["TSU_B200_NO_JIT"] = "1"  # the kernels population annealing runs, for the sweeps it is compared with
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tsu_emulator_b200.lattice import Ising2DEngine  # noqa: E402

HBM = 7.7e12
THETA, STEPS = 10, 10


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


def kernel_times(fn):
    """seconds per kernel name summed over one call of fn (torch.profiler, CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = defaultdict(float)
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            name = ev.name.split("(")[0].split("<")[0].replace("(anonymous namespace)::", "")
            out[name] += ev.device_time_total * 1e-6 if hasattr(ev, "device_time_total") else ev.cuda_time_total * 1e-6
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def sweeps_with_tables(eng, tables):
    for k in range(tables.shape[0]):
        eng.lut = tables[k:k + 1]
        eng.sweep(THETA)


def torch_loop(eng, Ts, tables, gen):
    """population annealing as a torch loop: no defined random stream, several launches and temporaries per step"""
    R = eng.n_replicas
    beta_prev = 0.0
    ar = torch.arange(R, device=eng.device, dtype=torch.float64)
    # the word-by-word counts take at most 65535 replicas per call (one grid row each)
    views = [eng.chunk_view(r0, min(32768, R - r0)) for r0 in range(0, R, 32768)]
    for k, T in enumerate(Ts):
        E = torch.cat([v.energy_tensor() for v in views])
        w = torch.exp(-(1.0 / T - beta_prev) * (E - E.min()))
        c = torch.cumsum(w, 0)
        u = (torch.rand(1, device=eng.device, dtype=torch.float64, generator=gen) + ar) / R * c[-1]
        idx = torch.searchsorted(c, u).clamp_(max=R - 1)
        eng.state.copy_(eng.state.index_select(0, idx))
        eng.lut = tables[k:k + 1]
        eng.sweep(THETA)
        beta_prev = 1.0 / T


def workload(name, eng, P, reps, info, loop=False):
    Ts = list(np.geomspace(3.0, 1.0, STEPS))
    R = eng.n_replicas
    state_bytes = eng.state.numel() * 4
    eng.init_random()
    eng.population_annealing(Ts, sweeps_per_step=THETA, n_populations=P)  # warm-up: tables, modules, allocator
    tables = eng._schedule_tables(np.asarray(Ts))
    sweeps_with_tables(eng, tables)
    gen = torch.Generator(device=eng.device).manual_seed(1)
    if loop:
        torch_loop(eng, Ts, tables, gen)
    t_pa, t_sw, t_loop = [], [], []
    for _ in range(reps):
        eng.init_random()
        t_pa.append(event_time(lambda: eng.population_annealing(Ts, sweeps_per_step=THETA, n_populations=P)) / STEPS)
        t_sw.append(event_time(lambda: sweeps_with_tables(eng, tables)) / STEPS)
        if loop:
            eng.init_random()
            t_loop.append(event_time(lambda: torch_loop(eng, Ts, tables, gen)) / STEPS)
    eng.init_random()
    kern = kernel_times(lambda: eng.population_annealing(Ts, sweeps_per_step=THETA, n_populations=P))
    pa, sw = float(np.median(t_pa)), float(np.median(t_sw))
    model_counts, model_gather, model_scan = state_bytes / HBM, 2 * state_bytes / HBM, 16 * R / HBM
    line = {
        **info, "workload": name, "replicas": R, "rows": eng.rows, "cols": eng.cols, "n_populations": P,
        "sweeps_per_step": THETA, "steps_per_call": STEPS, "pa_step_s": pa, "sweeps_per_step_s": sw,
        "non_sweep_s": pa - sw, "non_sweep_over_one_sweep": (pa - sw) / (sw / THETA),
        "model_non_sweep_s": model_counts + model_gather + model_scan, "model_counts_s": model_counts,
        "model_gather_s": model_gather, "model_scan_s": model_scan,
        "spread_pa": [min(t_pa), max(t_pa)], "spread_sweeps": [min(t_sw), max(t_sw)],
        "kernels_one_call_s": {k: round(v, 7) for k, v in kern.items()},
    }
    if loop:
        line.update({"torch_loop_step_s": float(np.median(t_loop)), "spread_torch_loop": [min(t_loop), max(t_loop)],
                     "torch_loop_over_pa": float(np.median(t_loop)) / pa})
    print(json.dumps(line), flush=True)


def main():
    quick = "--quick" in sys.argv
    info = gpu_info()
    print(json.dumps(info), flush=True)
    reps = 3 if quick else 7
    rng = np.random.default_rng(3)

    n_a = 8192 if quick else 131072
    signs = rng.choice(np.array([-1, 1], dtype=np.int8), size=(2, 32, 32))
    eng = Ising2DEngine(32, 32, n_replicas=n_a, temperature=3.0, seed=1, bonds=signs)
    workload("a", eng, 1, reps, info, loop=True)
    del eng

    K, r_pop = (8, 256) if quick else (64, 2048)
    signs = rng.choice(np.array([-1, 1], dtype=np.int8), size=(K, 2, 64, 64))
    eng = Ising2DEngine(64, 64, n_replicas=K * r_pop, temperature=3.0, seed=2, bonds=signs,
                        bond_index=np.repeat(np.arange(K), r_pop))
    workload("b", eng, K, reps, info)
    del eng

    P, r_pop = (4, 128) if quick else (16, 1024)
    eng = Ising2DEngine(256, 256, n_replicas=P * r_pop, temperature=3.0, seed=3)
    workload("c", eng, P, reps, info)
    del eng
    torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
