"""Swendsen-Wang cluster steps on the lattice kernels (Ising2DEngine.swendsen_wang) against heat-bath sweeps on the
same engine, same process, one JSON line per workload.

    python tools/lattice_cluster_bench.py [--quick]

Step time (T = 2.269, ferromagnet, periodic; CUDA-event medians of alternated runs):
  a  64 x 8192^2 (workspace chunks of the default 4 GiB budget)    (--quick: 8 replicas)
  b  256 x 1024^2                                                 (--quick: 32 replicas)
  c  148 x 50 x 50, one launch per call (10 steps per call)
Each line gives the SW step time, the Gibbs sweep time, their ratio, the byte model of a step at 7.7 TB/s (9.125 B per
site: state read for the bonds 0.125, activation words written and read 0.5, flip words written and read 0.25, labels
written by the local pass and read by the flips 8, state read and written by the flips 0.25; root lookups not counted)
and the summed time of every kernel of one call from torch.profiler, by name.

Physics payoff at T_c: 148 replicas of L x L (L = 64, 128) from random states; the per-step series of E and M^2 of every
replica (Gibbs: 2^16 sweeps, SW: 4096 steps; the first quarter dropped), the integrated autocorrelation time with
Sokal's windowed estimator (smallest W with W >= 6 tau(W)), and the device time per independent sample of one replica,
2 tau x step time / 148.  The GPU name and power limit are read in the same run.
"""
import json
import os
import subprocess
import sys
from collections import defaultdict

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tsu_emulator_b200.lattice import Ising2DEngine  # noqa: E402

HBM = 7.7e12
BYTES_PER_SITE = 0.125 + 0.5 + 0.25 + 8.0 + 0.25
TC = 2.0 / np.log(1.0 + np.sqrt(2.0))


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
            name = ev.name.replace("void ", "").replace("(anonymous namespace)::", "").split("(")[0].split("<")[0]
            out[name] += ev.device_time_total * 1e-6 if hasattr(ev, "device_time_total") else ev.cuda_time_total * 1e-6
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def step_workload(name, n_rep, L, per_call, reps, info):
    eng = Ising2DEngine(L, L, n_replicas=n_rep, temperature=2.269, periodic=True, seed=1)
    eng.init_random()
    eng.swendsen_wang(per_call)  # warm-up: workspace, threshold table, modules
    eng.sweep(per_call)
    torch.cuda.synchronize()
    t_sw, t_gibbs = [], []
    for _ in range(reps):
        t_sw.append(event_time(lambda: eng.swendsen_wang(per_call)) / per_call)
        t_gibbs.append(event_time(lambda: eng.sweep(per_call)) / per_call)
    sw, gibbs = float(np.median(t_sw)), float(np.median(t_gibbs))
    sites = n_rep * L * L
    return dict(info, workload=name, replicas=n_rep, L=L, sw_step_s=sw, gibbs_sweep_s=gibbs, ratio=sw / gibbs,
                sw_site_steps_per_s=sites / sw, byte_model_s=sites * BYTES_PER_SITE / HBM,
                model_share=sites * BYTES_PER_SITE / HBM / sw,
                kernels_s=kernel_times(lambda: eng.swendsen_wang(per_call)), steps_per_call=per_call)


def tau_int(x):
    """Sokal's windowed integrated autocorrelation time of series x [n_rep, n] (averaged autocorrelation)"""
    x = x - x.mean(axis=1, keepdims=True)
    n = x.shape[1]
    f = np.fft.rfft(x, 2 * n, axis=1)
    acf = np.fft.irfft(f * np.conj(f), axis=1)[:, :n].mean(axis=0)
    rho = acf / acf[0]
    tau = 0.5
    for W in range(1, n):
        tau += rho[W]
        if W >= 6 * tau:
            return float(tau), W
    return float(tau), n


def series(eng, n, step):
    """[n_rep, n] series of E and M^2 after every step (device copies, one host transfer at the end)"""
    obs = torch.empty((n, eng.n_replicas, 2), dtype=torch.int64, device=eng.device)
    for t in range(n):
        step()
        obs[t].copy_(eng.observables_tensor())
    o = obs.cpu().numpy().astype(np.float64).transpose(1, 0, 2)
    E = -(eng.n_bonds - 2.0 * o[..., 1])
    M = 2.0 * o[..., 0] - eng.n_sites
    return E, M * M


def payoff(L, n_rep, n_gibbs, n_sw, info):
    out = dict(info, workload=f"autocorrelation L={L}", replicas=n_rep, L=L, T=TC)
    for name, n, make_step in (("gibbs", n_gibbs, lambda e: (lambda: e.sweep(1))),
                               ("sw", n_sw, lambda e: (lambda: e.swendsen_wang(1)))):
        eng = Ising2DEngine(L, L, n_replicas=n_rep, temperature=TC, periodic=True, seed=3)
        eng.init_random()
        step = make_step(eng)
        step()
        t_step = float(np.median([event_time(lambda: [step() for _ in range(100)]) / 100 for _ in range(5)]))
        E, M2 = series(eng, n, step)
        keep = n // 4
        tE, wE = tau_int(E[:, keep:])
        tM, wM = tau_int(M2[:, keep:])
        out[name] = dict(steps=n, step_s=t_step, tau_E=tE, window_E=wE, tau_M2=tM, window_M2=wM,
                         s_per_independent_sample_E=2 * tE * t_step / n_rep,
                         s_per_independent_sample_M2=2 * tM * t_step / n_rep)
    return out


def main():
    quick = "--quick" in sys.argv
    torch.cuda.set_device(0)
    info = gpu_info()
    print(json.dumps(step_workload("a", 8 if quick else 64, 8192, 1, 3 if quick else 5, info)), flush=True)
    print(json.dumps(step_workload("b", 32 if quick else 256, 1024, 1, 3 if quick else 10, info)), flush=True)
    print(json.dumps(step_workload("c", 148, 50, 10, 10, info)), flush=True)
    for L in (64, 128):
        print(json.dumps(payoff(L, 148, (1 << 13) if quick else (1 << 16), 1024 if quick else 4096, info)), flush=True)


if __name__ == "__main__":
    main()
