"""Annealing and replica exchange on the tensor-core dense sampler, N = 4096, SK couplings rounded to bf16.

    python tools/tc_anneal.py [--steps 100] [--reps 5]

Prints the GPU name and power limit, then one line per measurement:
  * simulated annealing step at 2048 and 18944 chains, split into the sweep launch (tsu_dense_gibbs_tc_run, one sweep)
    and the energy / best-state pass (tsu_dense_tc_energy): CUDA-event medians over --steps alternated launches (the
    order an anneal runs them in), after warm-up;
  * GibbsSampler(precision="bf16").simulated_annealing end to end, per step: the difference of two anneals of
    different length (host clock around synchronised calls), so the coupling upload and set-up cancel;
  * the same for the float64 block kernel's simulated_annealing at 296 chains, per chain-step for comparison;
  * parallel_tempering(precision="bf16") with R = 32 temperatures, n_ladders = 64 and 592, 10 sweeps per iteration and
    one swap pass per iteration: time per iteration on the device (the iteration's launches between CUDA events) and end
    to end (the difference of two runs, which includes the copy of every sample to the host as int64).
The J matrix (32 MB) stays resident in the 126 MB L2 across launches, as it does in the sampler.
"""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tsu_emulator_b200 import GibbsConfig, GibbsSampler, _lib  # noqa: E402


def gpu_line():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return f"GPU: {name}, power limit {pl}"


def sk(N, seed=7):
    rng = np.random.default_rng(seed)
    J = np.triu(rng.standard_normal((N, N)), 1)
    J = (J + J.T) / np.sqrt(N)
    return torch.from_numpy(J).float().bfloat16().double().numpy()   # bf16-exact: every path sees the same model


def kernel_split(Jd, C, N, steps):
    """median sweep launch and energy pass of an anneal, CUDA events around every launch"""
    st = (torch.rand(C, N, device="cuda") < 0.5).to(torch.uint8)
    e = torch.empty(C, dtype=torch.float64, device="cuda")
    be = torch.full((C,), float("inf"), dtype=torch.float64, device="cuda")
    bs = torch.empty_like(st)
    s = _lib.current_stream()
    Ts = 4.0 * (0.05 / 4.0) ** (np.arange(steps) / steps)

    def step(k):
        _lib.call("tsu_dense_gibbs_tc_run", _lib.ptr(Jd), None, _lib.ptr(st), C, N, float(Ts[k]), None, 1, 3, k, 0,
                  None, s)

    def energy():
        _lib.call("tsu_dense_tc_energy", _lib.ptr(Jd), None, _lib.ptr(st), C, N, _lib.ptr(e), _lib.ptr(be),
                  _lib.ptr(bs), s)

    for k in range(5):                                   # warm-up: module load, tensor maps, L2
        step(k)
        energy()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * steps)]
    for k in range(steps):
        ev[3 * k].record()
        step(k)
        ev[3 * k + 1].record()
        energy()
        ev[3 * k + 2].record()
    torch.cuda.synchronize()
    sw = np.median([ev[3 * k].elapsed_time(ev[3 * k + 1]) for k in range(steps)])
    en = np.median([ev[3 * k + 1].elapsed_time(ev[3 * k + 2]) for k in range(steps)])
    return sw, en


def pt_iteration(Jd, K, R, N, reps):
    """median device time of one tempering iteration at the C-ABI level (CUDA events): 10 sweeps with per-chain T, the
    energy pass, the swap pass and the re-permutation of the per-chain temperatures - what parallel_tempering runs per
    iteration before the host-side copies of samples"""
    C = K * R
    st = (torch.rand(C, N, device="cuda") < 0.5).to(torch.uint8)
    T_slot = torch.from_numpy(np.geomspace(0.3, 3.0, R)).cuda()
    T_chain = T_slot.repeat(K)
    sr = torch.arange(C, dtype=torch.int32, device="cuda").view(K, R)
    e = torch.empty(C, dtype=torch.float64, device="cuda")
    s = _lib.current_stream()

    def it(k):
        _lib.call("tsu_dense_gibbs_tc_run", _lib.ptr(Jd), None, _lib.ptr(st), C, N, 1.0, _lib.ptr(T_chain), 10, 3,
                  10 * k, 0, None, s)
        _lib.call("tsu_dense_tc_energy", _lib.ptr(Jd), None, _lib.ptr(st), C, N, _lib.ptr(e), None, None, s)
        _lib.call("tsu_pt_swap", _lib.ptr(e), _lib.ptr(T_slot), _lib.ptr(sr), None, K, R, 3, k, None, None, 1, s)
        T_chain[sr.long()] = T_slot

    for k in range(3):
        it(k)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    ev[0].record()
    for k in range(reps):
        it(3 + k)
        ev[k + 1].record()
    torch.cuda.synchronize()
    return float(np.median([ev[k].elapsed_time(ev[k + 1]) for k in range(reps)]))


def wall(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t


def per_unit(fn, a, b, reps):
    """(time of fn(b) - time of fn(a)) / (b - a), median over reps alternated pairs, in ms"""
    fn(a)
    fn(b)
    d = []
    for _ in range(reps):
        ta = wall(lambda: fn(a))
        tb = wall(lambda: fn(b))
        d.append((tb - ta) / (b - a))
    return 1e3 * float(np.median(d))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    print(gpu_line(), flush=True)
    N = 4096
    J = sk(N)
    Jd = torch.from_numpy(J).cuda().float().bfloat16().contiguous()
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    for C in (2048, 128 * n_sm):
        sw, en = kernel_split(Jd, C, N, a.steps)
        print(f"anneal step N={N} chains={C}: sweep {sw:.3f} ms + energy/best pass {en:.3f} ms = {sw + en:.3f} ms "
              f"(energy pass = {en / sw:.2f} sweeps; CUDA-event medians of {a.steps} alternated launches)", flush=True)
        smp = GibbsSampler(seed=1, precision="bf16")
        ms = per_unit(lambda n: smp.simulated_annealing(J, T_initial=4.0, T_final=0.05, n_steps=n, n_chains=C),
                      a.steps // 2, a.steps + a.steps // 2, a.reps)
        print(f"simulated_annealing bf16 N={N} chains={C}: {ms:.3f} ms per step end to end, "
              f"{ms * 1e3 / C:.3f} us per chain-step", flush=True)
    f64 = GibbsSampler(seed=1, precision="float64")
    ms = per_unit(lambda n: f64.simulated_annealing(J, T_initial=4.0, T_final=0.05, n_steps=n, n_chains=296), 10, 30,
                  max(2, a.reps // 2))
    print(f"simulated_annealing float64 N={N} chains=296: {ms:.3f} ms per step, {ms * 1e3 / 296:.3f} us per chain-step",
          flush=True)
    temps = list(np.geomspace(0.3, 3.0, 32))
    for K in (64, 592):
        smp = GibbsSampler(GibbsConfig(n_burnin=0, n_sweeps=10), seed=2, precision="bf16")
        ms = per_unit(lambda n: smp.parallel_tempering(J, temps, n_samples=n, swap_interval=1, n_ladders=K,
                                                       criterion="metropolis"), 5, 15, a.reps)
        dev = pt_iteration(Jd, K, 32, N, 20)
        print(f"parallel_tempering bf16 N={N} R=32 ladders={K} ({32 * K} chains), 10 sweeps + 1 swap pass: "
              f"{dev:.3f} ms per iteration on the device (CUDA-event median of 20), {ms:.3f} ms end to end "
              f"(with the samples copied to the host as int64)", flush=True)


if __name__ == "__main__":
    main()
