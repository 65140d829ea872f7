"""Parallel tempering with and without Houdayer moves (ICM) on periodic 3-D +-J Edwards-Anderson glasses, on the
chromatic CSR back end (GibbsSampler.parallel_tempering(chromatic=True, houdayer_interval=1)).

Workload: L = 8 (N = 512) and L = 16 (N = 4096), 16 temperatures geometric from 0.2 to 2.0, 32 ladders, one sweep and
one exchange pass per iteration; moves on the slots with T <= 1.0 (below T_c ~ 1.1 of the 3-D +-J glass), between
ladders 2m and 2m + 1.  Prints one JSON line per measurement:
  tau      integrated autocorrelation time of q^2 between ladders 2m and 2m + 1 at the lowest T (Sokal window, c = 6),
           in iterations; "lower_bound" when the window did not close within the run
  iter     CUDA-event median cost of one iteration (the sweep, the move, the energy record and the exchange pass, as
           parallel_tempering runs them), over --timed iterations after --warm ones
  kernels  device time of the kernels alone, from torch.profiler over --timed back-to-back sweep + move pairs with the
           move's pairs built once: sparse_houdayer_kernel (one move of all pairs of all selected slots) and
           sparse_gibbs_kernel (one sweep of all chains with their energies); and the CUDA-event time per call of
           --timed back-to-back moves (the launch rate, issue overhead included)
  ground   L = 8 only, a few instances: the iteration at which each run first reaches the lowest energy any run found
Run on the GPU: python tools/sparse_houdayer_bench.py [--iters 1000] [--instances 3]
"""

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import scipy.sparse as sp

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

TEMPS = np.geomspace(0.2, 2.0, 16)
K = 32
T_MOVE = 1.0


def ea3d(L, seed):
    """periodic L^3 +-J glass as a symmetric scipy matrix"""
    rng = np.random.default_rng(seed)
    idx = np.arange(L ** 3).reshape(L, L, L)
    a = np.concatenate([idx.ravel()] * 3)
    b = np.concatenate([np.roll(idx, -1, axis=ax).ravel() for ax in range(3)])
    m = sp.coo_matrix((rng.choice([-1.0, 1.0], a.size), (a, b)), shape=(L ** 3, L ** 3)).tocsr()
    return (m + m.T).tocsr()


def tau_int(x, c=6.0):
    """(tau, closed): Sokal's automatic window on the mean autocorrelation of the rows of x [n_series, n_t]"""
    x = x - x.mean(axis=1, keepdims=True)
    n = x.shape[1]
    f = np.fft.rfft(x, 2 * n, axis=1)
    acf = np.fft.irfft(f * np.conj(f), axis=1)[:, :n].mean(axis=0)
    if acf[0] <= 0:
        return 0.5, True
    rho = acf / acf[0]
    tau = 0.5
    for w in range(1, n):
        tau += rho[w]
        if w >= c * tau:
            return float(tau), True
    return float(tau), False


def sampler(seed):
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler

    return GibbsSampler(GibbsConfig(n_burnin=0, n_sweeps=1), seed=seed)


def run_pt(J, iters, seed, moves):
    kw = dict(houdayer_interval=1, houdayer_max_temperature=T_MOVE) if moves else {}
    return sampler(seed).parallel_tempering(J, list(TEMPS), n_samples=iters, swap_interval=1, n_ladders=K,
                                            criterion="metropolis", chromatic=True, **kw)


def timings(J, warm, timed, seed):
    """iteration costs (CUDA-event medians) with and without the move, and the device time of the move and sweep
    kernels alone"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    from tsu_emulator_b200 import _lib
    from tsu_emulator_b200.sparse import SparseProblem

    dev = torch.device("cuda", 0)
    prob = SparseProblem(J, None, dev)
    R, N = TEMPS.size, J.shape[0]
    st = torch.randint(0, 2, (K * R, N), dtype=torch.uint8, device=dev)
    T_slot = torch.from_numpy(TEMPS).to(dev)
    sr = torch.arange(K * R, dtype=torch.int32, device=dev).view(K, R)
    T_chain = T_slot.repeat(K)
    stats = torch.zeros(2, dtype=torch.int64, device=dev)
    slots = torch.from_numpy(np.nonzero(TEMPS <= T_MOVE)[0]).to(dev)
    n_pairs = K // 2 * int(slots.numel())
    counter = [0]

    def sweep():
        counter[0] += 1
        _, e, _, _ = prob.run(st, T=1.0, seed=seed, sweep0=counter[0], chain0=0, n_burnin=1, n_samples=0,
                              sweeps_per_sample=0, T_chain=T_chain, want_energy=True)
        return e

    def pairs_now():
        sel = sr[:, slots]
        return torch.stack((sel[0::2], sel[1::2]), -1).reshape(-1, 2).contiguous()

    def move(pairs, e):
        prob.houdayer(st, pairs, n_pairs, seed=seed, step0=counter[0], n_steps=1, chain0=0, energy=e)

    def iteration(moves):
        e = sweep()
        if moves:
            move(pairs_now(), e)
        _ = e[sr.long()]
        _lib.call("tsu_pt_swap", e.data_ptr(), T_slot.data_ptr(), sr.data_ptr(), None, K, R, seed,
                  counter[0] & 0xFFFFFFFF, stats.data_ptr(), None, 1, _lib.current_stream())
        T_chain[sr.long()] = T_slot

    def median(fn, n):
        ts = []
        for _ in range(n):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        return float(np.median(ts))

    out = {}
    for name, fn in (("iter_us_pt", lambda: iteration(False)), ("iter_us_icm", lambda: iteration(True))):
        median(fn, warm)
        out[name] = median(fn, timed)
    pairs, e = pairs_now(), sweep()

    def back_to_back():
        for _ in range(timed):
            move(pairs, e)

    back_to_back()
    out["move_us_per_call_back_to_back"] = median(back_to_back, 3) / timed

    def sweep_and_move():
        for _ in range(timed):
            move(pairs, sweep())

    sweep_and_move()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sweep_and_move()
        torch.cuda.synchronize()
    dev_us = {"sparse_houdayer_kernel": 0.0, "sparse_gibbs_kernel": 0.0}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            for k in dev_us:
                if k in ev.name:
                    dev_us[k] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
    out["move_kernel_us"] = dev_us["sparse_houdayer_kernel"] / timed
    out["sweep_kernel_us"] = dev_us["sparse_gibbs_kernel"] / timed
    out["n_pairs"] = n_pairs
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=1000, help="iterations of the tau runs at L = 8 (a quarter at L = 16)")
    ap.add_argument("--instances", type=int, default=3, help="L = 8 instances of the ground-state race")
    ap.add_argument("--warm", type=int, default=20)
    ap.add_argument("--timed", type=int, default=200)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    for L, iters in ((8, args.iters), (16, max(args.iters // 4, 50))):
        J = ea3d(L, 100 + L)
        line = {"L": L, "N": L ** 3, "gpu": gpu, "temps": [0.2, 2.0, TEMPS.size], "ladders": K, "iters": iters}
        for moves in (False, True):
            samples, _ = run_pt(J, iters, 7, moves)
            s = 2 * samples[:, iters // 5:].astype(np.int8) - 1          # drop the first fifth as burn-in
            q = (s[0::2].astype(np.int32) * s[1::2]).mean(axis=2)
            tau, closed = tau_int(q * q)
            key = "icm" if moves else "pt"
            line[f"tau_q2_{key}"] = tau if closed else {"lower_bound": tau}
            line[f"q2_mean_{key}"] = float((q * q).mean())
        line.update(timings(J, args.warm, args.timed, 7))
        print(json.dumps(line), flush=True)
    race = []
    for inst in range(args.instances):
        J = ea3d(8, 500 + inst)
        first = {}
        lows = {}
        for moves in (False, True):
            _, info = run_pt(J, args.iters, 11 + inst, moves)
            e = np.asarray(info["energies"])                               # [K, R, iters]
            run_min = np.minimum.accumulate(e.min(axis=(0, 1)))
            lows[moves] = run_min
        best = min(lows[False][-1], lows[True][-1])
        for moves, run_min in lows.items():
            hit = np.nonzero(run_min <= best)[0]
            first["icm" if moves else "pt"] = int(hit[0]) + 1 if hit.size else None
        race.append({"instance": inst, "lowest_energy": float(best), "iterations_to_lowest": first})
    print(json.dumps({"L": 8, "gpu": gpu, "ground_race": race, "iters": args.iters}), flush=True)


if __name__ == "__main__":
    main()
