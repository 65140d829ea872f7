"""Houdayer cluster moves on the lattice kernels (Ising2DEngine.houdayer, LatticeTempering(houdayer_interval=)) against
heat-bath sweeps on the same engine, same process, one JSON line per workload.

    python tools/lattice_houdayer_bench.py [--quick]

Step time (2-D +-J, one shared realisation, periodic, T = 0.5; CUDA-event medians of alternated runs; the pairs start
from independent random states after 20 sweeps, so about half of the sites differ):
  a  64 pairs of 1024^2, four launches per step                    (--quick: 16 pairs)
  b  74 pairs of 50 x 50, one launch per call (10 steps per call)
Each line gives the Houdayer step time, the sweep time of all replicas, their ratio and the summed time of every
kernel of one call from torch.profiler, by name.

Physics payoff: replica exchange (LatticeTempering, one sweep and one exchange pass per iteration) of L = 32 +-J lattices
at 16 temperatures from 0.2 to 1.6 (geometric), 32 ladders, one realisation per ladder pair, with and without
houdayer_interval = 1.  The series of q^2 of the two slot-0 replicas of every ladder pair (2^16 iterations, the first
quarter dropped; --quick: 2^13), the integrated autocorrelation time with Sokal's windowed estimator (averaged
autocorrelation function, smallest W with W >= 6 tau(W)), the time per iteration (CUDA events around 500 iterations,
the exchange pass's host sync included) and the time per independent sample, 2 tau x iteration time.  The GPU name and
power limit are read in the same run.
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from lattice_cluster_bench import event_time, gpu_info, kernel_times, tau_int  # noqa: E402
from tsu_emulator_b200.distributed import LatticeTempering  # noqa: E402
from tsu_emulator_b200.lattice import Ising2DEngine  # noqa: E402


def signs(rng, *shape):
    return rng.choice(np.array([-1, 1], dtype=np.int8), size=shape)


def step_workload(name, n_pairs, L, per_call, reps, info):
    eng = Ising2DEngine(L, L, n_replicas=2 * n_pairs, temperature=0.5, periodic=True, seed=1,
                        bonds=signs(np.random.default_rng(1), 2, L, L))
    eng.init_random()
    eng.sweep(20)
    pairs = np.arange(2 * n_pairs).reshape(n_pairs, 2)
    eng.houdayer(pairs, per_call)  # warm-up: workspace, modules
    eng.sweep(per_call)
    torch.cuda.synchronize()
    diff = float(1.0 - eng.overlap(pairs).mean()) / 2
    t_h, t_s = [], []
    for _ in range(reps):
        t_h.append(event_time(lambda: eng.houdayer(pairs, per_call)) / per_call)
        t_s.append(event_time(lambda: eng.sweep(per_call)) / per_call)
    h, s = float(np.median(t_h)), float(np.median(t_s))
    return dict(info, workload=name, pairs=n_pairs, L=L, differing_fraction=diff, houdayer_step_s=h, sweep_s=s,
                ratio=h / s, kernels_s=kernel_times(lambda: eng.houdayer(pairs, per_call)), steps_per_call=per_call)


def q2_series(pt, n):
    """[n_ladders / 2, n] series of q^2 of the slot-0 replicas of ladders 2m and 2m+1 after every iteration (device
    popcounts, one host transfer at the end)"""
    eng = pt.engine
    pop = torch.tensor([bin(v).count("1") for v in range(256)], dtype=torch.int64, device=eng.device)
    out = torch.empty((n, pt.K // 2), dtype=torch.float64, device=eng.device)
    for t in range(n):
        pt.step()
        r0 = pt.slot_replica[:, 0].long()
        x = torch.bitwise_xor(eng.state[r0[0::2]], eng.state[r0[1::2]])
        d = pop[x.reshape(x.shape[0], -1).contiguous().view(torch.uint8).long()].sum(dim=1)
        q = 1.0 - 2.0 * d.to(torch.float64) / eng.n_sites
        out[t] = q * q
    return out.cpu().numpy().T


def payoff(L, temps, K, n_iter, houdayer_interval, info):
    rng = np.random.default_rng(7)
    real = signs(rng, K // 2, 2, L, L)
    R = len(temps)
    index = (np.arange(K * R) // (2 * R)).astype(np.int32)  # ladder k uses realisation k // 2

    def fac(n_local, replica0, temps_local):
        eng = Ising2DEngine(L, L, n_replicas=n_local, temperature=temps_local, periodic=True, seed=3,
                            replica0=replica0, bonds=real, bond_index=index[replica0:replica0 + n_local])
        eng.init_random()
        return eng

    pt = LatticeTempering(temps, n_ladders=K, engine_factory=fac, n_sweeps=1, swap_interval=1, seed=5,
                          houdayer_interval=houdayer_interval)
    for _ in range(100):  # warm-up: modules, workspace
        pt.step()
    t_iter = float(np.median([event_time(lambda: [pt.step() for _ in range(500)]) / 500 for _ in range(5)]))
    q2 = q2_series(pt, n_iter)
    keep = n_iter // 4
    tau, window = tau_int(q2[:, keep:])
    return dict(info, workload=f"tempering L={L} houdayer_interval={houdayer_interval}", L=L, ladders=K,
                temperatures=[float(t) for t in temps], iterations=n_iter, iteration_s=t_iter, tau_q2=tau,
                window_q2=window, mean_q2=float(q2[:, keep:].mean()), s_per_independent_sample=2 * tau * t_iter)


def main():
    quick = "--quick" in sys.argv
    torch.cuda.set_device(0)
    info = gpu_info()
    print(json.dumps(step_workload("a", 16 if quick else 64, 1024, 1, 3 if quick else 10, info)), flush=True)
    print(json.dumps(step_workload("b", 74, 50, 10, 10, info)), flush=True)
    temps = np.geomspace(0.2, 1.6, 16)
    n_iter = (1 << 13) if quick else (1 << 16)
    for k in (0, 1):
        print(json.dumps(payoff(32, temps, 32, n_iter, k, info)), flush=True)


if __name__ == "__main__":
    main()
