"""Population annealing on GibbsSampler (population_annealing) against its parts, same process, one JSON line per
workload.

    python tools/dense_population_bench.py [--quick]

Workloads (10 steps per call, from T = 3 down to T = 0.5, one population unless stated):
  a  SK, N = 4096, Gaussian couplings in bf16 (tensor cores), 18944 chains (one 128-chain tile per SM), theta = 1 and 10
  b  SK, N = 1024 in bf16, 16 populations x 4096 chains, theta = 10
  c  chromatic CSR, periodic 8 x 8 x 8 Edwards-Anderson +-J, 8 populations x 1024 chains, theta = 10
Each line gives CUDA-event medians of alternated runs: one population_annealing call, the coupling upload every call
starts with (GibbsSampler builds its problem per call), the PA step ((call - upload) / steps), theta sweeps alone, the
energy pass alone and the resampling (tsu_population_resample) alone; the summed time of every kernel of one PA call from
torch.profiler in a separate run; the resampling's byte model at 7.7 TB/s (24 B per chain for the energies, weights and
prefix sums, 2 row_bytes per chain for the gather) and the energy pass's FLOP count (2 N^2 per chain dense, 2 nnz
sparse).  The GPU name and power limit are read in the same run.
"""
import itertools
import json
import os
import subprocess
import sys
from collections import defaultdict

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tsu_emulator_b200 import GibbsSampler, _lib  # noqa: E402
from tsu_emulator_b200._lib import ptr  # noqa: E402

HBM = 7.7e12
STEPS = 10


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
            name = ev.name.replace("(anonymous namespace)::", "").removeprefix("void ").split("(")[0].split("<")[0]
            out[name] += ev.device_time_total * 1e-6 if hasattr(ev, "device_time_total") else ev.cuda_time_total * 1e-6
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def sk(N, seed):
    rng = np.random.default_rng(seed)
    J = np.triu(rng.standard_normal((N, N)), 1)
    return (J + J.T) / np.sqrt(N)


def ea_csr(L, seed):
    """periodic L^3 +-J couplings as a CSR tuple"""
    import scipy.sparse as sp

    rng = np.random.default_rng(seed)
    rows, cols = [], []
    for x, y, z in itertools.product(range(L), repeat=3):
        i = (x * L + y) * L + z
        for j in (((x + 1) % L * L + y) * L + z, (x * L + (y + 1) % L) * L + z, (x * L + y) * L + (z + 1) % L):
            rows.append(i)
            cols.append(j)
    v = rng.choice([-1.0, 1.0], len(rows))
    m = sp.coo_matrix((v, (rows, cols)), shape=(L ** 3, L ** 3)).tocsr()
    m = (m + m.T).tocsr()
    m.sort_indices()
    return (m.indptr, m.indices, m.data, L ** 3), int(m.nnz)


def workload(name, coupling, precision, chromatic, C, P, theta, reps, info, nnz=None):
    Ts = list(np.geomspace(3.0, 0.5, STEPS))
    smp = GibbsSampler(seed=1, precision=precision)
    run = lambda: smp.population_annealing(coupling, Ts, n_chains=C, n_populations=P, sweeps_per_step=theta,
                                           chromatic=chromatic)
    res = run()  # warm-up: modules, allocator
    prob = smp._problem(coupling, None, chromatic=chromatic, tensor_ok=True)
    st = smp._initial_states(prob, C)
    row_bytes = int(st.shape[1])
    other, fam, fam2 = torch.empty_like(st), res.family.clone(), torch.empty_like(res.family)
    energy = res.energy.clone()
    work_bytes = int(_lib.load().tsu_ising2d_population_work_bytes(C, P))
    work = torch.empty(work_bytes // 8, dtype=torch.int64, device=st.device)
    dbeta = torch.tensor([0.2], dtype=torch.float64, device=st.device)
    ws = torch.empty(P, dtype=torch.int64, device=st.device)
    er = torch.empty(P, dtype=torch.float64, device=st.device)

    def sweeps():
        for _ in range(STEPS):
            smp._run(prob, st, n_burnin=theta, n_samples=0, sweeps_per_sample=0, T=1.0, chain0=0)

    def energies():
        for _ in range(STEPS):
            smp._run(prob, st, n_burnin=0, n_samples=0, sweeps_per_sample=0, T=1.0, chain0=0, want_energy=True)

    def resamples():
        for k in range(STEPS):
            _lib.call("tsu_population_resample", ptr(st), ptr(other), ptr(fam), ptr(fam2), ptr(energy), ptr(dbeta), C,
                      P, row_bytes, 1, k, 0, ptr(ws), ptr(er), ptr(work), work_bytes, _lib.current_stream())

    upload = lambda: smp._problem(coupling, None, chromatic=chromatic, tensor_ok=True)
    sweeps(), energies(), resamples(), upload()
    t = defaultdict(list)
    for _ in range(reps):
        t["call"].append(event_time(run))
        t["upload"].append(event_time(upload))
        t["sweeps"].append(event_time(sweeps) / STEPS)
        t["energy"].append(event_time(energies) / STEPS)
        t["resample"].append(event_time(resamples) / STEPS)
    kern = kernel_times(run)
    med = {k: float(np.median(v)) for k, v in t.items()}
    med["pa"] = (med["call"] - med["upload"]) / STEPS
    N = res.n_sites
    model_resample = (24.0 + 2.0 * row_bytes) * C / HBM
    energy_flop = 2.0 * (nnz if chromatic else N * N) * C
    line = {
        **info, "workload": name, "backend": res.backend, "N": N, "chains": C, "n_populations": P,
        "sweeps_per_step": theta, "steps_per_call": STEPS, "call_s": med["call"], "coupling_upload_s": med["upload"],
        "pa_step_s": med["pa"], "sweeps_per_step_s": med["sweeps"],
        "energy_pass_s": med["energy"], "resample_s": med["resample"],
        "pa_step_over_sweeps": med["pa"] / med["sweeps"], "non_sweep_s": med["pa"] - med["sweeps"],
        "model_resample_s": model_resample, "resample_share_of_hbm": model_resample / med["resample"],
        "energy_flop": energy_flop, "energy_flop_per_s": energy_flop / med["energy"],
        "spread": {k: [min(v), max(v)] for k, v in t.items()},
        "kernels_one_call_s": {k: round(v, 7) for k, v in kern.items()},
    }
    print(json.dumps(line), flush=True)
    del smp, prob, st, other, res
    torch.cuda.empty_cache()


def main():
    quick = "--quick" in sys.argv
    info = gpu_info()
    print(json.dumps(info), flush=True)
    reps = 3 if quick else 7
    J = sk(4096, 1)
    C = 2048 if quick else 18944
    for theta in (1, 10):
        workload(f"a theta={theta}", J, "bf16", False, C, 1, theta, reps, info)
    workload("b", sk(1024, 2), "bf16", False, 16 * (512 if quick else 4096), 16, 10, reps, info)
    coupling, nnz = ea_csr(8, 3)
    workload("c", coupling, "float64", True, 8 * (128 if quick else 1024), 8, 10, reps, info, nnz=nnz)


if __name__ == "__main__":
    main()
