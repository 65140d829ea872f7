"""Edwards-Anderson +-J lattices against the ferromagnet on the same kernels, same process, one JSON line per run.

    python tools/lattice_bonds_bench.py [--quick]

Workloads (the first two time Ising2DEngine.sweep, the third LatticeTempering.step with its exchange passes):
  shared      4096 replicas of 8192^2 sharing one realisation (32 MB of bond words)
  per_replica  256 replicas of 8192^2, one realisation per replica (4 bond bits per site in HBM)
  tempering   16 ladders x 50 temperatures of 1024^2, one realisation per ladder, 10 sweeps per exchange pass
Every workload runs three ways, alternated and repeated: "ferro" (the engine's default choice, the run-time
specialised kernel where it compiles), "ferro_prebuilt" (TSU_B200_NO_JIT: the prebuilt kernel the bonded form is
derived from) and "bonded".  Times are CUDA-event medians.  Reported per line: spin updates/s (kernel rate of the
whole call) and the share of 7.7 TB/s HBM that the byte model implies: 2 bits per update for the state (read the
other colour, write this one) plus, with a realisation per replica, 4 bond bits per update (a shared realisation
stays in L2 and is not counted).  The first line carries the GPU name and power limit read in the same run.
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tsu_emulator_b200 import _lib  # noqa: E402
from tsu_emulator_b200._lib import ptr  # noqa: E402
from tsu_emulator_b200.distributed import LatticeTempering  # noqa: E402
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


def build(kind, make):
    if kind == "ferro_prebuilt":
        os.environ["TSU_B200_NO_JIT"] = "1"
    try:
        return make(kind == "bonded")
    finally:
        os.environ.pop("TSU_B200_NO_JIT", None)


def run(name, make, step, updates_per_step, bond_bits, reps, kinds=("ferro", "ferro_prebuilt", "bonded")):
    objs = {k: build(k, make) for k in kinds}
    for k in kinds:  # warm-up (module load, NVRTC build)
        step(objs[k])
    torch.cuda.synchronize()
    times = {k: [] for k in kinds}
    for _ in range(reps):
        for k in kinds:
            times[k].append(event_time(lambda: step(objs[k])))
    out = []
    for k in kinds:
        t = float(np.median(times[k]))
        rate = updates_per_step / t
        bits = 2 + (bond_bits if k == "bonded" else 0)
        out.append({"workload": name, "kind": k, "seconds_per_call": t, "updates_per_s": rate,
                    "hbm_bytes_per_update": bits / 8, "hbm_share_by_byte_model": rate * bits / 8 / HBM,
                    "spread": [float(min(times[k])), float(max(times[k]))]})
    del objs
    torch.cuda.empty_cache()
    return out


def main():
    quick = "--quick" in sys.argv
    info = gpu_info()
    print(json.dumps(info), flush=True)
    rng = np.random.default_rng(0)
    L = 1024 if quick else 8192
    n_shared, n_per, sweeps = (16, 4, 2) if quick else (4096, 256, 4)
    reps = 3 if quick else 5

    signs1 = rng.choice(np.array([-1, 1], dtype=np.int8), size=(2, L, L))

    def shared(bonded):
        e = Ising2DEngine(L, L, n_replicas=n_shared, temperature=1.0, seed=1, bonds=signs1 if bonded else None)
        return e.init_random()

    for line in run("shared", shared, lambda e: e.sweep(sweeps), sweeps * n_shared * L * L, 0, reps):
        print(json.dumps({**line, **info, "replicas": n_shared, "L": L}), flush=True)

    def per_replica(bonded):
        e = Ising2DEngine(L, L, n_replicas=n_per, temperature=1.0, seed=2,
                          bonds=signs1 if bonded else None, bond_index=np.zeros(n_per, dtype=np.int64) if bonded else None)
        if bonded:  # n_per x 2 L^2 signs would not fit the host as int8: drawn and packed on the device in chunks
            with torch.cuda.device(e.device):
                words = torch.empty((n_per,) + tuple(e.bonds.shape[1:]), dtype=torch.int32, device=e.device)
                gen = torch.Generator(device=e.device).manual_seed(5)
                for k0 in range(0, n_per, 16):
                    k1 = min(n_per, k0 + 16)
                    signs = (2 * torch.randint(0, 2, (k1 - k0, 2, L, L), generator=gen, device=e.device) - 1).to(torch.int8)
                    _lib.call("tsu_ising2d_pack_bonds", ptr(signs), ptr(words[k0:k1]), k1 - k0, L, L, int(e.wrap_rows),
                              int(e.wrap_cols), _lib.current_stream())
                    del signs
                e.bonds = words
                e.bond_index = torch.arange(n_per, dtype=torch.int32, device=e.device)
        return e.init_random()

    for line in run("per_replica", per_replica, lambda e: e.sweep(sweeps), sweeps * n_per * L * L, 4, reps):
        print(json.dumps({**line, **info, "replicas": n_per, "L": L}), flush=True)

    K, R, Lt = (4, 10, 256) if quick else (16, 50, 1024)
    temps = list(np.linspace(0.5, 2.0, R))
    signsT = rng.choice(np.array([-1, 1], dtype=np.int8), size=(K, 2, Lt, Lt))
    ladder = np.arange(K * R) // R

    def tempering(bonded):
        def fac(n_local, replica0, temps_local):
            kw = dict(bonds=signsT, bond_index=ladder[replica0:replica0 + n_local]) if bonded else {}
            return Ising2DEngine(Lt, Lt, n_replicas=n_local, temperature=temps_local, seed=3, replica0=replica0,
                                 **kw).init_random()
        return LatticeTempering(temps, n_ladders=K, engine_factory=fac, n_sweeps=10, swap_interval=1, seed=4)

    for line in run("tempering", tempering, lambda pt: pt.step(), 10 * K * R * Lt * Lt, 4, reps,
                    kinds=("ferro", "bonded")):
        print(json.dumps({**line, **info, "ladders": K, "temperatures": R, "L": Lt}), flush=True)


if __name__ == "__main__":
    main()
