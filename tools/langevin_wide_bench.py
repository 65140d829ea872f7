"""Throughput of the Langevin kernels above 64 coordinates (csrc/langevin_wide.cu), one JSON line per configuration.

    python tools/langevin_wide_bench.py [--quick]

Every line carries the GPU name and power limit read in the same run.  Times are CUDA-event medians of whole
tsu_langevin_run calls (Philox noise, no trajectory) after one warm-up call, repeated until 0.5 s have been timed.
Reported: chain-steps/s and coordinate-updates/s; for QUADRATIC_FORM also the achieved FLOP/s (2 dim^2 per
chain-step) against cuBLAS GEMM (torch.matmul, TF32 off) measured on the same card in the same run, and against
NVIDIA's HGX B200 data-sheet FP64 rate (296 TFLOP/s for eight GPUs: 37 TFLOP/s for one).  The last lines time the
register kernel at dim 64 and the wide kernel at dim 65: the cost at the boundary.
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

QUADRATIC, MIXTURE, DOUBLE_WELL, QUADRATIC_FORM = 0, 1, 2, 3
NAMES = {QUADRATIC: "quadratic", MIXTURE: "mixture", DOUBLE_WELL: "double_well", QUADRATIC_FORM: "quadratic_form"}
DATASHEET_FP64 = 37e12


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, check=True).stdout.splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unknown ({e})"}


def params_for(kind, dim, rng):
    if kind == QUADRATIC:
        return np.concatenate([[1.0], np.zeros(dim), np.ones(dim)])
    if kind == DOUBLE_WELL:
        return np.array([1.0, 1.0])
    if kind == MIXTURE:
        K = 8
        return np.concatenate([[K], np.full(K, 1.0 / K), 0.1 * rng.normal(size=K * dim)])
    A = np.eye(dim) + 0.1 * rng.normal(size=(dim, dim)) / np.sqrt(dim)
    return np.concatenate([A.ravel(), np.zeros(dim)])


def time_calls(fn, min_total=0.5, max_reps=50):
    fn()
    torch.cuda.synchronize()
    times = []
    while sum(times) < min_total * 1e3 and len(times) < max_reps:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)) * 1e-3, len(times)


def run(kind, dim, n_chains, steps, dtype, info, gemm_rate, note=None):
    rng = np.random.default_rng(dim)
    tdt = torch.float64 if dtype == "float64" else torch.float32
    p = torch.from_numpy(params_for(kind, dim, rng)).cuda()
    x0 = torch.zeros(dim, dtype=tdt, device="cuda")
    x = torch.empty((n_chains, dim), dtype=tdt, device="cuda")

    def call():
        _lib.call("tsu_langevin_run", ptr(x), 1 if dtype == "float64" else 0, n_chains, dim, kind, ptr(p),
                  int(p.numel()), ptr(x0), 0.1, 1, 1.0, 0.01, 1.0, 0, steps, 1, 0, None, None,
                  _lib.current_stream())

    t, reps = time_calls(call)
    assert torch.isfinite(x).all()
    line = dict(info, kernel="register" if dim <= 64 else "wide", energy=NAMES[kind], dtype=dtype, dim=dim,
                chains=n_chains, steps=steps, reps=reps, seconds_per_call=t,
                chain_steps_per_s=n_chains * steps / t, coordinate_updates_per_s=n_chains * steps * dim / t)
    if kind == QUADRATIC_FORM:
        flops = 2.0 * dim * dim * n_chains * steps / t
        line.update(flop_per_s=flops, cublas_gemm_flop_per_s=gemm_rate[dtype], share_of_cublas_gemm=flops / gemm_rate[dtype])
        if dtype == "float64":
            line.update(share_of_datasheet_fp64=flops / DATASHEET_FP64)
    if note:
        line["note"] = note
    print(json.dumps(line), flush=True)
    del x, p


def gemm_rates():
    torch.backends.cuda.matmul.allow_tf32 = False
    out = {}
    for dtype, tdt in (("float64", torch.float64), ("float32", torch.float32)):
        n = 8192
        a = torch.randn(n, n, dtype=tdt, device="cuda")
        b = torch.randn(n, n, dtype=tdt, device="cuda")
        t, _ = time_calls(lambda: torch.matmul(a, b), min_total=1.0, max_reps=20)
        out[dtype] = 2.0 * n ** 3 / t
        del a, b
    return out


def main():
    quick = "--quick" in sys.argv
    _lib.require_cuda()
    info = gpu_info()
    gemm = gemm_rates()
    print(json.dumps(dict(info, cublas_gemm_flop_per_s=gemm, gemm_shape="8192^3, TF32 off")), flush=True)
    big = 10000 if quick else 100000
    configs = [
        (QUADRATIC, 128, big, 100), (QUADRATIC, 1024, big, 50), (QUADRATIC, 8192, 10000, 50),
        (DOUBLE_WELL, 128, big, 100), (DOUBLE_WELL, 1024, big, 50), (DOUBLE_WELL, 8192, 10000, 50),
        (QUADRATIC_FORM, 256, big, 20), (QUADRATIC_FORM, 1024, big, 4), (QUADRATIC_FORM, 2048, 10000, 4),
        (MIXTURE, 1024, big, 10),
    ]
    for kind, dim, chains, steps in configs:
        for dtype in ("float64", "float32"):
            run(kind, dim, chains, steps, dtype, info, gemm)
    for kind, steps in ((QUADRATIC, 100), (QUADRATIC_FORM, 50), (MIXTURE, 50)):
        for dtype in ("float64", "float32"):
            for dim in (64, 65):
                run(kind, dim, big, steps, dtype, info, gemm, note="boundary")


if __name__ == "__main__":
    main()
