"""Tensor-core dense sweep: time the two tile heights (64 / 128 chains per CTA, forced with TSU_TC_M) at chain counts
where they differ in waves, alternating launches of the two so that drift and neighbours hit both alike.

    python tools/tc_tile_height.py [--n 4096] [--chains 2048,9473,12000,18816] [--sweeps 10] [--reps 30] [--out FILE]

Prints one JSON line: GPU name and power limit, then per chain count the CTAs and waves of each height, the median and
minimum time of one launch of `sweeps` sweeps (CUDA events, after warm-up) for each height and for the launcher's own
choice ("auto"), and whether all of them gave the same bits.
The 32 MB bf16 coupling matrix stays in L2 across launches, as it does in a sampling run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


HEIGHTS = (64, 128, "auto")   # forced tile heights and the launcher's default


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the measurement itself does not depend on it
        return {"gpu": "unknown", "power_limit": f"unknown ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--chains", default="2048,9473,12000,18816")
    ap.add_argument("--sweeps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    from tsu_emulator_b200 import _lib

    torch.manual_seed(0)
    N = a.n
    J = torch.randn(N, N, device="cuda", dtype=torch.float64)
    J = ((J.triu(1) + J.triu(1).T) / N**0.5).to(torch.float32).to(torch.bfloat16).contiguous()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    res = dict(gpu_info(), sms=sms, N=N, sweeps=a.sweeps, reps=a.reps, runs=[])

    def launch(st, m):
        if m == "auto":                      # the launcher's own rule
            os.environ.pop("TSU_TC_M", None)
        else:
            os.environ["TSU_TC_M"] = str(m)  # read by every launch
        _lib.call("tsu_dense_gibbs_tc_run", _lib.ptr(J), None, _lib.ptr(st), int(st.shape[0]), N, 1.0, None, a.sweeps,
                  1234, 0, 0, None, _lib.current_stream())

    for C in [int(c) for c in a.chains.split(",")]:
        init = (torch.rand(C, N, device="cuda") < 0.5).to(torch.uint8)
        outs = {}
        for m in HEIGHTS:                    # warm-up, and the bits of one launch from the same state
            st = init.clone()
            launch(st, m)
            outs[m] = st
        same = all(torch.equal(outs[64], outs[m]) for m in HEIGHTS)
        times = {m: [] for m in HEIGHTS}
        st = init.clone()
        for _ in range(a.reps):
            for m in HEIGHTS:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                launch(st, m)
                e1.record()
                e1.synchronize()
                times[m].append(e0.elapsed_time(e1))
        run = {"chains": C, "same_bits": same}
        for m in HEIGHTS:
            t = sorted(times[m])
            run[f"M{m}"] = {"median_ms": round(t[len(t) // 2], 4), "min_ms": round(t[0], 4)}
            if m != "auto":
                run[f"M{m}"].update(ctas=-(-C // m), waves=-(-C // m // sms))
        res["runs"].append(run)
    os.environ.pop("TSU_TC_M", None)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
