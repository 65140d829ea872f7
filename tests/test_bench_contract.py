"""bench.py contract that can be checked without a GPU: the reference arm prints ONE JSON line with the agreed keys
(timing the unmodified reference's GibbsSampler.gibbs_sweep, tsu/gibbs.py:128-162, on the host cores - its literal
port only where no reference tree exists), ranks other than 0 stay silent, and the B200 arm refuses to run without a
CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=e,
                          timeout=600)


def test_reference_arm_prints_one_json_line():
    r = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "spin_updates_per_s" and d["unit"] == "spin-updates/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 0
    assert d["config"]["workload"].startswith("ising2d_8192x8192")
    cb = d["cpu_baseline"]
    from oracle import make_ref
    assert cb["kind"] == ("reference" if make_ref.ref_root() else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "gibbs.py:128-162" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    r = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_b200_arm_needs_a_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = run_bench("--steps", "1", "--warmup", "3", "--no-cpu")
    assert r.returncode != 0 and "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_hold_what_the_timed_steps_computed(tmp_path):
    """--dump-outputs: the same files from run to run, spins equal to the oracle after (warmup + steps) x 10 sweeps on
    the sampled replicas and rows, observables of every replica consistent with them; --steps sets the timed steps"""
    import numpy as np

    from oracle import ising2d_oracle as O

    size, n_rep, steps, warmup, seed, T = 64, 16, 2, 3, 1234, 2.269
    dumps = []
    for k in range(2):
        out = tmp_path / str(k)
        r = run_bench("--size", str(size), "--replicas", str(n_rep), "--steps", str(steps), "--warmup", str(warmup),
                      "--no-cpu", "--no-secondary", "--dump-outputs", str(out))
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads(r.stdout.strip().splitlines()[-1])
        assert d["steps"] == steps and d["gpu_launches"] == steps * 10 * 2
        dumps.append({p.stem: np.load(p) for p in out.glob("*.npy")})
    a, b = dumps
    assert sorted(a) == ["energy", "magnetization", "spins", "spins_replicas", "spins_rows"]
    for name in a:
        assert a[name].dtype in (np.float32, np.float64) and np.array_equal(a[name], b[name]), name
    assert a["magnetization"].shape == a["energy"].shape == (n_rep,)
    rows = a["spins_rows"].astype(np.int64)
    for i, rep in enumerate(a["spins_replicas"].astype(np.int64)):
        want = O.checkerboard_sweeps_philox(O.init_bits(seed, rep, size, size), seed, rep, 0, (warmup + steps) * 10,
                                            1.0, 0.0, T, True)
        assert np.array_equal(a["spins"][i], 2.0 * want[rows] - 1), rep
        assert a["magnetization"][rep] == (2.0 * want.sum() - size * size) / (size * size)
        assert a["energy"][rep] == pytest.approx(O.energy(want, 1.0, 0.0, True), abs=1e-9)
