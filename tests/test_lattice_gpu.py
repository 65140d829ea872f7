"""GPU parity: the bit-packed lattice kernels (through the C-ABI) against the CPU oracle and the
reference's golden vectors.  Bit-exact: integer thresholds, no device transcendental."""
import glob
import os

import numpy as np
import pytest

from oracle import ising2d_oracle as O

pytestmark = pytest.mark.gpu


def make_engine(rows, cols, **kw):
    from tsu_emulator_b200.lattice import Ising2DEngine

    return Ising2DEngine(rows, cols, **kw)


def test_pack_unpack_and_layout():
    rng = np.random.default_rng(0)
    for shape in [(1, 1), (3, 5), (7, 50), (4, 64), (5, 65), (2, 300), (6, 512)]:
        bits = rng.integers(0, 2, (2,) + shape)
        eng = make_engine(*shape, n_replicas=2, periodic=False)
        eng.set_spins(bits)
        packed = eng.state.cpu().numpy().view(np.uint32)
        for r in range(2):
            assert (packed[r] == O.pack_spins(bits[r])).all()
        assert (eng.get_spins(pm1=False) == bits).all()
        assert (eng.get_spins(pm1=True) == 2 * bits - 1).all()


def test_init_random_matches_oracle():
    eng = make_engine(6, 70, n_replicas=3, periodic=False, seed=99, replica0=5)
    eng.init_random()
    got = eng.get_spins(pm1=False)
    for r in range(3):
        assert (got[r] == O.init_bits(99, 5 + r, 6, 70)).all()


def test_injected_uniforms_match_reference_goldens(golden_dir):
    paths = sorted(glob.glob(os.path.join(golden_dir, "lattice_*.npz")))
    assert len(paths) >= 9
    for path in paths:
        g = np.load(path)
        R, C = int(g["rows"]), int(g["cols"])
        eng = make_engine(R, C, coupling=float(g["J"]), field=float(g["h"]), temperature=float(g["T"]),
                          periodic=bool(g["periodic"]), bias_mode=str(g["bias_mode"]))
        eng.set_spins(g["bits0"])
        eng.sweep_injected(g["uniforms"])
        out = eng.get_spins(pm1=False)[0]
        assert (out == g["bits_out"]).all(), path
        assert eng.energy()[0] == pytest.approx(float(g["energy"]), abs=1e-9), path
        assert eng.magnetization()[0] == pytest.approx(float(g["magnetization"]), abs=1e-12), path


PHILOX_CASES = [
    # rows, cols, periodic, T, J, h   (fast path needs cols % 256 == 0 and periodic)
    (8, 256, True, 2.269, 1.0, 0.0),
    (6, 512, True, 0.1, 1.0, 0.0),      # p == 1.0 / 0.0 classes (sigmoid clamp)
    (10, 256, True, 2.269, 1.0, 0.2),
    (4, 768, True, 5.0, -1.0, 0.0),
    (50, 50, False, 2.5, 1.0, 0.0),     # BASELINE config 1 geometry (open, IsingGrid default)
    (50, 50, True, 2.5, 1.0, 0.0),
    (7, 5, False, 1.0, 0.7, -0.2),
    (12, 70, True, 2.0, 1.0, 0.1),
    (2, 6, True, 3.0, 1.0, 0.0),
    (1, 9, False, 1.5, 1.0, 0.0),
    (9, 1, False, 1.5, 1.0, 0.2),
    (3, 130, False, 2.269, 1.0, 0.0),
    (10, 256, False, 2.269, 1.0, 0.0),  # open lattices with full words: wide kernel + rim pass
    (64, 512, False, 2.0, 1.0, 0.15),
    (5, 768, False, 3.0, -1.0, 0.0),
    (2, 256, False, 1.5, 1.0, 0.0),     # no row has both vertical neighbours: generic kernel
    (10, 300, True, 2.269, 1.0, 0.0),   # ragged rows: wide kernel on the full 4-word groups + rim pass on the rest
    (9, 1000, False, 2.0, 1.0, 0.1),
    (6, 2050, True, 2.5, -1.0, 0.0),
    (7, 257, False, 1.5, 1.0, 0.0),
    (8, 510, True, 2.0, 1.0, 0.2),
]


@pytest.mark.parametrize("resident", ["1", "0"])   # one-launch resident kernel / one launch per half-sweep
@pytest.mark.parametrize("rows,cols,periodic,T,J,h", PHILOX_CASES)
def test_philox_mode_is_bit_exact_with_oracle(rows, cols, periodic, T, J, h, resident, tuning):
    tuning.setenv("TSU_LATTICE_RESIDENT", resident)
    n_rep, n_sweeps, seed = 2, 3, 1234
    eng = make_engine(rows, cols, n_replicas=n_rep, coupling=J, field=h, temperature=T, periodic=periodic,
                      seed=seed, replica0=7)
    eng.init_random()
    start = eng.get_spins(pm1=False)
    eng.sweep(n_sweeps)
    got = eng.get_spins(pm1=False)
    for r in range(n_rep):
        want = O.checkerboard_sweeps_philox(start[r], seed, 7 + r, 0, n_sweeps, J, h, T, periodic)
        assert (got[r] == want).all(), f"replica {r}: {(got[r] != want).sum()} mismatching spins"
    # continuing from sweep index 3 uses fresh counters
    eng.sweep(2)
    got2 = eng.get_spins(pm1=False)
    want2 = O.checkerboard_sweeps_philox(got[0], seed, 7, n_sweeps, 2, J, h, T, periodic)
    assert (got2[0] == want2).all()


def test_philox_and_injected_paths_agree_on_philox_uniforms():
    """independent implementations inside the library: bit-sliced compare vs per-lane compare"""
    rows, cols, seed = 16, 512, 5
    a = make_engine(rows, cols, temperature=2.269, periodic=True, seed=seed)
    b = make_engine(rows, cols, temperature=2.269, periodic=True, seed=seed)
    a.init_random()
    b.set_spins(a.get_spins())
    a.sweep(4)
    U = np.stack([O.philox_uniform_field(seed, 0, t, rows, cols) for t in range(4)])
    b.sweep_injected(U)
    assert (a.get_spins() == b.get_spins()).all()


def test_stragglers_exercised(tuning):
    """thresholds whose top byte ties often: every lane with top-8-bit tie must use the low bits (wide kernel: the
    tie queue; a lattice this small would otherwise take the resident kernel)"""
    tuning.setenv("TSU_LATTICE_RESIDENT", "0")
    rows, cols, seed = 64, 1024, 77
    eng = make_engine(rows, cols, temperature=2.269, periodic=True, seed=seed)
    eng.init_random()
    start = eng.get_spins(pm1=False)[0]
    eng.sweep(2)
    want = O.checkerboard_sweeps_philox(start, seed, 0, 0, 2, 1.0, 0.0, 2.269, True)
    assert (eng.get_spins(pm1=False)[0] == want).all()
    # 64*1024*2 sweeps = 131072 updates, ~512 expected top-byte ties


def test_per_replica_temperatures():
    temps = [0.5, 2.269, 4.0]
    eng = make_engine(8, 256, n_replicas=3, temperature=temps, periodic=True, seed=3)
    eng.init_random()
    start = eng.get_spins(pm1=False)
    eng.sweep(3)
    got = eng.get_spins(pm1=False)
    for r, T in enumerate(temps):
        want = O.checkerboard_sweeps_philox(start[r], 3, r, 0, 3, 1.0, 0.0, T, True)
        assert (got[r] == want).all()


def test_observables_match_oracle():
    rng = np.random.default_rng(5)
    for (rows, cols, periodic, J, h) in [(8, 256, True, 1.0, 0.0), (7, 5, False, 0.7, -0.2), (50, 50, False, 1.0, 0.3),
                                         (2, 6, True, 1.0, 0.1), (12, 70, True, -1.0, 0.0), (1, 9, False, 1.0, 0.0),
                                         (66, 512, True, 1.0, 0.2), (130, 256, True, -0.5, 0.0), (4, 768, True, 1.0, 0.0),
                                         (66, 512, False, 1.0, 0.2), (3, 256, False, -0.5, 0.1), (1, 256, False, 1.0, 0.0)]:
        bits = rng.integers(0, 2, (2, rows, cols))
        eng = make_engine(rows, cols, n_replicas=2, coupling=J, field=h, periodic=periodic)
        eng.set_spins(bits)
        E, M = eng.energy(), eng.magnetization()
        for r in range(2):
            assert E[r] == pytest.approx(O.energy(bits[r], J, h, periodic), abs=1e-9)
            assert M[r] == pytest.approx(O.magnetization(bits[r]), abs=1e-12)


def test_observables_vector_kernel_equals_generic_kernel(tuning):
    """the 16-byte-vector observables kernel (periodic columns, cols % 256 == 0) against the word-by-word kernel, for a
    whole lattice and for a row slab that gets its lower neighbour rows from another rank (next_rows)"""
    import torch
    rng = np.random.default_rng(9)
    rows, cols = 96, 1024
    bits = rng.integers(0, 2, (3, rows, cols))
    whole = make_engine(rows, cols, n_replicas=3, periodic=True)
    whole.set_spins(bits)
    slab = make_engine(40, cols, n_replicas=3, periodic=True, row0=17, global_rows=rows)   # rows 17..56 of the lattice
    slab.set_spins(bits[:, 17:57, :])
    below = make_engine(2, cols, n_replicas=3, periodic=True, row0=57, global_rows=rows)  # row 57 in the slab's layout
    below.set_spins(bits[:, 57:59, :])
    nxt = below.state[:, :, 0, :].contiguous()
    fast = [whole.observables_tensor().clone(), slab.observables_tensor(next_rows=nxt).clone(),
            slab.observables_tensor(next_rows=None).clone()]
    tuning.setenv("TSU_LATTICE_OBS_GENERIC", "1")
    slow = [whole.observables_tensor().clone(), slab.observables_tensor(next_rows=nxt).clone(),
            slab.observables_tensor(next_rows=None).clone()]
    for f, g in zip(fast, slow):
        assert torch.equal(f, g)
    for r in range(3):
        assert whole.energy()[r] == pytest.approx(O.energy(bits[r], 1.0, 0.0, True), abs=1e-9)


def test_open_lattice_wide_kernel_plus_rim_equals_generic_kernel(tuning):
    """open boundaries (the IsingGrid default) on full-word lattices: wide kernel for the rows with both vertical
    neighbours + rim pass with the true geometry == the word-by-word generic kernel == the oracle; also for a row slab
    that has a neighbour slab on one side only"""
    import torch
    tuning.setenv("TSU_LATTICE_RESIDENT", "0")
    seed = 5
    for rows, cols, periodic in ((66, 1024, False), (40, 1000, True), (33, 1379, False)):
        kw = dict(n_replicas=3, temperature=2.269, periodic=periodic, seed=seed, field=0.1)
        a = make_engine(rows, cols, **kw).init_random()
        start = a.get_spins(pm1=False)
        a.sweep(4)
        tuning.setenv("TSU_LATTICE_OPEN_GENERIC", "1")
        b = make_engine(rows, cols, **kw).init_random()
        b.sweep(4)
        tuning.delenv("TSU_LATTICE_OPEN_GENERIC")
        assert torch.equal(a.state, b.state), (rows, cols, periodic)
        want = O.checkerboard_sweeps_philox(start[2], seed, 2, 0, 4, 1.0, 0.1, 2.269, periodic)
        assert (a.get_spins(pm1=False)[2] == want).all(), (rows, cols, periodic)
    rows, cols = 66, 1024
    a = make_engine(rows, cols, n_replicas=3, temperature=2.269, periodic=False, seed=seed, field=0.1).init_random()
    a.sweep(4)
    # bottom slab of an open lattice: halo above, open edge below
    top = a.state[:, :, 40, :].contiguous()
    for generic in ("", "1"):
        if generic:
            tuning.setenv("TSU_LATTICE_OPEN_GENERIC", "1")
        slab = make_engine(25, cols, n_replicas=3, temperature=2.269, periodic=False, seed=seed, row0=41, global_rows=rows)
        slab.state.copy_(a.state[:, :, 41:66, :])
        for colour in (0, 1):
            slab.half_sweep(colour, halo_top=top[:, 1 - colour, :].contiguous(), halo_bot=None)
        if generic:
            assert torch.equal(slab.state, ref_state)
        else:
            ref_state = slab.state.clone()


def test_large_lattice_properties():
    """BASELINE config 2 geometry at reduced replica count: size-independent checks"""
    eng = make_engine(8192, 8192, n_replicas=2, temperature=2.269, periodic=True, seed=1)
    eng.init_random()
    m0 = eng.magnetization()
    assert np.all(np.abs(m0) < 1e-3)  # iid Bernoulli(1/2) over 6.7e7 spins
    e0 = eng.energy() / eng.n_sites
    assert np.all(np.abs(e0) < 1e-3)
    eng.sweep(10)
    e = eng.energy() / eng.n_sites
    assert np.all(e < -1.0) and np.all(e > -1.6)   # relaxing towards e(T_c) = -sqrt(2)
    # determinism: same seed, same bits
    eng2 = make_engine(8192, 8192, n_replicas=2, temperature=2.269, periodic=True, seed=1)
    eng2.init_random().sweep(10)
    import torch
    assert torch.equal(eng.state, eng2.state)


def test_cold_lattice_stays_ordered_and_hot_disorders():
    eng = make_engine(256, 256, temperature=0.5, periodic=True, seed=2)
    eng.set_spins(np.ones((256, 256)))
    eng.sweep(50)
    assert eng.magnetization()[0] > 0.99
    eng.set_temperature(10.0)
    eng.sweep(50)
    assert abs(eng.magnetization()[0]) < 0.05


def test_jit_specialised_and_prebuilt_kernels_agree(monkeypatch):
    """the NVRTC table-specialised build of the fast kernel and the prebuilt jump-table kernel are the same function"""
    import torch
    rows, cols, seed = 320, 1024, 31   # too large for the resident kernel: the wide kernels do the work
    a = make_engine(rows, cols, n_replicas=3, temperature=2.269, periodic=True, seed=seed)
    assert a._jit == 0                 # small lattice: no automatic compile (1-2 s per temperature would not pay back)
    if not a.specialise():
        pytest.skip("NVRTC specialisation unavailable here: " + getattr(a, "_jit_log", ""))
    small = make_engine(50, 50, temperature=2.269, periodic=True, seed=seed)
    assert not small.specialise()      # the generic kernels have no specialised form
    monkeypatch.setenv("TSU_B200_JIT", "1")   # from here on: compile at set_temperature whatever the size
    monkeypatch.setenv("TSU_B200_NO_JIT", "1")
    b = make_engine(rows, cols, n_replicas=3, temperature=2.269, periodic=True, seed=seed)
    assert b._jit == 0
    a.init_random().sweep(5)
    b.init_random().sweep(5)
    assert torch.equal(a.state, b.state)
    want = O.checkerboard_sweeps_philox(O.init_bits(seed, 1, rows, cols), seed, 1, 0, 5, 1.0, 0.0, 2.269, True)
    assert (a.get_spins(pm1=False)[1] == want).all()
    # a second engine at the same temperature reuses the cached module; a new temperature compiles a new one
    c = make_engine(rows, cols, temperature=2.269, periodic=True, seed=seed)
    monkeypatch.delenv("TSU_B200_NO_JIT")
    d = make_engine(rows, cols, temperature=2.269, periodic=True, seed=seed)
    e = make_engine(rows, cols, temperature=0.1, periodic=True, seed=seed)   # p == 1.0 classes
    assert d._jit == a._jit and e._jit > 0 and e._jit != a._jit
    e.init_random().sweep(3)
    want = O.checkerboard_sweeps_philox(O.init_bits(seed, 0, rows, cols), seed, 0, 0, 3, 1.0, 0.0, 0.1, True)
    assert (e.get_spins(pm1=False)[0] == want).all()


def test_binder_cumulant_crossing_at_tc():
    """statistical parity (SURVEY 8d): the Binder cumulant U4 = 1 - <m^4> / (3 <m^2>^2) of L = 32, 64, 128 periodic
    lattices orders by size below T_c, inverts above, and the curves cross at T_c = 2/ln(1+sqrt 2) = 2.269
    (ising.py:312) within jackknife error bars (replicas are independent Markov chains)."""
    import torch

    temps = (2.24, 2.269, 2.30)
    sizes = {32: (256, 4000, 60, 50), 64: (256, 30000, 60, 250), 128: (128, 120000, 50, 1000)}  # R, n_eq, n_meas, stride
    U, err = {}, {}
    for L, (R, n_eq, n_meas, stride) in sizes.items():
        for T in temps:
            eng = make_engine(L, L, n_replicas=R, temperature=T, periodic=True, seed=1000 * L + int(100 * T))
            eng.init_random()
            eng.sweep(n_eq)
            m2 = torch.zeros(R, dtype=torch.float64, device="cuda")
            m4 = torch.zeros_like(m2)
            for _ in range(n_meas):
                eng.sweep(stride)
                m = (2.0 * eng.observables_tensor()[:, 0].to(torch.float64) - L * L) / (L * L)
                m2 += m * m
                m4 += m ** 4
            m2, m4 = (m2 / n_meas).cpu().numpy(), (m4 / n_meas).cpu().numpy()
            u = lambda a2, a4: 1.0 - a4.mean() / (3.0 * a2.mean() ** 2)
            jk = np.array([u(np.delete(m2, r), np.delete(m4, r)) for r in range(R)])
            U[L, T] = u(m2, m4)
            err[L, T] = np.sqrt((R - 1) / R * ((jk - jk.mean()) ** 2).sum())
    print({k: (round(float(U[k]), 4), round(float(err[k]), 4)) for k in U})
    for a, b in ((32, 64), (64, 128)):
        lo, mid, hi = temps
        sig = lambda T: 4.0 * np.hypot(err[a, T], err[b, T])
        assert U[b, lo] > U[a, lo] - sig(lo), (a, b, U, err)           # ordered side: larger L -> larger U4 (-> 2/3)
        assert U[b, hi] < U[a, hi] + sig(hi), (a, b, U, err)           # disordered side: larger L -> smaller U4 (-> 0)
        # the sign of U_b - U_a flips between 2.24 and 2.30, and at T_c the difference is small against both ends:
        # the crossing lies within +-0.03 of 2.269
        d_lo, d_mid, d_hi = U[b, lo] - U[a, lo], U[b, mid] - U[a, mid], U[b, hi] - U[a, hi]
        assert d_lo > sig(lo) and d_hi < -sig(hi), (a, b, U, err)
        assert abs(d_mid) < 0.35 * min(d_lo, -d_hi) + sig(mid), (a, b, U, err)
    for L in sizes:
        assert abs(U[L, 2.269] - 0.61) < 0.04 + 4.0 * err[L, 2.269], (L, U[L, 2.269], err[L, 2.269])   # U* = 0.6107 (periodic square)


@pytest.mark.parametrize("rows,cols,periodic", [(50, 50, True), (50, 50, False), (37, 61, False), (256, 256, True)])
def test_resident_small_lattice_kernel_matches_per_half_sweep_launches(rows, cols, periodic, tuning):
    """C1-sized lattices run all sweeps of a call in ONE launch (one thread block per replica); the bits must equal
    the launch-per-half-sweep path (TSU_LATTICE_RESIDENT=0) and the oracle"""
    kw = dict(n_replicas=3, temperature=2.5, periodic=periodic, seed=77)
    a = make_engine(rows, cols, **kw)
    a.init_random()
    start = a.get_spins(pm1=False)
    a.sweep(7)
    tuning.setenv("TSU_LATTICE_RESIDENT", "0")
    b = make_engine(rows, cols, **kw)
    b.init_random()
    b.sweep(7)
    got = a.get_spins(pm1=False)
    assert (got == b.get_spins(pm1=False)).all()
    want = O.checkerboard_sweeps_philox(start[1], 77, 1, 0, 7, 1.0, 0.0, 2.5, periodic)
    assert (got[1] == want).all()


@pytest.mark.parametrize("rows,cols,periodic", [(40, 1024, True), (33, 1000, False), (24, 512, False), (12, 70, True),
                                                (9, 50, False)])
def test_row_ranges_compose_to_the_full_half_sweep(rows, cols, periodic, tuning):
    """tsu_ising2d_half_sweep over row ranges: boundary rows, interior and arbitrary splits, launched in any order, give
    the bits of the one-launch half-sweep (what the overlapped row-slab driver relies on)"""
    import torch
    tuning.setenv("TSU_LATTICE_RESIDENT", "0")
    kw = dict(n_replicas=2, temperature=2.269, periodic=periodic, seed=19, field=0.05)
    a = make_engine(rows, cols, **kw).init_random()
    b = make_engine(rows, cols, **kw).init_random()
    splits = [[(rows - 1, rows), (0, 1), (1, rows - 1)], [(0, rows // 3), (rows // 3, rows)], [(5, rows), (0, 5)]]
    for t in range(3):
        for colour in (0, 1):
            a.half_sweep(colour)
            for rng_ in splits[t]:
                b.half_sweep(colour, rows=rng_)
            assert torch.equal(a.state, b.state), (t, colour)
        a.sweep_index += 1
        b.sweep_index += 1
    want = O.checkerboard_sweeps_philox(O.init_bits(19, 1, rows, cols), 19, 1, 0, 3, 1.0, 0.05, 2.269, periodic)
    assert (b.get_spins(pm1=False)[1] == want).all()


def test_two_word_threads_equal_four_word_threads(tuning, monkeypatch):
    """W = 2 (64 spins per thread) and W = 4 (128) builds of the wide kernel, prebuilt and run-time specialised"""
    import torch
    tuning.setenv("TSU_LATTICE_RESIDENT", "0")
    rows, cols, seed = 130, 1536, 3
    ref = make_engine(rows, cols, n_replicas=2, temperature=2.269, periodic=True, seed=seed).init_random().sweep(4)
    tuning.setenv("TSU_LATTICE_W", "2")
    w2 = make_engine(rows, cols, n_replicas=2, temperature=2.269, periodic=True, seed=seed).init_random().sweep(4)
    assert torch.equal(ref.state, w2.state)
    tuning.setenv("TSU_JIT_W", "2")
    j2 = make_engine(rows, cols, n_replicas=2, temperature=2.3, periodic=True, seed=seed)   # a temperature no other test compiles
    if j2.specialise():
        tuning.delenv("TSU_LATTICE_W")
        want = make_engine(rows, cols, n_replicas=2, temperature=2.3, periodic=True, seed=seed).init_random().sweep(4)
        monkeypatch.setenv("TSU_B200_NO_JIT", "1")
        assert want._jit == 0
        j2.init_random().sweep(4)
        assert torch.equal(j2.state, want.state)


@pytest.mark.parametrize("rows,cols,periodic_cols,split", [(1200, 1024, True, 4), (1100, 1000, False, 3), (2100, 512, True, 8),
                                                          (700, 1024, True, 2), (64, 256, True, 0)])
def test_slab_driver_without_neighbours_equals_open_rows(rows, cols, periodic_cols, split, tuning):
    """tsu_ising2d_slab_sweeps_p2p with no rank above or below: interior row ranges on streams of their own, boundary
    rows on the side stream - the bits of the plain sweep of a lattice with open rows"""
    import ctypes

    import torch

    from tsu_emulator_b200 import _lib
    tuning.setenv("TSU_LATTICE_RESIDENT", "0")
    if split:
        tuning.setenv("TSU_LATTICE_SPLIT", str(split))
    kw = dict(n_replicas=2, temperature=2.269, periodic=periodic_cols, seed=23, field=0.02)
    ref = make_engine(rows, cols, **kw)
    ref.wrap_rows = False
    ref.init_random().sweep(5)
    eng = make_engine(rows, cols, **kw)
    eng.wrap_rows = False
    eng.init_random()
    wpr = eng.state.shape[-1]
    halo = torch.zeros(4 * 2 * wpr + 16, dtype=torch.int32, device="cuda")
    flags = halo[4 * 2 * wpr:]
    side = torch.cuda.Stream()
    for n in (2, 3):
        _lib.call("tsu_ising2d_slab_sweeps_p2p", 0, _lib.ptr(eng.state), 2, rows, cols, int(eng.wrap_cols), _lib.ptr(eng.lut),
                  None, eng.seed, eng.sweep_index, n, 0, 0, _lib.ptr(halo), _lib.ptr(flags), None, None, None, None, 0, 0,
                  int(torch.cuda.current_stream().cuda_stream), int(side.cuda_stream))
        eng.sweep_index += n
    torch.cuda.synchronize()
    assert torch.equal(eng.state, ref.state)
    assert int(flags[8]) == 0


@pytest.mark.parametrize("rows,cols,periodic,split", [(2048, 1024, True, 8), (1500, 1000, False, 5), (1024, 512, True, 3),
                                                     (1030, 1026, True, 4)])
def test_row_ranges_on_their_own_streams_equal_one_launch(rows, cols, periodic, split, tuning):
    """TSU_LATTICE_SPLIT: the half-sweeps of tsu_ising2d_sweeps cut into row ranges that only wait for their neighbours
    (what large single lattices do by default) - same bits as one launch per half-sweep, periodic rows included"""
    import torch
    tuning.setenv("TSU_LATTICE_RESIDENT", "0")
    tuning.setenv("TSU_LATTICE_SPLIT", "1")
    kw = dict(n_replicas=2, temperature=2.269, periodic=periodic, seed=29, field=-0.03)
    ref = make_engine(rows, cols, **kw).init_random().sweep(2).sweep(3)
    tuning.setenv("TSU_LATTICE_SPLIT", str(split))
    got = make_engine(rows, cols, **kw).init_random().sweep(2).sweep(3)
    assert torch.equal(got.state, ref.state)
    side = torch.cuda.Stream()      # and from a stream that is not the default one
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got.sweep(2)
    ref.sweep(2)
    torch.cuda.synchronize()
    assert torch.equal(got.state, ref.state)


@pytest.mark.parametrize("periodic,per_replica_T", [(True, False), (False, True), (True, True)])
def test_replica_chunks_on_their_own_streams_equal_one_launch(periodic, per_replica_T, tuning):
    """batches of lattices: chunks of replicas on streams of their own (TSU_LATTICE_SPLIT > 1 forces it on a small
    batch), per-replica threshold tables included - same bits as one launch per half-sweep"""
    import torch
    tuning.setenv("TSU_LATTICE_RESIDENT", "0")
    n_rep, rows, cols = 21, 70, 1024
    temps = list(np.linspace(1.5, 3.5, n_rep)) if per_replica_T else 2.269
    kw = dict(n_replicas=n_rep, temperature=temps, periodic=periodic, seed=31, replica0=5)
    tuning.setenv("TSU_LATTICE_SPLIT", "1")
    ref = make_engine(rows, cols, **kw).init_random().sweep(2).sweep(3)
    for split in (8, 3):
        tuning.setenv("TSU_LATTICE_SPLIT", str(split))
        got = make_engine(rows, cols, **kw).init_random().sweep(2).sweep(3)
        assert torch.equal(got.state, ref.state), split
