"""Argument rules of the lattice Swendsen-Wang update: they are checked before any device work, so these run without a
GPU."""
import ctypes

import numpy as np
import pytest

from oracle import cluster_oracle as SW


def bare_engine(field=0.0, bias_mode="physical", is_slab=False, rows=8, cols=8):
    """an Ising2DEngine with no device state: anything that got past the checks would fail on a missing attribute"""
    from tsu_emulator_b200.lattice import Ising2DEngine

    eng = object.__new__(Ising2DEngine)
    eng.field, eng.bias_mode, eng.is_slab = field, bias_mode, is_slab
    eng.rows, eng.cols, eng.n_replicas = rows, cols, 4
    return eng


def test_engine_arguments_raise():
    with pytest.raises(ValueError, match="field"):
        bare_engine(field=0.1).swendsen_wang()
    with pytest.raises(ValueError, match="bias_mode"):
        bare_engine(bias_mode="reference").swendsen_wang()
    with pytest.raises(ValueError, match="row-slab"):
        bare_engine(is_slab=True).swendsen_wang()
    with pytest.raises(ValueError, match="2\\^31"):
        bare_engine(rows=1 << 16, cols=1 << 15).swendsen_wang()


@pytest.mark.parametrize("n_steps", [-1, 1.0, 2.5, "3", None, True])
def test_bad_step_counts_raise(n_steps):
    with pytest.raises(ValueError, match="n_steps"):
        bare_engine().swendsen_wang(n_steps)


def test_zero_steps_do_nothing():
    eng = bare_engine()
    eng.sweep_index = 5
    assert eng.swendsen_wang(np.int64(0)) is eng and eng.sweep_index == 5


def test_cluster_threshold():
    from tsu_emulator_b200.lattice import cluster_threshold

    for J, T in [(1.0, 2.269), (-1.0, 1.0), (0.5, 5.0), (1.0, 0.02), (0.0, 1.0)]:
        assert cluster_threshold(J, T) == SW.threshold(J, T)
    assert cluster_threshold(1.0, 0.02) == 1 << 32  # p rounds to 1
    assert cluster_threshold(0.0, 1.0) == 0
    assert cluster_threshold(1.0, 2.0) == int(np.ceil(-np.expm1(-1.0) * 2.0 ** 32))
    with pytest.raises(ValueError):
        cluster_threshold(1.0, 0.0)


def test_work_bytes():
    from tsu_emulator_b200 import _lib

    lib = _lib.load()
    # labels (int32 per site, padded to 16 bytes) + activation and flip words (24 bytes per row and word)
    assert lib.tsu_ising2d_cluster_work_bytes(1, 8, 8) == 256 + 24 * 8 * 4
    assert lib.tsu_ising2d_cluster_work_bytes(3, 50, 50) == 3 * (10000 + 24 * 50 * 4)
    assert lib.tsu_ising2d_cluster_work_bytes(2, 3, 5) == 2 * (64 + 24 * 3 * 4)
    assert lib.tsu_ising2d_cluster_work_bytes(1, 8192, 8192) == 4 * 8192 * 8192 + 24 * 8192 * 128
    assert lib.tsu_ising2d_cluster_work_bytes(0, 8, 8) == 0
    assert lib.tsu_ising2d_cluster_work_bytes(1, 0, 8) == 0
    assert lib.tsu_ising2d_cluster_work_bytes(1, 46341, 46341) == 0  # labels are int32


def test_abi_rejects_bad_arguments_before_any_cuda_call():
    from tsu_emulator_b200 import _lib

    lib = _lib.load()
    fake = ctypes.c_void_p(256)  # never dereferenced: the arguments are rejected first
    work = int(lib.tsu_ising2d_cluster_work_bytes(1, 8, 8))
    good = dict(state=fake, n_replicas=4, rows=8, cols=8, wrap_rows=1, wrap_cols=1, thresholds=fake, lut_index=None,
                sign=1, bonds=None, bond_index=None, seed=1, sweep0=0, n_steps=2, replica0=0, work=fake,
                work_bytes=work, stream=0)

    def run(**kw):
        a = dict(good, **kw)
        return lib.tsu_ising2d_swendsen_wang(*a.values())

    bad = _lib.TSU_ERR_INVALID_ARG
    assert run(n_steps=-1) == bad
    for name in ("state", "thresholds", "work"):
        assert run(**{name: None}) == bad, name
    assert run(work_bytes=work - 1) == bad  # below one replica
    assert run(work_bytes=0) == bad
    for sign in (0, 2, -2):
        assert run(sign=sign) == bad
    assert run(rows=1 << 16, cols=1 << 15, wrap_rows=0, wrap_cols=0, work_bytes=1 << 62) == bad  # rows * cols >= 2^31
    assert run(n_replicas=0) == bad
    assert run(rows=7) == bad          # periodic rows must be even
    assert run(cols=2) == bad          # a periodic length-2 dimension has no wrap
    assert run(rows=1 << 25, wrap_rows=0) == bad  # rows of the lattice stream
    assert run(bond_index=fake) == bad  # a bond index needs bond words
    assert run(n_steps=0, work_bytes=work - 1) == bad  # the rules hold for a no-op too
