"""Argument rules of the lattice Houdayer move (Ising2DEngine.houdayer, tsu_ising2d_houdayer and
LatticeTempering(houdayer_interval=)): they are checked before any device work, so these run without a GPU."""
import ctypes

import numpy as np
import pytest


def bare_engine(bias_mode="physical", is_slab=False, rows=8, cols=8, n_replicas=6, temperatures=(1.0,),
                bond_index=None):
    """an Ising2DEngine with no device state: anything that got past the checks would fail on a missing attribute"""
    import torch

    from tsu_emulator_b200.lattice import Ising2DEngine

    eng = object.__new__(Ising2DEngine)
    eng.bias_mode, eng.is_slab = bias_mode, is_slab
    eng.rows, eng.cols, eng.n_replicas = rows, cols, n_replicas
    eng.temperatures = np.asarray(temperatures, dtype=np.float64)
    eng.bond_index = None if bond_index is None else torch.tensor(bond_index, dtype=torch.int32)
    eng.field = 0.3  # a field is allowed
    return eng


GOOD = [[0, 1], [2, 3]]


def test_engine_rules_raise():
    with pytest.raises(ValueError, match="bias_mode"):
        bare_engine(bias_mode="reference").houdayer(GOOD)
    with pytest.raises(ValueError, match="row-slab"):
        bare_engine(is_slab=True).houdayer(GOOD)
    with pytest.raises(ValueError, match="2\\^31"):
        bare_engine(rows=1 << 16, cols=1 << 15).houdayer(GOOD)


@pytest.mark.parametrize("pairs", [
    [0, 1],                          # not [n_pairs, 2]
    [[0, 1, 2]],
    np.zeros((0, 2), dtype=np.int64),
    [[0.0, 1.0]],                    # not integers
    [[True, False]],
    [["0", "1"]],
])
def test_bad_pair_shapes_and_types_raise(pairs):
    with pytest.raises(ValueError, match="pairs must be integers"):
        bare_engine().houdayer(pairs)


@pytest.mark.parametrize("pairs,match", [
    ([[0, 6]], "lie in"),
    ([[-1, 2]], "lie in"),
    ([[2, 2]], "two different"),
    ([[0, 1], [1, 2]], "disjoint"),
    ([[0, 1], [2, 0]], "disjoint"),
])
def test_bad_pair_indices_raise(pairs, match):
    with pytest.raises(ValueError, match=match):
        bare_engine().houdayer(pairs)


def test_pairs_need_equal_temperatures_and_bond_realisations():
    temps = [1.0, 1.0, 2.0, 2.0, 1.0, 2.0]
    bare_engine(temperatures=temps).houdayer([[0, 1], [2, 3]], n_steps=0)
    with pytest.raises(ValueError, match="temperature"):
        bare_engine(temperatures=temps).houdayer([[0, 1], [3, 4]])
    idx = [0, 0, 1, 1, 2, 0]
    bare_engine(bond_index=idx).houdayer([[0, 5], [3, 2]], n_steps=0)
    with pytest.raises(ValueError, match="bond_index"):
        bare_engine(bond_index=idx).houdayer([[0, 1], [2, 4]])


@pytest.mark.parametrize("n_steps", [-1, 1.0, 2.5, "3", None, True])
def test_bad_step_counts_raise(n_steps):
    with pytest.raises(ValueError, match="n_steps"):
        bare_engine().houdayer(GOOD, n_steps)


def test_zero_steps_do_nothing():
    eng = bare_engine()
    eng.sweep_index = 5
    assert eng.houdayer(np.array(GOOD, dtype=np.int16), np.int64(0)) is eng and eng.sweep_index == 5


def test_abi_rejects_bad_arguments_before_any_cuda_call():
    from tsu_emulator_b200 import _lib

    lib = _lib.load()
    fake = ctypes.c_void_p(256)  # never dereferenced: the arguments are rejected first
    work = int(lib.tsu_ising2d_cluster_work_bytes(1, 8, 8))
    good = dict(state=fake, n_replicas=4, rows=8, cols=8, wrap_rows=1, wrap_cols=1, pairs=fake, n_pairs=2, seed=1,
                sweep0=0, n_steps=2, replica0=0, work=fake, work_bytes=work, stream=0)

    def run(**kw):
        a = dict(good, **kw)
        return lib.tsu_ising2d_houdayer(*a.values())

    bad = _lib.TSU_ERR_INVALID_ARG
    assert run(n_steps=-1) == bad
    for name in ("state", "pairs", "work"):
        assert run(**{name: None}) == bad, name
    assert run(n_pairs=0) == bad
    assert run(n_pairs=-1) == bad
    assert run(n_pairs=3) == bad       # 2 n_pairs > n_replicas
    assert run(n_replicas=5, n_pairs=3) == bad
    assert run(work_bytes=work - 1) == bad  # below one pair
    assert run(work_bytes=0) == bad
    assert run(rows=1 << 16, cols=1 << 15, wrap_rows=0, wrap_cols=0, work_bytes=1 << 62) == bad  # rows * cols >= 2^31
    assert run(n_replicas=0) == bad
    assert run(rows=7) == bad          # periodic rows must be even
    assert run(cols=2) == bad          # a periodic length-2 dimension has no wrap
    assert run(rows=1 << 25, wrap_rows=0) == bad  # rows of the lattice stream
    assert run(n_steps=0, work_bytes=work - 1) == bad  # the rules hold for a no-op too
    assert run(n_steps=0) == _lib.TSU_OK  # a no-op with good arguments touches nothing


def pt_factory(rows=4, cols=4, bond_index=None, called=None):
    """engine factory of a LatticeTempering whose engine holds no device state (see bare_engine)"""
    import torch

    def fac(n_local, replica0, temps_local):
        if called is not None:
            called.append(n_local)
        eng = bare_engine(rows=rows, cols=cols, n_replicas=n_local, temperatures=temps_local, bond_index=bond_index)
        eng.state = torch.zeros((n_local, 2, rows, 4), dtype=torch.int32)
        eng.set_temperature_tables = lambda temps, idx: None
        return eng
    return fac


def test_tempering_rules_raise():
    from tsu_emulator_b200.distributed import LatticeTempering

    temps = [1.0, 2.0]
    for bad in (-1, 1.5, True, "1"):
        with pytest.raises(ValueError, match="houdayer_interval"):
            LatticeTempering(temps, 4, pt_factory(), houdayer_interval=bad)
    called = []
    with pytest.raises(ValueError, match="even n_ladders"):
        LatticeTempering(temps, 3, pt_factory(called=called), houdayer_interval=1)
    assert called == []  # checked before the engine is built
    LatticeTempering(temps, 3, pt_factory(), houdayer_interval=0)  # no cluster moves: any n_ladders
    # ladders 0, 1 share realisation 0 and ladders 2, 3 realisation 1 ...
    LatticeTempering(temps, 4, pt_factory(bond_index=[0, 0, 0, 0, 1, 1, 1, 1]), houdayer_interval=2)
    # ... but not here
    with pytest.raises(ValueError, match="bond realisation"):
        LatticeTempering(temps, 4, pt_factory(bond_index=[0, 0, 1, 1, 2, 2, 3, 3]), houdayer_interval=1)
    with pytest.raises(ValueError, match="bond realisation"):
        LatticeTempering(temps, 2, pt_factory(bond_index=[0, 1, 0, 0]), houdayer_interval=1)
    with pytest.raises(ValueError, match="int32"):
        LatticeTempering(temps, 2, pt_factory(rows=1 << 16, cols=1 << 15), houdayer_interval=1)
