"""Argument rules of the Houdayer move on sparse couplings (tsu_sparse_houdayer and
GibbsSampler.parallel_tempering(houdayer_interval=, chromatic=)): they are checked before any device work, so these run
without a GPU."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp


def ring(N=8, asymmetric=False):
    """a +-1 ring; asymmetric: one coupling of the transpose changed"""
    J = np.zeros((N, N))
    i = np.arange(N)
    J[i, (i + 1) % N] = J[(i + 1) % N, i] = 1.0
    if asymmetric:
        J[1, 0] = 0.5
    return J


def sampler(precision="float64"):
    from tsu_emulator_b200 import GibbsSampler

    return GibbsSampler(seed=1, precision=precision)


@pytest.mark.parametrize("interval", [-1, 1.5, True, "1", None])
def test_bad_intervals_raise(interval):
    with pytest.raises(ValueError, match="houdayer_interval"):
        sampler().parallel_tempering(ring(), [1.0, 2.0], n_samples=1, n_ladders=2, chromatic=True,
                                     houdayer_interval=interval)


def test_tempering_rules_raise():
    pt = sampler().parallel_tempering
    with pytest.raises(ValueError, match="chromatic=True"):
        pt(ring(), [1.0, 2.0], n_samples=1, n_ladders=2, houdayer_interval=1)
    for K in (1, 3):
        with pytest.raises(ValueError, match="even"):
            pt(ring(), [1.0, 2.0], n_samples=1, n_ladders=K, chromatic=True, houdayer_interval=1)
    for t in (0.0, -1.0, float("nan")):
        with pytest.raises(ValueError, match="houdayer_max_temperature"):
            pt(ring(), [1.0, 2.0], n_samples=1, n_ladders=2, chromatic=True, houdayer_interval=1,
               houdayer_max_temperature=t)
    with pytest.raises(ValueError, match="symmetric"):
        pt(ring(asymmetric=True), [1.0, 2.0], n_samples=1, n_ladders=2, chromatic=True, houdayer_interval=2)
    # the structure counts too: an explicit zero on one side only
    J = sp.csr_matrix(ring())
    J.data[0] = 0.0
    with pytest.raises(ValueError, match="symmetric"):
        pt(J, [1.0, 2.0], n_samples=1, n_ladders=2, chromatic=True, houdayer_interval=1)
    with pytest.raises(ValueError, match="'float64' sampler"):
        sampler("float32").parallel_tempering(ring(), [1.0, 2.0], n_samples=1, chromatic=True)
    with pytest.raises(ValueError, match="parity mode"):
        pt(ring(), [1.0, 2.0], n_samples=1, chromatic=True, _inject={})


def test_symmetry_check():
    from tsu_emulator_b200.sparse import is_symmetric_csr, to_csr

    rng = np.random.default_rng(0)
    A = sp.random(40, 40, density=0.1, random_state=1)
    S = (A + A.T).tocsr()
    S.setdiag(rng.normal(size=40))   # self couplings are symmetric by themselves
    assert is_symmetric_csr(*to_csr(S))
    assert not is_symmetric_csr(*to_csr(A))
    assert is_symmetric_csr(*to_csr(ring()))
    assert is_symmetric_csr(*to_csr(np.zeros((5, 5))))


def test_abi_rejects_bad_arguments_before_any_cuda_call():
    from tsu_emulator_b200 import _lib

    lib = _lib.load()
    fake = ctypes.c_void_p(256)  # never dereferenced: the arguments are rejected first
    big = 64000
    work = int(lib.tsu_sparse_houdayer_work_bytes(1, big))
    assert work >= 4 * big and work % 16 == 0
    assert int(lib.tsu_sparse_houdayer_work_bytes(3, big)) == 3 * work
    assert int(lib.tsu_sparse_houdayer_work_bytes(1, 32768)) == 0      # labels in shared memory
    assert int(lib.tsu_sparse_houdayer_work_bytes(1, 204801)) == 0     # beyond the sweep kernel
    assert int(lib.tsu_sparse_houdayer_work_bytes(0, big)) == 0
    good = dict(rowptr=fake, col=fake, val=fake, bias=None, state=fake, n_chains=4, N=100, pairs=fake, n_pairs=2,
                seed=1, step0=0, n_steps=2, chain0=0, energy=None, work=None, work_bytes=0, stream=0)

    def run(**kw):
        a = dict(good, **kw)
        return lib.tsu_sparse_houdayer(*a.values())

    bad = _lib.TSU_ERR_INVALID_ARG
    for name in ("rowptr", "col", "val", "state", "pairs"):
        assert run(**{name: None}) == bad, name
    assert run(n_steps=-1) == bad
    assert run(n_pairs=0) == bad
    assert run(n_pairs=-1) == bad
    assert run(n_pairs=3) == bad              # 2 n_pairs > n_chains
    assert run(n_chains=5, n_pairs=3) == bad
    assert run(N=0) == bad
    assert run(N=204801) == bad               # above the sweep kernel's cap
    assert run(N=big) == bad                  # labels in the workspace: none given
    assert run(N=big, work=fake, work_bytes=work - 1) == bad   # below one pair
    assert run(N=big, work_bytes=work) == bad  # a size without a buffer
    for off in (4, 8):                         # labels need a 16-byte aligned workspace
        assert run(N=big, work=ctypes.c_void_p(256 + off), work_bytes=work) == bad
    assert run(n_steps=0, N=big) == bad       # the rules hold for a no-op too
    assert run(n_steps=0) == _lib.TSU_OK      # a no-op with good arguments touches nothing
    assert run(n_steps=0, N=big, work=fake, work_bytes=work) == _lib.TSU_OK
