"""
ctypes binding of libtsu_b200.so (include/tsu_b200.h).

There is no CPU fallback: if the shared library is missing and cannot be built, importing any
compute entry point raises; if no CUDA device is visible, `require_cuda()` raises.
"""

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_uint32, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TSU_B200_LIB") or os.path.join(_HERE, "libtsu_b200.so")

c_uintptr = ctypes.c_size_t  # uintptr_t

TSU_OK = 0
TSU_ERR_INVALID_ARG = -1
TSU_ERR_UNSUPPORTED = -2
TSU_ERR_NO_DEVICE = -3


class TsuNativeError(RuntimeError):
    """a C-ABI call returned a non-zero status"""

    def __init__(self, fn, code, msg):
        super().__init__(f"{fn} failed with status {code}: {msg}")
        self.code = code


# name -> (restype, argtypes); must list every symbol declared in include/tsu_b200.h
SIGNATURES = {
    "tsu_version": (c_int, []),
    "tsu_error_string": (c_char_p, [c_int]),
    "tsu_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "tsu_philox4x32_10_host": (None, [POINTER(c_uint32), POINTER(c_uint32), POINTER(c_uint32)]),
    "tsu_philox_fill_u32": (c_int, [c_void_p, c_uint64, c_uint64, c_uint32, c_uintptr]),
    "tsu_peer_alloc": (c_int, [POINTER(c_void_p), ctypes.c_size_t]),
    "tsu_peer_free": (c_int, [c_void_p]),
    "tsu_peer_get_handle": (c_int, [c_void_p, c_char_p]),
    "tsu_peer_open_handle": (c_int, [c_char_p, POINTER(c_void_p)]),
    "tsu_peer_close_handle": (c_int, [c_void_p]),
    "tsu_peer_read_u32": (c_int, [c_void_p, POINTER(c_uint32)]),
    "tsu_ising2d_reload_tuning": (None, []),
    "tsu_ising2d_words_per_row": (c_int64, [c_int]),
    "tsu_ising2d_state_words": (c_int64, [c_int, c_int]),
    "tsu_ising2d_init_random": (c_int, [c_void_p, c_int, c_int, c_int, c_uint64, c_uint32, c_int, c_uintptr]),
    "tsu_ising2d_pack": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_uintptr]),
    "tsu_ising2d_unpack": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_uintptr]),
    "tsu_ising2d_half_sweep": (
        c_int,
        [c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_uint64,
         c_uint32, c_uint32, c_int, c_void_p, c_void_p, c_int, c_int, c_uintptr],
    ),
    "tsu_ising2d_slab_sweeps_p2p": (
        c_int,
        [c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_uint64, c_uint32, c_int, c_uint32, c_int,
         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_uint32, c_uint32, c_uintptr, c_uintptr],
    ),
    "tsu_ising2d_sweeps": (
        c_int,
        [c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_uint64, c_uint32,
         c_int, c_uint32, c_uintptr],
    ),
    "tsu_ising2d_jit_prepare": (c_int, [POINTER(c_uint32), c_char_p, c_char_p, c_int]),
    "tsu_ising2d_half_sweep_injected": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
         c_void_p, c_void_p, c_uintptr],
    ),
    "tsu_ising2d_observables": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_uintptr],
    ),
    "tsu_ising2d_energy_from_observables": (
        c_int,
        [c_void_p, c_int, c_double, c_double, c_int64, c_int64, c_void_p, c_uintptr],
    ),
    "tsu_ising2d_pack_bonds": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_uintptr]),
    "tsu_ising2d_overlap": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_uintptr]),
    "tsu_ising2d_anneal": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_uint64, c_uint32, c_uint32,
         c_double, c_double, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_uintptr],
    ),
    "tsu_ising2d_population_work_bytes": (c_int64, [c_int, c_int]),
    "tsu_ising2d_population_anneal": (
        c_int,
        [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
         c_void_p, c_uint64, c_uint32, c_uint32, c_double, c_double, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_size_t, c_uintptr],
    ),
    "tsu_ising2d_cluster_work_bytes": (c_int64, [c_int, c_int, c_int]),
    "tsu_ising2d_swendsen_wang": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_uint64, c_uint32,
         c_int, c_uint32, c_void_p, ctypes.c_size_t, c_uintptr],
    ),
    "tsu_dense_gibbs_run": (
        c_int,
        [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_double, c_void_p, c_void_p, c_int, c_int, c_int,
         c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_uint64, c_uint32, c_uint32, c_int,
         c_int, c_uintptr],
    ),
    "tsu_sparse_gibbs_run": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_double, c_void_p,
         c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_uint64, c_uint32,
         c_uint32, c_uintptr],
    ),
    "tsu_dense_energy": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_uintptr]),
    "tsu_dense_init_random": (c_int, [c_void_p, c_int, c_int, c_uint64, c_uint32, c_uintptr]),
    "tsu_dense_gibbs_tc_run": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int, c_int, c_double, c_void_p, c_int, c_uint64, c_uint32, c_uint32, c_void_p,
         c_uintptr],
    ),
    "tsu_dense_tc_debug_fields": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_uintptr]),
    "tsu_dense_tc_energy": (
        c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_uintptr]
    ),
    "tsu_pt_swap": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_uint64, c_uint32, c_void_p, c_void_p, c_int,
         c_uintptr],
    ),
    "tsu_langevin_jit_prepare": (c_int, [c_char_p, c_int, c_int, c_char_p, c_char_p, c_int]),
    "tsu_langevin_run_jit": (
        c_int,
        [c_int, c_void_p, c_int64, c_void_p, c_double, c_int, c_double, c_double, c_double, c_int, c_int, c_uint64,
         c_uint64, c_void_p, c_void_p, c_uintptr],
    ),
    "tsu_langevin_run": (
        c_int,
        [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_int, c_void_p, c_double, c_int, c_double, c_double,
         c_double, c_int, c_int, c_uint64, c_uint64, c_void_p, c_void_p, c_uintptr],
    ),
}

_lib = None


def load(build_if_missing: bool = True):
    """load (building first if the .so is absent and nvcc exists) and type the library."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if not build_if_missing:
            raise ImportError(f"{LIB_PATH} is missing: run `python -m tsu_emulator_b200.build`")
        from . import build as _build

        _build.build()
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.tsu_version() != 2:
        raise ImportError("libtsu_b200.so ABI version mismatch; rebuild with python -m tsu_emulator_b200.build --force")
    _lib = lib
    return lib


def check(fn_name: str, code: int):
    if code == TSU_OK:
        return
    msg = load().tsu_error_string(code).decode()
    if code == TSU_ERR_INVALID_ARG:
        raise ValueError(f"{fn_name}: {msg}")
    raise TsuNativeError(fn_name, code, msg)


def call(fn_name: str, *args):
    """call a status-returning entry point and raise on failure."""
    lib = load()
    check(fn_name, getattr(lib, fn_name)(*args))


def require_cuda():
    """torch CUDA device or a loud failure (no CPU fallback by design)."""
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError(
            "tsu_emulator_b200 needs a CUDA device (B200, sm_100a): there is no CPU fallback. "
            "Use the reference tsu package on CPU-only hosts."
        )
    return torch


def current_stream() -> int:
    import torch

    return int(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """device pointer of a torch tensor (or None -> NULL) for a c_void_p argument.  A plain int: ctypes converts it
    faster than a c_void_p built here, which matters on latency-bound calls (50 x 50 sweeps)."""
    return None if t is None else t.data_ptr()
