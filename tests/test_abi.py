"""The C-ABI library builds, loads and exports every symbol declared in include/tsu_b200.h."""
import os
import re

from tsu_emulator_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "tsu_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(tsu_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported_and_typed():
    lib = _lib.load()
    syms = declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in tsu_b200.h but not exported"
        assert s in _lib.SIGNATURES, f"{s} has no ctypes signature"
    assert set(_lib.SIGNATURES) == set(syms)


def test_abi_version_2_and_error_strings():
    lib = _lib.load()
    assert lib.tsu_version() == 2
    assert lib.tsu_error_string(0) == b"ok"
    assert b"invalid" in lib.tsu_error_string(-1)


def test_words_per_row_matches_oracle():
    from oracle.ising2d_oracle import words_per_row

    lib = _lib.load()
    for cols in (1, 2, 5, 50, 63, 64, 65, 256, 8192, 131072):
        assert lib.tsu_ising2d_words_per_row(cols) == words_per_row(cols)
        assert lib.tsu_ising2d_state_words(7, cols) == 2 * 7 * words_per_row(cols)


def test_invalid_arguments_return_error_codes_before_any_cuda_call():
    lib = _lib.load()
    # NULL state pointer is rejected before any CUDA call
    rc = lib.tsu_ising2d_init_random(None, 1, 4, 4, 0, 0, 0, 0)
    assert rc == _lib.TSU_ERR_INVALID_ARG
    rc = lib.tsu_ising2d_sweeps(0, None, 1, 4, 4, 1, 1, None, None, None, None, 0, 0, 1, 0, 0)
    assert rc == _lib.TSU_ERR_INVALID_ARG
