"""Limits of the Langevin sampler above 64 coordinates: they are checked before any device work, so these run
without a GPU."""
import ctypes

import numpy as np
import pytest


def test_traced_energy_above_64_coordinates_raises():
    from tsu_emulator_b200 import SamplingError, ThermalSamplingUnit

    with pytest.raises(SamplingError, match="traced Python energies are limited to 64 coordinates") as exc:
        ThermalSamplingUnit().sample_from_energy(lambda x: float(np.sum(np.cos(x))), np.zeros(65), 2)
    assert "quadratic forms" in str(exc.value) and "built-in energies" in str(exc.value)
    from tsu_emulator_b200.core import TracedEnergy

    traced = TracedEnergy(lambda x: np.sum(np.cos(x)), 65, np.zeros(65))
    with pytest.raises(SamplingError, match="limited to 64 coordinates"):
        ThermalSamplingUnit().sample_from_energy(traced, np.zeros(65), 2)


@pytest.mark.parametrize("dtype,cap", [("float64", 131072), ("float32", 262144)])
def test_each_kind_past_its_cap_raises(dtype, cap):
    from tsu_emulator_b200 import (DoubleWellEnergy, GaussianEnergy, MixtureEnergy, QuadraticEnergy,
                                   QuadraticFormEnergy, SamplingError, ThermalSamplingUnit)

    tsu = ThermalSamplingUnit(dtype=dtype)
    for energy in (QuadraticEnergy(), GaussianEnergy(), DoubleWellEnergy(), "double_well"):
        with pytest.raises(SamplingError, match=str(cap)):
            tsu.sample_from_energy(energy, np.zeros(cap + 1), 2)
    with pytest.raises(SamplingError, match=str(cap)):
        tsu.sample_from_energy(MixtureEnergy(np.zeros((2, cap + 1)), [1, 1]), np.zeros(cap + 1), 2)
    with pytest.raises(SamplingError, match="2048"):
        tsu.sample_from_energy(QuadraticFormEnergy(np.ones((2049, 2049)), np.zeros(2049)), np.zeros(2049), 2)
    with pytest.raises(SamplingError, match="16 centres"):
        tsu.sample_from_energy(MixtureEnergy(np.zeros((17, 65)), np.ones(17)), np.zeros(65), 2)
    assert tsu.sample_count == 0


def test_abi_rejects_dims_past_the_caps():
    from tsu_emulator_b200 import _lib

    lib = _lib.load()
    fake = ctypes.c_void_p(256)  # never dereferenced: the arguments are rejected first

    def run(dtype, dim, kind, n_params):
        return lib.tsu_langevin_run(fake, dtype, 4, dim, kind, fake, n_params, None, 0.1, 1, 1.0, 0.01, 1.0, 1, 1, 1,
                                    0, None, None, 0)

    bad = _lib.TSU_ERR_INVALID_ARG
    assert run(1, 131073, 0, 1 + 2 * 131073) == bad    # QUADRATIC, float64
    assert run(0, 262145, 0, 1 + 2 * 262145) == bad    # QUADRATIC, float32
    assert run(1, 131073, 2, 2) == bad                 # DOUBLE_WELL
    assert run(0, 262145, 2, 2) == bad
    assert run(1, 131073, 1, 1 + 2 * 131074) == bad    # MIXTURE, two centres
    assert run(1, 2049, 3, 2049 * 2049 + 2049) == bad  # QUADRATIC_FORM
    assert run(0, 2049, 3, 2049 * 2049 + 2049) == bad
    assert run(1, 65, 1, 1 + 17 * 66) == bad           # MIXTURE with 17 centres
    assert run(1, 65, 1, 1 + 2 * 66 + 1) == bad        # parameter count that is not 1 + K (1 + dim)
    assert run(1, 65, 3, 64 * 64 + 64) == bad          # parameter count of another dim
