"""The population-annealing oracle's building blocks (oracle/population_oracle.py), on the CPU: the spelled-out exp,
the quantised weights, the resampling draw and systematic resampling with integer weights."""
import math

import numpy as np
import pytest

from oracle import ising2d_oracle as O
from oracle import population_oracle as PA
from oracle.philox_ref import philox4x32_10


def test_exp_is_within_two_ulp_of_math_exp_and_exact_at_zero():
    assert PA.exp_neg(0.0) == 1.0
    xs = np.concatenate([np.linspace(0.0, 45.0, 200001), np.linspace(0.0, 1e-6, 1001), [math.log(2) * k for k in range(65)]])
    worst = max(abs(PA.exp_neg(float(x)) - math.exp(-x)) / math.ulp(math.exp(-x)) for x in xs)
    assert worst <= 2.0, worst


def test_weight_shift_and_quantisation():
    assert [PA.weight_shift(r) for r in (1, 2, 3, 4, 5, 1024, 1025, 1 << 20)] == [62, 61, 60, 60, 59, 52, 51, 42]
    for r_pop in (1, 3, 64, 2048, 1 << 20):
        s = PA.weight_shift(r_pop)
        assert r_pop * (1 << s) <= 1 << 62
        assert PA.quantised_weight(0.0, s) == 1 << s
        # weights with rint(x / ln 2) > s + 1 are dropped; just below, q is 0 or 1
        x_drop = (s + 1.5) * math.log(2.0)
        assert PA.quantised_weight(x_drop, s) == 0
        assert PA.quantised_weight((s + 1.4) * math.log(2.0), s) in (0, 1)
        x = 0.37
        assert PA.quantised_weight(x, s) == math.floor(math.ldexp(PA.exp_neg(x), s))


def test_resample_draw_is_the_lattice_stream_with_kind_3():
    seed, replica, sweep = 0x123456789ABCDEF0, 77, 1000
    c0, c1 = O.lattice_counter(0, 0, 3, 0)
    assert (int(c0), int(c1)) == (0, 3 << 26)
    out = philox4x32_10(0, 3 << 26, sweep, replica, seed & 0xFFFFFFFF, seed >> 32)
    assert PA.resample_draw(seed, replica, sweep) == int(out[0]) | (int(out[1]) << 32)
    assert PA.resample_draw(seed, replica, sweep) != PA.resample_draw(seed, replica + 1, sweep)


@pytest.mark.parametrize("r_pop", [1, 3, 7, 64, 1000])
def test_systematic_resampling_keeps_the_size_and_rounds_each_expected_count(r_pop):
    rng = np.random.default_rng(r_pop)
    s = PA.weight_shift(r_pop)
    for trial in range(20):
        x = rng.exponential(3.0, size=r_pop)
        x[rng.integers(r_pop)] = 0.0  # the replica at E_ref
        q = [PA.quantised_weight(float(v), s) for v in x]
        u64 = int(rng.integers(0, 1 << 63)) * 2 + int(rng.integers(0, 2))
        parents, W = PA.systematic_parents(q, u64)
        assert W == sum(q) and (1 << s) <= W <= 1 << 62
        assert len(parents) == r_pop and parents == sorted(parents)
        n = np.bincount(parents, minlength=r_pop)
        for i in range(r_pop):
            expected_num = r_pop * q[i]  # n_i in {floor, ceil} of r_pop q_i / W
            assert expected_num // W <= n[i] <= -(-expected_num // W)


@pytest.mark.parametrize("r_pop", [1, 3, 64, 5000])
def test_equal_weights_give_the_identity(r_pop):
    s = PA.weight_shift(r_pop)
    for u64 in (0, 1, (1 << 64) - 1, 0x9E3779B97F4A7C15):
        parents, W = PA.systematic_parents([1 << s] * r_pop, u64)
        assert parents == list(range(r_pop)) and W == r_pop << s


def test_exact_log_partition_limits():
    lz, mE = PA.exact_log_partition(2, 3, 1.0, 0.25, math.inf, False)
    assert lz == pytest.approx(6 * math.log(2.0)) and mE == pytest.approx(0.0)
    # T -> 0: ln Z -> -E_min / T for the ferromagnet's ground state (all up with h > 0)
    n_bonds = PA.n_bonds_of(2, 3, False)
    lz, mE = PA.exact_log_partition(2, 3, 1.0, 0.25, 0.01, False)
    e_min = -1.0 * n_bonds - 0.25 * 6
    assert lz == pytest.approx(-e_min / 0.01) and mE == pytest.approx(e_min)
