"""
ORACLE (test infrastructure, not product code): population annealing on the 2-D lattice, as
tsu_ising2d_population_anneal (csrc/ising2d.cu) runs it, restated in NumPy and Python integers.

One step k of a population of R_p replicas (Hukushima-Iba; Machta; Wang-Machta-Katzgraber):
  1. count   E_i of every replica from exact (up, anti) counts, with the float64 rounding of energy_of_counts;
             E_ref = min_i E_i
  2. weigh   x_i = dbeta_k (E_i - E_ref), q_i = floor(exp_neg(x_i) 2^s) with s = 62 - ceil(log2 R_p), W = sum q_i
  3. draw    one 64-bit Philox value (lattice stream, kind 3) per population and step, U = floor(u64 W / 2^64)
  4. resample (systematic, R_p fixed): the parent of child j is the smallest i with R_p C_i > j W + U, where C is the
             inclusive prefix sum of q
  5. sweep   theta sweeps at T_k; child j draws the Philox stream of its own position

exp_neg spells out every float64 operation (range reduction with a two-part ln 2, a degree-13 Horner polynomial,
ldexp), so that the CUDA kernel, which uses __dmul_rn / __dadd_rn in the same order, gives the same bits.  Everything
after it is integer arithmetic.
"""

import math
from bisect import bisect_right

import numpy as np

from . import ising2d_bonds_oracle as B
from . import ising2d_oracle as O
from .philox_ref import philox4x32_10

KIND_RESAMPLE = 3
INV_LN2 = float.fromhex("0x1.71547652b82fep+0")
LN2_HI = float.fromhex("0x1.62e42fee00000p-1")  # 32 significant bits: n * LN2_HI is exact for |n| < 2^21
LN2_LO = float.fromhex("0x1.a39ef35793c76p-33")
EXP_COEFFS = [1.0 / math.factorial(k) for k in range(14)]  # 1/k!, rounded to float64


def weight_shift(r_pop: int) -> int:
    """s = 62 - ceil(log2 R_p): W = sum q_i <= R_p 2^s <= 2^62"""
    return 62 - (int(r_pop) - 1).bit_length()


def exp_neg(x: float) -> float:
    """exp(-x) for x >= 0: n = rint(x / ln 2), r = x - n ln 2 (two parts), exp(-r) by Horner on t = -r, times 2^-n"""
    n = float(round(x * INV_LN2))  # round() on a float rounds half to even, as rint
    r = (x - n * LN2_HI) - n * LN2_LO
    t = -r
    p = EXP_COEFFS[13]
    for c in reversed(EXP_COEFFS[:13]):
        p = p * t + c
    return math.ldexp(p, -int(n))


def quantised_weight(x: float, s: int) -> int:
    """q = floor(exp_neg(x) 2^s); 0 when rint(x / ln 2) > s + 1"""
    n = round(x * INV_LN2)
    if n > s + 1:
        return 0
    return int(math.ldexp(exp_neg(x), s))  # exact: a power-of-two scaling of a float64 below 2^63


def resample_draw(seed: int, replica: int, sweep: int) -> int:
    """the 64-bit value of a population (first global replica `replica`) and step (first sweep index `sweep`)"""
    c0, c1 = O.lattice_counter(0, 0, KIND_RESAMPLE, 0)
    out = philox4x32_10(c0, c1, sweep & 0xFFFFFFFF, replica & 0xFFFFFFFF, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return int(out[0]) | (int(out[1]) << 32)


def systematic_parents(q, u64: int):
    """parents of the R_p children (systematic resampling, integers only) and W"""
    r_pop = len(q)
    W = sum(int(v) for v in q)
    U = (int(u64) * W) >> 64
    scaled, c = [], 0
    for v in q:
        c += int(v)
        scaled.append(r_pop * c)
    return [bisect_right(scaled, j * W + U) for j in range(r_pop)], W


def counts(bits, periodic: bool, signs=None):
    """(up, anti): up spins and anti-aligned bonds (with signs: unsatisfied bonds), as tsu_ising2d_observables"""
    bits = np.asarray(bits, dtype=np.int64)
    if signs is None:
        signs = np.ones((2,) + bits.shape, dtype=np.int8)
    return int(bits.sum()), B.unsatisfied_bonds(bits, periodic, signs)


def energy_of_counts(up: int, anti: int, J: float, h: float, n_bonds: int, n_sites: int) -> float:
    """fma(-J, n_bonds - 2 anti, -(h (2 up - n_sites))); equal to the kernel's rounding when J is a power of two"""
    return (-J * float(n_bonds - 2 * anti)) - (h * float(2 * up - n_sites))


def n_bonds_of(rows: int, cols: int, periodic: bool) -> int:
    return len(B.bond_list(rows, cols, periodic, np.ones((2, rows, cols), dtype=np.int8))[0])


def population_anneal(states, family, Ts, dbeta, theta, n_populations, seed, replica0, sweep0, J, h, periodic,
                      signs=None):
    """the whole run: states [R] of bit arrays, family [R] ints, temperatures Ts[n], dbeta[n] (float64).
    signs: None (ferromagnet) or a list of one (2, rows, cols) realisation per population.
    Returns (states, family, weight_sum [n, P], energy_ref [n, P], count_sums [n+1, P, 2], energy [R])."""
    states = [np.array(b, dtype=np.int64) for b in states]
    family = [int(f) for f in family]
    R = len(states)
    P = int(n_populations)
    r_pop = R // P
    s = weight_shift(r_pop)
    rows, cols = states[0].shape
    nb = n_bonds_of(rows, cols, periodic)
    n = len(Ts)
    weight_sum = np.zeros((n, P), dtype=object)
    energy_ref = np.zeros((n, P))
    count_sums = np.zeros((n + 1, P, 2), dtype=object)
    energy = np.zeros(R)

    def count_all(k):
        for i in range(R):
            p = i // r_pop
            up, anti = counts(states[i], periodic, None if signs is None else signs[p])
            energy[i] = energy_of_counts(up, anti, J, h, nb, rows * cols)
            count_sums[k, p, 0] += up
            count_sums[k, p, 1] += anti

    for k in range(n):
        count_all(k)
        new_states, new_family = list(states), list(family)
        for p in range(P):
            lo = p * r_pop
            E = energy[lo:lo + r_pop]
            e_ref = min(E)
            energy_ref[k, p] = e_ref
            q = [quantised_weight(float(dbeta[k]) * (float(e) - e_ref), s) for e in E]
            parents, W = systematic_parents(q, resample_draw(seed, replica0 + lo, sweep0 + k * theta))
            weight_sum[k, p] = W
            for j, i in enumerate(parents):
                new_states[lo + j] = states[lo + i].copy()
                new_family[lo + j] = family[lo + i]
        states, family = new_states, new_family
        for i in range(R):
            if signs is None:
                states[i] = O.checkerboard_sweeps_philox(states[i], seed, replica0 + i, sweep0 + k * theta, theta, J, h,
                                                         Ts[k], periodic)
            else:
                states[i] = B.checkerboard_sweeps_philox_bonds(states[i], seed, replica0 + i, sweep0 + k * theta, theta,
                                                               J, h, Ts[k], periodic, signs[i // r_pop])
    count_all(n)
    return states, family, weight_sum, energy_ref, count_sums, energy


def exact_log_partition(rows, cols, J, h, T, periodic, signs=None):
    """ln Z(T) and <E> by enumerating all 2^(rows cols) states (signs None: the ferromagnet); T = inf gives N ln 2"""
    n = rows * cols
    assert n <= 20
    if signs is None:
        signs = np.ones((2, rows, cols), dtype=np.int8)
    states = ((np.arange(1 << n)[:, None] >> np.arange(n)[None, :]) & 1).astype(np.int64)
    sp = 2 * states - 1
    a, b, g = B.bond_list(rows, cols, periodic, signs)
    E = -J * (g[None, :] * sp[:, a] * sp[:, b]).sum(axis=1) - h * sp.sum(axis=1)
    if math.isinf(T):
        return n * math.log(2.0), float(E.mean())
    x = -(E - E.min()) / T
    w = np.exp(x)
    return float(-E.min() / T + np.log(w.sum())), float((w * E).sum() / w.sum())
