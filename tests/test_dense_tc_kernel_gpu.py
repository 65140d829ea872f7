"""GPU parity of the tensor-core dense Gibbs kernel (csrc/dense_tc.cu: dense_tc_kernel<M>, thousands of chains sharing
one bf16 coupling matrix) at the shapes it serves, against the float64 rule of the reference (oracle/dense_oracle.py).

The kernel's moving parts each depend on something a small symmetric test never varies:
  * chunk g of the panel-major sequence goes to ring stage g % 3 and producer group g % 2, and both counters run on
    across panels and sweeps, so the phase pattern depends on n_panels mod 6: N = 128 k for k = 1 .. 8, 31, 32;
  * `panel_done` is a 4-deep parity ring: long launches at small N (128 x 100 sweeps, 640 x 13) wrap it many times;
  * row i of J holds the couplings INTO site i, the diagonal block is staged transposed and the correction MMA reads
    J[later, block]: only an asymmetric J tells a transpose from the original, so every dyadic problem here is one;
  * the tile height (64 / 128 chains per CTA) and the number of waves depend on the chain count: C = 1, 63 .. 65,
    127 .. 129, the C3 shape, the first two-wave counts of each height and the full wave (18944 chains);
  * the per-chain temperature of the second chain group of a threshold thread, the uint32 `sweep0` / `chain0` counters
    and the clamp of the threshold T logit(u) to +-20 T.

Dyadic couplings J = m / 2^k (|m| <= 3, k = ceil(log2 sqrt N), non-zero diagonal, bias in multiples of 2^-k) are exact
in bf16, and every partial sum of a field is a multiple of 2^-k below 2^(24 - k), so the TMEM accumulation, the x0.5,
the in-register corrections and the correction MMAs are all exact.  The kernel may then differ from the float64 rule
only through its acceptance threshold (fp32, lg2.approx): the field GEMM must equal S J^T exactly, and every update test
replays each sweep of the kernel's own trajectory against the reference's decision u < sigmoid(h / T).  A disagreement
must have |u - p| < TC_EPS_EXACT_J (Gaussian couplings: TC_EPS_GAUSSIAN_J), and their number is held to a budget.

Every update test also checks that the bits do not depend on how the work is launched: one launch of all sweeps against
one launch per sweep (`sweep0` offsets), against chain slices launched separately (`chain0` offsets), and the default
tile height against both forced ones (TSU_TC_M = 64 / 128).

The replay runs as two float64 GEMMs on the device: at the visit of site i the state is the kernel's new bits below i
and its old bits from i on, so h = after tril(J, -1)^T + start triu(J)^T + b.  Uniforms come from the oracle's Philox,
vectorised over (chain, site quad).  The CPU tests at the end of the file pin both helpers against the plain oracle.
"""
import functools
import math

import numpy as np
import pytest

from oracle import dense_oracle as D
from oracle.philox_ref import philox4x32_10

gpu = pytest.mark.gpu
M32 = 0xFFFFFFFF

# |u - sigmoid(h/T)| below which the kernel may disagree with the float64 rule (the budgets of tests/test_dense_gpu.py):
#   * exact fields (dyadic J): only the threshold T logit(u) is inexact - fp32 with lg2.approx, ~1e-6 of |logit| <= 17;
#   * Gaussian couplings rounded to bf16 (the reference gets the same rounded J): plus the fp32 accumulation error of
#     an N-term field, ~1e-6 sqrt(N) |J|, up to N = 4096.
TC_EPS_EXACT_J = 5e-6
TC_EPS_GAUSSIAN_J = 5e-5

# Disagreements per site visit that the count budgets allow (budget(): expectation + 5 sigma + 3).  A disagreement
# needs a uniform between the kernel's p and the reference's.  From the documented lg2.approx bound alone (2^-22
# absolute, twice, times ln 2) one would expect up to ~1e-7 per visit; measured on a B200 (1000 W) the whole file finds
# 4 disagreements in 4.4e8 visits with exact couplings (9e-9 per visit, max |u - p| = 2.6e-8) and 2 in 1.6e8 visits
# of the Gaussian full-wave workload (1.3e-8, max 2.9e-8).  The rates below are about twice those measurements: a
# systematic error in the fields or thresholds moves many more sites than that, while the count of a correct kernel
# stays far below the 5-sigma budget (e.g. 14 at the full wave).
RATE_EXACT_J = 2e-8
RATE_GAUSSIAN_J = 3e-8


def budget(visits, rate):
    expected = rate * visits
    return int(expected + 5.0 * math.sqrt(expected) + 3)


PANELS = [1, 2, 3, 4, 5, 6, 7, 8, 31, 32]            # N = 128 k: every residue mod 6 (ring phases) and mod 4 (panel_done)
SMALL_C = [1, 63, 64, 65, 127, 128, 129]              # tile boundaries at N = 256
# N = 4096: the C3 shape; 9473 = 148 * 64 + 1, the first count that runs two waves of 64-chain tiles; 18944 = 148 * 128,
# the full wave; 18945 the first two-wave count of 128-chain tiles
BIG_C = [2048, 9473, 18944, 18945]


# ------------------------------------------------------------------------------------------------ problems
def dyadic_problem(N, seed, *, asymmetric=True):
    """J = m / 2^k with |m| <= 3 and every diagonal entry non-zero (the self term is part of h, gibbs.py:97), bias in
    multiples of 2^-k with |b| <= 1; k = ceil(log2 sqrt N) keeps typical fields O(1).  Exact in bf16; every partial sum
    of a field is a multiple of 2^-k below 3 N / 2^k + 1 < 2^(24 - k): exact in fp32 in any order."""
    rng = np.random.default_rng(seed)
    k = int(np.ceil(np.log2(np.sqrt(N))))
    m = rng.integers(-3, 4, size=(N, N))
    if not asymmetric:
        m = np.triu(m) + np.triu(m, 1).T
    np.fill_diagonal(m, rng.integers(1, 4, N) * rng.choice([-1, 1], N))
    J = m * 2.0 ** -k
    b = rng.integers(-2**k, 2**k + 1, size=N) * 2.0 ** -k
    return J, b


def bf16_round(a):
    """float64 -> float32 -> bf16 -> float64: the rounding _TcProblem applies to the couplings"""
    import torch

    return torch.from_numpy(np.asarray(a, dtype=np.float64)).to(torch.float32).to(torch.bfloat16).double().numpy()


def sk_problem(N, seed):
    """symmetric J ~ N(0, 1/N) with zero diagonal, rounded to bf16 (so the reference sees the kernel's couplings)"""
    rng = np.random.default_rng(seed)
    J = rng.standard_normal((N, N))
    J = np.triu(J, 1)
    J += J.T
    J *= 1.0 / np.sqrt(N)
    return bf16_round(J)


def f32_temps(rng, C, lo=0.5, hi=2.0):
    """per-chain temperatures that are exact in fp32 (the kernel reads T_chain as float)"""
    return rng.uniform(lo, hi, C).astype(np.float32).astype(np.float64)


# ------------------------------------------------------------------------------------------------ host oracle helpers
def tc_uniforms(seed, chain0, C, sweep, N):
    """[C, N] float32 uniforms the kernel draws for chains chain0 .. chain0 + C - 1 (uint32, wrapping) in sweep `sweep`:
    D.philox_uniforms_tc vectorised over (chain, site quad) - word (i & 3) of Philox(i >> 2, chain, sweep, 'DENT'),
    top 24 bits / 2^24 (exact in float32)."""
    q = np.arange(N // 4, dtype=np.uint64)
    out = np.empty((C, N), dtype=np.float32)
    for a in range(0, C, 2048):
        z = min(C, a + 2048)
        chains = (np.uint64(chain0 & M32) + np.arange(a, z, dtype=np.uint64)) & np.uint64(M32)
        o = philox4x32_10(q[None, :], chains[:, None], sweep & M32, D.STREAM_DENSE_TC, seed & M32, (seed >> 32) & M32)
        w = np.stack(o, axis=-1).reshape(z - a, N)
        out[a:z] = (w >> 8).astype(np.float32) * np.float32(1.0 / 16777216.0)
    return out


_U_CACHE = {}


def uniforms(seed, chain0, C, sweep, N):
    """tc_uniforms, kept for the largest chain count asked so far: the N = 4096 tests share seed, chain0 and sweeps, so
    their 18945 x 4096 x 2 uniforms (about 12 s of host Philox) are drawn once"""
    if C * N < 1 << 24:
        return tc_uniforms(seed, chain0, C, sweep, N)
    key = (seed, chain0 & M32, sweep & M32, N)
    have = _U_CACHE.get(key, np.empty((0, N), dtype=np.float32))
    if have.shape[0] < C:                              # draw only the chains not drawn yet
        more = tc_uniforms(seed, chain0 + have.shape[0], C - have.shape[0], sweep, N)
        have = _U_CACHE[key] = np.concatenate([have, more])
    return have[:C]


def replay(start, after, J, b, T, U, chunk=4096):
    """One sweep of every chain replayed against the kernel's result (D.tc_sweep_disagreements for all chains at once).

    start / after: [C, N] bits before / after the sweep, J [N, N] and b [N] (or None) float64, T [C] float64, U [C, N]:
    torch tensors on one device.  At the visit of site i the kernel's state holds its new bits below i and the old ones
    from i on, so the reference's field (gibbs.py:97-99) is h = after tril(J, -1)^T + start triu(J)^T + b, in float64.
    Returns [(chain, site, |u - p|)] wherever u < sigmoid_ref(h / T) differs from the kernel's bit; |u - p| is evaluated
    with D.sigmoid_ref on the host."""
    import torch

    lower, upper = torch.tril(J, -1).T, torch.triu(J).T
    found = []
    for a in range(0, start.shape[0], chunk):
        s0, s1 = start[a:a + chunk].double(), after[a:a + chunk].double()
        h = s1 @ lower + s0 @ upper
        if b is not None:
            h += b
        x = h / T[a:a + chunk, None]
        p = torch.where(x > 20, 1.0, torch.where(x < -20, 0.0, 1.0 / (1.0 + torch.exp(-x))))
        u = U[a:a + chunk].double()
        c, i = torch.nonzero((u < p) != (s1 != 0), as_tuple=True)
        for cc, ii, xx, uu in zip(c.tolist(), i.tolist(), x[c, i].tolist(), u[c, i].tolist()):
            found.append((a + cc, ii, abs(uu - D.sigmoid_ref(xx))))
    return found


def energy_ref(S, J, b):
    """E = -1/2 s^T J s - b^T s (gibbs.py:215-236) of every chain, float64"""
    S = np.asarray(S, dtype=np.float64)
    e = -0.5 * np.einsum("cn,cn->c", S, S @ J.T)
    return e if b is None else e - S @ b


@functools.lru_cache(maxsize=None)
def find_extreme_uniform(seed, N, C, top, first_sweep=0, batch=256):
    """first (sweep, chain, site) with sweep >= first_sweep, chain < C, site < N whose uniform is exactly 0 (top=False) or
    1 - 2^-24 (top=True): words with all 24 used bits 0 / 1, once in 2^24 draws, found by searching the Philox counters"""
    q = np.arange(N // 4, dtype=np.uint64)
    want = np.uint32(0xFFFFFF if top else 0)
    s = first_sweep
    while True:
        sw = np.arange(s, s + batch, dtype=np.uint64)
        o = philox4x32_10(q[None, None, :], np.arange(C, dtype=np.uint64)[None, :, None], sw[:, None, None],
                          D.STREAM_DENSE_TC, seed & M32, (seed >> 32) & M32)
        hit = np.stack(o, axis=-1) >> np.uint32(8) == want       # [sweep, chain, quad, word]
        if hit.any():
            k, c, qq, w = np.argwhere(hit)[0]
            return int(s + k), int(c), int(4 * qq + w)
        s += batch


# ------------------------------------------------------------------------------------------------ device helpers
def _dev(a, dtype):
    import torch

    return None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).cuda()


def upload_j(J):
    """bf16 couplings as the kernel reads them (row i = couplings into site i) and the float64 matrix they stand for"""
    import torch

    Jd = torch.from_numpy(np.asarray(J, dtype=np.float64)).cuda().to(torch.float32).to(torch.bfloat16).contiguous()
    J64 = Jd.double()
    assert torch.equal(J64.cpu(), torch.from_numpy(np.asarray(J, dtype=np.float64))), "couplings are not bf16-exact"
    return Jd, J64


def tc_launch(Jd, bd, st, n_sweeps, seed, sweep0, chain0, Td=None, T=1.0):
    """one tsu_dense_gibbs_tc_run on the device state `st` ([C, N] uint8, updated in place); counters wrap at 2^32"""
    from tsu_emulator_b200 import _lib

    _lib.call("tsu_dense_gibbs_tc_run", _lib.ptr(Jd), _lib.ptr(bd), _lib.ptr(st), int(st.shape[0]), int(st.shape[1]),
              float(T), _lib.ptr(Td), int(n_sweeps), seed, sweep0 & M32, chain0 & M32, None, _lib.current_stream())
    return st


def tc_fields(Jd, S):
    """tsu_dense_tc_debug_fields: the fp32 field of every (chain, site) for the bits S, without bias"""
    import torch
    from tsu_emulator_b200 import _lib

    H = torch.full(S.shape, float("nan"), dtype=torch.float32, device="cuda")
    _lib.call("tsu_dense_tc_debug_fields", _lib.ptr(Jd), _lib.ptr(S), int(S.shape[0]), int(S.shape[1]), _lib.ptr(H),
              _lib.current_stream())
    return H


def check_update(label, J, b, init, n_sweeps, monkeypatch, *, seed, sweep0, chain0, T_chain=None, T=1.0,
                 eps=TC_EPS_EXACT_J, rate=RATE_EXACT_J, split=None):
    """The three launch comparisons and the float64 replay of every sweep of every chain (see the module docstring).
    `split`: chain indices where the chain slices start (default: one cut in the middle).  Returns the per-sweep
    trajectory [n_sweeps] of device states."""
    import torch

    C, N = init.shape
    Jd, J64 = upload_j(J)
    bd = _dev(None if b is None else np.asarray(b, dtype=np.float32), np.float32)
    Td = _dev(T_chain, np.float64)
    s0 = _dev(init, np.uint8)
    monkeypatch.delenv("TSU_TC_M", raising=False)
    one = tc_launch(Jd, bd, s0.clone(), n_sweeps, seed, sweep0, chain0, Td, T)
    for m in ("64", "128"):
        monkeypatch.setenv("TSU_TC_M", m)
        other = tc_launch(Jd, bd, s0.clone(), n_sweeps, seed, sweep0, chain0, Td, T)
        bad = int((other != one).any(1).sum())
        assert bad == 0, f"{label}: tile height {m} changes {bad} of {C} chains"
    monkeypatch.delenv("TSU_TC_M")
    seq, st = [], s0.clone()
    for s in range(n_sweeps):
        seq.append(tc_launch(Jd, bd, st, 1, seed, sweep0 + s, chain0, Td, T).clone())
    bad = int((seq[-1] != one).any(1).sum())
    assert bad == 0, f"{label}: one launch of {n_sweeps} sweeps and {n_sweeps} launches differ in {bad} of {C} chains"
    cuts = [0] + [a for a in (split if split is not None else [C // 2 + 1]) if 0 < a < C] + [C]
    parts = [tc_launch(Jd, bd, s0[a:z].clone(), n_sweeps, seed, sweep0, chain0 + a,
                       None if Td is None else Td[a:z].contiguous(), T) for a, z in zip(cuts, cuts[1:])]
    bad = int((torch.cat(parts) != one).any(1).sum())
    assert bad == 0, f"{label}: chain slices {cuts} launched separately differ in {bad} of {C} chains"
    Tv = Td if Td is not None else torch.full((C,), float(T), dtype=torch.float64, device="cuda")
    b64 = None if bd is None else bd.double()
    found = []
    for s in range(n_sweeps):
        U = torch.from_numpy(uniforms(seed, chain0, C, sweep0 + s, N)).cuda()
        found += [(s, *d) for d in replay(seq[s - 1] if s else s0, seq[s], J64, b64, Tv, U)]
        del U
    visits = C * N * n_sweeps
    worst = max([f[-1] for f in found], default=0.0)
    print(f"{label}: {len(found)} disagreeing visits of {visits} (budget {budget(visits, rate)}), "
          f"max |u - p| = {worst:.2e} (bound {eps:.0e})")
    assert all(f[-1] < eps for f in found), sorted(found, key=lambda f: -f[-1])[:10]
    assert len(found) <= budget(visits, rate), found[:20]
    return seq


# ------------------------------------------------------------------------------------------------ 1. the field GEMM
@gpu
@pytest.mark.parametrize("N,counts", [(128 * k, [70]) for k in PANELS] + [(256, SMALL_C), (4096, BIG_C)])
def test_fields_equal_float64_gemm_exactly(N, counts, monkeypatch):
    """tsu_dense_tc_debug_fields (the main GEMM alone: M x 128 x N per panel, A = spins expanded into TMEM, B = J tiles
    by TMA, x0.5 in the epilogue) must EQUAL S J^T in float64 for dyadic asymmetric J - at every panel count, chain count
    and both tile heights.  Any difference means the tensor core's accumulation is not exact for these inputs."""
    import torch

    J, _ = dyadic_problem(N, N)
    Jd, J64 = upload_j(J)
    rng = np.random.default_rng(N)
    for C in counts:
        S = _dev(rng.integers(0, 2, (C, N)), np.uint8)
        S[0] = 1                                       # every site set: the largest sums
        ref = S.double() @ J64.T
        for m in ("64", "128"):
            monkeypatch.setenv("TSU_TC_M", m)
            H = tc_fields(Jd, S).double()
            bad = int((H != ref).sum()) if not torch.isnan(H).any() else -1
            assert bad == 0, f"N={N} C={C} M={m}: {bad} fields differ from S J^T (-1: some never written)"


# ------------------------------------------------------------------------------------------------ 2. the panel ring
@gpu
@pytest.mark.parametrize("k", PANELS)
def test_panel_ring_phases(k, monkeypatch):
    """N = 128 k: every residue of n_panels mod 6 (stage and producer group of each chunk) and mod 4 (panel_done).
    Asymmetric dyadic J, bias, per-chain T in [0.5, 2], 3 sweeps in one launch, 70 chains (two tiles at M = 64, one
    partial tile with both chain groups of a threshold thread at M = 128)."""
    N, C = 128 * k, 70
    rng = np.random.default_rng(k)
    J, b = dyadic_problem(N, 10 + k)
    check_update(f"panel ring N={N}", J, b, rng.integers(0, 2, (C, N)), 3, monkeypatch, seed=1000 + k, sweep0=7 * k,
                 chain0=300 * k + 1, T_chain=f32_temps(rng, C), split=[33])


# ------------------------------------------------------------------------------------------------ 3. long launches
@gpu
@pytest.mark.parametrize("N,C,n_sweeps", [(128, 1000, 100), (640, 70, 13)])
def test_long_launches_wrap_panel_done(N, C, n_sweeps, monkeypatch):
    """many panels in one launch at small N: 100 sweeps of one panel (HardwareEmulator.sample_parallel's burn-in of 1000
    chains on N <= 128) and 13 sweeps of 5 panels wrap the 4-deep panel_done ring 25 and 16 times; every sweep replayed"""
    rng = np.random.default_rng(N)
    J, b = dyadic_problem(N, N + 1)
    check_update(f"long launch N={N} x {n_sweeps} sweeps", J, b, rng.integers(0, 2, (C, N)), n_sweeps, monkeypatch,
                 seed=77, sweep0=3, chain0=11, T_chain=f32_temps(rng, C), split=[300, 700] if C > 100 else [40])


# ------------------------------------------------------------------------------------------------ 6. counter wraps
@gpu
@pytest.mark.parametrize("what", ["sweep0", "chain0"])
def test_uint32_counter_wraps(what, monkeypatch):
    """sweep0 = 2^32 - 2 with 4 sweeps, and chain0 = 2^32 - 70 with 140 chains: the kernel's uint32 counters wrap, and
    the uniforms must be the oracle's at the masked counters (per-chain T, N = 384)"""
    N = 384
    C = 140 if what == "chain0" else 70
    sweep0, chain0 = (2**32 - 2, 5) if what == "sweep0" else (9, 2**32 - 70)
    rng = np.random.default_rng(1 if what == "sweep0" else 2)
    J, b = dyadic_problem(N, 384)
    check_update(f"{what} wrap", J, b, rng.integers(0, 2, (C, N)), 4 if what == "sweep0" else 2, monkeypatch, seed=2024,
                 sweep0=sweep0, chain0=chain0, T_chain=f32_temps(rng, C), split=[70] if C == 140 else [20])


# ------------------------------------------------------------------------------------------------ 7. threshold edges
EDGE_T = (0.37, 1.0, 3.3)
DELTAS = (0.0, 1e-7, -1e-7, 6e-6, -6e-6, 1e-3, -1e-3)
U_TOP = 1.0 - 2.0 ** -24


def _t16(t):
    """t with 16 significant bits: 20 t is then exact in fp32, so h / T = +-20 can be met exactly"""
    e = math.floor(math.log2(t))
    return round(t * 2.0 ** (15 - e)) * 2.0 ** (e - 15)


def _logit(u):
    with np.errstate(divide="ignore"):
        return np.log(u) - np.log1p(-u)


@gpu
@pytest.mark.parametrize("tile_m", ["64", "128"])
def test_threshold_edges(tile_m, monkeypatch):
    """J = 0, so h is the fp32 bias exactly.  Every site's bias is placed for one chain so that p = u + delta, delta in
    {0, +-1e-7, +-6e-6, +-1e-3}.  The uniforms u = 0 and u = 1 - 2^-24 (once in 2^24 draws; found by searching the Philox
    counters, then aimed at with sweep0 / chain0) are met with h / T = +-20 exactly, one fp32 ulp either side of it,
    inside the clamp, between 16 and 20 and on logit(u).  Per-chain T in {0.37, 1, 3.3} (second chain group of a
    threshold thread at M = 128).  Checks:
      * every visit with |u - p| >= TC_EPS_EXACT_J agrees with the reference;
      * the kernel's own rule h > T clamp(logit u, +-20) holds wherever lg2.approx cannot matter: |h/T - logit u| > 1e-4,
        or u = 0 (threshold exactly -20 T);
      * the disagreements inside the band are counted: at u = 0 and h = -20 T the reference accepts (p = 2e-9 > 0) and
        the kernel's strict h > -20 T does not, one per such launch."""
    import torch

    monkeypatch.setenv("TSU_TC_M", tile_m)
    N, C, seed = 128, 70, 99
    T = np.array([_t16(EDGE_T[c % 3]) for c in range(C)])
    Td = _dev(T, np.float64)
    Jd = torch.zeros((N, N), dtype=torch.bfloat16, device="cuda")
    checked = outside = in_band = rule_checked = expected_in_band = 0
    worst = 0.0
    for top in (False, True):
        sweep, c_hit, i_hit = find_extreme_uniform(seed, N, C, top)
        u_hit = U_TOP if top else 0.0
        sign = 1.0 if top else -1.0
        for pos in (67, 68, 69):                       # T = 1, 3.3, 0.37; chain group 1 of a 128-chain tile
            chain0 = (c_hit - pos) & M32
            U = uniforms(seed, chain0, C, sweep, N).astype(np.float64)
            assert U[pos, i_hit] == u_hit
            t = T[pos]
            h20 = np.float32(sign * 20.0 * t)          # exact: h / T = +-20
            targets = [h20, np.nextafter(h20, np.float32(sign * np.inf)), np.nextafter(h20, np.float32(0.0)),
                       np.float32(sign * 18.0 * t), np.float32(sign * 16.3 * t), np.float32(0.0)]
            if top:
                targets.append(np.float32(_logit(U_TOP) * t))
            for h_hit in targets:
                bias = np.zeros(N, dtype=np.float32)
                for i in range(N):
                    c = i % C
                    u = min(max(U[c, i] + DELTAS[(i // C + i) % len(DELTAS)], 2.0 ** -30), 1.0 - 2.0 ** -30)
                    bias[i] = np.float32(T[c] * _logit(u))
                bias[i_hit] = h_hit
                st = _dev(np.random.default_rng(i_hit).integers(0, 2, (C, N)), np.uint8)
                tc_launch(Jd, _dev(bias, np.float32), st, 1, seed, sweep, chain0, Td)
                got = st.cpu().numpy().astype(bool)
                x = bias.astype(np.float64)[None, :] / T[:, None]
                p = np.vectorize(D.sigmoid_ref)(x)
                want = U < p
                dist = np.abs(U - p)
                bad = got != want
                checked += got.size
                outside += int((dist >= TC_EPS_EXACT_J).sum())
                assert not (bad & (dist >= TC_EPS_EXACT_J)).any(), (top, pos, float(h_hit), np.argwhere(bad & (dist >= TC_EPS_EXACT_J)))
                in_band += int(bad.sum())
                worst = max(worst, float(dist[bad].max(initial=0.0)))
                # the kernel's rule with the exact logit: decided wherever the lg2.approx error cannot reach
                lg = np.clip(_logit(U), -20.0, 20.0)
                thr = (lg.astype(np.float32) * T.astype(np.float32)[:, None]).astype(np.float64)
                sure = (np.abs(x - lg) > 1e-4) | (U == 0.0)
                rule_checked += int(sure.sum())
                bad_rule = sure & (got != (bias.astype(np.float64)[None, :] > thr))
                assert not bad_rule.any(), (top, pos, float(h_hit), np.argwhere(bad_rule))
                expected_in_band += int(not top and h_hit == h20)
                if not top and h_hit == h20:           # u = 0, h = -20 T: p = sigmoid(-20) > 0 = u, the kernel says 0
                    assert not got[pos, i_hit] and want[pos, i_hit]
    print(f"threshold edges M={tile_m}: {checked} visits, {outside} with |u - p| >= {TC_EPS_EXACT_J:.0e} all agree, "
          f"{rule_checked} decided by the kernel's exact-logit rule; {in_band} disagree inside the band "
          f"({expected_in_band} of them at u = 0, h = -20 T), max |u - p| = {worst:.2e}")
    assert worst < TC_EPS_EXACT_J


# ------------------------------------------------------------------------------------------------ 4. chain counts
@gpu
@pytest.mark.parametrize("C", SMALL_C)
def test_chain_counts_tile_boundaries(C, monkeypatch):
    """C = 1 and both sides of 64 and 128 chains at N = 256: partial and exact tiles of both heights, 3 sweeps"""
    N = 256
    rng = np.random.default_rng(C)
    J, b = dyadic_problem(N, 256 + C)
    check_update(f"C={C} N={N}", J, b, rng.integers(0, 2, (C, N)), 3, monkeypatch, seed=5 + C, sweep0=1, chain0=C,
                 T_chain=f32_temps(rng, C), split=[C // 3 + 1])


# ------------------------------------------------------------------------------------------------ 8. host entry points
@gpu
@pytest.mark.parametrize("N", [129, 4000, 4096])
def test_sample_chains_energies_exact(N):
    """GibbsSampler(precision='bf16').sample_chains(return_energy=True): bits equal one C-ABI launch on the padded
    problem, and the energies (one more GEMM-only launch) equal the float64 energy EXACTLY for dyadic J - N = 129 is
    padded to 256 with uncoupled sites, 4000 to 4096"""
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler

    C, n_sweeps, T, seed = 70, 2, 1.25, 4321
    rng = np.random.default_rng(N)
    J, b = dyadic_problem(N, N + 9)
    init = rng.integers(0, 2, (C, N))
    out, e = GibbsSampler(GibbsConfig(temperature=T), seed=seed, precision="bf16").sample_chains(
        J, b, n_chains=C, n_sweeps=n_sweeps, initial_state=init, return_energy=True)
    Np = (N + 127) // 128 * 128
    Jp, bp, ip = np.zeros((Np, Np)), np.zeros(Np), np.zeros((C, Np), dtype=np.int64)
    Jp[:N, :N], bp[:N], ip[:, :N] = J, b, init
    Jd, _ = upload_j(Jp)
    st = tc_launch(Jd, _dev(bp, np.float32), _dev(ip, np.uint8), n_sweeps, seed, 0, 0, T=T)
    assert (st.cpu().numpy()[:, :N] == out).all()
    ref = energy_ref(out, J, b)
    print(f"sample_chains energies N={N}: max |E - E_float64| = {np.abs(e - ref).max():.1e}")
    assert (e == ref).all(), np.abs(e - ref).max()


@gpu
def test_sample_boltzmann_hardware_emulator_schedule():
    """The shape HardwareEmulator.sample_parallel routes to the tensor cores by default: N = 100 (padded to 128), 1000
    chains from the sampler's Philox initial state, 100 burn-in sweeps in one launch, then one sample after
    config.n_sweeps = 10 more.  The sample must equal the C-ABI launched one sweep at a time on the padded problem (whose
    110 sweeps are replayed against the float64 rule), and sample_parallel with numpy's global seed set must return the
    same samples as the sampler with the seed it draws."""
    import torch
    from tsu_emulator_b200 import GibbsConfig, GibbsSampler, HardwareEmulator

    N, C, T, burnin = 100, 1000, 1.0, 100
    J, _ = dyadic_problem(N, 100)
    saved = np.random.get_state()
    try:
        np.random.seed(20)
        seed = int(np.random.randint(0, 2**31 - 1))   # what GibbsSampler draws without seed=
        np.random.seed(20)
        hw_samples, timing = HardwareEmulator(n_bits=N, parallel_chains=C).sample_parallel(J, C, temperature=T)
    finally:
        np.random.set_state(saved)
    out = GibbsSampler(GibbsConfig(temperature=T), seed=seed, precision="bf16").sample_boltzmann(
        J, n_samples=1, burnin=burnin, n_chains=C)
    assert out.shape == (C, 1, N) and timing["batches_needed"] == 1
    assert (hw_samples == out[:, 0, :]).all()
    init = np.zeros((C, 128), dtype=np.int64)
    init[:, :N] = [D.philox_init_state(seed ^ 0x5DEECE66D, c, N) for c in range(C)]
    Jp = np.zeros((128, 128))
    Jp[:N, :N] = J
    Jd, J64 = upload_j(Jp)
    st = _dev(init, np.uint8)
    prev, found = st.clone(), []
    Tv = torch.full((C,), T, dtype=torch.float64, device="cuda")
    for s in range(burnin + 10):
        tc_launch(Jd, None, st, 1, seed, s, 0, T=T)
        U = torch.from_numpy(uniforms(seed, 0, C, s, 128)).cuda()
        found += replay(prev, st, J64, None, Tv, U)
        prev = st.clone()
    assert (st.cpu().numpy()[:, :N] == out[:, 0, :]).all()
    visits = C * 128 * (burnin + 10)
    print(f"sample_boltzmann N={N} x {C} chains, {burnin} + 10 sweeps: {len(found)} disagreeing visits of {visits}, "
          f"max |u - p| = {max([f[-1] for f in found], default=0.0):.2e}")
    assert all(f[-1] < TC_EPS_EXACT_J for f in found)
    assert len(found) <= budget(visits, RATE_EXACT_J)


# ------------------------------------------------------------------------------------------------ 4. N = 4096, many waves
BIG_SEED, BIG_SWEEP0, BIG_CHAIN0 = 8888, 12, 100


@gpu
@pytest.mark.parametrize("C", BIG_C)
def test_chain_counts_n4096(C, monkeypatch):
    """N = 4096 (32 panels), 2 sweeps, per-chain T: the C3 shape, the first two-wave counts of each tile height and the
    full wave; every chain of every sweep replayed"""
    rng = np.random.default_rng(C)
    J, b = dyadic_problem(4096, 4096)
    check_update(f"C={C} N=4096", J, b, rng.integers(0, 2, (C, 4096)), 2, monkeypatch, seed=BIG_SEED,
                 sweep0=BIG_SWEEP0, chain0=BIG_CHAIN0, T_chain=f32_temps(rng, C), split=[C // 3 + 1])


# ------------------------------------------------------------------------------------------------ 5. the full-wave workload
@gpu
def test_full_wave_gaussian_workload(monkeypatch):
    """The shape of the full-wave figure: Gaussian SK couplings rounded to bf16, N = 4096, one 128-chain tile per SM
    (18944 chains), 2 sweeps, scalar T.  Disagreements only within the fp32 field error TC_EPS_GAUSSIAN_J of p."""
    C, N = 18944, 4096
    rng = np.random.default_rng(18944)
    J = sk_problem(N, 18944)
    check_update(f"full wave SK C={C} N={N}", J, None, rng.integers(0, 2, (C, N)), 2, monkeypatch, seed=BIG_SEED,
                 sweep0=BIG_SWEEP0, chain0=BIG_CHAIN0, T=1.0, eps=TC_EPS_GAUSSIAN_J, rate=RATE_GAUSSIAN_J,
                 split=[9472])
    _U_CACHE.clear()


# ------------------------------------------------------------------------------------------------ CPU: the helpers
def test_dyadic_problem_is_exact():
    """dyadic_problem: bf16-exact couplings, non-zero diagonal, asymmetric unless asked otherwise, and every partial sum
    of a field a multiple of 2^-k below 2^(24 - k)"""
    for N in (128, 640, 4096):
        J, b = dyadic_problem(N, N)
        k = int(np.ceil(np.log2(np.sqrt(N))))
        assert (bf16_round(J) == J).all()
        assert (np.diag(J) != 0).all() and (J != J.T).any()
        assert (J * 2**k == np.round(J * 2**k)).all() and (b * 2**k == np.round(b * 2**k)).all()
        assert np.abs(J).sum(1).max() + np.abs(b).max() < 2.0 ** (24 - k)
        Js, _ = dyadic_problem(N, N, asymmetric=False)
        assert (Js == Js.T).all() and (np.diag(Js) != 0).all()
    J = sk_problem(256, 1)
    assert (J == J.T).all() and (bf16_round(J) == J).all()


def test_uniform_helper_matches_oracle():
    """tc_uniforms equals D.philox_uniforms_tc chain by chain, with chain and sweep counters that wrap at 2^32 and a
    seed above 2^32; find_extreme_uniform's hits are the extreme uniforms"""
    for seed, chain0, C, sweep, N in ((7, 0, 3, 0, 128), (2**40 + 5, 2**32 - 2, 5, 2**32 - 1, 256),
                                      (8888, 100, 2050, 13, 128)):
        U = tc_uniforms(seed, chain0, C, sweep, N)
        assert U.dtype == np.float32
        for c in (0, 1, C - 1):
            assert (U[c] == D.philox_uniforms_tc(seed, (chain0 + c) & M32, sweep, N)).all(), (seed, c)
    for top, u in ((False, 0.0), (True, U_TOP)):
        sweep, c, i = find_extreme_uniform(99, 128, 70, top)
        assert D.philox_uniforms_tc(99, c, sweep, 128)[i] == u


def test_replay_helper_matches_oracle():
    """replay (two float64 GEMMs, here on the CPU) finds the same disagreements as D.tc_sweep_disagreements, chain by
    chain: dyadic asymmetric J with bias and per-chain T, and Gaussian J without bias, on trajectories with flipped bits"""
    import torch

    rng = np.random.default_rng(3)
    total = 0
    for N, C, family in ((128, 5, "dyadic"), (256, 4, "gauss")):
        if family == "dyadic":
            J, b = dyadic_problem(N, 1)
        else:
            J, b = sk_problem(N, 2), None
        T = f32_temps(rng, C)
        start = rng.integers(0, 2, (C, N))
        U = tc_uniforms(11, 3, C, 4, N)
        after = start.copy()
        cur = start.astype(np.float64)
        for i in range(N):                              # the reference's sweep, then some bits flipped on purpose
            x = (cur @ J[i] + (0.0 if b is None else b[i])) / T
            cur[:, i] = U[:, i] < np.array([D.sigmoid_ref(v) for v in x])
        after = cur.astype(np.int64)
        after[rng.random((C, N)) < 0.05] ^= 1
        t = lambda a: torch.from_numpy(np.asarray(a))  # noqa: E731
        found = replay(t(start.astype(np.uint8)), t(after.astype(np.uint8)), t(J), None if b is None else t(b), t(T),
                       t(U))
        for c in range(C):
            ref = D.tc_sweep_disagreements(start[c], after[c], J, b, T[c], U[c].astype(np.float64))
            assert [(s, pytest.approx(e, abs=1e-12)) for s, e in ref] == [(s, e) for cc, s, e in found if cc == c]
            total += len(ref)
    assert total > 50


def test_count_budget():
    """budget() is the expectation plus five standard deviations plus three"""
    assert budget(0, RATE_EXACT_J) == 3
    assert budget(10**6, 1e-6) == 1 + 5 + 3
