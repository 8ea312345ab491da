"""The FP32 accept filter of the fused stretch-move kernels against the FP64 expression it stands in for (CPU).
tests/test_gpu_accept_filter.py places device decisions at the same margins.

The reference decides  ((N-1) log z + p1) - p0 >= log u  (src/samplers.jl:260) in FP64.  Write Lz = fl(log z),
Lu = fl(log u) and  t = (N-1) Lz + p1 - p0 - Lu  for the exact value of those FP64 operands.  Every filtered kernel
(kmc_kernels.cuh: filter_q, accept_decide) computes
    q  = fmaf(N-1, lg2.approx(float z), -lg2.approx(float u))      only for 1e-30 < float u, 1/16 < float z < 16
    tt = (p1 - p0) + ln2 q                                         FP64
and decides alone when |tt| > margin = float((N-1+64) 2e-6) and |p0| < 2^36; anything else takes the FP64 expression.
n = N-1, u32 = 2^-24 (half an ulp of FP32 at 1), hu(x) = half an ulp of x.

Filter error E_f = |tt - t|, in natural-log units (a log2 error times ln2):
  * float z = z (1 + e), |e| <= u32: log2 moves by <= 1.0001 u32 / ln2, n times; likewise float u, once.
  * lg2.approx.ftz: 2^-22.6 absolute on the mantissa part, then one FP32 rounding of the result:
    z: n (2^-22.6 + 2^-23) since |lg2 float z| < 4;  u: 2^-22.6 + 2^-18 since |lg2 float u| < 100.
  * the fmaf rounds once: hu32(|q|) <= hu32(4n + 100).
  * FP64: p1 - p0, ln2 q and their sum round at |.| < 10^3 and ln2 is a rounded constant: < 1e-12 together, and so
    are |ln2 log2(z) - Lz| n and |ln2 log2(u) - Lu| (a contracted DFMA for the sum changes nothing here).
  E_f(n) = ln2 [ n (1.0001 u32/ln2 + 2^-22.6 + 2^-23) + 1.0001 u32/ln2 + 2^-22.6 + 2^-18 + hu32(4n + 100) ] + 2e-12.
Reference rounding E_ref = |fl-expression - exact|, where a decision is close (|t| < margin + E_f):
  * S = fl(fl(n Lz) + p1) with |S| < |p0| + 71 (|Lu| < 69.1 inside the filter's range):  hu64(|p0| + 71);
  * fl(n Lz), |n Lz| < 127 ln 16 = 353: hu64(353) = 2^-45;  lhs = fl(S - p0), |lhs| < 71: 2^-47.
  E_ref(P) = hu64(P + 71) + 2^-45 + 2^-47  for |p0| < P.
The filter decides like the FP64 expression when margin > E_f + E_ref: tt > margin gives t > margin - E_f > E_ref,
so the rounded lhs - Lu stays > 0 (and symmetrically).  With P = 2^36, E_ref = 2^-17 + ... = 7.7e-6, and
E_f + E_ref <= margin / 5 for every n <= 127 (fused kernels serve d <= 16, K2F / K2G d <= 128).  Without the |p0| bound
E_ref grows with |p0|: hu64(2^41) = 2^-12 = 2.4e-4 exceeds margin(n = 1) = 1.3e-4 and decisions flip, which the
sweep below finds.  n = 0 is immune: 0 * Lz + p1 is exact.

The model restates the filter with lg2.approx at both ends of its error bound (the correctly rounded log2 shifted by
+-2^-22.6, then rounded to FP32) and the fmaf as one exact rounding; t is the exact rational value of the FP64
operands (fractions.Fraction)."""
import math
import re
from fractions import Fraction
from pathlib import Path

import numpy as np
import pytest

LN2 = 0.6931471805599453
LG2_ERR = 2.0 ** -22.6
U32 = 2.0 ** -24
KERNELS_H = Path(__file__).resolve().parent.parent / "kissmcmc.jl_b200" / "csrc" / "kmc_kernels.cuh"
# the bound the kernels compile (kFilterMaxLogp): the derivation and the sweeps below check that very value
FILTER_MAX_LOGP = float(re.search(r"constexpr double kFilterMaxLogp = ([0-9.eE+]+);", KERNELS_H.read_text()).group(1))
NM1S = (0, 1, 2, 5, 9, 15, 127)


def margin(nm1):
    """p.margin as the host sets it (kmc_api.cu): an FP32 value."""
    return float(np.float32((nm1 + 64.0) * 2e-6))


def _hu32(x):
    return 2.0 ** (math.floor(math.log2(x)) - 24)


def _hu64(x):
    return 2.0 ** (math.floor(math.log2(x)) - 53)


def e_filter(nm1):
    per = 1.0001 * U32 / LN2 + LG2_ERR
    return LN2 * (nm1 * (per + 2.0 ** -23) + per + 2.0 ** -18 + _hu32(4 * nm1 + 100)) + 2e-12


def e_ref(p0_bound):
    return _hu64(p0_bound + 71) + 2.0 ** -45 + 2.0 ** -47


def _round_f32(x: Fraction) -> np.float32:
    """x rounded to the nearest FP32 value, ties to even (no double rounding)."""
    c = np.float32(float(x))
    best = None
    for v in (np.nextafter(c, np.float32(-np.inf)), c, np.nextafter(c, np.float32(np.inf))):
        if not np.isfinite(v):
            continue
        dist = abs(Fraction(float(v)) - x)
        key = (dist, int(np.array(v).view(np.uint32)) & 1)
        if best is None or key < best[0]:
            best = (key, v)
    return best[1]


def _lg2_model(v: np.float32, shift: float) -> np.float32:
    return np.float32(math.log2(float(v)) + shift)     # lg2.approx: within 2^-22.6, then one FP32 rounding


def filter_q(nm1, z, u, end, replay=True):
    """filter_q of kmc_kernels.cuh with lg2.approx at one end (+1: q as large as the bound allows, -1: as small);
    NaN where the kernel sends the step to the exact path."""
    zf, uf = np.float32(z), np.float32(u)
    ok = bool(uf > np.float32(1e-30)) and (not replay or bool(uf < np.float32(1e30)))
    ok = ok and bool(zf > np.float32(0.0625)) and bool(zf < np.float32(16.0))
    if not ok:
        return math.nan
    lz, lu = _lg2_model(zf, end * LG2_ERR), _lg2_model(uf, -end * LG2_ERR)
    return float(_round_f32(Fraction(float(np.float32(nm1))) * Fraction(float(lz)) - Fraction(float(lu))))


def decide_fast(nm1, z, u, p1, p0, end, bounded=True):
    """accept_decide's fast path: True / False, or None for the exact path.  bounded=False drops |p0| < 2^36."""
    if bounded and not abs(p0) < FILTER_MAX_LOGP:
        return None
    tt = (p1 - p0) + filter_q(nm1, z, u, end) * LN2
    m = margin(nm1)
    if tt > m:
        return True
    if tt < -m:
        return False
    return None


def reference(nm1, z, u, p1, p0):
    """src/samplers.jl:260 in FP64 (kmc_oracle.c, accept_exact)."""
    return ((nm1 * math.log(z) + p1) - p0) >= math.log(u)


def t_exact(nm1, z, u, p1, p0) -> Fraction:
    return nm1 * Fraction(math.log(z)) + Fraction(p1) - Fraction(p0) - Fraction(math.log(u))


def place(nm1, z, u, p0, k):
    """(p1, u): p1 the double nearest to where t = k * margin; what p1's ulp leaves over is moved into u (when it
    is below 1), so t lands within a few 1e-16 of k * margin wherever p0's scale allows."""
    m = Fraction(margin(nm1))
    want = Fraction(p0) + Fraction(math.log(u)) - nm1 * Fraction(math.log(z)) + k * m
    p1 = float(want)
    r = t_exact(nm1, z, u, p1, p0) - k * m
    if 0 < abs(r) < 1 and u > 0:
        u = math.exp(math.log(u) + float(r))
    return p1, u


def _f32_next(v, toward):
    return float(np.nextafter(np.float32(v), np.float32(toward)))


ZS = (1.0, _f32_next(0.0625, 1), 0.0625 + 2.0 ** -40, _f32_next(16.0, 0), 16.0 - 2.0 ** -30)
US = (_f32_next(1e-30, 1), float(np.float32(1e-30)), 2.0 ** -53, 0.5, 1.0 - 2.0 ** -53, 1.0)
P0S = (0.0, 1.0, 1e6, 1e9, float(np.nextafter(FILTER_MAX_LOGP, 0)), FILTER_MAX_LOGP, 2.0 ** 41, 1e13, 1e15, 1e300)
KS = tuple(s * k for k in (0.5, 0.99, 1.01, 1.5, 3, 10) for s in (1, -1))


def sweep(bounded):
    """Every grid point at both ends of the lg2 bound: (nm1, |p0|, t / margin, fast decision, reference)."""
    out = []
    for nm1 in NM1S:
        for z in ZS:
            for u0 in US:
                for a in P0S:
                    for p0 in {a, -a}:
                        for k in KS:
                            p1, u = place(nm1, z, u0, p0, k)
                            ref = reference(nm1, z, u, p1, p0)
                            tm = float(t_exact(nm1, z, u, p1, p0) / Fraction(margin(nm1)))
                            for end in (1, -1):
                                out.append((nm1, abs(p0), tm, decide_fast(nm1, z, u, p1, p0, end, bounded), ref))
    return out


@pytest.fixture(scope="module")
def bounded_sweep():
    return sweep(True)


@pytest.fixture(scope="module")
def unbounded_sweep():
    return sweep(False)


@pytest.mark.parametrize("nm1", range(128))
def test_margin_covers_filter_and_reference_error(nm1):
    assert e_filter(nm1) + e_ref(FILTER_MAX_LOGP) <= margin(nm1) / 5
    assert margin(nm1) < (nm1 + 64.0) * 2e-6 * (1 + 2 ** -23)


def test_reference_rounding_outgrows_the_margin_without_the_bound():
    """Why |p0| is bounded at all: at 2^41 half an ulp of p1 alone is larger than the margin of d = 2.  The compiled
    bound is the one the derivation covers (2^36: E_ref stays below a tenth of the smallest margin)."""
    assert FILTER_MAX_LOGP == 2.0 ** 36
    assert e_ref(2.0 ** 41) > margin(1)
    assert e_ref(FILTER_MAX_LOGP) < margin(0) / 10


def test_filter_decides_like_reference(bounded_sweep):
    wrong = [r for r in bounded_sweep if r[3] is not None and r[3] != r[4]]
    assert not wrong, wrong[:10]
    # not vacuous: the sweep has fast decisions right outside the margin and exact-path decisions inside it
    near_fast = sum(1 for nm1, a, tm, fast, _ in bounded_sweep if fast is not None and 1 <= abs(tm) <= 4)
    inside = sum(1 for nm1, a, tm, fast, _ in bounded_sweep if fast is None and abs(tm) < 1)
    print(f"fast decisions with |t| in [margin, 4 margin]: {near_fast}; exact path with |t| < margin: {inside}")
    assert near_fast > 1000 and inside > 1000


def test_unbounded_filter_disagrees_at_large_logp(unbounded_sweep):
    """The same sweep without |p0| < 2^36: counterexamples at |p0| >= 2^41 for d >= 2, none for d = 1 and none where
    the bound would have let the filter decide."""
    wrong = [r for r in unbounded_sweep if r[3] is not None and r[3] != r[4]]
    print(f"filter decisions against the FP64 expression without the |p0| bound: {len(wrong)}")
    assert any(nm1 >= 1 and a >= 2.0 ** 41 for nm1, a, *_ in wrong)
    assert not [r for r in wrong if r[0] == 0]
    assert not [r for r in wrong if r[1] < FILTER_MAX_LOGP]


def test_model_tracks_exact_q():
    """The model's q is within its own bound of the exact (N-1) log2 z - log2 u at both ends."""
    for nm1 in NM1S:
        for z in ZS[:2] + ZS[3:4]:
            for u in (US[0], 0.5, 1.0 - 2.0 ** -53):
                exact = nm1 * math.log2(z) - math.log2(u)
                for end in (1, -1):
                    q = filter_q(nm1, z, u, end)
                    assert abs(q - exact) * LN2 <= e_filter(nm1)
