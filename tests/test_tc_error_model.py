"""Error bounds of the two approximate tcgen05 log-densities, derived from their arithmetic, and a numpy model of that
arithmetic that checks them (CPU).  tests/test_gpu_tc_error_bounds.py asserts the same bounds on a B200.

u = 2^-24 (half an ulp of FP32 at 1).  Every bound below is computed in FP64 from the inputs alone (theta, X, A, mu),
never from a kernel's output.

Logistic regression, K3 (`tc::logistic_tc_kernel`, kmc_tc.cuh).  The kernel returns
    R_tc ~ R = sum_n f(s_n),   f(s) = |s|/2 + log1p(e^-|s|),   s_n = theta . x_n,
in log2 units (s' = s log2 e); the exact FP64 finish adds theta . X^T (y - 1/2) and the prior.  |f'| <= 1/2, so a logit
error e (natural units) moves f by at most |e|/2.  With S_n = sum_k |theta_k x_nk|:
  * theta' = theta log2 e is split in FP64 into three round-to-nearest bf16 pieces; each leaves at most 2^-8 of what
    it splits, so the pieces miss theta' by at most u |theta'_k|: logit error <= u S_n.  X is bf16 and exact.
  * bf16 x bf16 products are exact in FP32.  Each tcgen05.mma (K = 16 columns) adds its products to the FP32
    accumulator with one rounding, allowed to truncate: at most one ulp, 2u, of a result no larger than
    (1 + 2^-7) S_n.  Pieces go in lo, mid, hi; the lo and mid partial sums are below 2^-7 S_n, so the MMAs cost
    <= 2.03 m u S_n in the logit, m = ceil(d/16) the MMAs per piece that meet a nonzero column (an MMA over
    padding adds exact zeros and rounds nothing).
    -> softplus error <= (1 + 2.03 m) u S_n / 2.
  * The epilogue sums |s'| of each 32-column chunk in FP32: two sequential sums of 16 (15 roundings each, every
    partial below the chunk's sum), one add and the final fmaf(0.5, sa + sb, lg): <= 8.5 u sum_n |s_n|.  This term
    is charged to |s_n| = |theta . x_n|, not to S_n: it is what the chunk sums add, and S_n is ~sqrt(d) times
    larger at random signs, which would make the bound ~2x looser at d = 32.
  Per row and independent of scale (beta): ex2.approx and the degree-5 polynomial variant (KMC_K3_POLY) are within
  2^-22 relative of 2^-|s'|, which moves log(1 + t) by <= 2u; the FP32 product of the 32 factors (1 + t) rounds once
  per row and once more per chunk (<= u each in log), the fmaf's lg term <= 0.7u, lg2.approx is within 2^-22 absolute
  (2.8u per chunk).  Per row 3.7u, per chunk 3.8u, at most ceil(N/32) chunks: beta N with beta = 5u for N >= 4.
      |R_tc - R| <= u [ (0.5 + 1.05 m) sum_n S_n + 8.5 sum_n |s_n| ] + 5 u N                    (per point)
                 <= 13.2 u sum_n sum_k |theta_k x_nk| + 5 u N               (|s_n| <= S_n, m <= 4)
  and a difference of two points gets the sum of their two bounds.  Most of it is the FP32 logits: the bound grows
  with the logit scale, so no fixed tolerance holds for every data set.  Bench configuration (BASELINE.json
  configs[3]: d = 32, N = 10^6, theta* ~ N(0,1)/sqrt(d), mean |logit| ~ 0.7): ~1.3 per point; with the data drawn
  from 16 theta* (mean |logit| ~ 11): ~13 per point.  What a B200 shows is far below this worst case (a common offset
  of ~3e-2 and 2e-3 on differences at the bench problem); the GPU tests print the headroom.

Dense Gaussian, K2 (`tc::gaussian_tc_kernel`, K2F, K2G, the batched Metropolis tc path).  logp = lognorm - |y|^2/2,
y = A (x - mu).  With P_i = (|A| |x - mu|)_i:
  * x - mu (FP64) is rounded once to FP32 and split exactly (split3_pair): <= u P_i in y_i;
  * A is split in FP64 into three round-to-nearest bf16 pieces: <= u P_i;
  * the three dropped piece pairs (lo,mid) (mid,lo) (lo,lo): <= 2.03 u P_i;
  * 6 piece pairs x ceil(d/16) <= 8 MMAs, one truncating rounding each; only the 8 (hi,hi) steps carry the full
    magnitude (the earlier partial sums are below 2^-7 P_i): <= 2.1 x 8 u P_i = 16.8 u P_i.
  So |dy_i| <= 21 u P_i, and |y_tc|^2/2 - |y|^2/2 <= sum_i |y_i| |dy_i| + dy_i^2 / 2.
  The epilogue sums y_i^2 in FP32 over each group of 32 columns: 32 sequential fmaf (K2 / K2F) or a depth-5
  butterfly plus three adds of the four quarters (K2G): <= 32 u sum y_i^2, halved: 16 u |y|^2.
      |logp_tc - logp| <= 21 u sum_i |y_i| P_i + 16 u |y|^2 + (21 u)^2 sum_i P_i^2 / 2          (per point)
  P_i / |y_i| is small unless A (x - mu) cancels, so the published 1e-5 (1 + |y|^2) = 168 u (1 + |y|^2) covers every
  case measured; the derived bound is the one that follows from the arithmetic alone.

The model below follows the kernels' comments operation by operation (FP32 rounding emulated on float64 values) and is
compared with an np.longdouble reference: (a) it stays inside the bound, (b) at the largest scale its error is at least
1/100 of the bound (the bound is not vacuous), (c) the FP64 oracle's own error is below 1e-3 of the bound, so the
oracle is a fit reference for the GPU tests."""
import math

import numpy as np
import pytest

from tests import cases

U = 2.0 ** -24
BETA_LOGISTIC = 5.0 * U
ALPHA_GAUSS, BETA_GAUSS = 21.0, 16.0
LOG2E = 1.4426950408889634


# ---------------------------------------------------------------------------------- the bounds (inputs only)

def logistic_bound(theta, X):
    """Per-point bound on |R_tc - R| for points theta [W, d] and data X [N, d]."""
    theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
    X = np.asarray(X, dtype=np.float64)
    m = -(-X.shape[1] // 16)
    S = np.abs(theta) @ np.abs(X).sum(axis=0)                          # sum_n sum_k |theta_k x_nk|
    s = np.abs(theta @ X.T).sum(axis=1)                                # sum_n |theta . x_n|
    return U * ((0.5 + 1.05 * m) * S + 8.5 * s) + BETA_LOGISTIC * X.shape[0]


def gaussian_terms(x, A, mu):
    """y = A (x - mu), |y|^2 and sum_i |y_i| (|A| |x - mu|)_i, sum_i (|A| |x - mu|)_i^2, per point (FP64)."""
    c = np.atleast_2d(np.asarray(x, dtype=np.float64)) - np.asarray(mu, dtype=np.float64)
    y = c @ A.T
    P = np.abs(c) @ np.abs(A).T
    return np.sum(y * y, axis=1), np.sum(np.abs(y) * P, axis=1), np.sum(P * P, axis=1)


def gaussian_bound(x, A, mu):
    """Per-point bound on |logp_tc - logp| of the dense Gaussian y = A (x - mu)."""
    yy, yP, PP = gaussian_terms(x, A, mu)
    a = ALPHA_GAUSS * U
    return a * yP + BETA_GAUSS * U * yy + 0.5 * a * a * PP


def gaussian_matrix(prm, d):
    """mu, A from the plugin's parameter vector [mu, A row-major, lognorm]."""
    prm = np.asarray(prm, dtype=np.float64)
    return prm[:d], prm[d:d + d * d].reshape(d, d)


# ---------------------------------------------------------------------------------- the arithmetic

def _bf16_rn(v):
    """Round-to-nearest-even to 8 significant bits (bf16; FP32's exponent range), exact on float64."""
    v = np.asarray(v, dtype=np.float64)
    m, e = np.frexp(v)
    r = np.ldexp(np.rint(np.ldexp(m, 8)), e - 8)
    return np.where(np.abs(r) > 3.3895313892515355e38, np.copysign(np.inf, v), r)


def _f32(v, mode="rn"):
    """FP32 rounding of float64 values: to nearest, or toward zero (a truncating accumulator)."""
    v = np.asarray(v, dtype=np.float64)
    f = v.astype(np.float32)
    if mode == "rz":
        over = np.abs(f.astype(np.float64)) > np.abs(v)
        f = np.where(over, np.nextafter(f, np.float32(0)), f)
    return f.astype(np.float64)


def _split3_f64(v):
    """split_theta_kernel / split_rows128 (matrix): three RN bf16 pieces of the FP64 value."""
    out = []
    for _ in range(3):
        h = _bf16_rn(v)
        out.append(h)
        v = v - h
    return out


def _split3_pair(v):
    """split3_pair: RN to FP32 once, then an exact bf16 split."""
    f = _f32(v)
    out = []
    for _ in range(3):
        h = _bf16_rn(f)
        out.append(h)
        f = _f32(f - h)
    return out


def _mma(steps, rows, cols, mode):
    """FP32 accumulator after the listed (left piece [rows, K], right piece [cols, K]) pairs, 16 columns per MMA,
    one rounding per MMA (products exact, their sum exact in float64 at these magnitudes)."""
    acc = np.zeros((rows, cols))
    for a, b in steps:
        for k0 in range(0, a.shape[1], 16):
            acc = _f32(acc + a[:, k0:k0 + 16] @ b[:, k0:k0 + 16].T, mode)
    return acc


def _ex2_neg_abs_poly(s):
    """ex2_neg_abs_poly of kmc_tc.cuh, FP32 operation by operation."""
    a = np.minimum(np.abs(s), 126.0)
    r = _f32(a + 12582912.0)
    x = _f32(_f32(r - 12582912.0) - a)
    q = 0.0013266970636323094
    for cf in (0.009675459936261177, 0.05550742521882057, 0.24022121727466583, 0.6931469440460205,
               1.0000001192092896):
        q = _f32(_f32(q) * x + _f32(cf))
    return q * np.exp2(-(r - 12582912.0))


def logistic_model(theta, X, mode="rz", ex2_err=0.0, lg2_err=0.0):
    """K3 + finish, softplus part only: sum_n (|s_n|/2 + log1p(e^-|s_n|)) as the kernel computes it.
    ex2_err / lg2_err: a relative error of MUFU ex2 and an absolute error of lg2 applied to every call (the
    worst case in one direction)."""
    theta = np.atleast_2d(theta)
    N, d = X.shape
    kp = 32 if d <= 32 else 64
    th = np.zeros((theta.shape[0], kp))
    th[:, :d] = theta * LOG2E
    Xp = np.zeros((N, kp))
    Xp[:, :d] = X
    hi, mid, lo = _split3_f64(th)
    s = _mma([(lo, Xp), (mid, Xp), (hi, Xp)], th.shape[0], N, mode)      # logits, log2 units
    npad = -N % 32
    s = np.pad(s, ((0, 0), (0, npad))).reshape(s.shape[0], -1, 32)
    valid = np.pad(np.ones(N, bool), (0, npad)).reshape(-1, 32)
    pa, pb, sa, sb = (np.ones(s.shape[:2]), np.ones(s.shape[:2]), np.zeros(s.shape[:2]), np.zeros(s.shape[:2]))
    for j in range(32):
        sj, ok = s[:, :, j], valid[:, j]
        if j % 4 == 3:                                                  # KMC_K3_POLY = 4
            t = _ex2_neg_abs_poly(sj)
        else:
            t = _f32(np.exp2(-np.abs(sj)) * (1.0 + ex2_err))
        if j % 2 == 0:
            pa = np.where(ok, _f32(pa * t + pa), pa)
            sa = np.where(ok, _f32(sa + np.abs(sj)), sa)
        else:
            pb = np.where(ok, _f32(pb * t + pb), pb)
            sb = np.where(ok, _f32(sb + np.abs(sj)), sb)
    lg = _f32(np.log2(_f32(pa * pb)) + lg2_err)
    chunk = _f32(0.5 * _f32(sa + sb) + lg)
    return chunk.sum(axis=1) * math.log(2.0)


def logistic_exact(theta, X, y=None, prior_sigma=None):
    """np.longdouble: the softplus part, or the whole log-density when y and prior_sigma are given."""
    th = np.atleast_2d(theta).astype(np.longdouble)
    s = th @ X.astype(np.longdouble).T
    a = np.abs(s)
    sp = (a / 2 + np.log1p(np.exp(-a))).sum(axis=1)
    if y is None:
        return sp
    yc = y.astype(np.longdouble) - np.longdouble(0.5)
    return (s * yc).sum(axis=1) - sp - (th * th).sum(axis=1) / (2 * np.longdouble(prior_sigma) ** 2)


def gaussian_model(x, A, mu, mode="rz", epilogue="seq"):
    """K2 / K2F (epilogue "seq": 32 sequential fmaf per group, FP64 across groups) or K2G ("tree": butterfly per 32
    columns, the four quarters added in FP32): -|y|^2 / 2 as the kernel computes it."""
    d = A.shape[0]
    C = _split3_pair(np.atleast_2d(x) - mu)
    M = _split3_f64(A)
    order = [(2, 0), (0, 2), (1, 1), (1, 0), (0, 1), (0, 0)]             # (C piece, A piece), 0 = hi
    y = _mma([(C[c], M[a]) for c, a in order], C[0].shape[0], d, mode)
    ypad = np.pad(y, ((0, 0), (0, -d % 32)))
    if epilogue == "seq":
        ss = np.zeros(y.shape[0])
        for g in range(0, d, 32):
            part = np.zeros(y.shape[0])
            for j in range(g, g + 32):
                part = _f32(ypad[:, j] * ypad[:, j] + part)
            ss += part
    else:
        quarters = []
        for g in range(0, 128, 32):
            v = _f32(ypad[:, g:g + 32] ** 2) if g < ypad.shape[1] else np.zeros((y.shape[0], 32))
            while v.shape[1] > 1:
                h = v.shape[1] // 2
                v = _f32(v[:, :h] + v[:, h:])
            quarters.append(v[:, 0])
        ss = _f32(_f32(_f32(quarters[0] + quarters[1]) + quarters[2]) + quarters[3])
    return -0.5 * ss


def gaussian_exact(x, A, mu):
    c = np.atleast_2d(x).astype(np.longdouble) - np.asarray(mu).astype(np.longdouble)
    y = c @ A.astype(np.longdouble).T
    return -(y * y).sum(axis=1) / 2


# ---------------------------------------------------------------------------------- problems shared with the GPU tests

SCALES = (1, 4, 16, 64)


def scaled_logistic_problem(N, d, scale, seed):
    """cases.logistic_problem with y drawn from scale * theta*: mean |logit| ~ 0.7 scale."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, d)).astype(np.float32)
    X = (X.view(np.uint32) & np.uint32(0xFFFF0000)).view(np.float32)
    tstar = scale * rng.standard_normal(d) / np.sqrt(d)
    y = (rng.random(N) < 1.0 / (1.0 + np.exp(-(X.astype(np.float64) @ tstar)))).astype(np.float32)
    return X, y, tstar


def logistic_points(tstar, N, npts, seed):
    """A ball about the mode (radius ~ the posterior scale) and two burn-in points: 0 and 100 theta*."""
    d = tstar.size
    ball = tstar + cases.ball(np.zeros(d), 1.0 / math.sqrt(N), npts, seed)
    return np.vstack([ball, np.zeros(d), 100.0 * tstar])


def equicorrelated(d, rho):
    return (1.0 - rho) * np.eye(d) + rho * np.ones((d, d))


def mvn_blocks(d):
    """Block-diagonal copies of the reference's mvn2 covariance (condition number ~1e3); a 1 x 1 block if d is odd."""
    cov = np.zeros((d, d))
    for i in range(0, d - 1, 2):
        cov[i:i + 2, i:i + 2] = cases.MVN_COV
    if d % 2:
        cov[-1, -1] = cases.MVN_COV[0][0]
    return cov


def gaussian_case(kind, d):
    """(mean, covariance) of the Gaussian error-bound cases."""
    mean = np.linspace(-1, 1, d)
    if kind == "spd":
        return mean, cases.spd_cov(d, 3)
    if kind == "rho0.99":
        return mean, equicorrelated(d, 0.99)
    if kind == "rho0.999":
        return mean, equicorrelated(d, 0.999)
    if kind == "mvn2_blocks":
        return mean, mvn_blocks(d)
    if kind == "scales":
        s = np.logspace(-3, 3, d)
        return mean * s, cases.spd_cov(d, 3) * np.outer(s, s)
    if kind == "mean1e3":
        return 1e3 + mean, cases.spd_cov(d, 3)
    raise ValueError(kind)


GAUSS_KINDS = ("spd", "rho0.99", "rho0.999", "mvn2_blocks", "scales", "mean1e3")


def gaussian_points(mean, cov, nsigma, npts, seed):
    """mean + nsigma L z with L L^T = cov, z ~ N(0, I)."""
    L = np.linalg.cholesky(cov)
    z = np.random.default_rng(seed).standard_normal((npts, mean.size))
    return mean + nsigma * z @ L.T


# ---------------------------------------------------------------------------------- the CPU checks

@pytest.mark.parametrize("N", [3001, 20_000])
@pytest.mark.parametrize("d", [5, 32, 33, 64])
def test_logistic_model_within_bound(orc, N, d):
    ratios = {}
    for scale in SCALES:
        X, y, tstar = scaled_logistic_problem(N, d, scale, seed=100 * d + scale)
        pts = logistic_points(tstar, N, 6, seed=d)
        ref = logistic_exact(pts, X)
        bound = logistic_bound(pts, X)
        for mode, e2, l2 in (("rz", 0.0, 0.0), ("rn", 0.0, 0.0), ("rz", 4 * U, 4 * U), ("rz", -4 * U, -4 * U)):
            err = np.abs((logistic_model(pts, X, mode, e2, l2) - ref).astype(np.float64))
            assert np.all(err <= bound), (scale, mode, np.max(err / bound))                     # (a)
            ratios[(scale, mode, e2)] = np.max(err / bound)
        # (c) the FP64 oracle, whole log-density, against long double
        od = orc.Density("logistic", d, [10.0], data=np.concatenate([X.ravel(), y]))
        full = logistic_exact(pts, X, y, 10.0)
        oerr = np.abs((od.eval(pts) - full).astype(np.float64))
        assert np.all(oerr <= 1e-3 * bound), (scale, np.max(oerr / bound))
    print(f"logistic model N={N} d={d}: max error / bound " +
          " ".join(f"{k[0]}{k[1]}{'+' if k[2] > 0 else '-' if k[2] < 0 else ''}={v:.3g}" for k, v in ratios.items()))
    assert ratios[(SCALES[-1], "rz", 0.0)] >= 1e-2                                                # (b)


@pytest.mark.parametrize("d", [17, 33, 64, 128])
@pytest.mark.parametrize("kind", GAUSS_KINDS)
def test_gaussian_model_within_bound(orc, kind, d):
    mean, cov = gaussian_case(kind, d)
    prm = cases.gaussian_params(mean, cov)
    mu, A = gaussian_matrix(prm, d)
    od = orc.Density("gaussian", d, prm)
    worst = {}
    for nsigma in (1.5, 1e3):
        x = gaussian_points(mean, cov, nsigma, 24, seed=d)
        ref = gaussian_exact(x, A, mu)
        bound = gaussian_bound(x, A, mu)
        yy = gaussian_terms(x, A, mu)[0]
        for mode in ("rz", "rn"):
            for epi in ("seq", "tree"):
                err = np.abs((gaussian_model(x, A, mu, mode, epi) - ref).astype(np.float64))
                assert np.all(err <= bound), (nsigma, mode, epi, np.max(err / bound))            # (a)
                assert np.all(err <= 1e-5 * (1.0 + yy))                                          # the published claim
                worst[(nsigma, mode, epi)] = np.max(err / bound)
        oerr = np.abs((od.eval(x) - (prm[-1] + ref)).astype(np.float64))
        assert np.all(oerr <= 1e-3 * bound), (nsigma, np.max(oerr / bound))                      # (c)
    print(f"gaussian model {kind} d={d}: max error / bound " +
          " ".join(f"{k[0]:g}{k[1]}{k[2]}={v:.3g}" for k, v in worst.items()))
    assert max(worst[(1e3, "rz", e)] for e in ("seq", "tree")) >= 1e-2                            # (b)


def test_model_reproduces_split_and_rounding():
    """The emulated pieces reconstruct what the kernels' comments promise: three RN bf16 pieces of an FP64 value within
    u of it, split3_pair exactly RN_f32(v); and the two FP32 roundings bracket the exact value."""
    v = np.random.default_rng(0).standard_normal(10_000) * np.logspace(-20, 20, 10_000)
    p = _split3_f64(v)
    assert np.all(np.abs(v - (p[0] + p[1] + p[2])) <= U * np.abs(v))
    assert np.all([np.all(_bf16_rn(q) == q) for q in p])
    q = _split3_pair(v)
    assert np.array_equal(q[0] + q[1] + q[2], v.astype(np.float32).astype(np.float64))
    rn, rz = _f32(v), _f32(v, "rz")
    assert np.all(np.abs(rz) <= np.abs(v)) and np.all(np.abs(rn - v) <= U * np.abs(v))
    assert np.all(np.abs(v - rz) < 2 * U * np.abs(v))
