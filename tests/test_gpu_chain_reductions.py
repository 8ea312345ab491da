"""The two device reductions over the stored chain, kmc_emcee_chain_moments and kmc_emcee_chain_covariance, against an
exact two-pass reference within bounds derived from the kernels' own arithmetic, across dimension, row count,
conditioning, sampler family and run progress.  GPU tests (`-m gpu`), except the reference's own check.

Notation.  u = 2^-53 (unit roundoff of binary64), gamma_m = m u / (1 - m u).  A sum of terms carried through at most m
roundings each, in any order, is sum t_i (1 + theta_i) with |theta_i| <= gamma_m; gamma_a + gamma_b <= gamma_(a+b) and
(1 + gamma_a)(1 + gamma_b) <= 1 + gamma_(a+b).  The rows are x_i (n of them), x0 = the first stored row, w = x - x0
exactly, A_a = sum |w_a|, B_ab = sum |w_a w_b|, S_a = sum w_a, S_ab = sum w_a w_b, and the exact mean and covariance
are mu = x0 + S_a / n and C_ab = (S_ab - S_a S_b / n) / (n - 1).

Device arithmetic.  Both kernels sum v = fl(x - x0) = w (1 + delta).  k is the longest chain of additions one term
goes through:
  chain_covariance  a CTA accumulates its contiguous range of at most ceil(n / 256) rows with one fma per row (v_a v_b
                    is exact inside the fma), then mh_cov_final_kernel adds the 256 partials in CTA order:
                    k = ceil(n / 256) + 256, and a product carries p = 2 roundings of its factors.
  chain_moments     each CTA adds its grid-stride elements into one shared-memory slot per column with atomics, in no
                    fixed order: J = ceil(n d / (256 G)) passes of 256 consecutive elements, at most ceil(256 / d) of
                    them in one column; then G global atomics, G = min(ceil(n d / 256), 1184):
                    k = J ceil(256 / d) + G, and v * v is rounded, p = 3.
So |S^_a - S_a| <= gamma_(k+1) A_a and |S^_ab - S_ab| <= gamma_(k+p) B_ab.  The host forms
(S^_ab - fl(fl(S^_a S^_b) / n)) / (n - 1): |S^_a S^_b - S_a S_b| <= ((1 + gamma_(k+1))^2 - 1) A_a A_b, the product and
the division by n add gamma_2 of S_a S_b / n, the subtraction and the final division gamma_2 of the result, so

    |cov_ab - C_ab| <= [gamma_(k+p+2) B_ab + gamma_(2k+6) A_a A_b / n] / (n - 1)          (variance: a = b)
    |mean_a - mu_a| <= gamma_(k+3) A_a / n + u |x0_a|                                       (fl(x0 + fl(S^_a / n)))

A bound in B_ab alone is not enough: S_a S_b / n is not bounded by B_ab off the diagonal, and the error of S^_a enters
it twice.  The one-pass formula loses what the shift by x0 does not remove: with x0 a far outlier, A_a^2 / n grows like
n |mean - x0|^2 while C_aa stays the spread.

Reference.  The stored rows as results() reads them back, sample-major.  Pass 1: each column's mean fsum(x) / n,
|m - mu| <= gamma_2 |mu| <= gamma_3 |m|.  Pass 2: the centred products d_a d_b (d = fl(x - m)) summed in blocks of
M = 256 rows in any order and the block sums added by math.fsum, then divided by n - 1.  Since
sum (x - m_a)(x - m_b) = (n - 1) C_ab + n (mu_a - m_a)(mu_b - m_b),

    |ref_ab - C_ab| <= [gamma_(M+5) sum |d_a d_b| + n gamma_3^2 |m_a m_b|] / (n - 1),   |ref_mean - mu| <= gamma_3 |m|

and every assertion allows the device bound plus the reference's.  The scales A, B and sum |d_a d_b| are evaluated in
floating point; their relative error is far below the slack of the bounds.

Each case prints its largest ratio of observed error to bound, and shows that the bound is not vacuous: leaving out
one row, or counting the row range of one covariance CTA twice, moves the reference by more than the bound.

The chains are controlled with Metropolis in replay mode: accept uniforms u = 0 make log u = -inf, so every proposal
of finite log-density is accepted, and the uploaded normals (sigma = 1) make x_t = x_(t-1) + z_t follow a chosen
sequence; the exponential target accepts any non-negative point.  Emcee runs are Philox runs, their offset and spread
set by the target and the start ball."""
import math
from fractions import Fraction

import numpy as np
import pytest

from tests import cases

U = 2.0 ** -53
BLOCK = 256
COV_GRID = 256
MOM_GRID = 148 * 8
KMC_ERR_UNSUPPORTED, KMC_ERR_STATE = 3, 4


def gamma(m):
    return m * U / (1.0 - m * U)


# ---------------------------------------------------------------------------------- reference and bounds

def _block_sums(a, b=None):
    """fsum over blocks of BLOCK rows of the column sums of a (or of a * b, per column)."""
    n = a.shape[0]
    p = a if b is None else a * b
    nb = -(-n // BLOCK)
    pad = np.zeros((nb * BLOCK,) + p.shape[1:])
    pad[:n] = p
    part = pad.reshape((nb, BLOCK) + p.shape[1:]).sum(1)
    return np.array([math.fsum(col) for col in part.reshape(nb, -1).T]).reshape(p.shape[1:])


def reference(rows, full=True):
    """(mean, cov or var, mean bound, cov or var bound) of rows [n, d] (ddof = 1): exact mean per column, then the
    centred products, block sums added by fsum.  full=False: the variances only."""
    n, d = rows.shape
    mean = np.array([math.fsum(rows[:, a]) for a in range(d)]) / n
    dev = rows - mean
    mb = gamma(3) * np.abs(mean)
    if n < 2:
        z = np.zeros((d, d)) if full else np.zeros(d)
        return mean, z, mb, z
    ad = np.abs(dev)
    if full:
        if d <= 8:
            s = np.array([[_block_sums(dev[:, a], dev[:, b]) for b in range(d)] for a in range(d)])
        else:
            nb = -(-n // BLOCK)
            pad = np.zeros((nb * BLOCK, d))
            pad[:n] = dev
            blk = pad.reshape(nb, BLOCK, d)
            part = np.matmul(blk.transpose(0, 2, 1), blk).reshape(nb, -1)
            s = np.array([math.fsum(part[:, e]) for e in range(d * d)]).reshape(d, d)
        D = ad.T @ ad
        mm = np.abs(np.outer(mean, mean))
    else:
        s = _block_sums(dev, dev)
        D = (ad * ad).sum(0)
        mm = mean * mean
    c = s / (n - 1)
    cb = (gamma(BLOCK + 5) * D + n * gamma(3) ** 2 * mm) / (n - 1) * (1 + 4 * U)
    return mean, c, mb, cb


def k_cov(n):
    return -(-n // COV_GRID) + COV_GRID


def k_mom(n, d):
    g = min(-(-n * d // 256), MOM_GRID)
    return -(-n * d // (256 * g)) * -(-256 // d) + g


def device_bound(rows, k, p, full=True):
    """(mean bound, cov or var bound) of a device reduction with longest accumulation k and p roundings per product."""
    n, d = rows.shape
    w = rows - rows[0]
    aw = np.abs(w)
    A = aw.sum(0)
    mb = gamma(k + 3) * A / n + U * np.abs(rows[0])
    if n < 2:
        return mb, np.zeros((d, d)) if full else np.zeros(d)
    if full:
        B, AA = aw.T @ aw, np.outer(A, A)
    else:
        B, AA = (aw * aw).sum(0), A * A
    return mb, (gamma(k + p + 2) * B + gamma(2 * k + 6) * AA / n) / (n - 1) * (1 + 1e-6)


def _ratio(err, bound):
    """Largest |err| / bound; an entry with a zero bound must be exact."""
    err, bound = np.abs(err), np.asarray(bound)
    r = np.where(bound > 0, err / np.where(bound > 0, bound, 1), np.where(err == 0, 0.0, np.inf))
    return float(np.max(r))


# ---------------------------------------------------------------------------------- the check every case runs

def stored_rows(th, m):
    """The first m stored samples of every walker, sample-major (the order of the device store)."""
    return np.ascontiguousarray(th[:, :m].transpose(1, 0, 2)).reshape(-1, th.shape[2])


def check_reductions(s, rows, label):
    """Both reductions of sampler s against the reference on rows, with every property asserted on each case."""
    n, d = rows.shape
    full = d <= 128
    mean_m, var_m, cnt_m = s.chain_moments()
    assert cnt_m == n, (label, cnt_m, n)
    assert np.all(var_m >= 0), label
    rm, rc, rmb, rcb = reference(rows, full)
    rvar, rvb = (np.diag(rc), np.diag(rcb)) if full else (rc, rcb)
    km_ = k_mom(n, d)
    mmb, mvb = device_bound(rows, km_, 3, full=False)
    r_mm = _ratio(mean_m - rm, mmb + rmb)
    r_mv = _ratio(var_m - rvar, mvb + rvb)
    assert r_mm <= 1 and r_mv <= 1, (label, r_mm, r_mv)
    out = f"moments k={km_}: mean {r_mm:.3g} var {r_mv:.3g}"
    if full:
        mean_c, cov_c, cnt_c = s.chain_covariance()
        assert cnt_c == n, (label, cnt_c, n)
        assert np.array_equal(cov_c, cov_c.T), label
        assert np.all(np.diag(cov_c) >= 0), label
        kc = k_cov(n)
        cmb, ccb = device_bound(rows, kc, 2)
        r_cm = _ratio(mean_c - rm, cmb + rmb)
        r_cc = _ratio(cov_c - rc, ccb + rcb)
        assert r_cm <= 1 and r_cc <= 1, (label, r_cm, r_cc)
        # the two device results against each other: both within their bounds of the exact values
        assert _ratio(np.diag(cov_c) - var_m, np.diag(ccb) + mvb) <= 1, label
        assert _ratio(mean_c - mean_m, cmb + mmb) <= 1, label
        again = s.chain_covariance()
        assert np.array_equal(again[0], mean_c) and np.array_equal(again[1], cov_c) and again[2] == cnt_c, label
        out += f" | covariance k={kc}: mean {r_cm:.3g} cov {r_cc:.3g}"
    # the bounds are not vacuous: one row less, or one CTA's row range counted twice, moves the reference beyond them
    if n >= 2 and np.any(rows != rows[0]):
        mbound = mmb + rmb
        vbound = (ccb + rcb) if full else (mvb + rvb)
        moved = []
        perturbed = [rows[np.r_[0:n - 2, n - 1]]] if n >= 3 else []
        perturbed.append(np.concatenate([rows, rows[n * (COV_GRID - 1) // COV_GRID:]]))
        for q in perturbed:
            pm, pc, _, _ = reference(q, full)
            a, b = _ratio(pm - rm, mbound), _ratio(pc - rc, vbound)
            assert a > 1 and b > 1, (label, a, b)
            moved.append(f"{min(a, b):.3g}")
        out += f" | perturbed reference / bound >= {', '.join(moved)}"
    print(f"\n{label}: n={n} d={d}  max error / bound  {out}")


def expect_state(km, s):
    """No sample stored yet: both reductions refuse."""
    for f in (s.chain_moments, s.chain_covariance):
        with pytest.raises(km.KmcError) as e:
            f()
        assert e.value.code == KMC_ERR_STATE, e.value


# ---------------------------------------------------------------------------------- designed Metropolis chains

SPREAD = 0.37


def design(rng, steps, nchains, d, offset, kind):
    """Chosen states [steps, nchains, d], all >= 0 (the exponential target): offset / spread = `offset`."""
    y = SPREAD * (offset + rng.uniform(-1.0, 1.0, (steps, nchains, d)))
    if kind == "outlier":      # the first stored row far out: x0 an outlier of the chain
        y[0] += SPREAD * 1e6
    elif kind == "const":      # every row the same
        y[:] = y[0, 0]
    elif kind == "onecol":     # column 0 constant, the others move
        y[:, :, 0] = y[0, 0, 0]
    return y


def metropolis_designed(km, y, nburnin=0, nthin=1):
    """A replay-mode Metropolis handle whose chain visits the states y [steps, nchains, d], and those states as the
    device computes them (x + 1.0 * z, rounded once)."""
    steps, nchains, d = y.shape
    x = y[0].copy()          # start at the first state: step 0 proposes z = 0
    z, xs = np.empty_like(y), np.empty_like(y)
    for t in range(steps):
        z[t] = y[t] - x
        x = x + z[t]
        xs[t] = x
    s = km.Metropolis(km.exponential(d), y[0], km.normal_proposal(1.0), steps, nburnin, nthin, mode=km.MODE_REPLAY)
    s.set_replay(z, np.zeros((steps, nchains)))
    return s, xs


def stored_steps(done, nburnin, nthin):
    """0-based iterations < done at which a sample is stored (the reference's n > 0 && rem(n, nthin) == 0)."""
    t = np.arange(done)
    n = t + 1 - nburnin
    return t[(n > 0) & (n % nthin == 0)]


MH_CASES = [  # (d, chains, steps, offset / spread, kind): rows = chains * steps
    (1, 1, 1, 1e4, "bulk"),           # 1 row: var = cov = 0, mean = the row
    (2, 2, 1, 1.0, "bulk"),           # 2
    (7, 3, 5, 1e8, "bulk"),           # 15, batched path
    (31, 4, 4, 1.0, "outlier"),       # 16
    (32, 17, 1, 1e4, "bulk"),         # 17
    (33, 15, 17, 1e8, "onecol"),      # 255
    (127, 16, 16, 1e4, "bulk"),       # 256
    (128, 257, 1, 1.0, "bulk"),       # 257; P = 8385 = 32 * 256 + 193 entries: the last per-thread slot partly filled
    (128, 64, 9, 1e8, "outlier"),
    (2, 17, 241, 1e8, "bulk"),        # 4097, fused path
    (16, 64, 33, 1e4, "outlier"),     # fused path at its largest d
    (3, 16, 16, 1e4, "const"),        # constant chain: 0 exactly
    (5, 16, 16, 1.0, "onecol"),
    (1, 1024, 297, 1e4, "bulk"),      # 304128 rows > 148 * 8 * 256: the moments grid-stride loop wraps
    (1, 1024, 297, 1.0, "outlier"),
    # moments only above d = 128 (the covariance refuses)
    (129, 3, 40, 1.0, "outlier"),
    (1000, 3, 20, 1e8, "bulk"),
    (3072, 2, 12, 1e4, "bulk"),       # 16 d = 48 KiB of shared memory: the last d without the opt-in
    (3073, 3, 10, 1.0, "bulk"),
    (4096, 2, 16, 1e8, "onecol"),     # the largest d a plugin accepts
    (4096, 3, 5, 1.0, "outlier"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("d,nchains,steps,offset,kind", MH_CASES)
def test_metropolis_designed_chain(km, d, nchains, steps, offset, kind):
    """A chosen chain on the fused (d <= 16) or batched Metropolis path: both reductions within their bounds; a
    constant chain and a single row exactly; above d = 128 the covariance refuses and the moments still hold."""
    rng = np.random.default_rng(d * 1000 + steps)
    y = design(rng, steps, nchains, d, offset, kind)
    s, xs = metropolis_designed(km, y)
    try:
        s.run(-1)
        th, _, _ = s.results()
        assert np.array_equal(th, xs.transpose(1, 0, 2)), "the replayed chain is not the designed one"
        rows = stored_rows(th, steps)
        if kind == "const":
            assert np.array_equal(s.chain_moments()[1], np.zeros(d))
            assert np.array_equal(s.chain_covariance()[1], np.zeros((d, d)))
        if d > 128:
            with pytest.raises(km.KmcError) as e:
                s.chain_covariance()
            assert e.value.code == KMC_ERR_UNSUPPORTED
        if rows.shape[0] == 1:
            m, v, n = s.chain_moments()
            mc, c, nc = s.chain_covariance()
            assert n == nc == 1 and np.array_equal(m, rows[0]) and np.array_equal(mc, rows[0])
            assert np.array_equal(v, np.zeros(d)) and np.array_equal(c, np.zeros((d, d)))
        check_reductions(s, rows, f"metropolis {kind} offset/spread={offset:g} chains={nchains} steps={steps}")
    finally:
        s.close()


# ---------------------------------------------------------------------------------- emcee families (Philox)

def _emcee(km, ld, x0, niter, nburnin, nthin, seed, **kw):
    s = km.Sampler(ld, x0, niter, nburnin, nthin, 2.0, seed, **kw)
    s.run(-1)
    th, _, _ = s.results()
    return s, th


@pytest.mark.gpu
def test_emcee_families(km):
    """One case per kernel family; the reductions read the same store whatever wrote it."""
    runs = [
        ("shared-memory kernel, rosenbrock", km.rosenbrock(), cases.ball([0.0, 0.0], 0.1, 512, 1), 40, 10, 3, {}),
        ("bulk kernel, 10-D gaussian at 1e4", km.gaussian(np.full(10, 1e4), cases.spd_cov(10, 2)),
         cases.ball(np.full(10, 1e4), 0.5, 1 << 18, 2), 8, 4, 1, {}),
        ("one launch per half-step, exponential d=5", km.exponential(5),
         1.0 + np.abs(cases.ball(np.zeros(5), 0.3, 600, 3)), 30, 6, 2, dict(launch_mode=1)),
        ("batched plugin, 31-D gaussian", km.gaussian(np.linspace(-3, 3, 31), cases.spd_cov(31, 4)),
         cases.ball(np.linspace(-3, 3, 31), 0.4, 256, 4), 24, 8, 2, {}),
        ("bench shape, rosenbrock 2^20 walkers x 32 samples", km.rosenbrock(), cases.ball([0.0, 0.0], 0.1, 1 << 20, 5),
         36, 4, 1, {}),
        ("batched plugin, exponential d=3073, 3076 walkers", km.exponential(3073),
         1.0 + np.abs(cases.ball(np.zeros(3073), 0.3, 3076, 6)), 3, 0, 1, {}),
    ]
    for i, (label, ld, x0, niter, nburnin, nthin, kw) in enumerate(runs):
        s, th = _emcee(km, ld, x0, niter, nburnin, nthin, seed=40 + i, **kw)
        try:
            check_reductions(s, stored_rows(th, s.ns), f"emcee {label}")
        finally:
            s.close()
        del th


# ---------------------------------------------------------------------------------- run progress

@pytest.mark.gpu
def test_metropolis_mid_run(km):
    """Before any run and during burn-in both reductions refuse; after each chunk past burn-in (nthin = 3) they reduce
    exactly the samples stored so far; reductions called mid-run leave the finished chain's result unchanged."""
    nburnin, nthin, nstored, nchains, d = 5, 3, 20, 40, 3
    steps = nburnin + nthin * nstored
    y = design(np.random.default_rng(7), steps, nchains, d, 1e4, "bulk")
    s, xs = metropolis_designed(km, y, nburnin, nthin)
    t_store = stored_steps(steps, nburnin, nthin)
    assert len(t_store) == nstored == s.ns
    try:
        expect_state(km, s)
        done = 0
        for chunk in (3, 2, 1, 7, 7, 11, 100):
            s.run(chunk)
            done = min(steps, done + chunk)
            m = len(stored_steps(done, nburnin, nthin))
            if m == 0:
                expect_state(km, s)
                continue
            th, _, _ = s.results()
            assert np.array_equal(th[:, :m], xs[t_store[:m]].transpose(1, 0, 2))
            check_reductions(s, stored_rows(th, m), f"metropolis after {done} of {steps} steps ({m} samples)")
        final = s.chain_covariance()
    finally:
        s.close()
    s, _ = metropolis_designed(km, y, nburnin, nthin)
    try:
        s.run(-1)
        whole = s.chain_covariance()
    finally:
        s.close()
    # the covariance's order is fixed, so its bits; the moments add with atomics in no fixed order (checked above)
    assert all(np.array_equal(u, v) for u, v in zip(final, whole))


@pytest.mark.gpu
def test_emcee_mid_run(km):
    """Emcee: refused before the first run and during burn-in; after run(k) past burn-in (nthin = 3) the samples
    stored so far; after an odd number of half-steps only the complete samples; the finished chain unchanged."""
    ld = km.gaussian([0.5, -0.25, 2.0], cases.spd_cov(3, 9))
    x0 = cases.ball([0.5, -0.25, 2.0], 0.3, 256, 9)
    nburnin, nthin, niter = 4, 3, 4 + 3 * 10
    s = km.Sampler(ld, x0, niter, nburnin, nthin, 2.0, 12)
    try:
        expect_state(km, s)
        s.run(3)
        expect_state(km, s)                     # iterations 0..2: burn-in
        done = 3
        for k in (1, 1, 5, 1, 1):
            s.run(k)
            done += k
            m = len(stored_steps(done, nburnin, nthin))
            if m == 0:
                expect_state(km, s)
                continue
            th, _, _ = s.results()
            check_reductions(s, stored_rows(th, m), f"emcee after {done} of {niter} iterations ({m} samples)")
        for h in (1, 5):                    # odd totals: the unfinished iteration (12, then 15) stores a sample
            s.run_half(h, sync=True)
            m = len(stored_steps(done + h // 2, nburnin, nthin))
            assert len(stored_steps(done + h // 2 + 1, nburnin, nthin)) == m + 1
            th, _, _ = s.results()
            check_reductions(s, stored_rows(th, m), f"emcee after {2 * done + h} half-steps ({m} complete samples)")
            s.run_half(1, sync=True)
            done += (h + 1) // 2
        s.run(-1)
        th_final, _, _ = s.results()
        check_reductions(s, stored_rows(th_final, s.ns), f"emcee chunked, finished ({s.ns} samples)")
        final = s.chain_covariance()
    finally:
        s.close()
    s = km.Sampler(ld, x0, niter, nburnin, nthin, 2.0, 12)
    try:
        s.run(-1)
        th_whole, _, _ = s.results()
        whole = s.chain_covariance()
    finally:
        s.close()
    assert np.array_equal(th_final, th_whole)
    assert all(np.array_equal(u, v) for u, v in zip(final, whole))


@pytest.mark.gpu
def test_stale_rows_of_a_reused_block(km):
    """Sampler A runs to the end with its chain at 1e6 and is closed; B, of the same shape, gets A's cached chain
    block and runs partway: B's reductions see only B's stored rows."""
    d, nchains, steps, nthin = 3, 256, 40, 2
    km.trim()
    ya = design(np.random.default_rng(1), steps, nchains, d, 1e6 / SPREAD, "bulk")
    a, _ = metropolis_designed(km, ya, 0, nthin)
    a.run(-1)
    a.close()
    yb = design(np.random.default_rng(2), steps, nchains, d, 3.0, "bulk")
    b, _ = metropolis_designed(km, yb, 0, nthin)
    try:
        b.run(15)
        m = len(stored_steps(15, 0, nthin))
        th, _, _ = b.results()
        assert np.all(th[:, m:] > 1e5), "B did not get A's chain block: the case tests nothing"
        check_reductions(b, stored_rows(th, m), f"stale block: B after 15 of {steps} steps ({m} samples)")
    finally:
        b.close()


# ---------------------------------------------------------------------------------- the reference itself (CPU)

def test_reference_against_exact_fractions():
    """The reference's mean and covariance against exact rational arithmetic, within its stated bound, on chains with
    a large offset (1e8 times the spread) and with a far outlier; and the device bound's scales on the same rows."""
    rng = np.random.default_rng(3)
    for kind in ("offset", "outlier"):
        n, d = 300, 4
        rows = 1e8 + rng.standard_normal((n, d)) * np.array([1.0, 1e-3, 7.0, 1.0])
        rows[:, 3] = 0.5 * rows[:, 0] + 1e-6 * rows[:, 3]
        if kind == "outlier":
            rows[0] += 1e6
        mean, cov, mb, cb = reference(rows)
        fr = [[Fraction(float(v)) for v in r] for r in rows]
        mu = [sum(r[a] for r in fr) / n for a in range(d)]
        for a in range(d):
            assert abs(Fraction(float(mean[a])) - mu[a]) <= Fraction(float(mb[a])), (kind, a)
            for b in range(d):
                c = sum((r[a] - mu[a]) * (r[b] - mu[b]) for r in fr) / (n - 1)
                err = abs(Fraction(float(cov[a, b])) - c)
                assert err <= Fraction(float(cb[a, b])), (kind, a, b, float(err), cb[a, b])
                assert cb[a, b] < 1e-6 * max(abs(float(c)), math.sqrt(abs(cov[a, a] * cov[b, b])))
        v_only = reference(rows, full=False)
        assert np.all(np.abs(v_only[1] - np.diag(cov)) <= 2 * np.diag(cb))
        np.testing.assert_allclose(v_only[3], np.diag(cb), rtol=1e-12)
    one = reference(rows[:1])
    assert np.array_equal(one[0], rows[0]) and not np.any(one[1])


def test_accumulation_lengths():
    """k of both kernels at the shapes the GPU cases use: the covariance CTA ranges and the moments grid."""
    assert k_cov(1) == 257 and k_cov(256) == 257 and k_cov(257) == 258 and k_cov(1 << 25) == (1 << 17) + 256
    assert k_mom(1, 1) == 256 + 1                  # one CTA: at most 256 elements of a column per pass
    assert k_mom(304128, 1) == 2 * 256 + 1184      # grid-stride loop wraps once
    assert k_mom(1 << 25, 2) == 222 * 128 + 1184
    assert k_mom(9228, 3073) == 94 + 1184
