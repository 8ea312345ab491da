"""The Gaussian-mixture plugin on the B200: device log-density against the oracle, the K = 1 identity with the
Gaussian plugin through eval, emcee and Metropolis, emcee parity with the oracle through every fused kernel family
(the shared-memory kernel K1, the general kernel, the bulk kernel, the push kernel), split runs, Metropolis parity with
both proposals, the statistics of the mixture's moments and weights, and a full-size run."""
import math

import numpy as np
import pytest

from tests import cases
from tests.test_metropolis_chol_host import random_chol
from tests.test_mixture_host import mixture_cases, mixture_points, random_mixture

pytestmark = pytest.mark.gpu

EVAL_TOL = 1e-14        # exp / log ulp budget, relative to 1 + |logp|


@pytest.fixture(scope="module")
def mxo():
    from mixture_oracle import oracle
    return oracle


def _pair(km, mxo, d, K, seed):
    w, mus, covs = random_mixture(d, K, seed)
    ld = km.gaussian_mixture(w, mus, covs)
    return ld, mxo.Density("gaussian_mixture", d, km.gaussian_mixture_params(w, mus, covs)), mus


def _close(got, want):
    assert np.array_equal(np.isfinite(got), np.isfinite(want))
    f = np.isfinite(want)
    np.testing.assert_array_less(np.abs(got[f] - want[f]), EVAL_TOL * (1 + np.abs(want[f])))


@pytest.mark.parametrize("d,K", mixture_cases())
def test_eval_matches_the_oracle(km, mxo, d, K):
    w, mus, covs = random_mixture(d, K, d * 7 + K)
    ld = km.gaussian_mixture(w, mus, covs)
    od = mxo.Density("gaussian_mixture", d, km.gaussian_mixture_params(w, mus, covs))
    x = mixture_points(w, mus, covs, seed=K)
    got, want = ld.eval(x), od.eval(x)
    assert np.all(np.isfinite(got)) and np.all(got[64:80] < -1490)      # far tails: every exp(l_k) underflows
    _close(got, want)
    x[3, 0] = math.nan
    assert math.isnan(ld.eval(x)[3])


def _emcee(km, ld, x0, nitw, nbw, nthin, seed=0, replay=None, launch_mode=0, split=None):
    s = km.Sampler(ld, x0, nitw, nbw, nthin, 2.0, seed, km.MODE_REPLAY if replay is not None else km.MODE_PHILOX,
                   launch_mode=launch_mode)
    try:
        if replay is not None:
            s.set_replay(*replay)
        if split:
            done = 0
            while done < nitw:
                s.run(min(split, nitw - done))
                done += split
        else:
            s.run(-1)
        th, lp, ar = s.results()
        x, l, na = s.state()
    finally:
        s.close()
    return th, lp, ar, x, l, na


def _check(got, want):
    th, lp, ar, x, l, na = got
    assert np.array_equal(th, want["chain_x"]) and np.array_equal(x, want["x"])          # states bit-exact
    assert np.array_equal(ar, want["accept_ratio"]) and np.array_equal(na, want["naccept"])
    _close(lp.ravel(), want["chain_lp"].ravel())
    _close(l, want["lp"])


def _same(a, b):
    for u, v in zip(a, b):
        assert np.array_equal(u, v)


@pytest.mark.parametrize("d", [1, 2, 3, 10, 16])
def test_k1_is_the_gaussian_bit_for_bit(km, d):
    mean, cov = np.linspace(-1, 1, d), cases.spd_cov(d, d)
    mix, gau = km.gaussian_mixture([1.0], mean[None], cov[None]), km.gaussian(mean, cov)
    x = mean + cases.ball(np.zeros(d), 1.5, 5000, d)
    assert np.array_equal(mix.eval(x), gau.eval(x))
    nw = max(64, 2 * d + 4)
    x0 = mean + cases.ball(np.zeros(d), 0.3, nw, 1)
    for mode_kw in (dict(), dict(launch_mode=1)):
        _same(_emcee(km, mix, x0, 60, 20, 2, seed=5, **mode_kw), _emcee(km, gau, x0, 60, 20, 2, seed=5, **mode_kw))
    L = random_chol(d, 2, 0.3)
    for prop in (km.normal_proposal(0.4), km.normal_proposal(chol=L)):
        runs = []
        for ld in (mix, gau):
            s = km.Metropolis(ld, x0, prop, 80, 20, 2, seed=6)
            s.run(-1)
            runs.append((*s.results(), *s.state()))
            s.close()
        _same(*runs)


# Which kernel runs (kmc_emcee_create): d <= 4 with launch_mode 0 runs the shared-memory kernel K1 in both modes (the
# state of these ensembles fits in shared memory); d = 10 with launch_mode 0 runs the bulk kernel in Philox mode and
# the general persistent kernel in replay mode; launch_mode 1 runs the general kernel, one launch per half-step.
EMCEE_CASES = [(1, 3, 0), (2, 4, 0), (10, 4, 0), (1, 3, 1), (2, 4, 1), (10, 4, 1)]


@pytest.mark.parametrize("replay", [False, True])
@pytest.mark.parametrize("d,K,launch_mode", EMCEE_CASES)
def test_emcee_matches_the_oracle(km, mxo, d, K, launch_mode, replay):
    ld, od, mus = _pair(km, mxo, d, K, 40 + d)
    nw, nitw, nbw, nthin, seed = 2048, 60, 20, 3, 11 + d
    x0 = mus[np.arange(nw) % K] + cases.ball(np.zeros(d), 0.5, nw, d)
    want = mxo.emcee(od, x0, nitw, nbw, nthin, 2.0, seed=seed, trace=replay, nthreads=8)
    if replay:          # draws of the Philox run, uploaded: the same decisions through the replay kernels
        want = mxo.emcee(od, x0, nitw, nbw, nthin, 2.0, replay=want["trace"][:3], nthreads=8) | dict(tr=want["trace"])
    print(f"d={d} K={K} launch_mode={launch_mode} replay={replay}: margin {want['min_margin']:.3e}, "
          f"accept {want['accept_ratio'].mean():.3f}")
    assert want["min_margin"] > 1e-11
    assert 0.01 < want["accept_ratio"].mean() < 0.99
    got = _emcee(km, ld, x0, nitw, nbw, nthin, seed=seed, replay=want["tr"][:3] if replay else None,
                 launch_mode=launch_mode)
    _check(got, want)


@pytest.mark.parametrize("d,K", [(2, 4), (10, 4)])
def test_split_runs_and_launch_mode_equal_the_one_shot_run(km, d, K):
    w, mus, covs = random_mixture(d, K, 3)
    ld = km.gaussian_mixture(w, mus, covs)
    x0 = mus[np.arange(4096) % K] + cases.ball(np.zeros(d), 0.5, 4096, 2)
    one = _emcee(km, ld, x0, 90, 30, 4, seed=8)
    for kw in (dict(split=7), dict(split=1), dict(launch_mode=1), dict(launch_mode=1, split=13)):
        _same(one, _emcee(km, ld, x0, 90, 30, 4, seed=8, **kw))


def _metro(km, ld, x0, prop, niter, nburnin, nthin, seed=0, replay=None):
    s = km.Metropolis(ld, x0, prop, niter, nburnin, nthin, seed, km.MODE_REPLAY if replay is not None else km.MODE_PHILOX)
    try:
        if replay is not None:
            s.set_replay(*replay)
        s.run(-1)
        th, lp, ar = s.results()
        x, l, na = s.state()
    finally:
        s.close()
    return th, lp, ar, x, l, na


@pytest.mark.parametrize("replay", [False, True])
@pytest.mark.parametrize("chol", [False, True])
@pytest.mark.parametrize("d,K", [(2, 4), (10, 4)])
def test_metropolis_matches_the_oracle(km, mxo, d, K, chol, replay):
    ld, od, mus = _pair(km, mxo, d, K, 60 + d)
    nc, niter, nburnin, nthin, seed = 1000, 80, 30, 2, 17
    x0 = mus[np.arange(nc) % K] + cases.ball(np.zeros(d), 0.5, nc, 3)
    L = random_chol(d, 5, 0.6 / math.sqrt(d))
    sigma = np.linspace(0.2, 0.6, d) / math.sqrt(d)
    if replay:
        rng = np.random.default_rng(d)
        normals, u = rng.standard_normal((niter, nc, d)), rng.random((niter, nc))
    else:
        normals, u = km.metropolis_draws(seed, 0, nc, 0, niter, d)
    want = mxo.metropolis(od, x0, None if chol else sigma, niter, nburnin, nthin, normals, u, nthreads=8,
                          chol=L if chol else None)
    assert want["min_margin"] > 1e-11
    assert 0.01 < want["accept_ratio"].mean() < 0.99
    prop = km.normal_proposal(chol=L) if chol else km.normal_proposal(sigma)
    _check(_metro(km, ld, x0, prop, niter, nburnin, nthin, seed=seed, replay=(normals, u) if replay else None), want)


def test_sharded_push_kernel_equals_the_single_gpu_run(km):
    d, K = 10, 4
    w, mus, covs = random_mixture(d, K, 9)
    ld = km.gaussian_mixture(w, mus, covs)
    nw, nitw, nbw, nthin = 8192, 40, 10, 3
    x0 = mus[np.arange(nw) % K] + cases.ball(np.zeros(d), 0.5, nw, 4)
    th, lp, ar, *_ = _emcee(km, ld, x0, nitw, nbw, nthin, seed=21)
    m = km.MultiSampler(ld, x0, nitw, nbw, nthin, 2.0, 21, devices=[0, 0], sharded=True)
    try:
        m.run(-1)
        _same((th, lp, ar), m.results())
    finally:
        m.close()


MOM_W = np.array([0.5, 0.3, 0.2])
MOM_MU = np.array([[0.0, 0.0], [1.5, 0.5], [-1.0, 1.5]])
MOM_COV = np.array([[[1.0, 0.3], [0.3, 0.8]], [[0.6, -0.2], [-0.2, 1.2]], [[0.9, 0.0], [0.0, 0.5]]])


def _sample_mixture(w, mus, covs, n, seed):
    rng = np.random.default_rng(seed)
    k = rng.choice(len(w), size=n, p=np.asarray(w) / np.sum(w))
    return np.stack([rng.multivariate_normal(mus[c], covs[c]) for c in k]) if mus.shape[1] > 1 else \
        (mus[k, 0] + np.sqrt(covs[k, 0, 0]) * rng.standard_normal(n))[:, None]


def _moment_check(km, s, label):
    """mean and covariance from chain_covariance() against the analytic mixture moments.  Tolerance: 5 standard errors
    of a correlated chain, sqrt(Var[f] * tau / N) with N the stored rows, tau the largest int_acorr time of the
    walkers' chains (in stored samples) and Var[f] the sample variance of f = x_i (means) or of
    f = (x_i - m_i)(x_j - m_j) (covariances)."""
    th, _, _ = s.results()
    mean, cov, n = s.chain_covariance()
    rows = th.reshape(-1, 2)
    assert n == rows.shape[0]
    tau, _ = km.int_acorr(th[:2048], warn=False)
    tmax = max(1.0, float(np.max(tau)))
    m = MOM_W @ MOM_MU
    C = sum(MOM_W[k] * (MOM_COV[k] + np.outer(MOM_MU[k], MOM_MU[k])) for k in range(3)) - np.outer(m, m)
    se_mean = np.sqrt(rows.var(0) * tmax / n)
    cen = rows - rows.mean(0)
    prod = cen[:, :, None] * cen[:, None, :]
    se_cov = np.sqrt(prod.reshape(n, 4).var(0).reshape(2, 2) * tmax / n)
    print(f"{label}: tau {tau}, mean {mean} (want {m}, 5 se {5 * se_mean}), cov {cov.ravel()} (want {C.ravel()}, "
          f"5 se {5 * se_cov.ravel()})")
    assert np.all(np.abs(mean - m) < 5 * se_mean)
    assert np.all(np.abs(cov - C) < 5 * se_cov)


def test_statistics_moments_emcee_and_metropolis(km):
    ld = km.gaussian_mixture(MOM_W, MOM_MU, MOM_COV)
    n = 2**14
    x0 = _sample_mixture(MOM_W, MOM_MU, MOM_COV, n, 1)
    s = km.Sampler(ld, x0, 2000, 500, 5, 2.0, 31)
    s.run(-1)
    _moment_check(km, s, "emcee")
    s.close()
    m = MOM_W @ MOM_MU
    Ctot = sum(MOM_W[k] * (MOM_COV[k] + np.outer(MOM_MU[k], MOM_MU[k])) for k in range(3)) - np.outer(m, m)
    s = km.Metropolis(ld, x0, km.normal_proposal(cov=2.38**2 / 2 * Ctot), 2000, 500, 5, seed=32)
    s.run(-1)
    _moment_check(km, s, "metropolis")
    s.close()


def test_statistics_weights_of_a_bimodal_target(km):
    """Modes at -3 and +3 (unit sigma), weights 0.3 / 0.7; the ensemble starts split 50 / 50, so only the weights can
    move the fraction above 0 to 0.7.  Error: the standard error of the mean of the walkers' own fractions, std / sqrt(nw)
    (it carries the autocorrelation of each walker's indicator chain, which int_acorr cannot take: a walker that never
    changes mode has a constant chain)."""
    ld = km.gaussian_mixture([0.3, 0.7], [-3.0, 3.0], [1.0, 1.0])
    nw = 2**14
    rng = np.random.default_rng(2)
    x0 = np.where(np.arange(nw) % 2 == 0, -3.0, 3.0) + rng.standard_normal(nw)
    th, ar, _, _ = km.emcee(ld, x0, niter=6000 * nw, nburnin=2000 * nw, nthin=10, use_progress_meter=False, seed=4)
    per_walker = (th > 0).mean(axis=1)                 # th [nw, ns]
    frac = per_walker.mean()
    se = per_walker.std(ddof=1) / math.sqrt(nw)
    print(f"fraction above 0: {frac:.5f}, se {se:.2e} (iid samples: {math.sqrt(0.21 / th.size):.2e}), "
          f"accept {ar.mean():.3f}")
    assert abs(frac - 0.7) < 5 * se


def test_full_size(km):
    d, K, nw, nitw, nthin = 2, 4, 2**20, 16, 1
    w, mus, covs = random_mixture(d, K, 12)
    ld = km.gaussian_mixture(w, mus, covs)
    x0 = km.make_theta0s(mus[0], 0.5, ld, nw, seed=3)
    assert x0.shape == (nw, d)
    assert np.all(np.isfinite(ld.eval(x0)))
    s = km.Sampler(ld, x0, nitw, 0, nthin, 2.0, 7)
    s.run(-1)
    th, lp, ar = s.results()
    _, _, na = s.state()
    s.close()
    assert np.array_equal(lp.ravel(), ld.eval(th.reshape(-1, d)))            # stored logp == eval(stored theta)
    tr = np.concatenate([x0[:, None, :], th], axis=1)
    changes = np.any(tr[:, 1:] != tr[:, :-1], axis=2).sum(1)
    assert np.array_equal(changes, na)                                          # accept counts == state changes
    assert np.array_equal(np.round(ar * nitw).astype(np.int64), na)
    assert 0.1 < ar.mean() < 0.9
