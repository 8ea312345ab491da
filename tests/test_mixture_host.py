"""The Gaussian-mixture plugin without a GPU: the oracle's log-density against scipy's logsumexp of MvNormal
log-densities (near the modes and in tails where every component underflows exp), its K = 1 identity with the
Gaussian plugin, the parameter packing, and every validation error of kmc_density_create and gaussian_mixture."""
import math

import numpy as np
import pytest
from scipy.special import logsumexp
from scipy.stats import multivariate_normal

from tests import cases

@pytest.fixture(scope="module")
def mxo():
    from mixture_oracle import oracle
    return oracle


KMAX = {1: 90, 2: 45, 3: 27, 4: 18, 5: 12, 6: 9, 8: 6, 10: 4, 12: 2, 16: 1}


def q(d):
    return d + d * (d + 1) // 2 + 1


def random_mixture(d, K, seed, spread=2.0):
    """weights [K], means [K, d], covs [K, d, d]: well-conditioned components with distinct means."""
    rng = np.random.default_rng(seed)
    w = 0.2 + rng.random(K)
    mus = spread * rng.standard_normal((K, d))
    covs = np.stack([cases.spd_cov(d, seed * 101 + k) * (0.3 + rng.random()) for k in range(K)])
    return w, mus, covs


def scipy_logpdf(w, mus, covs, x):
    lw = np.log(np.asarray(w) / np.sum(w))
    return logsumexp(np.stack([lw[k] + multivariate_normal(mus[k], covs[k]).logpdf(x) for k in range(len(w))]),
                     axis=0)


def mixture_points(w, mus, covs, n_near=64, seed=0):
    """Points near the modes and in the far tails (every l_k < -745 there: a naive sum of exp underflows to 0)."""
    rng = np.random.default_rng(seed)
    K, d = mus.shape
    near = mus[rng.integers(0, K, n_near)] + 0.7 * rng.standard_normal((n_near, d))
    dirs = rng.standard_normal((16, d))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    far = mus[0] + np.array([200.0, 1e3, 3e4, 1e6])[:, None, None] * dirs[None, :4]
    return np.concatenate([near, far.reshape(-1, d), mus])


def mixture_cases():
    """(d, K) pairs of the evaluation tests: K in {1, 3, Kmax} at d in {1, 2, 10}."""
    return [(d, K) for d in (1, 2, 10) for K in sorted({1, min(3, KMAX[d]), KMAX[d]})]


@pytest.mark.parametrize("d,K", mixture_cases())
def test_oracle_matches_scipy_logsumexp(km, mxo, d, K):
    w, mus, covs = random_mixture(d, K, d * 7 + K)
    od = mxo.Density("gaussian_mixture", d, km.gaussian_mixture_params(w, mus, covs))
    x = mixture_points(w, mus, covs, seed=K)
    got = od.eval(x)
    want = scipy_logpdf(w, mus, covs, x)
    assert np.all(np.isfinite(got))
    assert np.all(want[-(len(mus)):] > -50)                       # the modes themselves
    tails = got[64:64 + 16]
    assert np.all(tails < -745 * 2)                               # every component underflows exp() there
    np.testing.assert_array_less(np.abs(got - want), 1e-12 * (1 + np.abs(want)))


def test_oracle_nan_and_minus_inf(km, mxo):
    w, mus, covs = random_mixture(2, 3, 1)
    od = mxo.Density("gaussian_mixture", 2, km.gaussian_mixture_params(w, mus, covs))
    assert math.isnan(od.logpdf([math.nan, 0.0]))
    assert od.logpdf([math.inf, 0.0]) == -math.inf


@pytest.mark.parametrize("d", [1, 2, 3, 10, 16])
def test_oracle_k1_is_the_gaussian_bit_for_bit(km, orc, mxo, d):
    mean, cov = np.linspace(-1, 1, d), cases.spd_cov(d, d)
    mix = mxo.Density("gaussian_mixture", d, km.gaussian_mixture_params([1.0], mean[None], cov[None]))
    gau = orc.Density("gaussian", d, km.gaussian_params(mean, cov))
    x = mean + cases.ball(np.zeros(d), 1.5, 500, d)
    x = np.concatenate([x, mean + 1e3 * cases.ball(np.zeros(d), 1.0, 20, 1)])
    assert np.array_equal(mix.eval(x), gau.eval(x))


@pytest.mark.parametrize("name", ["rosenbrock", "mvn2", "mvn10", "lognormal", "exponential3"])
def test_oracle_loops_equal_the_emcee_and_metropolis_oracles_on_their_plugins(orc, mxo, name):
    """kmo_mix_emcee and kmo_mix_metropolis restate kmo_emcee and kmo_metropolis_loop: on every other plugin they give
    the same bits, in Philox and replay mode and with both proposals."""
    from metropolis_oracle import oracle as mo
    pname, d, params, theta0, _ = cases.plugin_specs()[name]
    base, mix = orc.Density(pname, d, params), mxo.Density(pname, d, params)
    x0 = cases.ball(theta0, 0.1, 64, 2)
    want = orc.emcee(base, x0, 40, 10, 3, 2.0, seed=9, trace=True, nthreads=2)
    got = mxo.emcee(mix, x0, 40, 10, 3, 2.0, seed=9, trace=True, nthreads=2)
    for k in ("chain_x", "chain_lp", "accept_ratio", "naccept", "x", "lp", "min_margin"):
        assert np.array_equal(got[k], want[k]), k
    assert all(np.array_equal(a, b) for a, b in zip(got["trace"], want["trace"]))
    rp = want["trace"][:3]
    a, b = orc.emcee(base, x0, 40, 10, 3, 2.0, replay=rp), mxo.emcee(mix, x0, 40, 10, 3, 2.0, replay=rp)
    assert all(np.array_equal(a[k], b[k]) for k in ("chain_x", "chain_lp", "naccept", "x", "lp"))
    rng = np.random.default_rng(d)
    normals, u = rng.standard_normal((50, 16, d)), rng.random((50, 16))
    L = np.tril(rng.standard_normal((d, d))) * 0.1 + np.diag(np.full(d, 0.3))
    for sigma, chol in ((np.linspace(0.2, 0.5, d), None), (None, L)):
        a = mo.metropolis(base, x0[:16], sigma, 50, 10, 2, normals, u, chol=chol)
        b = mxo.metropolis(mix, x0[:16], sigma, 50, 10, 2, normals, u, chol=chol)
        for k in ("chain_x", "chain_lp", "accept_ratio", "naccept", "x", "lp", "min_margin"):
            assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("d,K", [(1, 3), (2, 4), (3, 27), (10, 4), (16, 1)])
def test_packing_round_trips(km, d, K):
    w, mus, covs = random_mixture(d, K, 3 * d + K)
    p = km.gaussian_mixture_params(w, mus, covs)
    assert p.size == K * q(d)
    iu = np.triu_indices(d)
    for k, pk in enumerate(p.reshape(K, q(d))):
        assert np.array_equal(pk[:d], mus[k])
        A = np.zeros((d, d))
        A[iu] = pk[d:-1]                                         # row by row, j = i .. d-1
        assert np.all(np.diag(A) > 0)
        np.testing.assert_allclose(np.linalg.inv(A.T @ A), covs[k], rtol=1e-10, atol=1e-12)
        full = km.gaussian_params(mus[k], covs[k])              # the Gaussian plugin's per-component math
        assert np.array_equal(full[d:d + d * d].reshape(d, d)[iu], pk[d:-1])
        assert pk[-1] == math.log(w[k] / np.sum(w)) + full[-1]
    if d == 1:                                                    # [K] means and [K] variances
        assert np.array_equal(km.gaussian_mixture_params(w, mus[:, 0], covs[:, 0, 0]), p)


def test_scalar_weights_scale_out(km):
    w, mus, covs = random_mixture(2, 3, 5)
    a, b = km.gaussian_mixture_params(w, mus, covs), km.gaussian_mixture_params(4 * w, mus, covs)
    np.testing.assert_allclose(a, b, rtol=0, atol=1e-15)


def _params(km, d, K, seed=0):
    return km.gaussian_mixture_params(*random_mixture(d, K, seed))


@pytest.mark.parametrize("d", [1, 2, 10, 16])
def test_create_accepts_every_k_up_to_kmax(km, d):
    for K in sorted({1, 2 if KMAX[d] >= 2 else 1, KMAX[d]}):
        ld = km.LogDensity("gaussian_mixture", d, _params(km, d, K))
        assert ld.info("batched") == 0


@pytest.mark.parametrize("d,n", [(2, 5), (2, 7), (2, 0), (10, 65), (1, 4)])
def test_create_rejects_a_wrong_multiple_of_q(km, d, n):
    p = np.tile(_params(km, d, 1), 3)[:n] if n else np.zeros(0)
    with pytest.raises(km.KmcError) as e:
        km.LogDensity("gaussian_mixture", d, p)
    assert e.value.code == 1


@pytest.mark.parametrize("d", [1, 2, 5, 10, 12, 16])
def test_create_rejects_more_than_kmax_components(km, d):
    p = np.tile(_params(km, d, 1), KMAX[d] + 1)
    with pytest.raises(km.KmcError) as e:
        km.LogDensity("gaussian_mixture", d, p)
    assert e.value.code == 3 and f"Kmax={KMAX[d]}" in str(e.value)


@pytest.mark.parametrize("where", ["mu", "A", "c"])
@pytest.mark.parametrize("bad", [math.nan, math.inf, -math.inf])
def test_create_rejects_non_finite_parameters(km, where, bad):
    d, K = 2, 3
    p = _params(km, d, K).reshape(K, q(d))
    p[2, {"mu": 1, "A": d + 1, "c": -1}[where]] = bad
    with pytest.raises(km.KmcError) as e:
        km.LogDensity("gaussian_mixture", d, p.ravel())
    assert e.value.code == 1


@pytest.mark.parametrize("row", [0, 1, 2])
@pytest.mark.parametrize("value", [0.0, -0.5])
def test_create_rejects_a_non_positive_diagonal(km, row, value):
    d, K = 3, 2
    p = _params(km, d, K).reshape(K, q(d))
    diag = [d, d + 3, d + 5]                                      # row i of the upper triangle starts at its diagonal
    assert np.all(p[1, diag] > 0)
    p[1, diag[row]] = value
    with pytest.raises(km.KmcError) as e:
        km.LogDensity("gaussian_mixture", d, p.ravel())
    assert e.value.code == 1 and "component 1" in str(e.value)


@pytest.mark.parametrize("d", [7, 9, 17, 100])
def test_create_rejects_a_dimension_without_kernels(km, d):
    with pytest.raises(km.KmcError) as e:
        km.LogDensity("gaussian_mixture", d, np.zeros(q(d)) + 1.0)
    assert e.value.code == 3


@pytest.mark.parametrize("kw,k", [
    (dict(weights=[0.5, 0.0, 0.5]), 1),
    (dict(weights=[0.5, -1.0, 0.5]), 1),
    (dict(weights=[0.5, 1.0, math.nan]), 2),
    (dict(weights=[math.inf, 1.0, 1.0]), 0),
    (dict(covs=[np.eye(2), [[1.0, 2.0], [2.0, 1.0]], np.eye(2)]), 1),     # indefinite
    (dict(covs=[np.eye(2), np.eye(2), [[1.0, 0.5], [0.4, 1.0]]]), 2),      # not symmetric
    (dict(covs=[[[1.0, 0.0], [0.0, -1.0]], np.eye(2), np.eye(2)]), 0),     # negative
    (dict(covs=[np.eye(2), np.eye(2) * math.nan, np.eye(2)]), 1),
    (dict(means=[[0.0, 0.0], [math.inf, 0.0], [1.0, 1.0]]), 1),
])
def test_bad_weights_or_covariances_raise_value_error(km, kw, k):
    args = dict(weights=[0.2, 0.3, 0.5], means=[[0.0, 0.0], [1.0, 0.0], [0.0, 1.0]], covs=[np.eye(2)] * 3)
    args.update(kw)
    with pytest.raises(ValueError, match=f"component {k}"):
        km.gaussian_mixture(**args)


@pytest.mark.parametrize("kw", [dict(weights=[]), dict(means=[[0.0, 0.0], [1.0, 0.0]]),
                                dict(covs=[np.eye(3)] * 3), dict(covs=[np.eye(2)] * 2)])
def test_bad_shapes_raise_value_error(km, kw):
    args = dict(weights=[0.2, 0.3, 0.5], means=[[0.0, 0.0], [1.0, 0.0], [0.0, 1.0]], covs=[np.eye(2)] * 3)
    args.update(kw)
    with pytest.raises(ValueError):
        km.gaussian_mixture(**args)
