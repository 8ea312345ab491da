"""The correlated Metropolis proposal on the B200: replay and Philox parity of both device paths with the CPU oracle's
Cholesky loop, L = diag(sigma) against the diagonal walk, batch independence, the validation of L, the statistics
of the reference's correlated target, the pilot-then-tune workflow, and the device-side chain covariance."""
import math

import numpy as np
import pytest

from tests import cases
from tests.test_metropolis_chol_host import random_chol

pytestmark = pytest.mark.gpu

MVN_COV = np.asarray(cases.MVN_COV)


@pytest.fixture(scope="module")
def mo():
    from metropolis_oracle import oracle
    return oracle


def _pair(km, orc, name):
    pname, d, params, theta0, _ = cases.plugin_specs()[name]
    return km.LogDensity(pname, d, params), orc.Density(pname, d, params), d, theta0


def _run(km, ld, x0, prop, niter, nburnin, nthin, seed=0, replay=None, chain_id_base=0, split=None):
    s = km.Metropolis(ld, x0, prop, niter, nburnin, nthin, seed, km.MODE_REPLAY if replay is not None else km.MODE_PHILOX,
                      chain_id_base=chain_id_base)
    try:
        if replay is not None:
            s.set_replay(*replay)
        if split:
            done = 0
            while done < niter:
                s.run(min(split, niter - done))
                done += split
        else:
            s.run(-1)
        th, lp, ar = s.results()
        x, l, na = s.state()
    finally:
        s.close()
    return th, lp, ar, x, l, na


def _check(got, want, lp_rtol=0.0):
    th, lp, ar, x, l, na = got
    assert np.array_equal(ar, want["accept_ratio"]) and np.array_equal(na, want["naccept"])  # decisions exact
    assert np.array_equal(th, want["chain_x"]) and np.array_equal(x, want["x"])              # states bit-exact
    if lp_rtol:
        np.testing.assert_allclose(lp, want["chain_lp"], rtol=lp_rtol)
        np.testing.assert_allclose(l, want["lp"], rtol=lp_rtol)
    else:
        assert np.array_equal(lp, want["chain_lp"]) and np.array_equal(l, want["lp"])


def _same(a, b):
    for u, v in zip(a, b):
        assert np.array_equal(u, v)


@pytest.mark.parametrize("nchains", [1, 7, 1000])
@pytest.mark.parametrize("name", list(cases.plugin_specs()))
def test_chol_replay_parity_fused(km, orc, mo, name, nchains):
    ld, od, d, theta0 = _pair(km, orc, name)
    assert ld.info("batched") == 0
    niter, nburnin, nthin = 60, 20, 3
    rng = np.random.default_rng(nchains + d + 100)
    x0 = cases.ball(theta0, 0.1, nchains, 3)
    L = random_chol(d, nchains + d)
    normals, u = rng.standard_normal((niter, nchains, d)), rng.random((niter, nchains))
    want = mo.metropolis(od, x0, None, niter, nburnin, nthin, normals, u, nthreads=4, chol=L)
    print(f"{name} nchains={nchains}: smallest decision margin {want['min_margin']:.3e}")
    assert want["min_margin"] > 1e-12
    got = _run(km, ld, x0, km.normal_proposal(chol=L), niter, nburnin, nthin, replay=(normals, u))
    _check(got, want, lp_rtol=1e-14 if name == "lognormal" else 0.0)


@pytest.mark.parametrize("name,nchains", [("rosenbrock", 300), ("exponential3", 65), ("mvn10", 33), ("lognormal", 50)])
def test_chol_philox_mode_matches_oracle_fed_device_draws(km, orc, mo, name, nchains):
    ld, od, d, theta0 = _pair(km, orc, name)
    niter, nburnin, nthin, seed = 80, 30, 2, 4321
    x0 = cases.ball(theta0, 0.1, nchains, 4)
    L = random_chol(d, 7)
    normals, u = km.metropolis_draws(seed, 0, nchains, 0, niter, d)
    want = mo.metropolis(od, x0, None, niter, nburnin, nthin, normals, u, nthreads=4, chol=L)
    assert want["min_margin"] > 1e-12
    _check(_run(km, ld, x0, km.normal_proposal(chol=L), niter, nburnin, nthin, seed=seed), want,
           lp_rtol=1e-14 if name == "lognormal" else 0.0)


@pytest.mark.parametrize("which", ["rosenbrock", "mvn10", "gaussian32"])
def test_diag_chol_equals_the_diagonal_walk(km, which):
    if which == "gaussian32":
        d = 32
        mean = np.linspace(-1, 1, d)
        ld = km.gaussian(mean, cases.spd_cov(d, 2))
        assert ld.info("batched") == 1
        theta0 = mean
    else:
        pname, d, params, theta0, _ = cases.plugin_specs()[which]
        ld = km.LogDensity(pname, d, params)
        assert ld.info("batched") == 0
    sigma = np.linspace(0.1, 0.5, d) / math.sqrt(max(1.0, d / 2))
    x0 = cases.ball(theta0, 0.2, 777, 5)
    diag = _run(km, ld, x0, km.normal_proposal(sigma), 120, 40, 2, seed=9)
    chol = _run(km, ld, x0, km.normal_proposal(chol=np.diag(sigma)), 120, 40, 2, seed=9)
    _same(diag, chol)
    assert 0.05 < diag[2].mean() < 0.95


def test_chol_batch_independence_and_launch_split(km):
    ld = km.rosenbrock()
    nchains, niter, nburnin, nthin = 4096, 200, 50, 3
    x0 = cases.ball([1.0, 1.0], 0.5, nchains, 8)
    prop = km.normal_proposal(cov=[[0.16, 0.3], [0.3, 0.81]])
    full = _run(km, ld, x0, prop, niter, nburnin, nthin, seed=5)
    for c in (0, 1, 2047, 4095):                                  # chain c == a one-chain run with id c
        one = _run(km, ld, x0[c:c + 1], prop, niter, nburnin, nthin, seed=5, chain_id_base=c)
        for a, b in zip(full, one):
            assert np.array_equal(a[c:c + 1], b)
    _same(full, _run(km, ld, x0, prop, niter, nburnin, nthin, seed=5, split=37))   # run(37) repeated == run(-1)
    d = 32                                                        # the batched pipeline, the same two properties
    mean = np.zeros(d)
    ld = km.gaussian(mean, cases.spd_cov(d, 1))
    x0 = cases.ball(mean, 0.3, 300, 2)
    prop = km.normal_proposal(chol=random_chol(d, 3, 0.15))
    full = _run(km, ld, x0, prop, 40, 10, 2, seed=6)
    one = _run(km, ld, x0[123:124], prop, 40, 10, 2, seed=6, chain_id_base=123)
    for a, b in zip(full, one):
        assert np.array_equal(a[123:124], b)
    _same(full, _run(km, ld, x0, prop, 40, 10, 2, seed=6, split=7))


@pytest.mark.parametrize("d,nchains", [(32, 300), (100, 130)])
def test_chol_batched_gaussian_parity(km, orc, mo, d, nchains):
    mean, cov = np.linspace(-1, 1, d), cases.spd_cov(d, 2)
    ld = km.gaussian(mean, cov)
    od = orc.Density("gaussian", d, km.gaussian_params(mean, cov))
    assert ld.info("batched") == 1 and ld.info("tensor_cores") == 0
    niter, nburnin, nthin = 30, 10, 2
    L = random_chol(d, d, 0.08)
    prop = km.normal_proposal(chol=L)
    rng = np.random.default_rng(d)
    x0 = mean + cases.ball(np.zeros(d), 0.3, nchains, 1)
    normals, u = rng.standard_normal((niter, nchains, d)), rng.random((niter, nchains))
    want = mo.metropolis(od, x0, None, niter, nburnin, nthin, normals, u, nthreads=4, chol=L)
    assert want["min_margin"] > 1e-8
    assert 0.02 < want["accept_ratio"].mean() < 0.98
    _check(_run(km, ld, x0, prop, niter, nburnin, nthin, replay=(normals, u)), want, lp_rtol=1e-12)
    seed = 78                                     # Philox mode: the device's own draws
    normals, u = km.metropolis_draws(seed, 0, nchains, 0, niter, d)
    want = mo.metropolis(od, x0, None, niter, nburnin, nthin, normals, u, nthreads=4, chol=L)
    assert want["min_margin"] > 1e-8
    _check(_run(km, ld, x0, prop, niter, nburnin, nthin, seed=seed), want, lp_rtol=1e-12)


def test_chol_batched_logistic_parity(km, orc, mo):
    d, N, nchains, niter, nburnin, nthin = 8, 3000, 64, 20, 6, 3
    X, y, tstar = cases.logistic_problem(N=N, d=d, seed=4)
    ld = km.logistic(X, y, prior_sigma=10.0)
    od = orc.Density("logistic", d, [10.0], data=np.concatenate([X.ravel(), y]))
    x0 = tstar + cases.ball(np.zeros(d), 0.02, nchains, 7)
    L = random_chol(d, 11, 0.02)
    rng = np.random.default_rng(6)
    normals, u = rng.standard_normal((niter, nchains, d)), rng.random((niter, nchains))
    want = mo.metropolis(od, x0, None, niter, nburnin, nthin, normals, u, nthreads=4, chol=L)
    assert want["min_margin"] > 1e-6
    _check(_run(km, ld, x0, km.normal_proposal(chol=L), niter, nburnin, nthin, replay=(normals, u)), want,
           lp_rtol=1e-10)


def test_chol_batched_exponential_odd_dimension(km, orc, mo):
    d, nchains, niter = 7, 100, 40
    ld, od = km.exponential(d), orc.Density("exponential", d, [])
    assert ld.info("batched") == 3
    x0 = 1.0 + cases.ball(np.zeros(d), 0.1, nchains, 2)
    L = random_chol(d, 5, 0.5)
    normals, u = km.metropolis_draws(4, 0, nchains, 0, niter, d)
    want = mo.metropolis(od, x0, None, niter, 10, 1, normals, u, chol=L)
    _check(_run(km, ld, x0, km.normal_proposal(chol=L), niter, 10, 1, seed=4), want)


@pytest.mark.parametrize("bad", ["upper", "zero_diag", "negative_diag", "nan", "inf"])
@pytest.mark.parametrize("d", [2, 32])
def test_bad_chol_is_rejected_with_invalid(km, bad, d):
    ld = km.rosenbrock() if d == 2 else km.gaussian(np.zeros(d), np.eye(d))
    L = random_chol(d, 1)
    i, j = (0, 1) if bad == "upper" else (1, 1) if "diag" in bad else (1, 0)
    L[i, j] = {"upper": 0.1, "zero_diag": 0.0, "negative_diag": -0.2, "nan": math.nan, "inf": math.inf}[bad]
    with pytest.raises(km.KmcError) as e:
        km.Metropolis(ld, np.zeros((4, d)), km.normal_proposal(chol=L), 10, 5)
    assert e.value.code == 1
    with pytest.raises(km.KmcError) as e:                 # a full covariance passed by mistake
        km.Metropolis(ld, np.zeros((4, d)), km.normal_proposal(chol=np.eye(d) + 0.1), 10, 5)
    assert e.value.code == 1


def _mvn2(km, prop, nchains=256, niter=10**4, seed=11):
    pname, d, params, theta0, _ = cases.plugin_specs()["mvn2"]
    ld = km.LogDensity(pname, d, params)
    x0 = cases.ball(theta0, 0.1, nchains, 1)
    return km.metropolis(ld, prop, x0, niter=niter, nchains=nchains, use_progress_meter=False, seed=seed)


def test_statistics_of_the_correlated_target(km):
    """mvn2 (correlation 0.995): the proposal 2.38^2/d * Sigma mixes far faster than the diagonal [0.3, 1.2]."""
    std = np.sqrt(np.diag(MVN_COV))
    th, ar, _, _ = _mvn2(km, km.normal_proposal(cov=2.38**2 / 2 * MVN_COV))
    thd, ard, _, _ = _mvn2(km, km.normal_proposal([0.3, 1.2]))
    t = th.reshape(-1, 2)
    assert np.all(np.abs(t.mean(0) - cases.MVN_MEAN) < 0.3 * std), t.mean(0)
    assert np.all(np.abs(t.std(0) - std) < 0.3 * std), t.std(0)
    assert 0.28 < ar.mean() < 0.44, ar.mean()
    tau, _ = km.int_acorr(th, warn=False)
    taud, _ = km.int_acorr(thd, warn=False)
    print(f"tau chol {tau}, diagonal {taud}; accept {ar.mean():.3f} / {ard.mean():.3f}")
    assert np.all(tau < 20) and np.all(tau < taud / 5), (tau, taud)


def test_pilot_then_tune(km):
    """A diagonal pilot, its chain covariance, then normal_proposal(cov = 2.38^2/d * Sigma_hat): a shorter tau."""
    pname, d, params, theta0, _ = cases.plugin_specs()["mvn2"]
    ld = km.LogDensity(pname, d, params)
    x0 = cases.ball(theta0, 0.1, 256, 3)
    pilot = km.Metropolis(ld, x0, km.normal_proposal([0.3, 1.2]), 4000, 2000, 1, seed=21)
    pilot.run(-1)
    thp, _, _ = pilot.results()
    mean, cov, n = pilot.chain_covariance()
    pilot.close()
    assert n == 256 * 2000
    np.testing.assert_allclose(cov, MVN_COV, rtol=0.25)
    th, ar, _, _ = km.metropolis(ld, km.normal_proposal(cov=2.38**2 / d * cov), x0, niter=4000, nburnin=2000,
                                 nchains=256, use_progress_meter=False, seed=22)
    tau, _ = km.int_acorr(th, warn=False)
    taup, _ = km.int_acorr(thp, warn=False)
    print(f"tau tuned {tau}, pilot {taup}")
    assert np.all(tau < taup), (tau, taup)


def _cov_check(s, th):
    rows = th.reshape(-1, th.shape[-1])
    mean, cov, n = s.chain_covariance()
    assert n == rows.shape[0]
    want = np.cov(rows, rowvar=False, ddof=1)
    np.testing.assert_allclose(cov, want, rtol=1e-10, atol=1e-12 * np.abs(want).max())
    np.testing.assert_allclose(mean, rows.mean(0), rtol=1e-10, atol=1e-12)
    assert np.array_equal(cov, cov.T)
    m2, v2, n2 = s.chain_moments()
    assert n2 == n
    np.testing.assert_allclose(np.diag(cov), v2, rtol=1e-10)
    np.testing.assert_allclose(mean, m2, rtol=1e-10, atol=1e-12)
    again = s.chain_covariance()
    assert np.array_equal(again[0], mean) and np.array_equal(again[1], cov)   # fixed-order reduction: same bits


def test_chain_covariance_on_metropolis_and_emcee_handles(km):
    ld = km.gaussian(cases.MVN_MEAN, cases.MVN_COV)
    x0 = cases.ball(cases.MVN_MEAN, 0.5, 513, 2)
    s = km.Metropolis(ld, x0, km.normal_proposal(cov=MVN_COV), 400, 100, 2, seed=3)
    s.run(-1)
    th, _, _ = s.results()
    _cov_check(s, th)
    s.close()
    d = 10
    ld = km.gaussian(np.linspace(-1, 1, d), cases.spd_cov(d, 1))
    em = km.Sampler(ld, cases.ball(np.zeros(d), 0.5, 1024, 3), 300, 100, 2, 2.0, 4)
    em.run(-1)
    th, _, _ = em.results()
    _cov_check(em, th)
    em.close()
    d = 100                                       # the 100-D Gaussian workload, batched, d <= 128
    mean = np.linspace(-1, 1, d)
    ld = km.gaussian(mean, cases.spd_cov(d, 3))
    s = km.Metropolis(ld, mean + cases.ball(np.zeros(d), 0.3, 2000, 1), km.normal_proposal(0.05), 30, 10, 1, seed=2)
    s.run(-1)
    th, _, _ = s.results()
    _cov_check(s, th)
    s.close()


def test_chain_covariance_limits(km):
    d = 130
    ld = km.gaussian(np.zeros(d), np.eye(d))
    s = km.Metropolis(ld, cases.ball(np.zeros(d), 0.1, 8, 1), km.normal_proposal(0.05), 4, 2, 1)
    s.run(-1)
    with pytest.raises(km.KmcError) as e:
        s.chain_covariance()
    assert e.value.code == 3
    s.close()
    s = km.Metropolis(km.rosenbrock(), np.zeros((4, 2)), km.normal_proposal(0.5), 4, 4, 1)
    s.run(-1)
    with pytest.raises(km.KmcError) as e:         # nothing stored
        s.chain_covariance()
    assert e.value.code == 4
    s.close()


def test_full_size_rosenbrock_correlated(km, orc):
    ld, od = km.rosenbrock(), orc.Density("rosenbrock", 2, [1.0, 100.0, 20.0])
    nchains, niter, nthin = 2**20, 2000, 500
    rng = np.random.default_rng(3)
    x1 = 1.0 + math.sqrt(10.0) * rng.standard_normal(nchains)
    x0 = np.stack([x1, x1 * x1 + math.sqrt(0.1) * rng.standard_normal(nchains)], axis=1)
    prop = km.normal_proposal(cov=[[0.25, 0.4], [0.4, 0.81]])
    s = km.Metropolis(ld, x0, prop, niter, 0, nthin, seed=1)
    s.run(-1)
    th, lp, ar = s.results()
    _, _, na = s.state()
    s.close()
    idx = rng.integers(0, nchains, 4096)
    pts = th[idx].reshape(-1, 2)
    assert np.array_equal(lp[idx].reshape(-1), od.eval(pts, nthreads=4))     # stored logp == plugin(stored theta)
    assert np.array_equal(np.round(ar * niter).astype(np.int64), na)
    assert 0.05 < ar.mean() < 0.9
    for c in idx[:8]:                               # accept counts == state changes of the full chain
        one = _run(km, ld, x0[c:c + 1], prop, niter, 0, 1, seed=1, chain_id_base=int(c))
        tr = np.concatenate([x0[c:c + 1], one[0][0]])
        changes = int(np.any(tr[1:] != tr[:-1], axis=1).sum())
        assert changes == na[c] == one[5][0]
