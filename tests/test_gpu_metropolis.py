"""Metropolis on the B200: replay parity with the CPU oracle (metropolis_oracle/), Philox-mode parity through the
device's own draws, batch independence, the batched-plugin pipeline, and the reference's statistical cases."""
import math

import numpy as np
import pytest

from tests import cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mo():
    from metropolis_oracle import oracle
    return oracle


def _pair(km, orc, name):
    pname, d, params, theta0, _ = cases.plugin_specs()[name]
    return km.LogDensity(pname, d, params), orc.Density(pname, d, params), d, theta0


def _sigma(d):
    return np.linspace(0.2, 0.6, d) if d > 1 else 0.4


def _run(km, ld, x0, sigma, niter, nburnin, nthin, seed=0, replay=None, chain_id_base=0, split=None):
    s = km.Metropolis(ld, x0, km.normal_proposal(sigma), niter, nburnin, nthin, seed,
                      km.MODE_REPLAY if replay is not None else km.MODE_PHILOX, chain_id_base=chain_id_base)
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


@pytest.mark.parametrize("nchains", [1, 7, 1000])
@pytest.mark.parametrize("name", list(cases.plugin_specs()))
def test_replay_parity_fused(km, orc, mo, name, nchains):
    ld, od, d, theta0 = _pair(km, orc, name)
    assert ld.info("batched") == 0
    niter, nburnin, nthin = 60, 20, 3
    rng = np.random.default_rng(nchains + d)
    x0 = cases.ball(theta0, 0.1, nchains, 3)
    normals, u = rng.standard_normal((niter, nchains, d)), rng.random((niter, nchains))
    want = mo.metropolis(od, x0, _sigma(d), niter, nburnin, nthin, normals, u, nthreads=4)
    print(f"{name} nchains={nchains}: smallest decision margin {want['min_margin']:.3e}")
    assert want["min_margin"] > 1e-12             # no decision within reach of a 1-ulp log difference
    got = _run(km, ld, x0, _sigma(d), niter, nburnin, nthin, replay=(normals, u))
    _check(got, want, lp_rtol=1e-14 if name == "lognormal" else 0.0)


@pytest.mark.parametrize("name,nchains", [("rosenbrock", 300), ("exponential3", 65), ("mvn10", 33), ("lognormal", 50)])
def test_philox_mode_matches_oracle_fed_device_draws(km, orc, mo, name, nchains):
    ld, od, d, theta0 = _pair(km, orc, name)
    niter, nburnin, nthin, seed = 80, 30, 2, 1234
    x0 = cases.ball(theta0, 0.1, nchains, 4)
    normals, u = km.metropolis_draws(seed, 0, nchains, 0, niter, d)
    want = mo.metropolis(od, x0, _sigma(d), niter, nburnin, nthin, normals, u, nthreads=4)
    assert want["min_margin"] > 1e-12
    _check(_run(km, ld, x0, _sigma(d), niter, nburnin, nthin, seed=seed), want,
           lp_rtol=1e-14 if name == "lognormal" else 0.0)
    # the uniforms are integer-exact; the normals agree with numpy's Box-Muller to a few ulp
    hn, hu = km.metropolis_randn(seed, np.arange(nchains), np.arange(niter), d)
    assert np.array_equal(hu, u)
    np.testing.assert_allclose(normals, hn, rtol=1e-13, atol=1e-14)


def test_draws_are_a_function_of_chain_id_and_step(km):
    n_all, u_all = km.metropolis_draws(9, 100, 50, 10, 20, 5)
    n_sub, u_sub = km.metropolis_draws(9, 117, 3, 14, 2, 5)
    assert np.array_equal(n_sub, n_all[4:6, 17:20]) and np.array_equal(u_sub, u_all[4:6, 17:20])
    hn, hu = km.metropolis_randn(9, [2**32 - 1], [2**32 + 5], 5)
    dn, du = km.metropolis_draws(9, 2**32 - 1, 1, 2**32 + 5, 1, 5)
    assert np.array_equal(du, hu)
    np.testing.assert_allclose(dn, hn, rtol=1e-13, atol=1e-14)


def test_batch_independence_and_launch_split(km):
    ld = km.rosenbrock()
    nchains, niter, nburnin, nthin = 4096, 200, 50, 3
    x0 = cases.ball([1.0, 1.0], 0.5, nchains, 8)
    full = _run(km, ld, x0, [0.4, 0.9], niter, nburnin, nthin, seed=5)
    for c in (0, 1, 2047, 4095):                                  # chain c == a one-chain run with id c
        one = _run(km, ld, x0[c:c + 1], [0.4, 0.9], niter, nburnin, nthin, seed=5, chain_id_base=c)
        for a, b in zip(full, one):
            assert np.array_equal(a[c:c + 1], b)
    split = _run(km, ld, x0, [0.4, 0.9], niter, nburnin, nthin, seed=5, split=37)   # run(37) repeated == run(-1)
    for a, b in zip(full, split):
        assert np.array_equal(a, b)


def test_results_agree_with_squash_and_chain_moments(km):
    ld = km.gaussian(cases.MVN_MEAN, cases.MVN_COV)
    x0 = cases.ball(cases.MVN_MEAN, 0.5, 513, 2)
    s = km.Metropolis(ld, x0, km.normal_proposal([0.3, 1.2]), 400, 100, 2, seed=3)
    s.run(-1)
    th, lp, ar = s.results()
    t, amean, l, _ = s.squash()
    assert np.array_equal(t, th.reshape(-1, 2)) and np.array_equal(l, lp.reshape(-1))
    assert amean == pytest.approx(ar.mean(), rel=1e-12)
    mean, var, n = s.chain_moments()
    assert n == th.shape[0] * th.shape[1]
    np.testing.assert_allclose(mean, th.reshape(-1, 2).mean(0), rtol=1e-10)
    np.testing.assert_allclose(var, th.reshape(-1, 2).var(0, ddof=1), rtol=1e-10)
    it, na_mean, _, _ = s.progress()
    assert it == 400 and na_mean == pytest.approx(ar.mean() * 300, rel=1e-12)
    with pytest.raises(km.KmcError) as e:
        s.run_half(1)
    assert e.value.code == 4
    with pytest.raises(km.KmcError) as e:
        km.Sampler.set_replay(s, np.zeros(513, dtype=np.int64), np.ones(513), np.ones(513))
    assert e.value.code == 4
    s.close()
    em = km.Sampler(ld, x0[:512], 4, 2, 1, 2.0, 0, km.MODE_REPLAY)
    with pytest.raises(km.KmcError) as e:
        km.Metropolis.set_replay(em, np.zeros((1, 512, 2)), np.ones((1, 512)))
    assert e.value.code == 4
    em.close()


@pytest.mark.parametrize("d,nchains", [(32, 300), (100, 130)])
def test_batched_gaussian_replay_parity(km, orc, mo, d, nchains):
    mean, cov = np.linspace(-1, 1, d), cases.spd_cov(d, 2)
    ld = km.gaussian(mean, cov)
    od = orc.Density("gaussian", d, km.gaussian_params(mean, cov))
    assert ld.info("batched") == 1 and ld.info("tensor_cores") == 0
    niter, nburnin, nthin = 30, 10, 2
    rng = np.random.default_rng(d)
    x0 = mean + cases.ball(np.zeros(d), 0.3, nchains, 1)
    normals, u = rng.standard_normal((niter, nchains, d)), rng.random((niter, nchains))
    want = mo.metropolis(od, x0, 0.05, niter, nburnin, nthin, normals, u, nthreads=4)
    assert want["min_margin"] > 1e-8              # DESIGN.md section 4: FP64 batched log-densities within 1e-12 relative
    _check(_run(km, ld, x0, 0.05, niter, nburnin, nthin, replay=(normals, u)), want, lp_rtol=1e-12)
    seed = 77                                     # Philox mode: the device's own draws
    normals, u = km.metropolis_draws(seed, 0, nchains, 0, niter, d)
    want = mo.metropolis(od, x0, 0.05, niter, nburnin, nthin, normals, u, nthreads=4)
    assert want["min_margin"] > 1e-8
    _check(_run(km, ld, x0, 0.05, niter, nburnin, nthin, seed=seed), want, lp_rtol=1e-12)


def test_batched_logistic_replay_parity(km, orc, mo):
    d, N, nchains, niter, nburnin, nthin = 8, 3000, 64, 20, 6, 3
    X, y, tstar = cases.logistic_problem(N=N, d=d, seed=4)
    ld = km.logistic(X, y, prior_sigma=10.0)
    od = orc.Density("logistic", d, [10.0], data=np.concatenate([X.ravel(), y]))
    x0 = tstar + cases.ball(np.zeros(d), 0.02, nchains, 7)
    rng = np.random.default_rng(5)
    normals, u = rng.standard_normal((niter, nchains, d)), rng.random((niter, nchains))
    want = mo.metropolis(od, x0, 0.02, niter, nburnin, nthin, normals, u, nthreads=4)
    assert want["min_margin"] > 1e-6              # FP64 logistic kernel: 1e-10 relative
    _check(_run(km, ld, x0, 0.02, niter, nburnin, nthin, replay=(normals, u)), want, lp_rtol=1e-10)


def test_batched_exponential_odd_dimension(km, orc, mo):
    d, nchains, niter = 7, 100, 40
    ld, od = km.exponential(d), orc.Density("exponential", d, [])
    assert ld.info("batched") == 3
    x0 = 1.0 + cases.ball(np.zeros(d), 0.1, nchains, 2)
    normals, u = km.metropolis_draws(4, 0, nchains, 0, niter, d)
    want = mo.metropolis(od, x0, 0.5, niter, 10, 1, normals, u)
    _check(_run(km, ld, x0, 0.5, niter, 10, 1, seed=4), want)


def test_tensor_core_paths_store_consistent_logdensities(km, orc):
    """tensor_cores=1: every stored logp is the oracle density of the stored theta within the path's tolerance."""
    d = 32
    mean, cov = np.zeros(d), cases.spd_cov(d, 4)
    ld = km.gaussian(mean, cov)
    ld.set_option("tensor_cores", 1)
    od = orc.Density("gaussian", d, km.gaussian_params(mean, cov))
    th, ar, lp, _ = km.metropolis(ld, km.normal_proposal(0.2), cases.ball(mean, 0.5, 256, 3), niter=60, nburnin=20,
                                  nthin=4, nchains=256, use_progress_meter=False)
    pts = th.reshape(-1, d)
    want = od.eval(pts, nthreads=4)
    assert np.all(np.abs(lp.reshape(-1) - want) <= 1e-5 * (1 + np.sum(pts * pts, axis=1)))
    X, y, tstar = cases.logistic_problem(N=20000, d=32, seed=1)
    ld = km.logistic(X, y, prior_sigma=10.0, tensor_cores=True)
    od = orc.Density("logistic", 32, [10.0], data=np.concatenate([X.ravel(), y]))
    th, ar, lp, _ = km.metropolis(ld, km.normal_proposal(0.01), tstar + cases.ball(np.zeros(32), 0.02, 64, 2),
                                  niter=40, nburnin=10, nthin=5, nchains=64, use_progress_meter=False)
    assert ar.mean() > 0.05
    got, want = lp.reshape(-1), od.eval(th.reshape(-1, 32), nthreads=4)
    off = np.median(got - want)                    # the tensor path's common offset (~3e-8 per row)
    assert abs(off) < 1e-6 * 20000
    np.testing.assert_allclose(got - off, want, rtol=0, atol=2e-3)


STATS = [  # (name, sigma, truth mean, truth std, tolm)  -- the reference's test/metro.jl cases
    ("normal", 9.0, [-5.0], [3.0], 0.3),
    ("lognormal", 3.0, [math.exp(0.5)], [math.sqrt((math.e - 1) * math.e)], 0.3),
    ("mvn2", [0.3, 1.2], cases.MVN_MEAN, np.sqrt(np.diag(cases.MVN_COV)), 0.3),
    ("rosenbrock", 0.5, [1.0, 11.0], [math.sqrt(10.0), math.sqrt(2 * 10.0**2 + 4 * 10.0 + 0.1)], 0.6),
]


def _rosenbrock_exact(n, seed):
    """Draws from the Rosenbrock/20 target itself: x1 ~ N(1, 10), x2 | x1 ~ N(x1^2, 0.1)."""
    rng = np.random.default_rng(seed)
    x1 = 1.0 + math.sqrt(10.0) * rng.standard_normal(n)
    return np.stack([x1, x1 * x1 + math.sqrt(0.1) * rng.standard_normal(n)], axis=1)


@pytest.mark.parametrize("name,sigma,mean,std,tolm", STATS)
def test_statistics_of_the_reference_cases(km, name, sigma, mean, std, tolm):
    pname, d, params, theta0, _ = cases.plugin_specs()[name]
    ld = km.LogDensity(pname, d, params)
    nchains = 1024
    x0 = _rosenbrock_exact(nchains, 1) if name == "rosenbrock" else cases.ball(theta0, 0.1, nchains, 1)
    th, ar, lp, _ = km.metropolis(ld, km.normal_proposal(sigma), x0, niter=10**4, nthin=5, nchains=nchains,
                                  use_progress_meter=False, seed=11)
    assert 0.15 < ar.mean() < 0.45, ar.mean()
    t = th.reshape(-1, d)
    std = np.asarray(std, dtype=np.float64)
    assert np.all(np.abs(t.mean(0) - mean) < tolm * std), (t.mean(0), mean)
    assert np.all(np.abs(t.std(0) - std) < tolm * std), (t.std(0), std)
    if name != "rosenbrock":                       # R-hat of two independent chain batches
        th2, _, _, _ = km.metropolis(ld, km.normal_proposal(sigma), x0[:64], niter=4000, nthin=2, nchains=64,
                                     use_progress_meter=False, seed=12)
        rhat, _, _ = km.evaluate_convergence(th[:64, -1000:], th2)
        assert np.all(rhat < 1.1), rhat


def test_readme_call(km, capsys):
    """metropolis(logpdf, θ -> 1.5*randn() + θ, 0.5; niter=10^5) with logpdf(x) = x < 0 ? -Inf : -x."""
    thetas, accept_ratio, logdensities, blobs = km.metropolis(km.exponential(), km.normal_proposal(1.5), 0.5,
                                                              niter=10**5)
    assert thetas.shape == (50000,) and logdensities.shape == (50000,) and blobs is None
    assert isinstance(accept_ratio, float) and 0.1 < accept_ratio < 0.9
    assert abs(thetas.mean() - 1.0) < 0.3
    assert np.array_equal(logdensities, -thetas)
    assert "metropolis, niter=100000" in capsys.readouterr().err   # the coarse progress line


def test_full_size_rosenbrock(km, orc):
    ld, od = km.rosenbrock(), orc.Density("rosenbrock", 2, [1.0, 100.0, 20.0])
    nchains, niter, nthin = 2**20, 2000, 500
    x0 = _rosenbrock_exact(nchains, 3)
    s = km.Metropolis(ld, x0, km.normal_proposal(0.5), niter, 0, nthin, seed=1)
    s.run(-1)
    th, lp, ar = s.results()
    _, _, na = s.state()
    s.close()
    rng = np.random.default_rng(0)
    idx = rng.integers(0, nchains, 4096)
    pts = th[idx].reshape(-1, 2)
    assert np.array_equal(lp[idx].reshape(-1), od.eval(pts, nthreads=4))     # stored logp == plugin(stored theta)
    assert np.array_equal(np.round(ar * niter).astype(np.int64), na)
    for c in idx[:8]:                               # accept counts == state changes of the full chain
        one = _run(km, ld, x0[c:c + 1], 0.5, niter, 0, 1, seed=1, chain_id_base=int(c))
        tr = np.concatenate([x0[c:c + 1], one[0][0]])
        changes = int(np.any(tr[1:] != tr[:-1], axis=1).sum())
        assert changes == na[c] == one[5][0]
