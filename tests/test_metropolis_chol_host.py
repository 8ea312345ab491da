"""The correlated Metropolis proposal without a GPU: the oracle's Cholesky loop against a line-by-line restatement of
the proposal contract, L = diag(sigma) against the diagonal loop, and normal_proposal's argument checks."""
import math

import numpy as np
import pytest

from tests.cases import MVN_COV, plugin_specs

CASES = ["exponential", "exponential3", "rosenbrock", "mvn2", "mvn10", "lognormal"]


def random_chol(d, seed, scale=0.3):
    """A lower-triangular factor with a positive diagonal and non-zero entries below it."""
    rng = np.random.default_rng(seed)
    L = np.tril(rng.standard_normal((d, d))) * scale / math.sqrt(d)
    L[np.diag_indices(d)] = scale * (0.5 + rng.random(d))
    return L


def python_metropolis_chol(logpdf, theta0, L, niter, nburnin, nthin, normals, u):
    """The Metropolis loop with y[i] = x[i] + s, s = 0.0; s = s + L[i][j] * z[j] for j = 0 .. i (Python floats:
    IEEE binary64, one rounding per operation, never fused)."""
    d = len(theta0)
    theta0 = [float(v) for v in theta0]
    p0 = logpdf(np.array(theta0))
    naccept = 0
    thetas, lps = [], []
    t = 0
    for ni in range(1 - nburnin, niter - nburnin + 1):
        z = [float(v) for v in normals[t]]
        theta1 = []
        for i in range(d):
            s = 0.0
            for j in range(i + 1):
                s = s + float(L[i, j]) * z[j]
            theta1.append(theta0[i] + s)
        p1 = logpdf(np.array(theta1))
        lu = math.log(u[t]) if u[t] > 0 else -math.inf
        if p1 - p0 > lu:
            theta0, p0 = theta1, p1
            naccept += 1
        if ni > 0 and ni % nthin == 0:
            thetas.append(list(theta0))
            lps.append(p0)
        if ni == 0:
            naccept = 0
        t += 1
    return np.array(thetas).reshape(len(thetas), d), np.array(lps), naccept / (niter - nburnin), np.array(theta0), p0


@pytest.mark.parametrize("name", CASES)
def test_oracle_chol_loop_matches_the_python_loop_bit_for_bit(name):
    from metropolis_oracle import oracle as mo
    from oracle.oracle import Density
    pname, d, params, theta0, _ = plugin_specs()[name]
    dens = Density(pname, d, params)
    nc, niter, nburnin, nthin = 3, 90, 29, 4
    rng = np.random.default_rng(21)
    normals = rng.standard_normal((niter, nc, d))
    u = rng.random((niter, nc))
    u[5, 0] = 0.0
    x0 = np.tile(np.atleast_1d(theta0), (nc, 1)).astype(np.float64)
    L = random_chol(d, d + 3)
    got = mo.metropolis(dens, x0, None, niter, nburnin, nthin, normals, u, nthreads=2, chol=L)
    for c in range(nc):
        th, lp, ar, xf, pf = python_metropolis_chol(dens.logpdf, x0[c], L, niter, nburnin, nthin, normals[:, c],
                                                    u[:, c])
        assert np.array_equal(got["chain_x"][c], th)
        assert np.array_equal(got["chain_lp"][c], lp)
        assert got["accept_ratio"][c] == ar
        assert np.array_equal(got["x"][c], xf) and got["lp"][c] == pf
    assert 0.0 < got["accept_ratio"].mean() < 1.0


@pytest.mark.parametrize("name", CASES)
def test_oracle_chol_of_diag_sigma_equals_the_diagonal_loop(name):
    from metropolis_oracle import oracle as mo
    from oracle.oracle import Density
    pname, d, params, theta0, _ = plugin_specs()[name]
    dens = Density(pname, d, params)
    nc, niter, nburnin, nthin = 16, 150, 50, 3
    rng = np.random.default_rng(d)
    normals, u = rng.standard_normal((niter, nc, d)), rng.random((niter, nc))
    x0 = np.atleast_1d(theta0) + 0.05 * rng.standard_normal((nc, d))
    sigma = np.linspace(0.2, 0.7, d)
    diag = mo.metropolis(dens, x0, sigma, niter, nburnin, nthin, normals, u)
    chol = mo.metropolis(dens, x0, None, niter, nburnin, nthin, normals, u, chol=np.diag(sigma))
    for k in ("chain_x", "chain_lp", "accept_ratio", "naccept", "x", "lp"):
        assert np.array_equal(diag[k], chol[k]), k


def test_normal_proposal_forms(km):
    p = km.normal_proposal([0.3, 1.2])
    assert p.chol is None and np.array_equal(p.sigma, [0.3, 1.2])
    assert km.normal_proposal(0.5).chol is None
    cov = 2.38**2 / 2 * np.asarray(MVN_COV)
    p = km.normal_proposal(cov=cov)
    assert p.sigma is None and np.allclose(p.chol @ p.chol.T, cov, rtol=1e-14)
    assert np.array_equal(p.chol, np.tril(p.chol)) and np.all(np.diag(p.chol) > 0)
    L = random_chol(3, 1)
    assert np.array_equal(km.normal_proposal(chol=L).chol, L)


@pytest.mark.parametrize("kw", [dict(), dict(sigma=0.5, cov=np.eye(2)), dict(sigma=0.5, chol=np.eye(2)),
                                dict(cov=np.eye(2), chol=np.eye(2))])
def test_normal_proposal_takes_exactly_one_form(km, kw):
    with pytest.raises(ValueError, match="exactly one"):
        km.normal_proposal(**kw)


@pytest.mark.parametrize("cov", [[[1.0, 2.0], [2.0, 1.0]],          # indefinite
                                 [[1.0, 0.5], [0.4, 1.0]],          # not symmetric
                                 [[1.0, 0.0], [0.0, -1.0]],         # negative
                                 np.ones((2, 3)),                   # not square
                                 [[1.0, math.nan], [math.nan, 1.0]]])
def test_normal_proposal_rejects_a_bad_covariance(km, cov):
    with pytest.raises(ValueError):
        km.normal_proposal(cov=cov)


def test_chol_shape_must_match_the_density(km):
    with pytest.raises(ValueError):
        km.normal_proposal(chol=np.ones((2, 3)))
    with pytest.raises(ValueError):
        km.Metropolis(km.rosenbrock(), np.zeros((4, 2)), km.normal_proposal(chol=np.eye(3)), 10, 5)
