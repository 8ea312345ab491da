"""Metropolis without a GPU: the oracle against a line-by-line restatement of the reference loop, the sample-count
arithmetic, the draw layout, and the API's argument checks."""
import math

import numpy as np
import pytest

from tests.cases import plugin_specs

CASES = ["exponential", "exponential3", "rosenbrock", "mvn2", "lognormal"]


def python_metropolis(logpdf, theta0, sigma, niter, nburnin, nthin, normals, u):
    """src/samplers.jl:9-128 (the restatement in metropolis_oracle/kmo_metropolis.c), one chain, line by line."""
    theta0 = np.array(theta0, dtype=np.float64)
    p0 = logpdf(theta0)
    naccept = 0
    thetas, lps = [], []
    t = 0
    for ni in range(1 - nburnin, niter - nburnin + 1):
        theta1 = theta0 + sigma * normals[t]           # mul, then add (two numpy ufuncs: never fused)
        p1 = logpdf(theta1)
        lu = math.log(u[t]) if u[t] > 0 else -math.inf
        if p1 - p0 > lu:                                # strict >; NaN (-Inf - -Inf) rejects
            theta0, p0 = theta1, p1
            naccept += 1
        if ni > 0 and ni % nthin == 0:
            thetas.append(theta0.copy())
            lps.append(p0)
        if ni == 0:
            naccept = 0
        t += 1
    return np.array(thetas).reshape(len(thetas), -1), np.array(lps), naccept / (niter - nburnin), theta0, p0


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_the_python_loop_bit_for_bit(name):
    from metropolis_oracle import oracle as mo
    from oracle.oracle import Density
    pname, d, params, theta0, _ = plugin_specs()[name]
    dens = Density(pname, d, params)
    nc, niter, nburnin, nthin = 3, 120, 37, 4
    rng = np.random.default_rng(11)
    normals = rng.standard_normal((niter, nc, d))
    u = rng.random((niter, nc))
    u[5, 0] = 0.0                                            # log(0) = -Inf: any finite p1 - p0 accepts
    x0 = np.tile(np.atleast_1d(theta0), (nc, 1)).astype(np.float64)
    if pname in ("exponential", "lognormal"):
        x0[1, 0] = -0.05                                     # p0 = -Inf at the start: the first finite proposal accepts
    sigma = np.linspace(0.3, 0.9, d) if d > 1 else 0.5
    got = mo.metropolis(dens, x0, sigma, niter, nburnin, nthin, normals, u, nthreads=2)
    for c in range(nc):
        th, lp, ar, xf, pf = python_metropolis(dens.logpdf, x0[c], sigma, niter, nburnin, nthin, normals[:, c], u[:, c])
        assert np.array_equal(got["chain_x"][c], th)
        assert np.array_equal(got["chain_lp"][c], lp)
        assert got["accept_ratio"][c] == ar
        assert np.array_equal(got["x"][c], xf) and got["lp"][c] == pf
    if pname in ("exponential", "lognormal"):
        assert np.isfinite(got["chain_lp"][1]).all()         # the -Inf start was left


@pytest.mark.parametrize("niter,nburnin,nthin", [(10, 5, 1), (10, 0, 3), (11, 4, 2), (7, 7, 1), (100, 50, 7),
                                                 (9, 2, 10)])
def test_sample_count_and_accept_ratio_arithmetic(niter, nburnin, nthin):
    from metropolis_oracle import oracle as mo
    from oracle.oracle import Density
    dens = Density("gaussian", 1, plugin_specs()["normal"][2])
    u = np.zeros((niter, 2))                                 # log(0) = -Inf: every finite proposal is accepted
    out = mo.metropolis(dens, [[-5.0], [-4.0]], 0.1, niter, nburnin, nthin, np.ones((niter, 2, 1)), u)
    ns = (niter - nburnin) // nthin
    assert out["chain_x"].shape == (2, ns, 1)
    if niter > nburnin:
        assert np.array_equal(out["accept_ratio"], [1.0, 1.0])  # naccept counts the niter - nburnin post-burn-in steps
        if ns:                                                  # sample s is the state after step nburnin + (s+1)*nthin
            steps = nburnin + nthin * np.arange(1, ns + 1)
            assert np.allclose(out["chain_x"][0, :, 0], -5.0 + 0.1 * steps)


def test_metropolis_uniform_counter_layout_is_integer_exact(km):
    """The uniform of pair 0 of step t of chain c: ((r2 & 0xFFFF) << 32 | r3) * 2^-48 of Philox(c, t lo, t hi, tag)."""
    from oracle.oracle import philox4x32_10
    seed = 0x123456789
    n, u = km.metropolis_randn(seed, [0, 7, 2**32 - 1], [0, 5, 2**33 + 3], 3)
    assert n.shape == (3, 3, 3) and u.shape == (3, 3)
    for i, t in enumerate([0, 5, 2**33 + 3]):
        for j, c in enumerate([0, 7, 2**32 - 1]):
            r = philox4x32_10([c, t & 0xFFFFFFFF, t >> 32, 0x4D480000], [seed & 0xFFFFFFFF, seed >> 32])
            assert u[i, j] == (((r[2] & 0xFFFF) << 32) | r[3]) * 2.0 ** -48
            r1 = philox4x32_10([c, t & 0xFFFFFFFF, t >> 32, 0x4D480001], [seed & 0xFFFFFFFF, seed >> 32])
            u1, u2 = (r1[0] + 1.0) * 2.0 ** -32, r1[1] * 2.0 ** -32
            assert n[i, j, 2] == pytest.approx(math.sqrt(-2.0 * math.log(u1)) * math.cos(2 * math.pi * u2), rel=1e-13)


def test_callable_proposal_raises_type_error(km):
    with pytest.raises(TypeError, match="proposal descriptor"):
        km.metropolis(km.exponential(), lambda th: th + 1.5 * np.random.randn(), 0.5, niter=10)


def test_hasblob_raises(km):
    with pytest.raises(NotImplementedError):
        km.metropolis(km.exponential(), km.normal_proposal(1.5), 0.5, niter=10, hasblob=True)


@pytest.mark.parametrize("sigma", [[1.0, 2.0], 0.0, -1.0, math.nan, math.inf, [0.5, 0.5, -0.5]])
def test_bad_sigma_is_rejected_with_invalid(km, sigma):
    d = 3 if np.size(sigma) == 3 else 1
    with pytest.raises(km.KmcError) as e:
        km.metropolis(km.exponential(d), km.normal_proposal(sigma), np.ones(d) if d > 1 else 0.5, niter=10)
    assert e.value.code == 1


def test_theta0_shape_must_match_nchains(km):
    with pytest.raises(ValueError):
        km.metropolis(km.rosenbrock(), km.normal_proposal(0.5), np.zeros((3, 2)), niter=10, nchains=4)
    with pytest.raises(ValueError):
        km.metropolis(km.rosenbrock(), km.normal_proposal(0.5), np.zeros(2), niter=10, nchains=2)
    with pytest.raises(ValueError):
        km.metropolis(km.rosenbrock(), km.normal_proposal(0.5), np.zeros(3), niter=10)


def test_chain_ids_must_fit_32_bits(km):
    with pytest.raises(km.KmcError) as e:
        km.Metropolis(km.exponential(), np.ones((2, 1)), km.normal_proposal(1.0), 10, 5, chain_id_base=2**32 - 1)
    assert e.value.code == 1


def test_without_a_device_metropolis_raises(km):
    if _has_device(km):
        pytest.skip("a CUDA device is present")
    with pytest.raises(km.KmcError):
        km.metropolis(km.exponential(), km.normal_proposal(1.5), 0.5, niter=100)


def _has_device(km):
    try:
        return km.device_count() > 0
    except km.KmcError:
        return False
