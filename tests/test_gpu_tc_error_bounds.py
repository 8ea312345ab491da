"""GPU tests (`-m gpu`): the tcgen05 log-densities against the FP64 oracle within the bounds derived from their
arithmetic (tests/test_tc_error_model.py holds the derivation and the bound functions), across logit scale,
conditioning, shape and every path that evaluates them.  Each case prints its largest ratio of observed error to bound,
so the log records the headroom.  Wherever the published 1e-5 (1 + |y|^2) of the Gaussian path applies, it is asserted
as well."""
import numpy as np
import pytest

from tests import cases
from tests.test_tc_error_model import (GAUSS_KINDS, SCALES, gaussian_bound, gaussian_case, gaussian_matrix,
                                       gaussian_points, gaussian_terms, logistic_bound, logistic_points,
                                       scaled_logistic_problem)

pytestmark = pytest.mark.gpu

F32_MAX = float(np.finfo(np.float32).max)


def _ratio(err, bound):
    return float(np.max(np.abs(err) / bound))


# ---------------------------------------------------------------------------------- logistic regression (K3)

def _logistic(km, orc, X, y):
    ld = km.logistic(X, y, prior_sigma=10.0, tensor_cores=True)
    assert ld.info("tensor_cores") == 1.0
    return ld, orc.Density("logistic", X.shape[1], [10.0], data=np.concatenate([X.ravel(), y]))


@pytest.mark.parametrize("d", [5, 16, 32, 33, 64])
@pytest.mark.parametrize("N", [3001, 50_001, 1_000_000])
def test_logistic_eval_within_derived_bound(km, orc, N, d):
    """Points: a ball about the mode (radius ~ the posterior scale) and two burn-in points (0 and 100 theta*), for data
    drawn from theta* scaled by 1, 4, 16 and 64.  Each point within its bound, each neighbour difference in the ball
    within the sum of the two bounds."""
    out = []
    for scale in SCALES:
        X, y, tstar = scaled_logistic_problem(N, d, scale, seed=1000 + d)
        ld, od = _logistic(km, orc, X, y)
        pts = logistic_points(tstar, N, 14, seed=d)
        got, want = ld.eval(pts), od.eval(pts, nthreads=8)
        bound = logistic_bound(pts, X)
        err = got - want
        assert np.all(np.abs(err) <= bound), (scale, _ratio(err, bound))
        dd = err[1:14] - err[:13]
        dbound = bound[1:14] + bound[:13]
        assert np.all(np.abs(dd) <= dbound), (scale, _ratio(dd, dbound))
        out.append(f"x{scale}: point {_ratio(err, bound):.3g} diff {_ratio(dd, dbound):.3g} "
                   f"(max |err| {np.max(np.abs(err)):.3g}, |diff err| {np.max(np.abs(dd)):.3g})")
    print(f"\nlogistic eval N={N} d={d}: max error / bound  " + "; ".join(out))


def _check_logistic_chain(od, X, th, lp, label):
    d = X.shape[1]
    pts, got = th.reshape(-1, d), lp.reshape(-1)
    want = od.eval(pts, nthreads=8)
    bound = logistic_bound(pts, X)
    assert np.all(np.isfinite(got))
    assert np.all(np.abs(got - want) <= bound), _ratio(got - want, bound)
    print(f"\n{label}: {got.size} stored log-densities, max error / bound {_ratio(got - want, bound):.3g}")


def test_logistic_sampling_at_scale_16(km, orc):
    """emcee and metropolis on the tcgen05 path, data drawn from 16 theta* (mean |logit| ~ 11): every stored
    log-density is the oracle's at the stored theta within the bound."""
    N, d = 50_001, 32
    X, y, tstar = scaled_logistic_problem(N, d, 16, seed=77)
    ld, od = _logistic(km, orc, X, y)
    r = 1.0 / np.sqrt(N)
    nw = 128
    x0 = tstar + cases.ball(np.zeros(d), r, nw, 1)
    th, ar, lp, _ = km.emcee(ld, x0, niter=16 * nw, nburnin=4 * nw, nthin=2, use_progress_meter=False, seed=3)
    assert ar.mean() > 0.05
    _check_logistic_chain(od, X, th, lp, "logistic emcee x16")
    th, ar, lp, _ = km.metropolis(ld, km.normal_proposal(0.3 * r), x0[:64], niter=40, nburnin=10, nthin=2, nchains=64,
                                  use_progress_meter=False)
    assert ar.mean() > 0.05
    _check_logistic_chain(od, X, th, lp, "logistic metropolis x16")


# ---------------------------------------------------------------------------------- dense Gaussian (K2, K2F, K2G)

GAUSS_D = [17, 31, 32, 33, 63, 64, 65, 100, 127, 128]


def _gaussian(km, orc, kind, d):
    mean, cov = gaussian_case(kind, d)
    prm = cases.gaussian_params(mean, cov)
    ld = km.LogDensity("gaussian", d, prm)
    ld.set_option("tensor_cores", 1)
    assert ld.info("tensor_cores") == 1.0
    return mean, cov, prm, ld, orc.Density("gaussian", d, prm)


def _check_gaussian(prm, d, pts, got, want):
    """Both bounds; returns (error / derived bound, error / published bound)."""
    mu, A = gaussian_matrix(prm, d)
    bound = gaussian_bound(pts, A, mu)
    claim = 1e-5 * (1.0 + gaussian_terms(pts, A, mu)[0])
    err = got - want
    assert np.all(np.isfinite(got))
    assert np.all(np.abs(err) <= bound), _ratio(err, bound)
    assert np.all(np.abs(err) <= claim), _ratio(err, claim)
    return _ratio(err, bound), _ratio(err, claim)


@pytest.mark.parametrize("d", GAUSS_D)
@pytest.mark.parametrize("kind", GAUSS_KINDS)
def test_gaussian_paths_within_derived_bound(km, orc, kind, d):
    """Covariances: spd_cov, equicorrelated at rho = 0.99 and 0.999, block copies of mvn2's, spd_cov at per-coordinate
    scales 1e-3 .. 1e3, and a mean at 1e3.  eval at 1.5 sigma and 1e3 sigma; then every stored log-density of the
    emcee pipeline (launch_mode 1), the fused kernels K2F and K2G, and Metropolis on the batched path."""
    mean, cov, prm, ld, od = _gaussian(km, orc, kind, d)
    out = []
    for nsigma in (1.5, 1e3):
        pts = gaussian_points(mean, cov, nsigma, 300, seed=d)
        r = _check_gaussian(prm, d, pts, ld.eval(pts), od.eval(pts))
        out.append(f"eval {nsigma:g}sigma {r[0]:.3g}/{r[1]:.3g}")
    nw = 256
    x0 = gaussian_points(mean, cov, 1.0, nw, seed=d + 1)
    for label, variant, mode in (("launch_mode=1", 2, 1), ("K2F", 1, 0), ("K2G", 2, 0)):
        ld.set_option("fused_variant", variant)
        s = km.Sampler(ld, x0, 6, 2, 1, 2.0, seed=5, launch_mode=mode)
        s.run(-1)
        th, lp, ar = s.results()
        s.close()
        pts = th.reshape(-1, d)
        r = _check_gaussian(prm, d, pts, lp.reshape(-1), od.eval(pts, nthreads=8))
        out.append(f"{label} {r[0]:.3g}/{r[1]:.3g}")
    m = km.Metropolis(ld, x0, km.normal_proposal(np.sqrt(np.diag(cov) / d)), 8, 2, 1, seed=5)
    m.run(-1)
    th, lp, ar = m.results()
    m.close()
    pts = th.reshape(-1, d)
    r = _check_gaussian(prm, d, pts, lp.reshape(-1), od.eval(pts, nthreads=8))
    out.append(f"metropolis {r[0]:.3g}/{r[1]:.3g}")
    print(f"\ngaussian {kind} d={d}: max error / derived bound / 1e-5 (1 + |y|^2)  " + "; ".join(out))


# ---------------------------------------------------------------------------------- inputs outside the FP32 range

def _bad_rows(d, good):
    """Rows with one coordinate at 1e39, -1e39, NaN, and one row at 1e39 throughout."""
    rows = np.repeat(good[None], 4, axis=0)
    rows[0, 0], rows[1, d // 2], rows[2, d - 1] = 1e39, -1e39, np.nan
    rows[3] = 1e39
    return rows


def _never_finite(v):
    assert np.all(np.isnan(v) | (v == -np.inf)), v


def _check_never_accepted(x0, th, lp):
    """A stored state that is not the walker's starting point was accepted: it must be inside the FP32 range with a
    finite log-density.  A walker that starts outside the range may only leave it for a state inside."""
    same = (th == x0[:, None, :]) | (np.isnan(th) & np.isnan(x0[:, None, :]))
    moved = ~np.all(same, axis=2)
    inside = np.all(np.abs(th) <= F32_MAX, axis=2)
    assert np.all(inside[moved]) and np.all(np.isfinite(lp[moved]))


def test_outside_fp32_range_is_never_finite_nor_accepted(km, orc):
    d = 33
    mean, cov, prm, ld, od = _gaussian(km, orc, "spd", d)
    _never_finite(ld.eval(_bad_rows(d, mean)))
    X, y, tstar = scaled_logistic_problem(5000, 32, 4, seed=9)
    ll, _ = _logistic(km, orc, X, y)
    _never_finite(ll.eval(_bad_rows(32, tstar)))
    # ensembles with walkers outside the range: a partner there puts the stretch proposal outside it too
    nw = 128
    for dens, centre, scale, modes in ((ld, mean, 1.0, ((2, 1), (1, 0), (2, 0))), (ll, tstar, 0.02, ((0, 0),))):
        dd = centre.size
        x0 = centre + cases.ball(np.zeros(dd), scale, nw, 3)
        for w in (0, 5, nw // 2 + 1, nw // 2 + 7):
            x0[w, w % dd] = 1e39 if w % 2 else -1e39
        x0[nw // 2 + 3, 0] = np.nan
        for variant, mode in modes:
            if dens is ld:
                ld.set_option("fused_variant", variant)
            s = km.Sampler(dens, x0, 8, 0, 1, 2.0, seed=11, launch_mode=mode)
            s.run(-1)
            th, lp, ar = s.results()
            s.close()
            _check_never_accepted(x0, th, lp)
    # Metropolis: every proposal lies outside the range, so no chain moves
    x0 = mean + cases.ball(np.zeros(d), 0.5, 64, 4)
    th, ar, lp, _ = km.metropolis(ld, km.normal_proposal(1e39), x0, niter=6, nburnin=0, nthin=1, nchains=64,
                                  use_progress_meter=False)
    assert np.all(ar == 0) and np.all(th == x0[:, None, :])
