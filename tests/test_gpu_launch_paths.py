"""Launch counts of every host run path.  `last_run_ms()[1]` is the one public record of which path a run took:
one launch for the persistent and fused kernels, one per half-step for launch_mode 1, and propose + log-density +
accept kernels per half-step (emcee) or step (Metropolis) for the batched plugins."""
import numpy as np
import pytest

from tests import cases

pytestmark = pytest.mark.gpu

K = 3  # iterations (emcee) or steps (Metropolis) of the measured run(K); the handles are built for 2 K


def _gaussian(km, d, tensor_cores=False, fused_variant=None):
    ld = km.LogDensity("gaussian", d, cases.gaussian_params(np.linspace(-1, 1, d), cases.spd_cov(d, 3)))
    if tensor_cores:
        ld.set_option("tensor_cores", 1)
    if fused_variant:
        ld.set_option("fused_variant", fused_variant)
    return ld


def _logistic(km, d, tensor_cores):
    X, y, _ = cases.logistic_problem(N=3000, d=d, seed=1)  # X exact in bf16: the tcgen05 path is available
    return km.logistic(X, y, tensor_cores=tensor_cores)


def _x0(ld, n):
    return cases.ball(np.full(ld.d, 0.5), 0.1, n, 7)


def _emcee(km, ld, nw=64, **kw):
    return km.Sampler(ld, _x0(ld, nw), 2 * K, 1, 1, 2.0, 5, **kw)


def _metropolis(km, ld, proposal, nchains=64):
    return km.Metropolis(ld, _x0(ld, nchains), proposal, 2 * K, 1, 1, 5)


def _emcee_replay(km, nw=64):
    s = _emcee(km, km.rosenbrock(), nw, mode=km.MODE_REPLAY)
    half = nw // 2
    partner = np.tile(np.concatenate([np.arange(half, nw), np.arange(half)]), 2 * K)  # the other half's walker
    s.set_replay(partner, np.full(partner.size, 1.25), np.full(partner.size, 0.5))
    return s


# id -> (sampler factory, the density's info("batched"), expected launches of run(K))
PATHS = {
    "rosenbrock": (lambda km: _emcee(km, km.rosenbrock()), 0, 1),
    "rosenbrock-replay": (_emcee_replay, 0, 1),
    "rosenbrock-launch_mode1": (lambda km: _emcee(km, km.rosenbrock(), launch_mode=1), 0, 2 * K),
    "gaussian10-fused": (lambda km: _emcee(km, _gaussian(km, 10)), 0, 1),
    "exponential7": (lambda km: _emcee(km, km.exponential(7)), 3, 3 * 2 * K),
    "gaussian20": (lambda km: _emcee(km, _gaussian(km, 20)), 1, 3 * 2 * K),
    "gaussian200-l2": (lambda km: _emcee(km, _gaussian(km, 200), nw=256), 1, 3 * 2 * K),
    "gaussian20-tc-launch_mode1": (lambda km: _emcee(km, _gaussian(km, 20, True), launch_mode=1), 1, 3 * 2 * K),
    "gaussian20-tc-K2G": (lambda km: _emcee(km, _gaussian(km, 20, True)), 1, 1),
    "gaussian20-tc-K2F": (lambda km: _emcee(km, _gaussian(km, 20, True, fused_variant=1)), 1, 1),
    "logistic5": (lambda km: _emcee(km, _logistic(km, 5, False)), 2, 4 * 2 * K),
    "logistic16-tc": (lambda km: _emcee(km, _logistic(km, 16, True)), 2, 5 * 2 * K),
    "mh-rosenbrock-diag": (lambda km: _metropolis(km, km.rosenbrock(), km.normal_proposal(0.1)), 0, 1),
    "mh-rosenbrock-chol": (lambda km: _metropolis(km, km.rosenbrock(), km.normal_proposal(chol=0.1 * np.eye(2))), 0, 1),
    "mh-gaussian20-diag": (lambda km: _metropolis(km, _gaussian(km, 20), km.normal_proposal(0.1)), 1, 3 * K),
    "mh-gaussian20-chol": (lambda km: _metropolis(km, _gaussian(km, 20), km.normal_proposal(chol=0.1 * np.eye(20))),
                           1, 4 * K),
    "mh-logistic16-tc": (lambda km: _metropolis(km, _logistic(km, 16, True), km.normal_proposal(0.05)), 2, 5 * K),
}


@pytest.mark.parametrize("path", list(PATHS))
def test_launch_count(km, path):
    make, batched, want = PATHS[path]
    s = make(km)
    try:
        assert s.logdensity.info("batched") == batched
        s.run(K)
        ms, launches = s.last_run_ms()
        assert launches == want
        assert ms > 0.0
        s.run(0)  # nothing left to run in this call: no launches, no timed window
        assert s.last_run_ms() == (0.0, 0)
    finally:
        s.close()
