"""Benchmark of the Gaussian-mixture plugin against its unimodal counterparts; prints ONE JSON line.  Not run by bench.py.

Each mixture workload alternates, in the same process, with unimodal runs of the same geometry (walker-steps /
chain-steps per second from the sampler's CUDA events around its kernels; one warm-up run of every shape; the 126 MB L2
overwritten before every timed launch; the median of `--reps` alternations):
  emcee_d2      2^20 walkers x 10^4 iterations, nthin = 1000, d = 2: mixture K = 4 vs rosenbrock vs the mvn2 gaussian
                (the shared-memory kernel K1)
  metro_d2      2^20 chains x 10^4 steps, nthin = 1000, diagonal proposal: the same three densities
  emcee_d10     2^24 walkers x 200 iterations, nthin = 100, d = 10: mixture K = 4 vs gaussian (the bulk kernel)
The card's name, power limit and SM clock are read before and after, in the same call.

Usage: python profiles/mixture_bench.py [--quick] [--reps N]
"""
from __future__ import annotations

import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "profiles"))

import kissmcmc_b200 as km  # noqa: E402
from metropolis_bench import L2Flush, gpu_info  # noqa: E402
from tests import cases  # noqa: E402
from tests.test_mixture_host import random_mixture  # noqa: E402


def emcee_ms(ld, x0, niter, nthin, flush):
    s = km.Sampler(ld, x0, niter, 0, nthin, 2.0, 1)
    try:
        flush()
        s.run(-1)
        return s.last_run_ms()[0]
    finally:
        s.close()


def metro_ms(ld, x0, niter, nthin, flush):
    s = km.Metropolis(ld, x0, km.normal_proposal(0.5), niter, 0, nthin, seed=1)
    try:
        flush()
        s.run(-1)
        return s.last_run_ms()[0]
    finally:
        s.close()


def alternate(run, arms, n, steps, reps):
    """arms: name -> (density, x0).  Median ms and rate of each arm over `reps` alternations after one warm-up each."""
    for ld, x0 in arms.values():
        run(ld, x0, 2)
    ms = {k: [] for k in arms}
    for _ in range(reps):
        for k, (ld, x0) in arms.items():
            ms[k].append(run(ld, x0, steps))
    out = {}
    for k, v in ms.items():
        med = float(np.median(v))
        out[k] = dict(ms_median=med, ms_all=v, steps_per_s=n * steps / (med * 1e-3))
    mix = out["mixture_k4"]["ms_median"]
    for k in out:
        out[k]["time_vs_mixture"] = out[k]["ms_median"] / mix
    return out


def main(quick=False, reps=3):
    flush = L2Flush()
    res = dict(gpu_info(), metric="walker_or_chain_steps_per_s", workloads={})
    W = res["workloads"]
    sc = 16 if quick else 1

    d, K = 2, 4
    w, mus, covs = random_mixture(d, K, 12)
    mix = km.gaussian_mixture(w, mus, covs)
    mvn2 = km.gaussian(cases.MVN_MEAN, cases.MVN_COV)
    rosen = km.rosenbrock()
    n, steps = 2**20 // sc, 10**4 // sc
    x_mix = mus[np.arange(n) % K] + cases.ball(np.zeros(d), 0.5, n, 1)
    x_mvn = cases.ball(cases.MVN_MEAN, 0.5, n, 2)
    x_ros = cases.ball([1.0, 1.0], 0.5, n, 3)
    arms = dict(mixture_k4=(mix, x_mix), gaussian_mvn2=(mvn2, x_mvn), rosenbrock=(rosen, x_ros))
    W["emcee_d2_2e20_1e4"] = dict(walkers=n, iterations=steps, nthin=1000 // sc, kernel="emcee_smem_kernel (K1)",
                                  arms=alternate(lambda ld, x0, s: emcee_ms(ld, x0, s, 1000 // sc, flush), arms, n,
                                                 steps, reps))
    W["metro_d2_2e20_1e4"] = dict(chains=n, steps=steps, nthin=1000 // sc, kernel="metropolis_kernel (diagonal)",
                                  arms=alternate(lambda ld, x0, s: metro_ms(ld, x0, s, 1000 // sc, flush), arms, n,
                                                 steps, reps))

    d = 10
    w, mus, covs = random_mixture(d, K, 13)
    mix = km.gaussian_mixture(w, mus, covs)
    gau = km.gaussian(np.linspace(-1, 1, d), cases.spd_cov(d, 1))
    n, steps = 2**24 // sc, 200
    x_mix = mus[np.arange(n) % K] + cases.ball(np.zeros(d), 0.5, n, 4)
    x_gau = np.linspace(-1, 1, d) + cases.ball(np.zeros(d), 0.5, n, 5)
    arms = dict(mixture_k4=(mix, x_mix), gaussian_d10=(gau, x_gau))
    W["emcee_d10_2e24_200"] = dict(walkers=n, iterations=steps, nthin=100, kernel="emcee_bulk_kernel",
                                   arms=alternate(lambda ld, x0, s: emcee_ms(ld, x0, s, 100, flush), arms, n, steps,
                                                  reps))
    res.update(gpu_info_after=gpu_info())
    print(json.dumps(res))


if __name__ == "__main__":
    r = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 3
    main(quick="--quick" in sys.argv, reps=r)
