"""Benchmark of the correlated Metropolis proposal against the diagonal one; prints ONE JSON line.

Every workload alternates diagonal and Cholesky runs of the same chains in one process (REPS rounds), with the GPU's
name and power limit read in the same run.  Rates are chain-steps/s from CUDA events around the sampler's kernels
(kmc_emcee_last_run_ms), the 126 MB L2 overwritten before every timed launch (before every step of a batched run):
  rosenbrock20  Rosenbrock/20, 2^20 chains x 10^4 steps, nthin = 1000: the fused kernel (metropolis_chol_kernel)
  gauss100      100-D Gaussian, 2^16 chains: the batched pipeline.  The split of a step into propose / density /
                accept is the kernel time torch.profiler records for each stage, in a separate profiled pass.
  mvn2          the reference's correlated target (correlation 0.995), 2^20 chains: rate, plus the integrated
                autocorrelation time tau of 1024 chains x 10^4 steps (int_acorr), and effective samples per second
                = chain-steps/s / max(tau).
Usage: python profiles/metropolis_chol_bench.py [--quick]
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

REPS = 3


def timed(ld, x0, prop, niter, nburnin, nthin, flush, per_step):
    s = km.Metropolis(ld, x0, prop, niter, nburnin, nthin, seed=1)
    try:
        ms = 0.0
        if per_step:
            for _ in range(niter):
                flush()
                s.run(1)
                ms += s.last_run_ms()[0]
        else:
            flush()
            s.run(-1)
            ms = s.last_run_ms()[0]
    finally:
        s.close()
    return ms


def alternate(ld, x0, props, niter, nburnin, nthin, flush, per_step):
    """{name: [chain-steps/s of each round]}, the proposals run in turn within every round."""
    for p in props.values():                                  # warm-up of every shape the timed rounds use
        timed(ld, x0, p, 2, 0, 1, flush, per_step)
    out = {k: [] for k in props}
    for _ in range(REPS):
        for k, p in props.items():
            out[k].append(len(x0) * niter / (timed(ld, x0, p, niter, nburnin, nthin, flush, per_step) * 1e-3))
    return out


def summary(rates):
    r = np.asarray(rates)
    return dict(chain_steps_per_s=float(np.median(r)), spread=[float(r.min()), float(r.max())])


def stage_split(ld, x0, prop, steps):
    """ms per step of each stage from a torch.profiler pass (kernel names: the propose kernels, mh_accept_kernel,
    everything else is the density)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    s = km.Metropolis(ld, x0, prop, steps, 0, 1, seed=2)
    try:
        s.run(1)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            s.run(-1)
            torch.cuda.synchronize()
    finally:
        s.close()
    split = dict(propose=0.0, density=0.0, accept=0.0)
    for e in prof.key_averages():
        if e.device_type.name != "CUDA":
            continue
        us = e.self_device_time_total if hasattr(e, "self_device_time_total") else e.self_cuda_time_total
        k = "propose" if any(n in e.key for n in ("mh_propose", "mh_normals", "mh_chol")) else \
            "accept" if "mh_accept" in e.key else "density"
        split[k] += us * 1e-3 / (steps - 1)
    return split


def main(quick=False):
    flush = L2Flush()
    out = dict(gpu_info(), metric="chain_steps_per_s", reps=REPS, workloads={})
    W = out["workloads"]
    sc = 10 if quick else 1

    # Rosenbrock/20, fused ----------------------------------------------------------------------------------------
    ld = km.rosenbrock()
    nc, steps, nthin = 2**20 // sc, 10**4 // sc, 1000 // sc
    x0 = cases.ball([1.0, 1.0], 0.5, nc, 1)
    props = dict(diag=km.normal_proposal(0.5), chol=km.normal_proposal(cov=[[0.25, 0.4], [0.4, 0.81]]))
    r = alternate(ld, x0, props, steps, 0, nthin, flush, False)
    W["rosenbrock20_2e20"] = dict(chains=nc, steps=steps, nthin=nthin, path="fused",
                                  diag=summary(r["diag"]), chol=summary(r["chol"]))

    # 100-D Gaussian, batched FP64 --------------------------------------------------------------------------------
    d = 100
    mean, cov = np.linspace(-1, 1, d), cases.spd_cov(d, 3)
    ld = km.gaussian(mean, cov)
    nc, steps = 2**16 // sc, 20
    x0 = mean + cases.ball(np.zeros(d), 0.3, nc, 1)
    props = dict(diag=km.normal_proposal(0.05), chol=km.normal_proposal(cov=0.05**2 * cov / np.diag(cov).mean()))
    r = alternate(ld, x0, props, steps, 0, 1, flush, True)
    W["gaussian100_2e16_fp64"] = dict(chains=nc, steps=steps, path="batched",
                                      diag=dict(summary(r["diag"]), ms_per_step_profiled=stage_split(ld, x0, props["diag"], 6)),
                                      chol=dict(summary(r["chol"]), ms_per_step_profiled=stage_split(ld, x0, props["chol"], 6)),
                                      propose_flop_per_chain_step=d * (d + 1))

    # mvn2: rate and effective samples ----------------------------------------------------------------------------
    pname, d, params, theta0, _ = cases.plugin_specs()["mvn2"]
    ld = km.LogDensity(pname, d, params)
    mvn = np.asarray(cases.MVN_COV)
    props = dict(diag=km.normal_proposal([0.3, 1.2]), chol=km.normal_proposal(cov=2.38**2 / 2 * mvn))
    nc, steps = 2**20 // sc, 2000
    x0 = cases.ball(theta0, 0.1, nc, 1)
    r = alternate(ld, x0, props, steps, 0, 1000, flush, False)
    ent = dict(chains=nc, steps=steps, path="fused")
    for k, p in props.items():
        th, ar, _, _ = km.metropolis(ld, p, cases.ball(theta0, 0.1, 1024, 2), niter=10**4 // sc, nchains=1024,
                                     use_progress_meter=False, seed=3)
        tau, _ = km.int_acorr(th, warn=False)
        rate = summary(r[k])
        ent[k] = dict(rate, tau=tau.tolist(), accept_ratio=float(ar.mean()),
                      eff_samples_per_s=rate["chain_steps_per_s"] / float(np.max(tau)))
    W["mvn2_2e20"] = ent
    out.update(gpu_info_after=gpu_info())
    print(json.dumps(out))


if __name__ == "__main__":
    main(quick="--quick" in sys.argv)
