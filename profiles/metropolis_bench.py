"""Benchmark of the batched Metropolis sampler; prints ONE JSON line.  bench.py (the emcee workload) is separate.

Workloads (chain-steps/s from CUDA events around the sampler's kernels, inputs resident in HBM, one warm-up run of
every shape, the 126 MB L2 overwritten before every timed launch -- before the single launch of a fused run, before
every step of a batched run; end-to-end = wall time of the public metropolis() call, results copied to the host):
  readme      Exp(1), ONE chain, sigma = 1.5, niter = 10^5 (the reference README call): a latency case, us per step
  rosenbrock  Rosenbrock/20, 2^20 chains x 10^4 steps, nthin = 1000: the fused thread-per-chain kernel
  gauss100    100-D Gaussian, 2^16 chains: the batched FP64 pipeline (propose -> dense contraction -> accept per step)
  logistic    logistic regression d = 32, N = 10^6, 8192 chains, FP64 and tensor_cores=1
The bound of the fused kernel is issue rate: per chain-step one Philox4x32-10 per coordinate pair, Box-Muller (log,
sqrt, sincospi), the density and one log for the accept test, all FP64 except Philox; DRAM traffic is only the
thinned store, (8d + 8) / nthin bytes per chain-step.  The batched workloads are bound by their density kernel.
The CPU column is the oracle (metropolis_oracle/, OpenMP over chains, -march=native) fed pre-drawn normals and
uniforms -- it does not pay for its random numbers -- on a sub-sample of chains/steps, reported as chain-steps/s.

Usage: python profiles/metropolis_bench.py [--quick]
"""
from __future__ import annotations

import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import kissmcmc_b200 as km  # noqa: E402
from tests import cases  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    name, plim, sm, smmax = [v.strip() for v in r.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=plim, sm_clock=sm, sm_clock_max=smmax)


class L2Flush:
    def __init__(self):
        import torch
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def __call__(self):
        import torch
        self.buf.random_(0, 255)
        torch.cuda.synchronize()


def timed(ld, x0, sigma, niter, nburnin, nthin, flush, per_step):
    """Device ms of the whole run (sum of per-step launches for the batched pipeline) and the launch count."""
    s = km.Metropolis(ld, x0, km.normal_proposal(sigma), niter, nburnin, nthin, seed=1)
    try:
        ms, launches = 0.0, 0
        if per_step:
            for _ in range(niter):
                flush()
                s.run(1)
                m, n = s.last_run_ms()
                ms, launches = ms + m, launches + n
        else:
            flush()
            s.run(-1)
            ms, launches = s.last_run_ms()
    finally:
        s.close()
    return ms, launches


def e2e(ld, x0, sigma, niter, nburnin, nthin):
    t0 = time.perf_counter()
    one = len(x0) == 1
    km.metropolis(ld, km.normal_proposal(sigma), x0[0] if one else x0, niter=niter, nburnin=nburnin, nthin=nthin,
                  use_progress_meter=False, seed=1, nchains=None if one else len(x0))
    return time.perf_counter() - t0


def cpu_rate(od, x0, sigma, niter, nburnin, nthin):
    from metropolis_oracle import oracle as mo
    nc, d = x0.shape
    rng = np.random.default_rng(0)
    n, u = rng.standard_normal((niter, nc, d)), rng.random((niter, nc))
    nt = mo.max_threads(native=True)
    mo.metropolis(od, x0, sigma, min(niter, 2), 0, 1, n[:2], u[:2], nthreads=nt, native=True)  # warm-up / page-in
    t0 = time.perf_counter()
    mo.metropolis(od, x0, sigma, niter, nburnin, nthin, n, u, nthreads=nt, native=True)
    return nc * niter / (time.perf_counter() - t0), nt, nc, niter


def main(quick=False):
    flush = L2Flush()
    out = dict(gpu_info(), metric="chain_steps_per_s", workloads={})
    W = out["workloads"]
    sc = 10 if quick else 1

    # README call -------------------------------------------------------------------------------------------------
    ld = km.exponential()
    x0 = np.array([[0.5]])
    timed(ld, x0, 1.5, 1000, 500, 1, flush, False)
    ms, nl = timed(ld, x0, 1.5, 10**5 // sc, 10**5 // sc // 2, 1, flush, False)
    r, nt, cc, cn = cpu_rate(km_oracle("exponential", 1), x0, 1.5, 10**5 // sc, 10**5 // sc // 2, 1)
    W["readme_exp1"] = dict(chains=1, steps=10**5 // sc, kernel_ms=ms, launches=nl, us_per_step=ms * 1e3 / (10**5 // sc),
                            chain_steps_per_s=(10**5 // sc) / (ms * 1e-3),
                            e2e_s=e2e(ld, x0, 1.5, 10**5 // sc, 10**5 // sc // 2, 1),
                            cpu_chain_steps_per_s=r, cpu_threads=nt, bound="latency: one thread, serial steps")

    # Rosenbrock/20, fused ----------------------------------------------------------------------------------------
    ld = km.rosenbrock()
    nc, steps = 2**20 // sc, 10**4 // sc
    x0 = cases.ball([1.0, 1.0], 0.5, nc, 1)
    timed(ld, x0, 0.5, 100, 0, 100, flush, False)
    ms, nl = timed(ld, x0, 0.5, steps, 0, 1000 // sc, flush, False)
    r, nt, cc, cn = cpu_rate(km_oracle("rosenbrock", 2, [1.0, 100.0, 20.0]), x0[:2**14], 0.5, 200, 0, 100)
    W["rosenbrock20_2e20"] = dict(chains=nc, steps=steps, nthin=1000 // sc, kernel_ms=ms, launches=nl,
                                  chain_steps_per_s=nc * steps / (ms * 1e-3), dram_bytes_per_chain_step=(8 * 2 + 8) / (1000 // sc),
                                  e2e_s=e2e(ld, x0, 0.5, steps, 0, 1000 // sc),
                                  cpu_chain_steps_per_s=r, cpu_threads=nt, cpu_sample=[cc, cn],
                                  bound="issue rate (Philox + Box-Muller + density + log per chain-step)")

    # 100-D Gaussian, batched FP64 --------------------------------------------------------------------------------
    d = 100
    mean, cov = np.linspace(-1, 1, d), cases.spd_cov(d, 3)
    ld = km.gaussian(mean, cov)
    nc, steps = 2**16 // sc, 20
    x0 = mean + cases.ball(np.zeros(d), 0.3, nc, 1)
    timed(ld, x0, 0.05, 2, 0, 1, flush, True)
    ms, nl = timed(ld, x0, 0.05, steps, 0, 1, flush, True)
    r, nt, cc, cn = cpu_rate(km_oracle("gaussian", d, km.gaussian_params(mean, cov)), x0[:1024], 0.05, 5, 0, 1)
    W["gaussian100_2e16_fp64"] = dict(chains=nc, steps=steps, kernel_ms=ms, launches=nl, launches_per_step=nl / steps,
                                      chain_steps_per_s=nc * steps / (ms * 1e-3), e2e_s=e2e(ld, x0, 0.05, steps, 0, 1),
                                      cpu_chain_steps_per_s=r, cpu_threads=nt, cpu_sample=[cc, cn],
                                      bound="FP64 dense contraction (2 d^2 flop per chain-step)")

    # logistic d = 32, N = 10^6 -----------------------------------------------------------------------------------
    N, d = 10**6 // sc, 32
    X, y, tstar = cases.logistic_problem(N=N, d=d, seed=0)
    nc = 8192 // sc
    x0 = tstar + cases.ball(np.zeros(d), 0.001, nc, 1)
    r, nt, cc, cn = cpu_rate(km_oracle("logistic", d, [10.0], np.concatenate([X.ravel(), y])), x0[:64], 0.001, 2, 0, 1)
    for tc in (False, True):
        ld = km.logistic(X, y, prior_sigma=10.0, tensor_cores=tc)
        steps = 20 if tc else 5
        timed(ld, x0, 0.001, 1, 0, 1, flush, True)
        ms, nl = timed(ld, x0, 0.001, steps, 0, 1, flush, True)
        W["logistic32_N1e6_8192" + ("_tc" if tc else "_fp64")] = dict(
            chains=nc, steps=steps, kernel_ms=ms, launches=nl, launches_per_step=nl / steps,
            chain_steps_per_s=nc * steps / (ms * 1e-3), e2e_s=e2e(ld, x0, 0.001, steps, 0, 1),
            cpu_chain_steps_per_s=r, cpu_threads=nt, cpu_sample=[cc, cn],
            bound="logits GEMM (2 N d flop per chain-step)" + (", tcgen05 bf16x3" if tc else ", FP64"))
    out.update(gpu_info_after=gpu_info())
    print(json.dumps(out))


def km_oracle(name, d, params=(), data=None):
    from oracle.oracle import Density
    return Density(name, d, params, data=data)


if __name__ == "__main__":
    main(quick="--quick" in sys.argv)
