"""kissmcmc.jl_b200 -- B200-native emcee stretch-move hot path of KissMCMC.jl.

Holds only what the path needs: csrc/ (CUDA kernels + the C-ABI of libkissmcmc_cuda.so), the
Python host mirror of the reference's public API (api.py) and the Julia `CUDABackend` module
source (julia/).  Import it as `kissmcmc_b200` (the directory name has a dot in it; the
repo-root shim kissmcmc_b200.py registers it).
"""
from ._lib import (EXCHANGE_PUSH, EXCHANGE_REPLICA, KmcError, MODE_PHILOX, MODE_REPLAY, MULTI_INDEPENDENT, MULTI_SHARDED,
                   SYMBOLS, LIB_PATH, device_count, lib, trim)
from .api import (LogDensity, Metropolis, MultiSampler, NormalProposal, Sampler, ball_randn, ball_randn_device, cdf_g_inv, g_pdf, sample_g, emcee, exponential, gaussian, gaussian_mixture,
                  gaussian_mixture_params, gaussian_params, logistic, lognormal,
                  make_theta0s, metropolis, metropolis_draws, metropolis_randn, normal_proposal, philox4x32_10, rosenbrock,
                  squash_walkers)

from .analysis import acor1d, auto_window, eff_samples, evaluate_convergence, int_acorr  # noqa: E402


def __getattr__(name):
    # the one-process-per-GPU drivers need torch.distributed; everything else (including the library-owned
    # multi-GPU path, MultiSampler / emcee(devices=...)) works without torch, so the import is lazy
    if name == "distributed":
        import importlib
        return importlib.import_module(__name__ + ".distributed")
    raise AttributeError(name)


__all__ = [
    "distributed", "MultiSampler", "EXCHANGE_PUSH", "EXCHANGE_REPLICA", "MULTI_SHARDED", "MULTI_INDEPENDENT", "int_acorr", "acor1d", "auto_window", "eff_samples", "evaluate_convergence",
    "emcee", "make_theta0s", "squash_walkers", "LogDensity", "Sampler", "exponential", "rosenbrock", "gaussian",
    "gaussian_params", "gaussian_mixture", "gaussian_mixture_params", "lognormal", "logistic", "KmcError", "MODE_PHILOX", "MODE_REPLAY", "device_count", "trim", "ball_randn", "ball_randn_device", "g_pdf", "cdf_g_inv", "sample_g",
    "philox4x32_10", "SYMBOLS", "LIB_PATH", "lib", "metropolis", "normal_proposal", "NormalProposal", "Metropolis",
    "metropolis_draws", "metropolis_randn",
]
