"""Host-side mirror of KissMCMC.jl's public emcee API over libkissmcmc_cuda.so.

Drop-in names, argument meaning and error behaviour of the reference
(/root/reference/src/samplers.jl):

    emcee(logdensity, theta0s; niter, nburnin, nthin, a_scale, use_progress_meter, hasblob,
          init_blobs, reduce_blob!)                               :188-216
    make_theta0s(theta0, ball_radius, logdensity, nwalkers; ...)  :311-349
    squash_walkers(thetas, accept_ratio, logdensities, blobs; ...) :372-428
    metropolis(pdf, sample_ppdf, theta0; niter, nburnin, nthin, ...) :9-128

The one deliberate difference: `logdensity` is a device plugin descriptor (`LogDensity`) and
not a closure -- user closures cannot cross the C-ABI onto the GPU and there is no CPU
fallback.  `hasblob=True` raises (arbitrary host objects cannot live on the device).
"""
from __future__ import annotations

import ctypes as C
import math
import sys
import time
import warnings

import numpy as np

from . import _lib
from ._lib import (EXCHANGE_PUSH, EXCHANGE_REPLICA, EmceeOpts, KmcError, MODE_PHILOX, MODE_REPLAY, MULTI_INDEPENDENT,
                   MULTI_SHARDED, check, lib)

_dp = C.POINTER(C.c_double)
_i64p = C.POINTER(C.c_int64)


def _ptr(a, typ=_dp):
    return a.ctypes.data_as(typ) if a is not None else None


# ------------------------------------------------------------------------------------------
# Log-density plugin registry (replaces the closure `pdf`, src/samplers.jl:257)

class LogDensity:
    """A device log-density plugin instance: name + parameters (+ optional data array)."""

    def __init__(self, name: str, d: int, params=(), data: np.ndarray | None = None, device: int = 0):
        self.name, self.d, self.device = name, int(d), int(device)
        self.params = np.ascontiguousarray(np.asarray(params, dtype=np.float64).ravel())
        self.data = None if data is None else np.ascontiguousarray(data)
        h = C.c_void_p()
        check(lib.kmc_density_create(
            name.encode(), self.d, _ptr(self.params) if self.params.size else None, self.params.size,
            self.data.ctypes.data_as(C.c_void_p) if self.data is not None else None,
            self.data.nbytes if self.data is not None else 0, self.device, C.byref(h)))
        self._h = h

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib.kmc_density_destroy(h)

    def __call__(self, theta):
        """logdensity(theta) like the reference closure: one point -> float, [n,d] -> [n]."""
        th = np.asarray(theta, dtype=np.float64)
        single = th.ndim == 0 or (th.ndim == 1 and self.d > 1)  # for d == 1 a 1-D array is a batch
        out = self.eval(th.reshape(-1, self.d))
        return float(out[0]) if single else out

    def set_option(self, key: str, value: float):
        check(lib.kmc_density_set_option(self._h, key.encode(), float(value)))

    def info(self, key: str) -> float:
        v = C.c_double()
        check(lib.kmc_density_get_info(self._h, key.encode(), C.byref(v)))
        return v.value

    def eval(self, thetas) -> np.ndarray:
        th = np.ascontiguousarray(np.asarray(thetas, dtype=np.float64).reshape(-1, self.d))
        out = np.empty(th.shape[0])
        check(lib.kmc_density_eval(self._h, _ptr(th), th.shape[0], _ptr(out)))
        return out


def exponential(d: int = 1, device: int = 0) -> LogDensity:
    """README.md:15  logpdf(x) = x<0 ? -Inf : -x."""
    return LogDensity("exponential", d, device=device)


def rosenbrock(a: float = 1.0, b: float = 100.0, temper: float = 20.0, device: int = 0) -> LogDensity:
    """test/runtests.jl:68  -(b*(x2-x1^2)^2 + (a-x1)^2)/temper."""
    return LogDensity("rosenbrock", 2, [a, b, temper], device=device)


def gaussian_params(mean, cov) -> np.ndarray:
    """[mu, A row-major, lognorm] with A = chol(cov^-1)^T so that |A(x-mu)|^2 is the Mahalanobis form."""
    mu = np.atleast_1d(np.asarray(mean, dtype=np.float64))
    cov = np.atleast_2d(np.asarray(cov, dtype=np.float64))
    d = mu.size
    prec = np.linalg.inv(cov)
    L = np.linalg.cholesky((prec + prec.T) / 2)  # prec = L L^T,  x^T prec x = |L^T x|^2
    A = L.T
    lognorm = float(np.sum(np.log(np.diag(L))) - 0.5 * d * math.log(2 * math.pi))
    return np.concatenate([mu, A.ravel(), [lognorm]])


def gaussian(mean, cov, device: int = 0) -> LogDensity:
    """MvNormal(mean, cov) (test/runtests.jl:53,61); a scalar mean/variance gives Normal."""
    mu = np.atleast_1d(np.asarray(mean, dtype=np.float64))
    return LogDensity("gaussian", mu.size, gaussian_params(mean, cov), device=device)


def lognormal(mu: float = 0.0, sigma: float = 1.0, device: int = 0) -> LogDensity:
    """LogNormal(mu, sigma) (test/runtests.jl:56)."""
    return LogDensity("lognormal", 1, [mu, sigma, math.log(sigma) + 0.5 * math.log(2 * math.pi)], device=device)


def logistic(X, y, prior_sigma: float = 10.0, device: int = 0, tensor_cores: bool = False) -> LogDensity:
    """Bayesian logistic regression (BASELINE.json configs[3]): X [N, d], y [N] in {0, 1}, prior N(0, sigma^2 I).
    logp(theta) = sum_n (y_n s_n - softplus(s_n)) - |theta|^2 / (2 sigma^2),  s_n = x_n . theta.

    Exact FP64 by default.  Any d <= 512.  tensor_cores=True opts in to the tcgen05 kernel (needs d <= 64 and every X value
    bf16-representable, else KmcError): theta split into three bf16 pieces, FP32 accumulation, FP32 softplus.
    It is APPROXIMATE, and its error grows with the size of the logits.  Per point, with u = 2^-24 and m = ceil(d/16):
        |logp - logp_fp64| <= u [(0.5 + 1.05 m) sum_n sum_k |theta_k x_nk| + 8.5 sum_n |theta . x_n|] + 5 u N
    (at most 13.2 u sum_n sum_k |theta_k x_nk| + 5 u N), and the sum of the two bounds on a difference of two points.
    At d = 32, N = 10^6, theta* ~ N(0, 1/d) (mean |logit| 0.7) that is ~1.3 per point; a B200 shows a common offset of
    about +3e-2 (+3e-8 per data row, in the stored `logdensities` and the initial p0s, cancelling in every accept test)
    and 2e-3 on differences between nearby points.  With the data drawn from 16 theta* (mean |logit| 11) the bound is
    ~13 per point."""
    X = np.ascontiguousarray(X, dtype=np.float32)
    y = np.ascontiguousarray(y, dtype=np.float32).ravel()
    assert X.ndim == 2 and y.size == X.shape[0]
    data = np.concatenate([X.ravel(), y])
    ld = LogDensity("logistic", X.shape[1], [prior_sigma], data=data, device=device)
    if tensor_cores:
        ld.set_option("tensor_cores", 1)
    return ld


# ------------------------------------------------------------------------------------------
# Low-level sampler handle

class Sampler:
    """Owns a kmc_sampler_t.  Counts are PER WALKER (niter_walker = niter // nwalkers)."""

    def __init__(self, logdensity: LogDensity, theta0s, niter_walker, nburnin_walker, nthin=1, a_scale=2.0,
                 seed=0, mode=MODE_PHILOX, device=None, walker_id_base=0, launch_mode=0, shard=None,
                 exchange=EXCHANGE_REPLICA, push_chunk=0, push_cap=0, push_lag=0):
        x = np.ascontiguousarray(np.asarray(theta0s, dtype=np.float64))
        if x.ndim == 1:
            x = x.reshape(-1, 1)
        self.nw, self.d = x.shape
        self.logdensity = logdensity
        self.opts = EmceeOpts(int(niter_walker), int(nburnin_walker), int(nthin), float(a_scale), int(seed),
                              int(mode), int(logdensity.device if device is None else device),
                              int(walker_id_base), int(launch_mode), int(exchange),
                              int(shard[0]) if shard else 0, int(shard[1]) if shard else 0,
                              int(push_chunk), int(push_cap), int(push_lag), 0)
        h = C.c_void_p()
        check(lib.kmc_emcee_create(logdensity._h, _ptr(x), self.nw, self.d, C.byref(self.opts), C.byref(h)))
        self._h = h
        n = C.c_int64()
        check(lib.kmc_emcee_nsamples(h, C.byref(n)))
        self.ns = n.value
        check(lib.kmc_emcee_nlocal(h, C.byref(n)))
        self.nl = n.value            # walkers whose chains this sampler stores (2*shard_count if sharded)

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib.kmc_emcee_destroy(h)

    __del__ = close

    def set_stream(self, cuda_stream: int | None):
        check(lib.kmc_emcee_set_stream(self._h, C.c_void_p(cuda_stream or 0)))

    def set_replay(self, partner, z, u):
        p = np.ascontiguousarray(partner, dtype=np.int64)
        z = np.ascontiguousarray(z, dtype=np.float64)
        u = np.ascontiguousarray(u, dtype=np.float64)
        if not (p.size == z.size == u.size) or p.size % self.nw:
            raise ValueError("replay arrays must each hold niters*nwalkers draws")
        check(lib.kmc_emcee_set_replay(self._h, _ptr(p, _i64p), _ptr(z), _ptr(u), p.size // self.nw))

    def run(self, niters: int = -1, sync: bool = True):
        check(lib.kmc_emcee_run(self._h, int(niters)))
        if sync:
            check(lib.kmc_emcee_sync(self._h))

    def run_half(self, nhalfsteps: int = 1, sync: bool = False):
        """Advance half-ensemble sweeps (two per outer iteration); asynchronous by default."""
        check(lib.kmc_emcee_run_half(self._h, int(nhalfsteps)))
        if sync:
            check(lib.kmc_emcee_sync(self._h))

    def sync(self):
        check(lib.kmc_emcee_sync(self._h))

    def ipc_export(self):
        """(handle_x, handle_flags): two 64-byte CUDA IPC handles for peer mode."""
        hx, hf = C.create_string_buffer(64), C.create_string_buffer(64)
        check(lib.kmc_emcee_ipc_export(self._h, hx, hf))
        return hx.raw, hf.raw

    def set_peers(self, handles_x, handles_flags, rank: int):
        """All ranks' IPC handles (lists of 64-byte strings, rank-major)."""
        n = len(handles_x)
        check(lib.kmc_emcee_set_peers(self._h, b"".join(handles_x), b"".join(handles_flags), n, rank))

    def window_export(self) -> bytes:
        """The 64-byte CUDA IPC handle of a push-exchange sampler's window (positions + receive ring + flags)."""
        hw = C.create_string_buffer(64)
        check(lib.kmc_emcee_window_export(self._h, hw))
        return hw.raw

    def window_attach(self, handles, rank: int):
        """All ranks' window handles (list of 64-byte strings, rank-major)."""
        check(lib.kmc_emcee_window_attach(self._h, b"".join(handles), len(handles), rank))

    def device_ptrs(self):
        """(x, logp, naccept) device addresses: x [nw][d] f64, logp [nw] f64, naccept [nw] u32."""
        x, lp, na = C.c_void_p(), C.c_void_p(), C.c_void_p()
        check(lib.kmc_emcee_device_ptrs(self._h, C.byref(x), C.byref(lp), C.byref(na)))
        return x.value, lp.value, na.value

    def last_run_ms(self):
        ms, n = C.c_double(), C.c_int64()
        check(lib.kmc_emcee_last_run_ms(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def progress(self):
        it, mean, sd, outl = C.c_int64(), C.c_double(), C.c_double(), C.c_int64()
        check(lib.kmc_emcee_progress(self._h, C.byref(it), C.byref(mean), C.byref(sd), C.byref(outl)))
        return it.value, mean.value, sd.value, outl.value

    def results(self, out_thetas=None, out_logp=None, out_ratio=None):
        th = np.empty((self.nl, self.ns, self.d)) if out_thetas is None else out_thetas
        lp = np.empty((self.nl, self.ns)) if out_logp is None else out_logp
        ar = np.empty(self.nl) if out_ratio is None else out_ratio
        check(lib.kmc_emcee_copy_results(self._h, _ptr(th), _ptr(lp), _ptr(ar)))
        return th, lp, ar

    def squash(self, drop_low_accept_ratio=False, drop_fact=2, order=False, with_logp=True):
        """squash_walkers (src/samplers.jl:372-428) of the stored chains ON THE DEVICE: the per-walker chains never
        cross PCIe un-squashed.  Returns the reference 4-tuple (thetas [nkept*ns, d], mean accept ratio of the kept
        walkers, logdensities [nkept*ns] | None, None); `self.squash_stats` holds (nkept, median, std) of the accept
        ratios (what `verbose` prints in the reference, :386)."""
        nk, mean, med, sd = C.c_int64(), C.c_double(), C.c_double(), C.c_double()
        args = (int(bool(drop_low_accept_ratio)), float(drop_fact), int(bool(order)))
        check(lib.kmc_emcee_squash(self._h, *args, None, None, C.byref(nk), C.byref(mean), C.byref(med), C.byref(sd)))
        th = np.empty((nk.value * self.ns, self.d))
        lp = np.empty(nk.value * self.ns) if with_logp else None
        check(lib.kmc_emcee_squash(self._h, *args, _ptr(th), _ptr(lp), C.byref(nk), C.byref(mean), C.byref(med),
                                   C.byref(sd)))
        self.squash_stats = (nk.value, med.value, sd.value)
        return th, mean.value, lp, None

    def chain_moments(self):
        """(mean[d], var[d], nsamples) of the whole stored chain, reduced on the device."""
        mean, var, n = np.empty(self.d), np.empty(self.d), C.c_int64()
        check(lib.kmc_emcee_chain_moments(self._h, _ptr(mean), _ptr(var), C.byref(n)))
        return mean, var, n.value

    def chain_covariance(self):
        """(mean[d], cov[d, d], nsamples) of the whole stored chain (the rows of chain_moments; unbiased, ddof=1),
        reduced on the device in a fixed order: the same chain gives the same bits.  d <= 128."""
        mean, cov, n = np.empty(self.d), np.empty((self.d, self.d)), C.c_int64()
        check(lib.kmc_emcee_chain_covariance(self._h, _ptr(mean), _ptr(cov), C.byref(n)))
        return mean, cov, n.value

    def state(self):
        """Current ensemble (x, logp, naccept); a push-exchange sampler returns the rows it holds
        (its slice of half 0, then of half 1)."""
        n = self.nl if self.opts.exchange == EXCHANGE_PUSH else self.nw
        x, lp, na = np.empty((n, self.d)), np.empty(n), np.empty(n, dtype=np.int64)
        check(lib.kmc_emcee_copy_state(self._h, _ptr(x), _ptr(lp), _ptr(na, _i64p)))
        return x, lp, na


class MultiSampler:
    """Owns a kmc_multi_t: one emcee run over several GPUs of THIS process (library-owned multi-GPU).

    sharded=True   ONE ensemble sharded by walker index over `devices` (push exchange over peer memory); results are
                   those of the single-GPU run of the same ensemble, bit for bit.  theta0s [nw, d].
    sharded=False  len(devices) independent ensembles, theta0s [ndev, nw, d]; results concatenated ensemble-major.
    A device ordinal may repeat (its sub-samplers share the GPU) -- that is how the sharded path runs on one GPU."""

    def __init__(self, logdensity, theta0s, niter_walker, nburnin_walker, nthin=1, a_scale=2.0, seed=0, devices=(0,),
                 sharded=True, push_chunk=0, push_cap=0, push_lag=0):
        devices = [int(v) for v in devices]
        lds = list(logdensity) if isinstance(logdensity, (list, tuple)) else [logdensity] * len(devices)
        assert len(lds) == len(devices)
        x = np.ascontiguousarray(np.asarray(theta0s, dtype=np.float64))
        if sharded:
            x = x.reshape(len(x), -1)
            self.nw, self.d = x.shape
        else:
            x = x.reshape(len(devices), x.shape[1], -1)
            _, self.nw, self.d = x.shape
        self._keep = lds
        self.opts = EmceeOpts(int(niter_walker), int(nburnin_walker), int(nthin), float(a_scale), int(seed), MODE_PHILOX,
                              0, 0, 0, 0, 0, 0, int(push_chunk), int(push_cap), int(push_lag), 0)
        hs = (C.c_void_p * len(devices))(*[ld._h for ld in lds])
        dv = (C.c_int32 * len(devices))(*devices)
        h = C.c_void_p()
        check(lib.kmc_emcee_create_multi(hs, _ptr(x), self.nw, self.d, C.byref(self.opts), dv, len(devices),
                                         MULTI_SHARDED if sharded else MULTI_INDEPENDENT, C.byref(h)))
        self._h = h
        ns, nwo = C.c_int64(), C.c_int64()
        check(lib.kmc_multi_shape(h, C.byref(ns), C.byref(nwo)))
        self.ns, self.nw_out = ns.value, nwo.value

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib.kmc_multi_destroy(h)

    __del__ = close

    def run(self, niters: int = -1, sync: bool = True):
        check(lib.kmc_multi_run(self._h, int(niters)))
        if sync:
            check(lib.kmc_multi_sync(self._h))

    def last_run_ms(self) -> float:
        ms = C.c_double()
        check(lib.kmc_multi_last_run_ms(self._h, C.byref(ms)))
        return ms.value

    def results(self):
        th, lp, ar = np.empty((self.nw_out, self.ns, self.d)), np.empty((self.nw_out, self.ns)), np.empty(self.nw_out)
        check(lib.kmc_multi_copy_results(self._h, _ptr(th), _ptr(lp), _ptr(ar)))
        return th, lp, ar


# ------------------------------------------------------------------------------------------
# emcee  (src/samplers.jl:188-216)

def _require_plugin(logdensity):
    if not isinstance(logdensity, LogDensity):
        raise TypeError(
            "the CUDA backend takes a LogDensity plugin descriptor (exponential(), rosenbrock(), gaussian(), "
            "lognormal(), ...) in place of a closure: user code cannot run on the device and there is no CPU "
            "fallback")


def emcee(logdensity, theta0s, *, niter=10**5, nburnin=None, nthin=1, a_scale=2.0, use_progress_meter=True,
          hasblob=False, init_blobs=None, reduce_blob=None, seed=0, replay=None, launch_mode=0, devices=None,
          sharded=True):
    """The affine-invariant ensemble sampler; same call shape and 4-tuple as the reference.

    devices=[0, 1, ...] runs on several GPUs of this process (library-owned, no torch): sharded=True shards the ONE
    ensemble by walker index (same chains as a single GPU, bit for bit); sharded=False runs len(devices) independent
    ensembles from theta0s [ndev, nw(, d)] and returns them concatenated.

    Returns (thetas, accept_ratio, logdensities, None): thetas[w] is walker w's chain
    ([nw, ns] for scalar theta, [nw, ns, d] otherwise), accept_ratio [nw], logdensities [nw, ns],
    ns = ((niter // nw) - (nburnin // nw)) // nthin.  niter/nburnin are TOTAL walker-steps (:203-204).
    `seed` keys the Philox draws; `replay=(partner, z, u)` uploads the draws instead.
    """
    _require_plugin(logdensity)
    if hasblob or init_blobs is not None or reduce_blob is not None:
        raise NotImplementedError("hasblob=True is not supported by the CUDA backend: blobs are arbitrary host "
                                  "objects (src/samplers.jl:194-196)")
    th = np.asarray(theta0s, dtype=np.float64)  # np.asarray + ascontiguousarray below = the deepcopy at :198
    if devices is not None and not sharded:     # len(devices) independent ensembles, theta0s [ndev, nw(, d)]
        if nburnin is None:
            nburnin = niter // 2
        scalar_theta = th.ndim == 2
        nwalkers = th.shape[1]
        assert a_scale > 1 and nwalkers % 2 == 0, "Use an even number of walkers."
        m = MultiSampler(logdensity, th, niter // nwalkers, nburnin // nwalkers, nthin, a_scale, seed, devices=devices,
                         sharded=False)
        try:
            m.run(-1)
            thetas, logp, ratio = m.results()
        finally:
            m.close()
        return (thetas[:, :, 0] if scalar_theta else thetas), ratio, logp, None
    scalar_theta = th.ndim == 1
    if nburnin is None:
        nburnin = niter // 2                    # :190
    assert a_scale > 1                          # :200
    nwalkers = len(th)                          # :201
    assert nwalkers % 2 == 0, "Use an even number of walkers."    # :202
    niter_walker = niter // nwalkers            # :203
    nburnin_walker = nburnin // nwalkers        # :204
    npar = 1 if scalar_theta else th.shape[1]
    assert nwalkers >= npar + 2, "Use more walkers: at least DOF+2, but better many more."  # :205

    if devices is not None:
        if replay is not None:
            raise NotImplementedError("replay mode runs on one device")
        m = MultiSampler(logdensity, th, niter_walker, nburnin_walker, nthin, a_scale, seed, devices=devices,
                         sharded=True)
        try:
            m.run(-1)
            thetas, logp, ratio = m.results()
        finally:
            m.close()
        if scalar_theta:
            thetas = thetas[:, :, 0]
        return thetas, ratio, logp, None
    mode = MODE_REPLAY if replay is not None else MODE_PHILOX
    s = Sampler(logdensity, th, niter_walker, nburnin_walker, nthin, a_scale, seed, mode,
                launch_mode=launch_mode)
    try:
        if replay is not None:
            s.set_replay(*replay)
        if use_progress_meter and niter_walker > 0:     # :213, :275-284 -- coarse, never per iteration
            chunks = min(20, niter_walker)
            done, t0 = 0, time.time()
            for c in range(chunks):
                upto = (niter_walker * (c + 1)) // chunks
                s.run(upto - done)
                done = upto
                it, mean, sd, outl = s.progress()
                nn = max(1, it - nburnin_walker if it > nburnin_walker else it)
                sys.stderr.write(
                    f"\remcee, niter={niter}, nwalkers={nwalkers}: {100 * done // niter_walker:3d}%  "
                    f"accept_ratio_mean={mean / nn:.3g} accept_ratio_std={sd / nn:.3g} "
                    f"accept_ratio_outliers={outl} burnin_phase={it <= nburnin_walker} "
                    f"[{time.time() - t0:.1f}s]")
            sys.stderr.write("\n")
        else:
            s.run(-1)
        thetas, logp, ratio = s.results()
    finally:
        s.close()
    if scalar_theta:
        thetas = thetas[:, :, 0]
    return thetas, ratio, logp, None


# ------------------------------------------------------------------------------------------
# metropolis  (src/samplers.jl:9-128)

class NormalProposal:
    """The proposal of a random-walk Metropolis chain in place of the closure `sample_ppdf`:
    theta1 = theta0 .+ sigma .* randn(d), sigma a scalar or one scale per component; or, with `chol` (the lower
    Cholesky factor L of the proposal covariance, d x d), the correlated walk theta1 = theta0 .+ L * randn(d).
    `chol` is None for the diagonal walk and `sigma` is None for the correlated one."""

    def __init__(self, sigma, chol=None):
        self.sigma = None if sigma is None else np.ascontiguousarray(
            np.atleast_1d(np.asarray(sigma, dtype=np.float64)).ravel())
        self.chol = None if chol is None else np.ascontiguousarray(np.asarray(chol, dtype=np.float64))
        if self.chol is not None and (self.chol.ndim != 2 or self.chol.shape[0] != self.chol.shape[1]):
            raise ValueError(f"chol must be a square d x d matrix, got shape {self.chol.shape}")

    def __repr__(self):
        if self.chol is not None:
            return f"NormalProposal(chol={self.chol.tolist()})"
        return f"NormalProposal({self.sigma.tolist() if self.sigma.size > 1 else float(self.sigma[0])})"


def normal_proposal(sigma=None, *, cov=None, chol=None) -> NormalProposal:
    """Symmetric Gaussian random walk.  Give exactly one of
    sigma  scale, scalar or length d (finite and > 0, checked at the call): theta1 = theta0 .+ sigma .* randn(d);
    cov    proposal covariance, d x d symmetric positive definite (e.g. 2.38^2 / d times a pilot run's
           chain_covariance()), factored here with numpy's Cholesky;
    chol   its lower Cholesky factor L (lower-triangular, positive diagonal, checked at the call):
           theta1 = theta0 .+ L * randn(d), each component summed in ascending order without FMA."""
    if sum(a is not None for a in (sigma, cov, chol)) != 1:
        raise ValueError("normal_proposal takes exactly one of sigma, cov= and chol=")
    if cov is not None:
        c = np.asarray(cov, dtype=np.float64)
        if c.ndim != 2 or c.shape[0] != c.shape[1] or not np.all(np.isfinite(c)):
            raise ValueError(f"cov must be a finite square d x d matrix, got shape {c.shape}")
        if not np.allclose(c, c.T, rtol=1e-12, atol=1e-14 * np.abs(c).max()):
            raise ValueError("cov is not symmetric")
        try:
            chol = np.linalg.cholesky(0.5 * (c + c.T))
        except np.linalg.LinAlgError:
            raise ValueError("cov is not positive definite") from None
    if chol is not None:
        return NormalProposal(None, chol=chol)
    return NormalProposal(sigma)


def _require_proposal(sample_ppdf) -> NormalProposal:
    if not isinstance(sample_ppdf, NormalProposal):
        raise TypeError(
            "the CUDA backend takes a proposal descriptor (normal_proposal(sigma)) in place of the closure "
            "sample_ppdf: user code cannot run on the device and there is no CPU fallback")
    return sample_ppdf


class Metropolis(Sampler):
    """Owns a kmc_sampler_t of nchains independent random-walk Metropolis chains.  Counts are PER CHAIN.
    Chain c draws with id chain_id_base + c, so it is the same chain whatever the batch it runs in.  Running, results,
    state, squash, chain moments / covariance and progress are those of Sampler; there are no half-steps and nothing
    to exchange.  A proposal with `chol` creates the handle with kmc_metropolis_create_chol."""

    def __init__(self, logdensity: LogDensity, theta0s, proposal, niter, nburnin, nthin=1, seed=0, mode=MODE_PHILOX,
                 device=None, chain_id_base=0):
        x = np.ascontiguousarray(np.asarray(theta0s, dtype=np.float64))
        if x.ndim == 1:
            x = x.reshape(-1, 1)
        self.nw, self.d = x.shape
        self.logdensity = logdensity
        self.proposal = _require_proposal(proposal)
        self.opts = EmceeOpts(int(niter), int(nburnin), int(nthin), 0.0, int(seed), int(mode),
                              int(logdensity.device if device is None else device), int(chain_id_base),
                              0, 0, 0, 0, 0, 0, 0, 0)
        h = C.c_void_p()
        if self.proposal.chol is not None:
            L = self.proposal.chol
            if L.shape != (self.d, self.d):
                raise ValueError(f"the proposal's Cholesky factor is {L.shape[0]} x {L.shape[1]}, the density has d={self.d}")
            check(lib.kmc_metropolis_create_chol(logdensity._h, _ptr(x), self.nw, self.d, _ptr(L), C.byref(self.opts),
                                                 C.byref(h)))
        else:
            sig = self.proposal.sigma
            check(lib.kmc_metropolis_create(logdensity._h, _ptr(x), self.nw, self.d, _ptr(sig), sig.size,
                                            C.byref(self.opts), C.byref(h)))
        self._h = h
        n = C.c_int64()
        check(lib.kmc_emcee_nsamples(h, C.byref(n)))
        self.ns = n.value
        self.nl = self.nw

    def set_replay(self, normals, u):
        """normals [steps, nchains, d] and accept uniforms [steps, nchains] from the current step on."""
        n = np.ascontiguousarray(normals, dtype=np.float64)
        u = np.ascontiguousarray(u, dtype=np.float64)
        if u.size % self.nw or n.size != u.size * self.d:
            raise ValueError("replay arrays must hold [steps, nchains, d] normals and [steps, nchains] uniforms")
        check(lib.kmc_metropolis_set_replay(self._h, _ptr(n), _ptr(u), u.size // self.nw))


def metropolis_draws(seed: int, chain0: int, nchains: int, t0: int, nsteps: int, d: int, device: int = 0):
    """The normals [nsteps, nchains, d] and accept uniforms [nsteps, nchains] the DEVICE draws for chain ids
    [chain0, chain0 + nchains) at 0-based steps [t0, t0 + nsteps)."""
    n, u = np.empty((int(nsteps), int(nchains), int(d))), np.empty((int(nsteps), int(nchains)))
    check(lib.kmc_metropolis_draws(int(seed), int(chain0), int(nchains), int(t0), int(nsteps), int(d), int(device),
                                   _ptr(n), _ptr(u)))
    return n, u


def metropolis_randn(seed: int, chains, steps, d: int):
    """Host restatement of the Metropolis draws of chain ids `chains` at 0-based steps `steps`: (normals
    [len(steps), len(chains), d], uniforms [len(steps), len(chains)]).  Philox counter (chain, t lo, t hi,
    0x4D48 << 16 | pair); the uniform ((r2 & 0xFFFF) << 32 | r3) * 2^-48 of pair 0 is exact integer arithmetic; the
    normals are numpy's Box-Muller of words r0, r1 (the device's log / sqrt / sincospi may differ by a few ulp)."""
    c = np.atleast_1d(np.asarray(chains, dtype=np.uint64))
    t = np.atleast_1d(np.asarray(steps, dtype=np.uint64))
    pair = np.arange((d + 1) // 2, dtype=np.uint64)
    m32 = np.uint64(0xFFFFFFFF)
    r0, r1, r2, r3 = philox4x32_10(c[None, :, None], (t & m32)[:, None, None], (t >> np.uint64(32))[:, None, None],
                                   np.uint64(0x4D480000) | pair[None, None, :], seed, seed >> 32)
    u = (((r2[:, :, 0] & np.uint64(0xFFFF)) << np.uint64(32)) | r3[:, :, 0]).astype(np.float64) * 2.0 ** -48
    u1 = (r0.astype(np.float64) + 1.0) * 2.0 ** -32
    u2 = r1.astype(np.float64) * 2.0 ** -32
    rad = np.sqrt(-2.0 * np.log(u1))
    z = np.stack([rad * np.cos(2 * np.pi * u2), rad * np.sin(2 * np.pi * u2)], axis=-1).reshape(len(t), len(c), -1)
    return z[:, :, :d], u


def metropolis(logdensity, sample_ppdf, theta0, *, niter=10**5, nburnin=None, nthin=1, use_progress_meter=True,
               hasblob=False, seed=0, replay=None, nchains=None):
    """Random-walk Metropolis; same call shape and 4-tuple as the reference, on the device.

    `sample_ppdf` is normal_proposal(sigma), normal_proposal(cov=...) or normal_proposal(chol=...) (a Python
    callable raises TypeError).  niter / nburnin count the steps of
    ONE chain; ns = (niter - nburnin) // nthin.
    nchains=None: the reference call, one chain from theta0 (scalar or [d]): returns (thetas [ns] or [ns, d],
    accept_ratio: float, logdensities [ns], None).
    nchains=k: k independent chains from theta0 [k] or [k, d] (chain c draws with id c): returns ([k, ns(, d)], [k],
    [k, ns], None) -- the per-walker layout of emcee, so squash_walkers, int_acorr, eff_samples and
    evaluate_convergence take it directly.
    `seed` keys the Philox draws; `replay=(normals [niter, k, d], u [niter, k])` uploads the draws instead.
    """
    _require_plugin(logdensity)
    proposal = _require_proposal(sample_ppdf)
    if hasblob:
        raise NotImplementedError("hasblob=True is not supported by the CUDA backend: blobs are arbitrary host objects")
    if nburnin is None:
        nburnin = niter // 2
    d = logdensity.d
    th = np.asarray(theta0, dtype=np.float64)  # + ascontiguousarray in Metropolis: the deepcopy of theta0
    if nchains is None:
        scalar_theta = th.ndim == 0
        if th.size != d or th.ndim > 1:
            raise ValueError(f"theta0 must be a scalar or a vector of length d={d} for one chain")
        k = 1
    else:
        k = int(nchains)
        scalar_theta = th.ndim == 1
        if k < 1 or th.shape not in [(k, d)] + ([(k,)] if d == 1 else []):
            raise ValueError(f"with nchains={k}, theta0 must have shape ({k}, {d})" + (f" or ({k},)" if d == 1 else ""))
    mode = MODE_REPLAY if replay is not None else MODE_PHILOX
    s = Metropolis(logdensity, th.reshape(k, d), proposal, niter, nburnin, nthin, seed, mode)
    try:
        if replay is not None:
            s.set_replay(*replay)
        if use_progress_meter and niter > 0:    # coarse, never per step
            chunks = min(20, niter)
            done, t0 = 0, time.time()
            for c in range(chunks):
                upto = (niter * (c + 1)) // chunks
                s.run(upto - done)
                done = upto
                it, mean, sd, outl = s.progress()
                nn = max(1, it - nburnin if it > nburnin else it)
                sys.stderr.write(
                    f"\rmetropolis, niter={niter}, nchains={k}: {100 * done // niter:3d}%  "
                    f"accept_ratio_mean={mean / nn:.3g} accept_ratio_std={sd / nn:.3g} "
                    f"accept_ratio_outliers={outl} burnin_phase={it <= nburnin} [{time.time() - t0:.1f}s]")
            sys.stderr.write("\n")
        else:
            s.run(-1)
        thetas, logp, ratio = s.results()
    finally:
        s.close()
    if scalar_theta:
        thetas = thetas[:, :, 0]
    if nchains is None:
        return thetas[0], float(ratio[0]), logp[0], None
    return thetas, ratio, logp, None


# ------------------------------------------------------------------------------------------
# make_theta0s  (src/samplers.jl:311-349)

_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10 (numpy uint64 lanes holding 32-bit words)."""
    c0, c1, c2, c3 = (np.asarray(v, dtype=np.uint64) & np.uint64(0xFFFFFFFF) for v in (c0, c1, c2, c3))
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    mask, sh = np.uint64(0xFFFFFFFF), np.uint64(32)
    for _ in range(10):
        p0 = np.uint64(_M0) * c0
        p1 = np.uint64(_M1) * c2
        n0 = (p1 >> sh) ^ c1 ^ np.uint64(k0)
        n2 = (p0 >> sh) ^ c3 ^ np.uint64(k1)
        c0, c1, c2, c3 = n0, p1 & mask, n2, p0 & mask
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return c0, c1, c2, c3


def ball_randn(seed: int, walkers, k: int, j: int, d: int) -> np.ndarray:
    """Counter-based standard normals for make_theta0s: [len(walkers), d], a pure function of
    (seed, walker, halving step k, try j, component).  Philox words -> two 32-bit uniforms in
    (0,1] / [0,1) -> Box-Muller.  Stream tag 0x4D54 keeps it apart from the sampler's draws."""
    w = np.atleast_1d(np.asarray(walkers, dtype=np.uint64))
    comp = np.arange((d + 1) // 2, dtype=np.uint64)
    r0, r1, r2, r3 = philox4x32_10(w[:, None], comp[None, :], np.uint64(k) << np.uint64(16) | np.uint64(j),
                                   np.uint64(0x4D540000), seed, seed >> 32)
    u1 = (r0.astype(np.float64) + 1.0) * 2.0 ** -32
    u2 = r1.astype(np.float64) * 2.0 ** -32
    rad = np.sqrt(-2.0 * np.log(u1))
    z = np.stack([rad * np.cos(2 * np.pi * u2), rad * np.sin(2 * np.pi * u2)], axis=-1).reshape(len(w), -1)
    return z[:, :d]


def ball_randn_device(seed: int, walker0: int, n: int, k: int, j: int, d: int, device: int = 0) -> np.ndarray:
    """The standard normals the DEVICE make_theta0s uses for walkers [walker0, walker0 + n), halving step k, try j:
    the same counter layout as ball_randn, Box-Muller evaluated with the device's log / sqrt / sincospi."""
    out = np.empty((n, d))
    check(lib.kmc_ball_randn(int(seed), int(walker0), int(n), int(k), int(j), int(d), int(device), _ptr(out)))
    return out


def g_pdf(z, a_scale: float = 2.0):
    """src/samplers.jl:224: the density g(z) = 1/sqrt(z) / (2 (sqrt(a) - sqrt(1/a))) on [1/a, a], else 0."""
    zz = np.ascontiguousarray(np.atleast_1d(np.asarray(z, dtype=np.float64)))
    out = np.empty_like(zz)
    check(lib.kmc_g_pdf(_ptr(zz), zz.size, float(a_scale), _ptr(out)))
    return float(out[0]) if np.ndim(z) == 0 else out.reshape(np.shape(z))


def cdf_g_inv(u, a_scale: float = 2.0):
    """src/samplers.jl:227: (u (sqrt(a) - sqrt(1/a)) + sqrt(1/a))^2."""
    uu = np.ascontiguousarray(np.atleast_1d(np.asarray(u, dtype=np.float64)))
    out = np.empty_like(uu)
    check(lib.kmc_cdf_g_inv(_ptr(uu), uu.size, float(a_scale), _ptr(out)))
    return float(out[0]) if np.ndim(u) == 0 else out.reshape(np.shape(u))


def sample_g(a_scale: float = 2.0, n: int | None = None, seed: int = 0, device: int = 0):
    """src/samplers.jl:230: z ~ g, drawn on the device through the sampler's own draw path."""
    out = np.empty(1 if n is None else int(n))
    check(lib.kmc_sample_g(float(a_scale), int(seed), out.size, int(device), _ptr(out)))
    return float(out[0]) if n is None else out


def make_theta0s(theta0, ball_radius, logdensity, nwalkers, *, ball_radius_halfing_steps=7, ntries=100,
                 hasblob=False, seed=0, randn=None, on_device=None):
    """Initial ensemble inside a Gaussian ball around theta0, rejecting points of zero density.

    With a device plugin and no `randn` callback the whole loop runs ON THE DEVICE (kmc_make_theta0s: Philox /
    Box-Muller normals, rejection through the plugin, all pending walkers tried at once); `on_device=False` or a
    `randn` callback selects the host loop below, which batches only the density calls.

    Same loop semantics as the reference, including its quirks (cumulative, never-reset radius
    halving at :326; a walker that exhausts every try is skipped, :344-345 cannot fire), but the
    density calls are batched through the device plugin: all pending walkers are tried at once
    and the sequential order is only replayed for the rare walker that needs a smaller ball.
    randn(walkers, k, j) -> [len(walkers), d] normals (default: counter-based ball_randn).
    Scalar theta0 -> array [nwalkers]; vector theta0 -> [nwalkers, d].
    """
    _require_plugin(logdensity)
    if hasblob:
        raise NotImplementedError("hasblob=True is not supported by the CUDA backend")
    scalar = np.ndim(theta0) == 0
    th0 = np.atleast_1d(np.asarray(theta0, dtype=np.float64))
    npara = th0.size                                         # :315
    br = np.asarray(ball_radius, dtype=np.float64)
    br = np.ones(npara) * br if br.ndim == 0 else br.copy()  # :316-318
    assert br.size == npara                                  # :319
    if on_device is None:
        on_device = randn is None and bool(getattr(logdensity, "_h", None))
    if on_device:
        if randn is not None:
            raise ValueError("a randn callback runs on the host: pass on_device=False")
        res = np.empty((nwalkers, npara))
        nf = C.c_int64()
        th0c, brc = np.ascontiguousarray(th0), np.ascontiguousarray(br)
        check(lib.kmc_make_theta0s(logdensity._h, _ptr(th0c), _ptr(brc), int(nwalkers), int(ball_radius_halfing_steps),
                                   int(ntries), int(seed), _ptr(res), C.byref(nf)))
        if nf.value < nwalkers:
            warnings.warn("make_theta0s: could not find a point of non-zero density for "
                          f"{nwalkers - nf.value} walker(s); like the reference they are silently skipped")
        res = res[:nf.value]
        return res[:, 0] if scalar else res
    if randn is None:
        randn = lambda w, k, j: ball_randn(seed, w, k, j, npara)

    out = np.empty((nwalkers, npara))
    found = np.zeros(nwalkers, dtype=bool)
    i0 = 0
    while i0 < nwalkers:
        pend = np.arange(i0, nwalkers)
        for j in range(1, ntries + 1):                       # k = 1: radius factor 1/2^0 = 1
            tmp = th0[None, :] + randn(pend, 1, j) * br[None, :]
            ok = logdensity.eval(tmp) > -np.inf              # :338
            out[pend[ok]] = tmp[ok]
            found[pend[ok]] = True
            pend = pend[~ok]
            if pend.size == 0:
                break
        if pend.size == 0:
            break
        f = int(pend[0])            # first walker whose k=1 tries all failed: later ones must be redone
        found[f + 1:] = False
        for k in range(2, ball_radius_halfing_steps + 1):    # :324
            br = br * (1.0 / 2.0 ** (k - 1))                 # :326 (cumulative, never reset)
            for j in range(1, ntries + 1):
                tmp = th0[None, :] + randn(np.array([f]), k, j) * br[None, :]
                if logdensity.eval(tmp)[0] > -np.inf:
                    out[f] = tmp[0]
                    found[f] = True
                    break
            if found[f]:
                break
        i0 = f + 1
    if not found.all():
        warnings.warn("make_theta0s: could not find a point of non-zero density for "
                      f"{int((~found).sum())} walker(s); like the reference they are silently skipped")
    res = out[found]
    return res[:, 0] if scalar else res


# ------------------------------------------------------------------------------------------
# squash_walkers  (src/samplers.jl:372-428)

def squash_walkers(thetas, accept_ratio, logdensities=None, blobs=None, *, drop_low_accept_ratio=False,
                   drop_fact=2, verbose=True, order=False, merge_blobs=None):
    """Puts the samples of all walkers into one array (walker-major; time-major if order=True).

    Returns (thetas, mean(accept_ratio[kept]), logdensities | None, None)."""
    if blobs is not None:
        raise NotImplementedError("blobs are not supported by the CUDA backend")
    thetas = np.asarray(thetas)
    accept_ratio = np.asarray(accept_ratio, dtype=np.float64)
    nwalkers = len(accept_ratio)                                             # :378
    if drop_low_accept_ratio:                                                # :379-393
        ma, sa = np.median(accept_ratio), np.std(accept_ratio, ddof=1)
        if verbose:
            print(f"Median accept ratio is {ma}, standard deviation is {sa}\n")
        drop = accept_ratio <= ma - drop_fact * sa
        if verbose:
            for nc in np.nonzero(drop)[0]:
                print(f"Dropping walker {nc + 1} with low accept ratio {accept_ratio[nc]}")
        keep = np.nonzero(~drop)[0]
    else:
        keep = np.arange(nwalkers)                                           # :395
    t = thetas[keep]
    l = None if logdensities is None else np.asarray(logdensities)[keep]
    if order:   # :415-426 stable sortperm of (1:ns repeated) == time-major, walkers in kept order
        t = np.swapaxes(t, 0, 1)
        l = None if l is None else np.swapaxes(l, 0, 1)
    t = t.reshape((-1,) + thetas.shape[2:])                                  # :398-399
    l = None if l is None else l.reshape(-1)
    return t, float(np.mean(accept_ratio[keep])), l, None                    # :427
