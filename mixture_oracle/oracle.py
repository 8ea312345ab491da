"""ctypes front end of the Gaussian-mixture CPU oracle (mixture_oracle/kmo_mixture.c).  TEST INFRASTRUCTURE ONLY.

Only tests/ and profiles/ may import this module; the product never does.  The library is compiled on first use into
a temporary directory (the tree may be read-only), with the flags of the emcee oracle: -ffp-contract=off, OpenMP.
`Density`, `emcee` and `metropolis` take the arguments of oracle.oracle.Density / oracle.oracle.emcee and
metropolis_oracle.oracle.metropolis, and accept "gaussian_mixture" besides every plugin those know.
"""
from __future__ import annotations

import atexit
import ctypes as C
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from oracle import oracle as _emcee_oracle

_HERE = Path(__file__).resolve().parent
_GCC = "/usr/bin/gcc"
_FLAGS = ["-O3", "-march=x86-64-v3", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared"]
KIND_GAUSSIAN_MIXTURE = 5
_lib: C.CDLL | None = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="kmo_mixture_")
        atexit.register(shutil.rmtree, tmp, True)
        out = Path(tmp) / "libkmo_mixture.so"
        subprocess.run([_GCC, *_FLAGS, "-o", str(out), str(_HERE / "kmo_mixture.c"), "-lm"], check=True)
        L = C.CDLL(str(out))
        L.kmo_mix_logpdf.restype = C.c_double
        L.kmo_mix_emcee.restype = C.c_int
        L.kmo_mix_metropolis.restype = C.c_int
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _i64p(a):
    return a.ctypes.data_as(C.POINTER(C.c_int64)) if a is not None else None


class Density(_emcee_oracle.Density):
    """A plugin instance for this oracle: "gaussian_mixture" (params as kissmcmc_b200.gaussian_mixture_params packs
    them) or any plugin of oracle.oracle.Density, evaluated through kmo_mix_logpdf."""

    def __init__(self, name: str, d: int, params=(), data: np.ndarray | None = None):
        if name != "gaussian_mixture":
            super().__init__(name, d, params, data)
            return
        self.name, self.d, self.data = name, int(d), None
        self.params = np.ascontiguousarray(np.asarray(params, dtype=np.float64).ravel())
        self._s = _emcee_oracle._Density(KIND_GAUSSIAN_MIXTURE, self.d, _dp(self.params), self.params.size, None, 0)

    def logpdf(self, theta) -> float:
        th = np.ascontiguousarray(np.atleast_1d(np.asarray(theta, dtype=np.float64)))
        assert th.size == self.d
        return float(lib().kmo_mix_logpdf(C.byref(self._s), _dp(th)))

    def eval(self, thetas, nthreads=1) -> np.ndarray:
        th = np.ascontiguousarray(np.asarray(thetas, dtype=np.float64).reshape(-1, self.d))
        out = np.empty(th.shape[0])
        lib().kmo_mix_eval(C.byref(self._s), _dp(th), C.c_int64(th.shape[0]), _dp(out), C.c_int32(nthreads))
        return out


def emcee(dens: Density, theta0s, niter_walker, nburnin_walker, nthin=1, a_scale=2.0, seed=0, replay=None,
          trace=False, store=True, nthreads=1):
    """oracle.oracle.emcee over kmo_mix_emcee: the same arguments and the same returned dict."""
    x = np.array(np.asarray(theta0s, dtype=np.float64).reshape(len(theta0s), -1), order="C")
    nw, d = x.shape
    assert d == dens.d
    lp = dens.eval(x, nthreads=nthreads)
    ns = (niter_walker - nburnin_walker) // nthin
    nslots = niter_walker * nw
    chain_x = np.empty((nw, ns, d)) if store else None
    chain_lp = np.empty((nw, ns)) if store else None
    naccept, ratio = np.zeros(nw, dtype=np.int64), np.empty(nw)
    if replay is not None:
        rp = [np.ascontiguousarray(replay[0], dtype=np.int64), np.ascontiguousarray(replay[1], dtype=np.float64),
              np.ascontiguousarray(replay[2], dtype=np.float64)]
        assert all(a.size == nslots for a in rp)
        mode = _emcee_oracle.MODE_REPLAY
    else:
        rp, mode = [None, None, None], _emcee_oracle.MODE_PHILOX
    tr = None
    if trace:
        tr = (np.empty(nslots, dtype=np.int64), np.empty(nslots), np.empty(nslots), np.empty(nslots, dtype=np.uint8))
    margin = C.c_double()
    rc = lib().kmo_mix_emcee(
        C.byref(dens._s), _dp(x), _dp(lp), C.c_int64(nw), C.c_int64(niter_walker), C.c_int64(nburnin_walker),
        C.c_int64(nthin), C.c_double(a_scale), C.c_int32(mode), C.c_uint64(seed), _i64p(rp[0]), _dp(rp[1]),
        _dp(rp[2]), _dp(chain_x), _dp(chain_lp), _i64p(naccept), _dp(ratio), _i64p(tr[0]) if tr else None,
        _dp(tr[1]) if tr else None, _dp(tr[2]) if tr else None,
        tr[3].ctypes.data_as(C.POINTER(C.c_uint8)) if tr else None, C.byref(margin), C.c_int32(nthreads))
    if rc != 0:
        raise ValueError(f"kmo_mix_emcee rejected its arguments (rc={rc})")
    return dict(chain_x=chain_x, chain_lp=chain_lp, accept_ratio=ratio, naccept=naccept, x=x, lp=lp, trace=tr,
                min_margin=margin.value)


def metropolis(dens, theta0s, sigma, niter, nburnin, nthin, normals, u, nthreads=1, store=True, chol=None):
    """metropolis_oracle.oracle.metropolis over kmo_mix_metropolis: the same arguments and the same returned dict."""
    x = np.array(np.asarray(theta0s, dtype=np.float64).reshape(len(theta0s), -1), order="C")
    nc, d = x.shape
    assert d == dens.d
    assert (sigma is None) != (chol is None), "give sigma or chol"
    n = np.ascontiguousarray(normals, dtype=np.float64)
    uu = np.ascontiguousarray(u, dtype=np.float64)
    assert n.size == niter * nc * d and uu.size == niter * nc
    ns = (niter - nburnin) // nthin if niter > nburnin else 0
    chain_x = np.empty((nc, ns, d)) if store else None
    chain_lp = np.empty((nc, ns)) if store else None
    lp, na, ratio, margin = np.empty(nc), np.zeros(nc, dtype=np.int64), np.empty(nc), C.c_double()
    sig = None if sigma is None else np.ascontiguousarray(np.atleast_1d(np.asarray(sigma, dtype=np.float64)).ravel())
    L = None if chol is None else np.ascontiguousarray(chol, dtype=np.float64)
    assert L is None or L.shape == (d, d)
    rc = lib().kmo_mix_metropolis(C.byref(dens._s), _dp(x), _dp(lp), C.c_int64(nc), C.c_int64(niter),
                                  C.c_int64(nburnin), C.c_int64(nthin), _dp(sig), C.c_int64(0 if sig is None else sig.size),
                                  _dp(L), _dp(n), _dp(uu), _dp(chain_x), _dp(chain_lp), _i64p(na), _dp(ratio),
                                  C.byref(margin), C.c_int32(nthreads))
    if rc != 0:
        raise ValueError(f"kmo_mix_metropolis rejected its arguments (rc={rc})")
    return dict(chain_x=chain_x, chain_lp=chain_lp, accept_ratio=ratio, naccept=na, x=x, lp=lp,
                min_margin=margin.value)
