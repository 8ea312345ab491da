"""ctypes front end of the Metropolis CPU oracle (metropolis_oracle/kmo_metropolis.c).  TEST INFRASTRUCTURE ONLY.

Only tests/ and profiles/ may import this module; the product never does.  The library is compiled on first use into
a temporary directory (the tree may be read-only), with the flags of the emcee oracle: -ffp-contract=off, OpenMP.
"""
from __future__ import annotations

import atexit
import ctypes as C
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from oracle.oracle import Density  # noqa: F401  (the plugin instances the oracle takes)

_HERE = Path(__file__).resolve().parent
_GCC = "/usr/bin/gcc"
_FLAGS = ["-O3", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared"]
_libs: dict[bool, C.CDLL] = {}


def lib(native: bool = False) -> C.CDLL:
    """native=True: a -march=native build for the machine it runs on (CPU rates); default x86-64-v3."""
    if native not in _libs:
        tmp = tempfile.mkdtemp(prefix="kmo_metropolis_")
        atexit.register(shutil.rmtree, tmp, True)
        out = Path(tmp) / "libkmo_metropolis.so"
        march = "-march=native" if native else "-march=x86-64-v3"
        subprocess.run([_GCC, *_FLAGS, march, "-o", str(out), str(_HERE / "kmo_metropolis.c"), "-lm"], check=True)
        L = C.CDLL(str(out))
        L.kmo_metropolis.restype = C.c_int
        L.kmo_metropolis_chol.restype = C.c_int
        L.kmo_max_threads.restype = C.c_int32
        _libs[native] = L
    return _libs[native]


def max_threads(native: bool = False) -> int:
    return int(lib(native).kmo_max_threads())


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def metropolis(dens, theta0s, sigma, niter, nburnin, nthin, normals, u, nthreads=1, store=True, native=False,
               chol=None):
    """nchains independent chains fed the draws normals [niter, nchains, d], u [niter, nchains].

    theta0s [nchains, d] (or [nchains]).  sigma: the diagonal proposal x + sigma .* n; or sigma=None and chol=L
    ([d, d] lower-triangular): the correlated proposal x + L n (kmo_metropolis_chol).  Returns dict(chain_x
    [nchains, ns, d], chain_lp [nchains, ns], accept_ratio [nchains], naccept [nchains], x, lp (final state),
    min_margin)."""
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
    common = (C.c_int64(nc), C.c_int64(niter), C.c_int64(nburnin), C.c_int64(nthin))
    tail = (_dp(n), _dp(uu), _dp(chain_x), _dp(chain_lp), na.ctypes.data_as(C.POINTER(C.c_int64)), _dp(ratio),
            C.byref(margin), C.c_int32(nthreads))
    if chol is None:
        sig = np.ascontiguousarray(np.atleast_1d(np.asarray(sigma, dtype=np.float64)).ravel())
        rc = lib(native).kmo_metropolis(C.byref(dens._s), _dp(x), _dp(lp), *common, _dp(sig), C.c_int64(sig.size),
                                        *tail)
    else:
        L = np.ascontiguousarray(chol, dtype=np.float64)
        assert L.shape == (d, d)
        rc = lib(native).kmo_metropolis_chol(C.byref(dens._s), _dp(x), _dp(lp), *common, _dp(L), *tail)
    if rc != 0:
        raise ValueError(f"kmo_metropolis rejected its arguments (rc={rc})")
    return dict(chain_x=chain_x, chain_lp=chain_lp, accept_ratio=ratio, naccept=na, x=x, lp=lp,
                min_margin=margin.value)
