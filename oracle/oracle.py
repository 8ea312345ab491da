"""ctypes front end of the CPU oracle (oracle/kmc_oracle.c).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product (kissmcmc.jl_b200, libkissmcmc_cuda.so) never does.

Also holds plain-numpy restatements of the two host-side reference functions:
  make_theta0s     /root/reference/src/samplers.jl:311-349
  squash_walkers   /root/reference/src/samplers.jl:372-428
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
KINDS = {"exponential": 0, "rosenbrock": 1, "gaussian": 2, "lognormal": 3, "logistic": 4}
MODE_PHILOX, MODE_REPLAY = 0, 1
_GCC = "/usr/bin/gcc"
_FLAGS = ["-O3", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared"]


class _Density(C.Structure):
    _fields_ = [("kind", C.c_int32), ("d", C.c_int32), ("params", C.POINTER(C.c_double)),
                ("nparams", C.c_int64), ("data", C.POINTER(C.c_float)), ("ndata", C.c_int64)]


def build(native: bool = False, out_dir: Path = _HERE) -> Path:
    """Compile the oracle into out_dir.  native=True builds a -march=native copy for the machine it
    runs on (bench.py's CPU baseline); the default is a portable x86-64-v3 build."""
    out = Path(out_dir) / ("libkmc_oracle_native.so" if native else "libkmc_oracle.so")
    src = _HERE / "kmc_oracle.c"
    if out.exists() and out.stat().st_mtime >= src.stat().st_mtime:
        return out
    march = "-march=native" if native else "-march=x86-64-v3"
    subprocess.run([_GCC, *_FLAGS, march, "-o", str(out), str(src), "-lm"], check=True)
    return out


_libs: dict[bool, C.CDLL] = {}


def lib(native: bool = False) -> C.CDLL:
    if native not in _libs:
        if native:
            # the native build belongs to the host it runs on, and the tree may be read-only there (bench.py):
            # it is compiled into a temporary directory, which goes once the library is loaded
            with tempfile.TemporaryDirectory(prefix="kmc_oracle_") as tmp:
                try:
                    L = C.CDLL(str(build(True, Path(tmp))))
                except Exception:
                    L = C.CDLL(str(build(False)))
        else:
            L = C.CDLL(str(build(False)))
        L.kmo_g_pdf.restype = C.c_double
        L.kmo_g_pdf.argtypes = [C.c_double, C.c_double]
        L.kmo_cdf_g_inv.restype = C.c_double
        L.kmo_cdf_g_inv.argtypes = [C.c_double, C.c_double]
        L.kmo_logpdf.restype = C.c_double
        L.kmo_max_threads.restype = C.c_int32
        L.kmo_emcee.restype = C.c_int
        _libs[native] = L
    return _libs[native]


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


class Density:
    """A log-density plugin instance for the oracle (same names/params as the CUDA registry)."""

    def __init__(self, name: str, d: int, params=(), data: np.ndarray | None = None):
        self.name, self.d = name, int(d)
        self.params = np.ascontiguousarray(np.asarray(params, dtype=np.float64).ravel())
        self.data = None if data is None else np.ascontiguousarray(data, dtype=np.float32).ravel()
        n = 0
        if name == "logistic":
            n = self.data.size // (self.d + 1)
            assert n * (self.d + 1) == self.data.size
        self._s = _Density(KINDS[name], self.d, _dp(self.params) if self.params.size else None,
                           self.params.size,
                           self.data.ctypes.data_as(C.POINTER(C.c_float)) if self.data is not None else None,
                           n)

    def logpdf(self, theta, native=False) -> float:
        th = np.ascontiguousarray(np.atleast_1d(np.asarray(theta, dtype=np.float64)))
        assert th.size == self.d
        return float(lib(native).kmo_logpdf(C.byref(self._s), _dp(th)))

    def eval(self, thetas, nthreads=1, native=False) -> np.ndarray:
        th = np.ascontiguousarray(np.asarray(thetas, dtype=np.float64).reshape(-1, self.d))
        out = np.empty(th.shape[0])
        lib(native).kmo_density_eval(C.byref(self._s), _dp(th), C.c_int64(th.shape[0]), _dp(out),
                                     C.c_int32(nthreads))
        return out


def philox4x32_10(ctr, key):
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    o = (C.c_uint32 * 4)()
    lib().kmo_philox4x32_10(c, k, o)
    return [int(v) for v in o]


def draw(seed, walker, it, batch, nhalf):
    pl, uz, ua = C.c_int64(), C.c_double(), C.c_double()
    lib().kmo_draw(C.c_uint64(seed), C.c_uint64(walker), C.c_uint64(it), C.c_uint32(batch),
                   C.c_uint64(nhalf), C.byref(pl), C.byref(uz), C.byref(ua))
    return pl.value, uz.value, ua.value


def g_pdf(z, a):
    return lib().kmo_g_pdf(z, a)


def cdf_g_inv(u, a):
    return lib().kmo_cdf_g_inv(u, a)


def emcee(dens: Density, theta0s, niter_walker, nburnin_walker, nthin=1, a_scale=2.0, seed=0,
          replay=None, trace=False, store=True, nthreads=1, native=False):
    """_emcee (src/samplers.jl:232-293) on per-walker counts.  theta0s: [nw, d] (or [nw]).

    replay = (partner[int64, global 0-based], z, u), each of length T*2*(nw/2).
    Returns dict(chain_x[nw,ns,d], chain_lp[nw,ns], accept_ratio[nw], naccept[nw], x, lp,
                 trace=(partner,z,u,accept) or None, min_margin).
    """
    x = np.array(np.asarray(theta0s, dtype=np.float64).reshape(len(theta0s), -1), order="C")
    nw, d = x.shape
    assert d == dens.d
    lp = dens.eval(x, nthreads=nthreads, native=native)  # src/samplers.jl:209-210
    ns = (niter_walker - nburnin_walker) // nthin
    T = niter_walker
    nslots = T * nw
    chain_x = np.empty((nw, ns, d)) if store else None
    chain_lp = np.empty((nw, ns)) if store else None
    naccept = np.zeros(nw, dtype=np.int64)
    ratio = np.empty(nw)
    if replay is not None:
        rp = [np.ascontiguousarray(replay[0], dtype=np.int64),
              np.ascontiguousarray(replay[1], dtype=np.float64),
              np.ascontiguousarray(replay[2], dtype=np.float64)]
        assert all(a.size == nslots for a in rp)
        mode = MODE_REPLAY
    else:
        rp = [None, None, None]
        mode = MODE_PHILOX
    tr = None
    if trace:
        tr = (np.empty(nslots, dtype=np.int64), np.empty(nslots), np.empty(nslots),
              np.empty(nslots, dtype=np.uint8))
    margin = C.c_double()
    i64p = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64)) if a is not None else None
    rc = lib(native).kmo_emcee(
        C.byref(dens._s), _dp(x), _dp(lp), C.c_int64(nw), C.c_int64(niter_walker),
        C.c_int64(nburnin_walker), C.c_int64(nthin), C.c_double(a_scale), C.c_int32(mode),
        C.c_uint64(seed), i64p(rp[0]), _dp(rp[1]), _dp(rp[2]), _dp(chain_x), _dp(chain_lp),
        i64p(naccept), _dp(ratio), i64p(tr[0]) if tr else None, _dp(tr[1]) if tr else None,
        _dp(tr[2]) if tr else None,
        tr[3].ctypes.data_as(C.POINTER(C.c_uint8)) if tr else None, C.byref(margin),
        C.c_int32(nthreads))
    if rc != 0:
        raise ValueError(f"kmo_emcee rejected its arguments (rc={rc})")
    return dict(chain_x=chain_x, chain_lp=chain_lp, accept_ratio=ratio, naccept=naccept, x=x,
                lp=lp, trace=tr, min_margin=margin.value)


# ----------------------------------------------------------------------------------------
# Host-side reference functions, restated in numpy (pure-Python loops: small cases only).

def make_theta0s(theta0, ball_radius, logpdf, nwalkers, randn, ball_radius_halfing_steps=7,
                 ntries=100):
    """src/samplers.jl:311-349, line by line, including its quirks:
    the radius shrink `ball_radius *= 1/2^(k-1)` (:326) is cumulative and never reset between
    walkers, and a walker that exhausts every try is silently skipped (the error at :344-345
    cannot fire because the inner loop variable shadows `j`).
    randn(i, k, j) -> d standard normals for walker i (0-based), halving step k, try j
    (1-based like the reference loops); the reference uses Julia's global RNG here (:329-331).
    """
    scalar = np.ndim(theta0) == 0
    th0 = np.atleast_1d(np.asarray(theta0, dtype=np.float64))
    npara = th0.size
    br = np.asarray(ball_radius, dtype=np.float64)
    br = np.ones(npara) * br if br.ndim == 0 else br.copy()      # :316-318
    assert br.size == npara                                        # :319
    out = []
    for i in range(nwalkers):                                      # :323
        for k in range(1, ball_radius_halfing_steps + 1):          # :324
            br = br * (1.0 / 2.0 ** (k - 1))                       # :326
            for j in range(1, ntries + 1):                         # :327
                tmp = th0 + randn(i, k, j) * br                    # :328-332
                if logpdf(tmp) > -np.inf:                          # :338
                    out.append(tmp)
                    break
            if len(out) == i + 1:                                  # :343
                break
    arr = np.array(out).reshape(len(out), npara)
    return arr[:, 0] if scalar else arr


def squash_walkers(thetas, accept_ratio, logdensities=None, drop_low_accept_ratio=False,
                   drop_fact=2, order=False):
    """src/samplers.jl:372-428 for blobs=nothing.  thetas: [nw][ns](,d) per-walker chains."""
    accept_ratio = np.asarray(accept_ratio, dtype=np.float64)
    nwalkers = len(accept_ratio)
    if drop_low_accept_ratio:                                      # :379-393
        ma, sa = np.median(accept_ratio), np.std(accept_ratio, ddof=1)
        keep = [nc for nc in range(nwalkers) if not accept_ratio[nc] <= ma - drop_fact * sa]
    else:
        keep = list(range(nwalkers))                               # :395
    t = np.concatenate([np.asarray(thetas[w]) for w in keep], axis=0)      # :398-399
    l = None if logdensities is None else np.concatenate([np.asarray(logdensities[w]) for w in keep])
    if order:                                                      # :415-426
        ns = len(thetas[0])
        perm = np.argsort(np.concatenate([np.arange(ns)] * len(keep)), kind="stable")
        t = t[perm]
        l = None if l is None else l[perm]
    return t, float(np.mean(accept_ratio[keep])), l, None          # :427
