"""ctypes binding of libkissmcmc_cuda.so (include/kissmcmc_cuda.h).

There is no CPU fallback: if the shared library is missing this module raises on import, and
every compute call fails with KmcError when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["KMC_LIB"]) if os.environ.get("KMC_LIB") else PKG / "libkissmcmc_cuda.so"

MODE_PHILOX, MODE_REPLAY = 0, 1
EXCHANGE_REPLICA, EXCHANGE_PUSH = 0, 1
MULTI_SHARDED, MULTI_INDEPENDENT = 0, 1

# every symbol include/kissmcmc_cuda.h declares
SYMBOLS = [
    "kmc_version", "kmc_last_error", "kmc_device_count", "kmc_trim",
    "kmc_density_create", "kmc_density_destroy", "kmc_density_eval", "kmc_density_set_option",
    "kmc_density_get_info",
    "kmc_emcee_create", "kmc_emcee_destroy", "kmc_emcee_set_stream", "kmc_emcee_set_replay",
    "kmc_emcee_run", "kmc_emcee_run_half", "kmc_emcee_device_ptrs", "kmc_emcee_ipc_export", "kmc_emcee_set_peers", "kmc_emcee_nlocal", "kmc_emcee_sync", "kmc_emcee_last_run_ms", "kmc_emcee_progress",
    "kmc_emcee_nsamples", "kmc_emcee_copy_results", "kmc_emcee_copy_state", "kmc_emcee_chain_moments",
    "kmc_emcee_window_export", "kmc_emcee_window_attach",
    "kmc_emcee_create_multi", "kmc_multi_destroy", "kmc_multi_run", "kmc_multi_sync", "kmc_multi_last_run_ms",
    "kmc_multi_shape", "kmc_multi_copy_results",
    "kmc_g_pdf", "kmc_cdf_g_inv", "kmc_sample_g", "kmc_emcee_squash", "kmc_make_theta0s", "kmc_ball_randn",
    "kmc_metropolis_create", "kmc_metropolis_set_replay", "kmc_metropolis_draws", "kmc_metropolis_create_chol",
    "kmc_emcee_chain_covariance",
]


class KmcError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libkissmcmc_cuda error {code}: {msg}")
        self.code = code


class EmceeOpts(C.Structure):
    _fields_ = [
        ("niter_walker", C.c_int64), ("nburnin_walker", C.c_int64), ("nthin", C.c_int64),
        ("a_scale", C.c_double), ("seed", C.c_uint64), ("mode", C.c_int32), ("device", C.c_int32),
        ("walker_id_base", C.c_int64), ("launch_mode", C.c_int32), ("exchange", C.c_int32),
        ("shard_begin", C.c_int64), ("shard_count", C.c_int64),
        ("push_chunk", C.c_int32), ("push_cap", C.c_int32), ("push_lag", C.c_int32), ("reserved", C.c_int32),
    ]


if not LIB_PATH.exists():
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(nvcc, sm_100a).  There is no CPU fallback.")

lib = C.CDLL(str(LIB_PATH))
_dp = C.POINTER(C.c_double)
_i64p = C.POINTER(C.c_int64)

lib.kmc_version.restype = C.c_int32
lib.kmc_last_error.restype = C.c_char_p
lib.kmc_device_count.argtypes = [C.POINTER(C.c_int32)]
lib.kmc_density_create.argtypes = [C.c_char_p, C.c_int32, _dp, C.c_int64, C.c_void_p, C.c_int64,
                                   C.c_int32, C.POINTER(C.c_void_p)]
lib.kmc_density_destroy.argtypes = [C.c_void_p]
lib.kmc_density_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_double]
lib.kmc_density_get_info.argtypes = [C.c_void_p, C.c_char_p, _dp]
lib.kmc_density_eval.argtypes = [C.c_void_p, _dp, C.c_int64, _dp]
lib.kmc_emcee_create.argtypes = [C.c_void_p, _dp, C.c_int64, C.c_int32, C.POINTER(EmceeOpts),
                                 C.POINTER(C.c_void_p)]
lib.kmc_emcee_destroy.argtypes = [C.c_void_p]
lib.kmc_emcee_set_stream.argtypes = [C.c_void_p, C.c_void_p]
lib.kmc_emcee_set_replay.argtypes = [C.c_void_p, _i64p, _dp, _dp, C.c_int64]
lib.kmc_emcee_run.argtypes = [C.c_void_p, C.c_int64]
lib.kmc_emcee_sync.argtypes = [C.c_void_p]
lib.kmc_emcee_run_half.argtypes = [C.c_void_p, C.c_int64]
lib.kmc_emcee_device_ptrs.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
lib.kmc_emcee_nlocal.argtypes = [C.c_void_p, _i64p]
lib.kmc_emcee_ipc_export.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
lib.kmc_emcee_set_peers.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
lib.kmc_emcee_last_run_ms.argtypes = [C.c_void_p, _dp, _i64p]
lib.kmc_emcee_progress.argtypes = [C.c_void_p, _i64p, _dp, _dp, _i64p]
lib.kmc_emcee_nsamples.argtypes = [C.c_void_p, _i64p]
lib.kmc_emcee_copy_results.argtypes = [C.c_void_p, _dp, _dp, _dp]
lib.kmc_emcee_copy_state.argtypes = [C.c_void_p, _dp, _dp, _i64p]
lib.kmc_emcee_chain_moments.argtypes = [C.c_void_p, _dp, _dp, _i64p]
lib.kmc_emcee_window_export.argtypes = [C.c_void_p, C.c_void_p]
lib.kmc_emcee_window_attach.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
lib.kmc_emcee_create_multi.argtypes = [C.POINTER(C.c_void_p), _dp, C.c_int64, C.c_int32, C.POINTER(EmceeOpts),
                                       C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]
lib.kmc_multi_destroy.argtypes = [C.c_void_p]
lib.kmc_multi_run.argtypes = [C.c_void_p, C.c_int64]
lib.kmc_multi_sync.argtypes = [C.c_void_p]
lib.kmc_multi_last_run_ms.argtypes = [C.c_void_p, _dp]
lib.kmc_multi_shape.argtypes = [C.c_void_p, _i64p, _i64p]
lib.kmc_multi_copy_results.argtypes = [C.c_void_p, _dp, _dp, _dp]
lib.kmc_g_pdf.argtypes = [_dp, C.c_int64, C.c_double, _dp]
lib.kmc_cdf_g_inv.argtypes = [_dp, C.c_int64, C.c_double, _dp]
lib.kmc_sample_g.argtypes = [C.c_double, C.c_uint64, C.c_int64, C.c_int32, _dp]
lib.kmc_emcee_squash.argtypes = [C.c_void_p, C.c_int32, C.c_double, C.c_int32, _dp, _dp, _i64p, _dp, _dp, _dp]
lib.kmc_make_theta0s.argtypes = [C.c_void_p, _dp, _dp, C.c_int64, C.c_int32, C.c_int32, C.c_uint64, _dp, _i64p]
lib.kmc_ball_randn.argtypes = [C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _dp]
lib.kmc_metropolis_create.argtypes = [C.c_void_p, _dp, C.c_int64, C.c_int32, _dp, C.c_int64, C.POINTER(EmceeOpts),
                                      C.POINTER(C.c_void_p)]
lib.kmc_metropolis_create_chol.argtypes = [C.c_void_p, _dp, C.c_int64, C.c_int32, _dp, C.POINTER(EmceeOpts),
                                           C.POINTER(C.c_void_p)]
lib.kmc_emcee_chain_covariance.argtypes = [C.c_void_p, _dp, _dp, _i64p]
lib.kmc_metropolis_set_replay.argtypes = [C.c_void_p, _dp, _dp, C.c_int64]
lib.kmc_metropolis_draws.argtypes = [C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, _dp,
                                     _dp]
for _name in SYMBOLS:
    if _name not in ("kmc_version", "kmc_last_error"):
        getattr(lib, _name).restype = C.c_int32


def check(rc: int) -> None:
    if rc != 0:
        raise KmcError(rc, (lib.kmc_last_error() or b"").decode())


def trim() -> None:
    """Release the library's cached device blocks (buffers of destroyed samplers) back to the driver."""
    check(lib.kmc_trim())


def device_count() -> int:
    n = C.c_int32(0)
    check(lib.kmc_device_count(C.byref(n)))
    return n.value
