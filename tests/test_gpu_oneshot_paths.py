"""GPU tests (`-m gpu`) of the one-shot entry points' staging and compaction at sizes the other tests do not reach:

  - squash over several 1024-walker keep blocks, with a walker-major output larger than one 64 MiB staging chunk;
  - squash and copy_results of a shard sampler, whose accept counters sit in two non-adjacent segments;
  - an allocation the device refuses, which is an ordinary error return.
"""
import ctypes as C

import numpy as np
import pytest

from tests import cases

pytestmark = pytest.mark.gpu

KEEP_BLOCK = 1024              # walkers per block of the device keep list (kmc_aux.cu)
STAGE_BYTES = 64 << 20         # the device squash and copy_results stage through at most this much


def _mvn10_run(km, nw, nitw, nbw, spread, seed=3, **kw):
    name, d, params, th0, rad = cases.plugin_specs()["mvn10"]
    x0 = cases.ball(th0, rad, nw, seed)
    x0[::17] += spread             # a few walkers start far out: they accept rarely and fall under the drop threshold
    s = km.Sampler(km.LogDensity(name, d, params), x0, nitw, nbw, 1, 2.0, seed, **kw)
    s.run(-1)
    return s


def _check_squash(km, s, th, lp, ar, drop, order):
    got_t, got_a, got_l, _ = s.squash(drop_low_accept_ratio=drop, drop_fact=1.0, order=order)
    nk, med, sd = s.squash_stats
    want_t, want_a, want_l, _ = km.squash_walkers(th, ar, lp, drop_low_accept_ratio=drop, drop_fact=1.0, order=order,
                                                  verbose=False)
    assert got_t.shape == want_t.shape and np.array_equal(got_t, want_t)
    assert np.array_equal(got_l, want_l)
    np.testing.assert_allclose(got_a, want_a, rtol=1e-13)
    assert med == np.median(ar)
    np.testing.assert_allclose(sd, np.std(ar, ddof=1), rtol=1e-12)
    assert (nk < len(ar)) if drop else (nk == len(ar))
    return nk


@pytest.mark.parametrize("drop", [False, True])
@pytest.mark.parametrize("order", [False, True])
def test_squash_over_keep_blocks_and_staging_chunks(km, drop, order):
    nw, ns, d = 20000, 100, 10
    s = _mvn10_run(km, nw, ns + 20, 20, spread=40.0)
    th, lp, ar = s.results()
    assert th.shape == (nw, ns, d) and nw > 3 * KEEP_BLOCK
    nk = _check_squash(km, s, th, lp, ar, drop, order)
    s.close()
    assert nk * ns * d * 8 > STAGE_BYTES            # the kept chains took more than one staging chunk


@pytest.mark.parametrize("drop", [False, True])
def test_shard_squash_and_results_read_both_counter_segments(km, drop):
    nw, nitw, nbw = 8192, 60, 20
    b, c = 1024, 1536                                 # positions [b, b + c) of each half: rows b.. and nw/2 + b..
    s = _mvn10_run(km, nw, nitw, nbw, spread=40.0, shard=(b, c), launch_mode=1)
    th, lp, ar = s.results()
    x, lp_now, nacc = s.state()
    rows = np.r_[b:b + c, nw // 2 + b:nw // 2 + b + c]
    assert th.shape[0] == 2 * c > KEEP_BLOCK
    assert np.array_equal(ar, nacc[rows] / (nitw - nbw))          # the counters of both segments, in chain order
    assert np.array_equal(th[:, -1], x[rows]) and np.array_equal(lp[:, -1], lp_now[rows])  # nthin = 1: last = now
    _check_squash(km, s, th, lp, ar, drop, order=False)
    _check_squash(km, s, th, lp, ar, drop, order=True)
    s.close()


def test_ball_randn_refused_allocation_is_an_error_return(km):
    """2^40 walkers of one double ask for an 8 TiB block, which cudaMalloc refuses at once: KMC_ERR_CUDA, nothing
    written, and the library keeps working."""
    want = km.ball_randn_device(5, 0, 1000, 1, 1, 3)
    out = np.full(1, 7.0)
    rc = km.lib.kmc_ball_randn(5, 0, 2 ** 40, 1, 1, 1, 0, out.ctypes.data_as(C.POINTER(C.c_double)))
    assert rc == 2                                                # KMC_ERR_CUDA
    assert "out of memory" in km.lib.kmc_last_error().decode()
    assert out[0] == 7.0
    assert np.array_equal(km.ball_randn_device(5, 0, 1000, 1, 1, 3), want)
