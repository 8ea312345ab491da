"""GPU tests (`-m gpu`) of the accept decision of every filtered stretch-move kernel (kmc_kernels.cuh: filter_q,
accept_decide) at its margin: decisions placed just inside and just outside the FP32 filter's margin, at log-densities
from ~1 to ~1e15, compared bit for bit with the FP64 oracle or with a bit-identical twin.
tests/test_accept_filter_model.py derives the margin and the |p0| < 2^36 bound on the CPU.

Every case prints how many decisions have the exact t (tests/test_accept_filter_model.t_exact) in [margin, 4 margin]
(the filter decides them alone) and how many have |t| < margin (the exact path), and at |logp| >= 2^41 how many the
FP64 expression's own rounding decides against the sign of t; it asserts each is non-zero."""
import math
from fractions import Fraction

import numpy as np
import pytest

from tests import cases
from tests.test_accept_filter_model import margin, t_exact
from tests.test_oracle import edge_case_draws

pytestmark = pytest.mark.gpu
KS = np.array([0.5, 0.99, 1.01, 1.5, 3.0, 10.0])
SCALES = [1.0, 1e6, 2.5e12, 1e13, 1e15]   # 2.5e12: just above 2^41, where the FP64 rounding starts to flip decisions


def _density(km, orc, plugin, d):
    if plugin == "exponential":
        params = []
    elif plugin == "gaussian":
        params = cases.gaussian_params(np.linspace(-1, 1, d), cases.spd_cov(d, d))
    else:
        params = [1.0, 100.0, 20.0]
    return km.LogDensity(plugin, d, params), orc.Density(plugin, d, params), params


def _cloud(plugin, d, params, scale, nw, rng):
    """nw walkers whose log-densities are all ~ -scale and differ by O(1): every proposal's p1 - p0 is O(1), so u can
    put lhs - log u anywhere near the margin."""
    if plugin == "exponential":
        c = np.full(d, scale / d)
        eps = 1.0 / math.sqrt(d)
    elif plugin == "gaussian":
        mu = np.asarray(params[:d])
        Lt = np.asarray(params[d:d + d * d]).reshape(d, d)
        e = rng.standard_normal(d)
        e /= np.linalg.norm(e)
        c = mu + math.sqrt(2 * scale) / np.linalg.norm(Lt @ e) * e
        eps = 1.0 / max(1.0, np.linalg.norm(Lt.T @ (Lt @ (c - mu))))
    else:  # rosenbrock, x1 ~ (20 scale / 100)^(1/4): scale 5e12 at x1 ~ 1e3
        c = np.array([(0.2 * scale) ** 0.25 + 1.0, 0.0])
        eps = 1.0 / (20 * c[0] ** 3 + 1)
    x = c + eps * rng.standard_normal((nw, d))
    return np.abs(x) if plugin == "exponential" else x


def _design(od, x0, nm1, partner, z, rng):
    """u of one iteration's draws so that the FP64 lhs - log u of each step lands at +-KS * margin (batch by batch,
    the reference's decisions applied in between).  Returns u and the (z, p1, p0, u) of every designed step."""
    x, lp = x0.copy(), od.eval(x0)
    nw = len(x)
    nh = nw // 2
    m = margin(nm1)
    u = np.empty(nw)
    steps = []
    for b in (0, 1):
        act = np.arange(nh) + b * nh
        sl = slice(b * nh, (b + 1) * nh)
        j = partner[sl]
        zz = z[sl][:, None]
        y = x[j] + zz * (x[act] - x[j])
        p1 = od.eval(y)
        k = rng.choice(np.concatenate([KS, -KS]), nh)
        for i in range(nh):
            lhs = (nm1 * math.log(z[sl][i]) + p1[i]) - lp[act[i]]
            ui = math.exp(lhs - k[i] * m) if math.isfinite(lhs) else 0.5
            u[b * nh + i] = ui
            if i < 4000:
                steps.append((z[sl][i], p1[i], lp[act[i]], ui))
            if ui == 0.0 or lhs >= math.log(ui):
                x[act[i]], lp[act[i]] = y[i], p1[i]
    return u, steps


def _window_counts(nm1, steps):
    m = Fraction(margin(nm1))
    near = inside = flipped = 0
    for z, p1, p0, u in steps:
        if not (math.isfinite(p1) and math.isfinite(p0) and u > 0):
            continue
        t = t_exact(nm1, z, u, p1, p0)
        near += m <= abs(t) <= 4 * m
        inside += abs(t) < m
        ref = ((nm1 * math.log(z) + p1) - p0) >= math.log(u)
        flipped += t != 0 and ref != (t > 0)
    return near, inside, flipped


def _run(km, ld, x0, a=2.0, seed=0, replay=None, launch_mode=0, niter=1):
    s = km.Sampler(ld, x0, niter, 0, 1, a, seed, km.MODE_REPLAY if replay is not None else km.MODE_PHILOX,
                   launch_mode=launch_mode)
    if replay is not None:
        s.set_replay(*replay)
    lp0 = s.state()[1]
    s.run(-1)
    th, lp, ar = s.results()
    x, l, na = s.state()
    s.close()
    return dict(chain_x=th, chain_lp=lp, accept_ratio=ar, x=x, lp=l, naccept=na, lp0=lp0)


def _assert_same(got, want, what):
    for k in ("chain_x", "chain_lp", "accept_ratio", "x", "lp", "naccept"):
        assert np.array_equal(got[k], want[k], equal_nan=True), f"{what}: {k}"


def _check_counts(nm1, scale, steps, what):
    near, inside, flipped = _window_counts(nm1, steps)
    print(f"{what}: |t| in [m, 4m]: {near}, |t| < m: {inside}, FP64 rounding against sign(t): {flipped}")
    assert near > 0 and inside > 0
    if scale >= 2.0 ** 41 and nm1 >= 1:
        assert flipped > 0


REPLAY_CASES = [("exponential", d) for d in (1, 2, 3, 6, 10, 16)] + [("gaussian", 2), ("gaussian", 8), ("rosenbrock", 2)]


@pytest.mark.parametrize("scale", SCALES)
@pytest.mark.parametrize("plugin,d", REPLAY_CASES)
def test_replay_decisions_at_the_margin(km, orc, plugin, d, scale):
    """Shared-memory kernel K1 (small ensemble, launch_mode 0) and the general kernel (launch_mode 1) with designed u."""
    ld, od, params = _density(km, orc, plugin, d)
    rng = np.random.default_rng(d * 7 + int(math.log10(scale)))
    nw = 8192
    x0 = _cloud(plugin, d, params, scale, nw, rng)
    nh = nw // 2
    partner = np.concatenate([nh + rng.integers(0, nh, nh), rng.integers(0, nh, nh)]).astype(np.int64)
    z = rng.uniform(0.5, 2.0, nw)
    u, steps = _design(od, x0, d - 1, partner, z, rng)
    want = orc.emcee(od, x0, 1, 0, 1, 2.0, replay=(partner, z, u))
    _check_counts(d - 1, scale, steps, f"{plugin} d={d} |logp|~{scale:g}")
    bad = []
    for lm in (0, 1):
        try:
            _assert_same(_run(km, ld, x0, replay=(partner, z, u), launch_mode=lm), want, f"launch_mode {lm}")
        except AssertionError as e:
            bad.append(str(e).splitlines()[0])
    assert not bad, bad


@pytest.mark.parametrize("d,nw", [(2, 1 << 21), (16, 1 << 19)])
@pytest.mark.parametrize("scale", [1.0, 1e13])
def test_replay_general_kernel_large_ensemble(km, orc, d, nw, scale):
    """An ensemble too large for the shared-memory kernel: replay takes the general kernel in launch_mode 0."""
    ld, od, params = _density(km, orc, "exponential", d)
    rng = np.random.default_rng(d + 100)
    x0 = _cloud("exponential", d, params, scale, nw, rng)
    nh = nw // 2
    partner = np.concatenate([nh + rng.integers(0, nh, nh), rng.integers(0, nh, nh)]).astype(np.int64)
    z = rng.uniform(0.5, 2.0, nw)
    u, steps = _design(od, x0, d - 1, partner, z, rng)
    want = orc.emcee(od, x0, 1, 0, 1, 2.0, replay=(partner, z, u), nthreads=8)
    _check_counts(d - 1, scale, steps, f"general kernel d={d} nw={nw} |logp|~{scale:g}")
    _assert_same(_run(km, ld, x0, replay=(partner, z, u)), want, "general kernel")


@pytest.mark.parametrize("scale", [1.0, 1e13])
def test_replay_edges_at_scale(km, orc, scale):
    """Exact ties (z = 1 and a partner at the walker's own position: y == x_k, lhs = 0 >= log 1 accepts), u = 0, -Inf
    proposals, NaN u, and a_scale = 20, where ~12 % of the z fall outside the filter's range (1/16, 16), on top of a
    cloud at |logp| ~ scale."""
    ld, od, params = _density(km, orc, "exponential", 2)
    rng = np.random.default_rng(5)
    x0 = _cloud("exponential", 2, params, scale, 512, rng)
    nh = 256
    partner = np.concatenate([nh + rng.integers(0, nh, nh), rng.integers(0, nh, nh)]).astype(np.int64)
    z = np.sqrt(1 / 20) + rng.random(512) * (math.sqrt(20) - math.sqrt(1 / 20))
    z = z * z
    assert 0.05 < np.mean((z <= 1 / 16) | (z >= 16)) < 0.25
    u, _ = _design(od, x0, 1, partner, z, rng)
    partner[:8] = nh + np.arange(8)
    x0[nh:nh + 8] = x0[:8]                       # ties: y = x_j + 1 (x_k - x_j) = x_k exactly
    z[:8], u[:8] = 1.0, 1.0
    u[8:16] = 0.0
    u[16:20] = np.nan
    partner[20:24] = nh + 20 + np.arange(4)
    x0[nh + 20:nh + 24] = -2.0 * x0[20:24]       # partners outside the support and z = 1/2: y = (x_j + x_k) / 2 < 0,
    z[20:24] = 0.5                               # the proposals are -Inf
    want = orc.emcee(od, x0, 1, 0, 1, 20.0, replay=(partner, z, u))
    assert np.all(want["naccept"][:16] == 1)     # ties accept on >=; u = 0 accepts (log 0 = -Inf)
    assert np.all(want["naccept"][16:24] == 0)   # NaN u and -Inf proposals reject
    for lm in (0, 1):
        _assert_same(_run(km, ld, x0, a=20.0, replay=(partner, z, u), launch_mode=lm), want, f"launch_mode {lm}")
    ex = edge_case_draws()
    x1 = np.array([[1.0], [6.0], [3.0], [4.0]]) + (scale if scale > 1 else 0.0)
    want = orc.emcee(orc.Density("exponential", 1, []), x1, 1, 0, 1, 2.0, replay=ex)
    _assert_same(_run(km, km.exponential(), x1, replay=ex), want, "edge_case_draws")


def _philox_positions(orc, d, nw, seed, scale, a=2.0):
    """Exponential walkers for one Philox iteration: the passive half at one base point B, each active walker k of
    batch 0 placed so that lhs - log u = (N-1) log z + (1 - z)(S_k - B) - log u lands at +-KS * margin."""
    rng = np.random.default_rng(seed)
    nh = nw // 2
    nm1 = d - 1
    m = margin(nm1)
    sia = math.sqrt(1 / a)
    span = math.sqrt(a) - sia
    base = scale / d
    x = np.full((nw, d), base)
    B = float(np.sum(x[0]))
    steps = []
    k = rng.choice(np.concatenate([KS, -KS]), nh)
    for i in range(nh):
        _, uz, ua = orc.draw(seed, i, 0, 0, nh)
        s = uz * span + sia
        z = s * s
        if abs(1 - z) < 0.05:
            continue
        sk = B + (k[i] * m + math.log(ua) - nm1 * math.log(z)) / (1 - z)
        x[i] = base + (sk - B) / d
        if len(steps) < 4000:
            steps.append(i)
    return x, steps


def _philox_counts(orc, od, x, nm1, seed, steps, a=2.0):
    nh = len(x) // 2
    sia = math.sqrt(1 / a)
    span = math.sqrt(a) - sia
    lp = od.eval(x)
    out = []
    for i in steps:
        pl, uz, ua = orc.draw(seed, i, 0, 0, nh)
        s = uz * span + sia
        z = s * s
        j = nh + pl
        y = x[j] + z * (x[i] - x[j])
        out.append((z, float(od.eval(y[None])[0]), lp[i], ua))
    return out


@pytest.mark.parametrize("scale", [1.0, 1e13])
def test_philox_bulk_kernel_at_the_margin(km, orc, scale):
    """The bulk (TMA) kernel: even d >= 6, Philox draws, an ensemble too large for the shared-memory kernel."""
    d, nw, seed = 10, (1 << 18) + 154, 17
    ld, od, _ = _density(km, orc, "exponential", d)
    x0, steps = _philox_positions(orc, d, nw, seed, scale)
    _check_counts(d - 1, scale, _philox_counts(orc, od, x0, d - 1, seed, steps), f"bulk |logp|~{scale:g}")
    want = orc.emcee(od, x0, 1, 0, 1, 2.0, seed=seed, nthreads=8)
    _assert_same(_run(km, ld, x0, seed=seed), want, "bulk kernel")


@pytest.mark.parametrize("scale", [1.0, 1e13])
def test_philox_push_kernel_at_the_margin(km, orc, scale):
    """The push kernel: one ensemble sharded over two sub-samplers on one GPU."""
    d, nw, seed = 10, 8192, 23
    ld, od, _ = _density(km, orc, "exponential", d)
    x0, steps = _philox_positions(orc, d, nw, seed, scale)
    _check_counts(d - 1, scale, _philox_counts(orc, od, x0, d - 1, seed, steps), f"push |logp|~{scale:g}")
    want = orc.emcee(od, x0, 1, 0, 1, 2.0, seed=seed, nthreads=8)
    m = km.MultiSampler(ld, x0, 1, 0, 1, 2.0, seed, devices=[0, 0], sharded=True)
    m.run(-1)
    th, lp, ar = m.results()
    m.close()
    assert np.array_equal(th, want["chain_x"]) and np.array_equal(lp, want["chain_lp"])
    assert np.array_equal(ar, want["accept_ratio"])


def _tc_gaussian(km, d, variant):
    prm = cases.gaussian_params(np.linspace(-1, 1, d), cases.spd_cov(d, 3))
    ld = km.LogDensity("gaussian", d, prm)
    ld.set_option("tensor_cores", 1)
    ld.set_option("fused_variant", variant)
    return ld, prm


def _tc_cloud(d, prm, scale, nw, rng):
    """Walkers at |logp| ~ scale whose every proposal y has the same FP32 (y - mu) as its walker: the tensor path
    rounds y - mu to FP32 before it splits it into bf16 pieces, so K(y) == K(x_k) bit for bit and p1 == p0 on the
    kernel's own bits.  Each coordinate is an FP32 value v_i (not a power of two) plus at most ulp(v_i) / 64: one
    stretch, y = x_j + z (x_k - x_j) with z <= 2, moves at most 5x as far from v_i, so after the two half-steps of
    iteration 0 the walkers are within 5/64 ulp and iteration 1's proposals within 25/64 ulp of v_i."""
    mu = np.asarray(prm[:d])
    Lt = np.asarray(prm[d:d + d * d]).reshape(d, d)
    e = rng.standard_normal(d)
    e /= np.linalg.norm(e)
    v = (math.sqrt(2 * scale) / np.linalg.norm(Lt @ e) * e).astype(np.float32)
    mant = np.frexp(v)[0]
    v = np.where(np.abs(mant) == 0.5, np.nextafter(v, np.float32(0)), v)
    ulp = np.spacing(np.abs(v)).astype(np.float64)
    x = (mu + v.astype(np.float64)) + ulp * rng.uniform(-1 / 64, 1 / 64, (nw, d))
    assert np.all(((x - mu).astype(np.float32)) == v)
    return x


@pytest.mark.parametrize("d", [33, 100])
@pytest.mark.parametrize("scale", [1.0, 1e5, 1e13])
def test_fused_tensor_kernels_at_the_margin(km, d, scale):
    """K2F and K2G in two replay passes of two iterations.  Pass 1 accepts everything (u = 0), so in iteration 1 each
    batch-0 walker's p0 is the kernel's own p1 of iteration 0, and the chain holds iteration 1's p1.  Pass 2 repeats
    iteration 0 and places iteration 1's batch-0 u around the FP64 expression on those bits.  K2F == the launch_mode 1
    pipeline (exact FP64 decisions on the same p1) bit for bit; for both kernels, the batch-0 accept counts of pass 2
    are those of the FP64 expression on the kernel's own p1 and p0.  The walkers share their FP32 coordinates
    (_tc_cloud), so p1 - p0 is exactly 0 at any scale and lhs - log u can be placed even at |logp| ~ 1e13."""
    nw, nm1 = 2 * 1000, d - 1
    nh = nw // 2
    rng = np.random.default_rng(d)
    bad = []
    for variant in (1, 2):
        ld, prm = _tc_gaussian(km, d, variant)
        x0 = _tc_cloud(d, prm, scale, nw, rng)
        partner = np.tile(np.concatenate([nh + rng.integers(0, nh, nh), rng.integers(0, nh, nh)]), 2).astype(np.int64)
        z = rng.uniform(0.5, 2.0, 2 * nw)
        first = _run(km, ld, x0, replay=(partner, z, np.zeros(2 * nw)), niter=2)
        p0, p1 = first["chain_lp"][:nh, 0], first["chain_lp"][:nh, 1]
        k = rng.choice(np.concatenate([KS, -KS]), nh)
        u = np.zeros(2 * nw)
        steps = []
        for i in range(nh):
            zi = z[nw + i]
            lhs = (nm1 * math.log(zi) + p1[i]) - p0[i]
            u[nw + i] = math.exp(lhs - k[i] * margin(nm1))
            steps.append((zi, p1[i], p0[i], u[nw + i]))
        name = f"K2{'FG'[variant - 1]}"
        _check_counts(nm1, scale, steps, f"{name} d={d} |logp|~{scale:g}")
        got = _run(km, ld, x0, replay=(partner, z, u), niter=2)
        acc = np.array([((nm1 * math.log(zi) + b) - a) >= math.log(ui) for zi, b, a, ui in steps])
        lost = first["naccept"][:nh] - got["naccept"][:nh]     # pass 1 accepted every one of these steps
        if not np.array_equal(lost, (~acc).astype(lost.dtype)):
            bad.append(f"{name}: {int(np.sum(lost != ~acc))} decisions differ from the FP64 expression")
        if variant == 1:
            try:
                _assert_same(got, _run(km, ld, x0, replay=(partner, z, u), launch_mode=1, niter=2), "K2F vs launch_mode 1")
            except AssertionError as e:
                bad.append(str(e))
    assert not bad, bad
