"""CPU checks of the arithmetic and index maps that the tcgen05 kernels hard-code, read from the CUDA sources so that an
edit of a constant or a layout formula shows up here (the GPU parity tests then say whether the kernel still agrees
with the FP64 path).  float32 emulation with numpy; no GPU, no oracle."""
import re
from pathlib import Path

import numpy as np

CSRC = Path(__file__).resolve().parent.parent / "kissmcmc.jl_b200" / "csrc"
TC = (CSRC / "kmc_tc.cuh").read_text()
FUSED = (CSRC / "kmc_fused_gauss.cuh").read_text()
f32 = np.float32


def _fma32(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def _poly_coeffs():
    body = TC[TC.index("float ex2_neg_abs_poly(float s)"):]
    body = body[:body.index("return __int_as_float")]
    lead = float(re.search(r"float q = ([-0-9.e]+)f;", body).group(1))
    rest = [float(v) for v in re.findall(r"q = fmaf\(q, x, ([-0-9.e]+)f\);", body)]
    assert len(rest) == 5
    return [lead] + rest


def _ex2_neg_abs_poly(s):
    """ex2_neg_abs_poly of kmc_tc.cuh, operation by operation, in float32."""
    a = np.minimum(np.abs(s).astype(f32), f32(126.0))
    magic = f32(12582912.0)
    r = (a + magic).astype(f32)
    x = ((r - magic).astype(f32) - a).astype(f32)
    c = _poly_coeffs()
    q = np.full_like(a, f32(c[0]))
    for ck in c[1:]:
        q = _fma32(q, x, np.full_like(a, f32(ck)))
    bits = q.view(np.int32) - (r.view(np.int32) << 23)
    return bits.view(np.float32)


def test_k3_polynomial_exp2_matches_its_stated_error():
    """2^-|s| on the FMA pipe: relative error <= 2.5e-7 (the MUFU.EX2 it replaces has 2^-22 = 2.4e-7) over the whole
    range of logits, exact at integers, harmless (tiny, finite, >= 0) beyond the clamp."""
    s = np.concatenate([np.linspace(-60, 60, 400001), np.arange(-40, 41, dtype=np.float64)]).astype(f32)
    got = _ex2_neg_abs_poly(s).astype(np.float64)
    want = np.exp2(-np.abs(s.astype(np.float64)))
    assert np.max(np.abs(got / want - 1.0)) < 2.5e-7
    ints = np.arange(0, 41, dtype=np.float64).astype(f32)
    assert np.max(np.abs(_ex2_neg_abs_poly(ints).astype(np.float64) / np.exp2(-ints.astype(np.float64)) - 1)) < 1.3e-7
    far = _ex2_neg_abs_poly(np.array([126.0, 127.5, 1e4, 3e38, np.inf], dtype=f32))
    assert np.all(np.isfinite(far)) and np.all(far >= 0) and np.all(far < 1e-37)


def test_k3_product_form_equals_softplus_sum():
    """sum_n softplus(s_n) = sum_n s_n/2 + ln2 * sum over 32-logit chunks of (0.5 * sum|s'| + lg2 prod(1 + 2^-|s'|)),
    s' = s * log2(e): the identity behind the epilogue, and its float32 error per chunk (two chains of 16, one lg2)."""
    rng = np.random.default_rng(0)
    s = (rng.standard_normal((4000, 32)) * 6.0)
    s[0] = 0.0                                        # all terms 2: the largest product, 2^16 per chain
    s[1] = 40.0 * np.sign(rng.standard_normal(32))    # saturated logits
    sp = (s * 1.4426950408889634).astype(f32)
    t = np.exp2(-np.abs(sp.astype(np.float64))).astype(f32)
    pa, pb = np.ones(len(s), f32), np.ones(len(s), f32)
    sa, sb = np.zeros(len(s), f32), np.zeros(len(s), f32)
    for j in range(0, 32, 2):
        pa = _fma32(pa, t[:, j], pa)
        pb = _fma32(pb, t[:, j + 1], pb)
        sa = (sa + np.abs(sp[:, j])).astype(f32)
        sb = (sb + np.abs(sp[:, j + 1])).astype(f32)
    assert np.all(pa <= 65536.0) and np.all(pb <= 65536.0)
    lg = np.log2((pa * pb).astype(f32).astype(np.float64)).astype(f32)
    part = _fma32(np.full_like(lg, f32(0.5)), (sa + sb).astype(f32), lg).astype(np.float64) * 0.6931471805599453
    want = np.sum(np.logaddexp(0.0, s) - 0.5 * s, axis=1)
    assert np.all(np.abs(part - want) < 2e-5 + 3e-7 * np.abs(want))   # per 32 logits: a few float32 ulps of the sum
    assert abs(np.mean(part - want)) < 2e-6            # no systematic offset from the formulation itself


def test_sw128_chunk_offset_is_a_bijection_onto_the_piece():
    """The manual SWIZZLE_128B operand build of the fused Gaussian kernels: (row, 16-byte chunk) -> byte offset is a
    bijection onto the 32 KB piece, 16-byte aligned, and the eight chunks of a row half stay inside the row's 128 bytes
    of its k-half (what the UMMA descriptor with SBO = 1024 expects)."""
    m = re.search(r"return kh \* \(GPIECE_BYTES / 2\) \+ \(r >> 3\) \* 1024 \+ \(r & 7\) \* 128 \+ \(\(c8 \^ \(r & 7\)\) << 4\);", FUSED)
    assert m, "sw128_chunk_offset changed: update this test together with the kernels"
    piece = 2 * 128 * 128
    seen = set()
    for r in range(128):
        for ck in range(16):
            kh, c8 = ck >> 3, ck & 7
            off = kh * (piece // 2) + (r >> 3) * 1024 + (r & 7) * 128 + ((c8 ^ (r & 7)) << 4)
            assert off % 16 == 0 and 0 <= off < piece
            assert (off % (piece // 2)) // 128 == r          # stays in row r of its k-half
            seen.add(off)
    assert len(seen) == 128 * 16


def test_lane_butterfly_leaves_column_l_in_lane_l():
    """K2G's transpose-and-add (kmc_fused_gauss2.cuh): after the 5 shuffle stages lane l holds the sum over the 32
    lanes of column l.  Emulated with one array row per lane."""
    rng = np.random.default_rng(1)
    v = rng.integers(-50, 50, size=(32, 32)).astype(np.float64)     # v[lane][column]
    s = v.copy()
    lanes = np.arange(32)
    hh = 16
    while hh >= 1:
        new = s.copy()
        for e in range(hh):
            up = (lanes & hh) != 0
            send = np.where(up, s[:, e], s[:, e + hh])
            keep = np.where(up, s[:, e + hh], s[:, e])
            new[:, e] = keep + send[lanes ^ hh]                      # __shfl_xor_sync(send, hh)
        s = new
        hh >>= 1
    assert np.array_equal(s[:, 0], v.sum(axis=0))


def test_balanced_tiling_of_the_fused_gaussian_kernels_covers_every_walker_once():
    """K2F / K2G tile the active half as `waves` tiles per CTA of `tr <= 128` walkers (kmc_fused_gauss*.cuh); the host
    launches min(ceil(W / 128), SMs) CTAs (kmc_api.cu).  Emulated for many sizes: every walker position belongs to exactly
    one (CTA, tile), no CTA gets more than `waves` tiles, and the MMA's N (tr rounded up to 16) stays legal."""
    for src in (FUSED, (CSRC / "kmc_fused_gauss2.cuh").read_text()):
        assert "const unsigned waves = ((W + BM - 1) / BM + gridDim.x - 1) / gridDim.x;" in src
        assert "(W + waves * gridDim.x - 1) / (waves * gridDim.x)" in src
    BM, nsm = 128, 148
    sizes = list(range(1, 700)) + [1000, 2 ** 15, 148 * 128, 148 * 128 + 1, 148 * 128 * 2 + 777, 148 * 128 * 3 - 50, 10 ** 6 + 3]
    for W in sizes:
        grid = min((W + BM - 1) // BM, nsm)
        waves = ((W + BM - 1) // BM + grid - 1) // grid
        tr = min(BM, (W + waves * grid - 1) // (waves * grid))
        ntiles = (W + tr - 1) // tr
        assert 1 <= tr <= BM and 16 <= ((tr + 15) & ~15) <= 128
        covered = 0
        for cta in range(grid):
            T = (ntiles - cta + grid - 1) // grid if ntiles > cta else 0
            assert T <= waves
            for k in range(T):
                w0 = (cta + k * grid) * tr
                covered += max(0, min(tr, W - w0))
        assert covered == W, (W, grid, waves, tr, ntiles)
        assert (ntiles - 1) * tr < W <= ntiles * tr


def test_chain_gather_launch_geometry_covers_long_chains():
    """kmc_emcee_copy_results and the walker-major squash transpose the sample-major chain (chain_gather) in launches
    of at most kTransposeMaxSamples samples (gridDim.y <= 65535 blocks of 32 samples): every sample exactly once, for
    chains far beyond 2.09 M samples."""
    src = (CSRC / "kmc_kernels.cuh").read_text()
    m = re.search(r"kTransposeMaxSamples = (\d+)LL \* (\d+);", src)
    max_samples = int(m.group(1)) * int(m.group(2))
    assert max_samples == 65535 * 32
    api = (CSRC / "kmc_api.cu").read_text()
    gather = api[api.index("int32_t chain_gather("):]
    gather = gather[:gather.index("\n}\n")]
    assert api.count("s0 += kmc::kTransposeMaxSamples") == 1 and "s0 += kmc::kTransposeMaxSamples" in gather
    assert "what == 0 ? s->chain_x : s->chain_lp" in gather            # thetas and logp both loop over sample chunks
    assert "chain_gather(s, nullptr, nl, thetas, logp)" in api
    for ns in (1, 31, 32, max_samples - 1, max_samples, max_samples + 1, 5_000_000, 3 * max_samples + 7):
        covered = 0
        for s0 in range(0, ns, max_samples):
            sc = min(max_samples, ns - s0)
            grid_y = (sc + 31) // 32
            assert 1 <= grid_y <= 65535
            assert grid_y * 32 >= sc                                    # the launch reaches the chunk's last sample
            covered += sc
        assert covered == ns


def _smem_geometry(scnt, nsm=148):
    """Host mirror of the persistent-launch geometry of kmc_emcee_create (kmc_api.cu, `geometry` lambda) for the
    shared-memory kernel, with the constants read from kmc_kernels.cuh."""
    src = (CSRC / "kmc_kernels.cuh").read_text()
    threads = int(re.search(r"#define KMC_SMEM_THREADS (\d+)", src).group(1))
    rounds_max = int(re.search(r"#define KMC_SMEM_ROUNDS (\d+)", src).group(1))
    ctas = int(re.search(r"#define KMC_SMEM_CTAS (\d+)", src).group(1))
    split = int(re.search(r"#define KMC_SMEM_SPLIT (\d+)", src).group(1))
    ahead = int(re.search(r"#define KMC_SMEM_AHEAD (\d+)", src).group(1))
    grid = min(-(-scnt // threads), ctas * nsm)
    per_cta = -(-scnt // grid)
    grid = -(-scnt // per_cta)
    rounds = -(-per_cta // threads)
    block = min(threads, -(-(-(-per_cta // rounds)) // 32) * 32)
    return dict(threads=threads, rounds_max=rounds_max, split=split, ahead=ahead, grid=grid, per_cta=per_cta,
                rounds=rounds, block=block)


def test_shared_memory_kernel_geometry_of_the_bench_config():
    """BASELINE.json configs[1] (2^20 walkers, 2^19 per half-step) on 148 SMs: 296 CTAs x 256 threads, 7 rounds, and every
    round full -- the reason for 256 x 7 (the 384 x 5 of round 1 ran its fifth round 61 % full)."""
    g = _smem_geometry(1 << 19)
    assert (g["grid"], g["block"], g["rounds"], g["per_cta"]) == (296, 256, 7, 1772)
    assert g["rounds"] <= g["rounds_max"]
    assert g["per_cta"] / (g["rounds"] * g["block"]) > 0.98                 # rounds 98.9 % full
    assert 2 * g["per_cta"] * 28 <= 113 * 1024                              # x, logp, counter of both halves: 2 CTAs per SM
    assert g["ahead"] <= g["split"] <= g["rounds_max"]                      # the first gathers' draws are made in the shadow
    # every owned position is covered exactly once by (round, thread)
    owned = [q * g["block"] + t for q in range(g["rounds"]) for t in range(g["block"]) if q * g["block"] + t < g["per_cta"]]
    assert owned == list(range(g["per_cta"]))
    # the README example (100 walkers) and a ragged size: one CTA / a last warp that exists (it is the polling warp)
    assert _smem_geometry(50)["grid"] == 1 and _smem_geometry(50)["block"] == 64
    for scnt in (33, 257, 1000, 12345, 300000):
        gg = _smem_geometry(scnt)
        assert gg["block"] % 32 == 0 and gg["block"] >= 32 and gg["rounds"] * gg["block"] >= gg["per_cta"]
