"""CPU checks of bench.py's contract pieces that need no GPU: workloads = BASELINE.json's configs, the roofline arithmetic
(SURVEY.md section 8d), the kernel labels, the reference arm's JSON line, the order of operations in the rank barrier and
the files of --dump-outputs; and on a GPU, that those files hold what the last timed step computed."""
import inspect
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402


def test_workloads_are_the_baseline_configs():
    w = bench.WORKLOADS
    assert (w["exponential1d"]["nw"], w["exponential1d"]["d"]) == (100, 1)                  # configs[0]
    assert (w["rosenbrock2d"]["nw"], w["rosenbrock2d"]["d"], w["rosenbrock2d"]["niter_walker"]) == (1 << 20, 2, 10_000)
    assert (w["gaussian100d"]["nw"], w["gaussian100d"]["d"]) == (1 << 16, 100)              # configs[2]
    assert (w["logistic32d"]["nw"], w["logistic32d"]["d"], w["logistic32d"]["ndata"]) == (8192, 32, 10**6)
    assert (w["gaussian10d"]["nw"], w["gaussian10d"]["d"]) == (1 << 24, 10)                 # configs[4]
    cfgs = json.loads((ROOT / "BASELINE.json").read_text())["configs"]
    assert len(cfgs) == 5 and "2^20 walkers" in cfgs[1] and "2^24-walker 10-D" in cfgs[4]


def test_roofline_arithmetic():
    wl = bench.WORKLOADS["rosenbrock2d"]
    assert bench.b_step(2) == 72 and bench.b_step(10) == 264 and bench.b_step(100) == 2424   # 24 d + 24
    r = bench.roofline_of(wl, "rosenbrock2d", False, 0, 118.5, None)
    steps = (1 << 20) * 10_000
    alg = 72 * steps + (8 * 2 + 8) * (1 << 20) * 5                   # + 5 stored samples per walker
    assert r["algorithmic_bytes_per_launch"] == alg == 755100549120
    assert r["bound"] == "hbm" and r["unit"] == "GB/s"
    assert r["achieved"] == pytest.approx(alg / 0.1185 / 1e9) and r["frac"] == pytest.approx(r["achieved"] / r["peak"])
    rl = bench.roofline_of(bench.WORKLOADS["logistic32d"], "logistic32d", True, 0, 8.8, None)
    assert rl["bound"] == "tensor" and rl["algorithmic_flops_per_step"] == 2.0 * 32 * 10**6 * 8192 * 4


def test_dominant_kernel_labels_follow_the_library_rules():
    w = bench.WORKLOADS
    assert bench.dominant_kernel(w["rosenbrock2d"], False, 0) == "emcee_smem_kernel"
    assert bench.dominant_kernel(w["exponential1d"], False, 0) == "emcee_smem_kernel"
    assert bench.dominant_kernel(w["gaussian10d"], False, 0) == "emcee_bulk_kernel"
    assert bench.dominant_kernel(w["gaussian100d"], True, 0) == "tc::gaussian_fused2_kernel"
    big = dict(w["rosenbrock2d"], nw=1 << 22)                         # does not fit 7 rounds of 256 per CTA any more
    assert bench.dominant_kernel(big, False, 0) == "emcee_run_kernel"


def test_rank_barrier_synchronizes_before_the_collective():
    """dist.barrier() with this rank's cooperative launches still queued cost one random rank +12 ms per step
    (profiles/r2_call34.log): the device is drained first."""
    src = inspect.getsource(bench.Env.barrier)
    code = [ln.strip() for ln in src.splitlines() if ln.strip() and not ln.strip().startswith("#")]
    assert code.index("self.torch.cuda.synchronize()") < code.index("self.dist.barrier()")
    assert code.count("self.torch.cuda.synchronize()") == 2            # and again after it


def test_dump_outputs_writes_a_fixed_bounded_sample(tmp_path):
    """--dump-outputs: float64 .npy files, all walkers while they fit the budget, else the same seeded walker sample in
    every file and on every run."""
    rng = np.random.default_rng(1)
    chain, logp, ratio = rng.standard_normal((1000, 5, 2)), rng.standard_normal((1000, 5)), rng.random(1000)
    bench.dump_outputs(tmp_path / "all", chain, logp, ratio)
    got = {p.stem: np.load(p) for p in (tmp_path / "all").glob("*.npy")}
    assert np.array_equal(got["chain"], chain) and np.array_equal(got["log_density"], logp)
    assert np.array_equal(got["accept_ratio"], ratio) and np.array_equal(got["walker_index"], np.arange(1000))
    budget = 100 * 8 * (10 + 5 + 2)
    for run in ("a", "b"):
        bench.dump_outputs(tmp_path / run, chain, logp, ratio.astype(np.float32), budget=budget)
    a = {p.stem: np.load(p) for p in (tmp_path / "a").glob("*.npy")}
    b = {p.stem: np.load(p) for p in (tmp_path / "b").glob("*.npy")}
    assert sorted(a) == ["accept_ratio", "chain", "log_density", "walker_index"]
    assert all(a[k].dtype == np.float64 and np.array_equal(a[k], b[k]) for k in a)
    assert sum(v.nbytes for v in a.values()) <= budget
    keep = a["walker_index"].astype(np.int64)
    assert len(keep) == 100 and np.all(np.diff(keep) > 0)
    assert np.array_equal(a["chain"], chain[keep]) and np.array_equal(a["log_density"], logp[keep])
    assert np.array_equal(a["accept_ratio"], ratio.astype(np.float32)[keep])


@pytest.mark.gpu
def test_dumped_outputs_are_those_of_the_last_timed_step(km, tmp_path):
    """bench.py --dump-outputs on the default workload: the files hold, bit for bit, the sampled walkers of the job of
    the last timed step (seed (warmup + steps - 1) << 8 on rank 0), and the line reports the steps asked for."""
    steps, warmup = 2, 1
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                          "--no-others", "--no-sharded", "--no-traffic", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=600,
                         cwd=tmp_path)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warmup
    got = {p.stem: np.load(p) for p in (tmp_path / "out").glob("*.npy")}
    assert sum(v.nbytes for v in got.values()) <= 64 << 20
    wl = bench.WORKLOADS["rosenbrock2d"]
    params, x0 = bench.make_inputs(wl, 1000)
    nitw = wl["niter_walker"]
    s = km.Sampler(km.LogDensity("rosenbrock", 2, params), x0, nitw, nitw // 2, wl["nthin"], 2.0,
                   seed=(warmup + steps - 1) << 8)
    s.run(-1)
    th, lp, ar = s.results()
    s.close()
    keep = got["walker_index"].astype(np.int64)
    assert len(keep) > 0 and np.array_equal(got["walker_index"], keep)
    assert np.array_equal(got["chain"], th[keep]) and np.array_equal(got["log_density"], lp[keep])
    assert np.array_equal(got["accept_ratio"], ar[keep])


def test_reference_arm_line():
    """`bench.py --impl reference`: the oracle timed on the host cores, same metric / unit / config keys, no GPU touched."""
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == bench.UNIT
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 1e6
    assert d["config"]["workload"] == "rosenbrock2d"
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
