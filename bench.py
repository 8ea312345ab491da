#!/usr/bin/env python
"""bench.py -- walker-steps/s of the emcee stretch-move hot path on N B200s.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload rosenbrock2d] [--dump-outputs DIR]

One "step" is one complete emcee job of the workload: BASELINE.json configs[1], the 2-D
Rosenbrock density with 2^20 walkers and 10^4 iterations per walker (API niter = 10^4 * 2^20,
default burn-in niter/2, nthin=1000 so that 5 samples per walker are stored -- the unthinned
chain would be 126 GB).  At N>1 every rank runs its own ensemble of that size with its own
Philox key and walker-id range (independent-ensembles mode: no data-path collective, weak
scaling); value = walker-steps of all ranks / max-over-ranks device time.

value     device-timed (CUDA events on the launch stream), inputs already resident in HBM.
e2e       the same metric through the public API with HOST buffers: pinned theta0s -> H2D ->
          initial log-densities -> run -> chain transpose -> D2H into pinned result buffers.
roofline  of the dominant kernel (named in roofline.kernel): algorithmic bytes per launch
          (24d+24 per walker-step + 8d+8 per stored sample, SURVEY.md section 8d) over the
          launch duration measured with the library's own CUDA events on the launch stream.
cpu_baseline / --impl reference: the Julia reference cannot run here (no Julia in the image);
          the C restatement of its loop (oracle/kmc_oracle.c, OpenMP over the active half like
          Threads.@threads at src/samplers.jl:248) is timed on the host cores on a bounded
          sample (same ensemble, fewer iterations).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "walker_steps_per_s"
UNIT = "walker-steps/s"

WORKLOADS = {
    # name: plugin, d, nwalkers, niter_walker, nthin
    "rosenbrock2d": dict(plugin="rosenbrock", d=2, nw=1 << 20, niter_walker=10_000, nthin=1000,
                         desc="BASELINE.json configs[1]: 2-D Rosenbrock/20, 2^20 walkers, 10^4 iterations per walker"),
    "gaussian10d": dict(plugin="gaussian", d=10, nw=1 << 24, niter_walker=200, nthin=100,
                        desc="BASELINE.json configs[4] ensemble: 10-D Gaussian, 2^24 walkers (per GPU), 200 iterations"),
    "gaussian100d": dict(plugin="gaussian", d=100, nw=1 << 16, niter_walker=400, nthin=100,
                         desc="BASELINE.json configs[2]: 100-D dense correlated Gaussian, 2^16 walkers, 400 iterations"),
    "logistic32d": dict(plugin="logistic", d=32, nw=8192, niter_walker=4, nthin=1, ndata=1_000_000,
                        desc="BASELINE.json configs[3]: Bayesian logistic regression d=32, N=10^6, 8192 walkers, 4 iterations"),
    "exponential1d": dict(plugin="exponential", d=1, nw=100, niter_walker=1000, nthin=1,
                          desc="BASELINE.json configs[0]: README exponential, 100 walkers, niter=10^5"),
}


def b_step(d: int) -> int:
    """Algorithmic bytes per walker-step (SURVEY.md section 8d)."""
    return 24 * d + 24


def dominant_kernel(wl, tensor, launch_mode):
    """Name of the kernel the roofline object describes (selection logic: csrc/kmc_api.cu, kmc_emcee_create/run)."""
    d = wl["d"]
    if d > 16:
        if tensor:
            return "tc::gaussian_fused2_kernel" if launch_mode == 0 else \
                "propose_split_kernel + tc::gaussian_tc_kernel + accept_kernel"
        return "propose_kernel + gaussian_wide_logp_kernel + accept_kernel"
    # shared-memory-resident state: 2 CTAs per SM, <= 7 rounds of 256 threads per half, 8d + 12 bytes per walker position
    per_cta = -(-(wl["nw"] // 2) // (2 * 148))
    if launch_mode == 0 and d <= 4 and per_cta <= 7 * 256 and 2 * per_cta * (8 * d + 12) <= 113 * 1024:
        return "emcee_smem_kernel"
    if launch_mode == 0 and d >= 6 and d % 2 == 0:
        return "emcee_bulk_kernel"
    return "emcee_run_kernel"


def gaussian_params(mean, cov):
    """[mu, A row-major, lognorm], A = chol(cov^-1)^T: logp = lognorm - |A (x - mu)|^2 / 2 (include/kissmcmc_cuda.h)."""
    mu = np.atleast_1d(np.asarray(mean, dtype=np.float64))
    prec = np.linalg.inv(np.atleast_2d(np.asarray(cov, dtype=np.float64)))
    L = np.linalg.cholesky((prec + prec.T) / 2)
    lognorm = float(np.sum(np.log(np.diag(L))) - 0.5 * mu.size * np.log(2 * np.pi))
    return np.concatenate([mu, L.T.ravel(), [lognorm]])


def spd_cov(d, seed=0):
    """Sigma = A A^T / d + I (SURVEY.md section 8d, config C3), stated seed."""
    a = np.random.default_rng(seed).standard_normal((d, d))
    return a @ a.T / d + np.eye(d)


def logistic_problem(N, d, seed=0):
    """Synthetic Bayesian logistic regression (SURVEY.md section 8d, config C4): X ~ N(0,1) rounded to
    bf16-representable values, theta* ~ N(0,1)/sqrt(d), y ~ Bernoulli(sigmoid(X theta*))."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, d)).astype(np.float32)
    X = (X.view(np.uint32) & np.uint32(0xFFFF0000)).view(np.float32)
    tstar = rng.standard_normal(d) / np.sqrt(d)
    y = (rng.random(N) < 1.0 / (1.0 + np.exp(-(X.astype(np.float64) @ tstar)))).astype(np.float32)
    return X, y, tstar


def make_inputs(wl, seed):
    rng = np.random.default_rng(seed)
    d, nw = wl["d"], wl["nw"]
    if wl["plugin"] == "rosenbrock":
        params = [1.0, 100.0, 20.0]
        x0 = 0.1 * rng.standard_normal((nw, d))
    elif wl["plugin"] == "gaussian":
        params = gaussian_params(np.linspace(-1, 1, d), spd_cov(d, 1))
        x0 = 0.1 * rng.standard_normal((nw, d))
    elif wl["plugin"] == "logistic":
        X, y, tstar = logistic_problem(N=wl["ndata"], d=d, seed=seed)
        wl["_data"] = np.concatenate([X.ravel(), y])
        params = [10.0]
        x0 = tstar + 1e-3 * rng.standard_normal((nw, d))
    else:
        params = []
        x0 = np.abs(0.5 + 0.1 * rng.standard_normal((nw, d)))
    return params, x0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.path = gpu_index, None, None

    def start(self):
        if os.environ.get("KMC_BENCH_NO_CLOCKS"):   # experiment: is the sampler itself a perturbation?
            return
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.idx)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def wait_ready(self, timeout=8.0):
        """Blocks until nvidia-smi has printed its first sample: its start-up (NVML attaches to every GPU of the box) must
        not overlap the timed region -- measured on 2- and 8-GPU boxes: kernels running during that start-up were 11 %
        slower (131.6 instead of 118.5 ms per step)."""
        if not self.proc:
            return
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < timeout:
            try:
                if os.path.getsize(self.path) > 0:
                    return
            except OSError:
                return
            time.sleep(0.02)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [v.strip() for v in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def run_reference(args, wl):
    """--impl reference: the C restatement of the reference loop on all host cores, bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle
    nthreads = os.cpu_count() or 1
    # each step ~4 s of CPU work (the whole run stays within a few minutes)
    dens, x0, nw, iters = _cpu_sample(wl, 4.0, nthreads)
    iters, _ = _cpu_run(wl, dens, x0, iters, 4.0, nthreads, 99)      # settles the sample size (untimed)
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        oracle.emcee(dens, x0, iters, iters // 2, max(1, iters // 5), 2.0, seed=i, store=True, nthreads=nthreads,
                     native=True)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    value = nw * iters * args.steps / total
    sample = (f"{wl['plugin']} d={wl['d']}, {nw} walkers (of {wl['nw']}) x {iters} iterations per step "
              f"(of {wl['niter_walker']})")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "description": wl["desc"], "nwalkers": nw, "d": wl["d"],
                   "note": "C restatement of the reference loop (oracle/kmc_oracle.c, -O3 -march=native -fopenmp, "
                           "-ffp-contract=off); the Julia reference cannot run in this image"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": nthreads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def _cpu_sample(wl, seconds, nthreads):
    """Bounded sample of the workload for the CPU leg: (walkers, iterations) worth ~`seconds` of host time.
    Calibrated in two steps (single-thread cost on the smallest legal ensemble, then all threads on a sub-ensemble
    sized from it) so that even the calibration of an expensive density stays short; the sample keeps the full
    ensemble unless two iterations of it would already exceed the budget."""
    from oracle import oracle
    params, x0 = make_inputs(wl, 1)
    dens = oracle.Density(wl["plugin"], wl["d"], params, data=wl.get("_data"))
    nw = wl["nw"]
    # 1) one thread, the smallest legal ensemble: a reliable per-walker-step cost without OpenMP noise
    n1 = min(nw, 2 * ((wl["d"] + 3) // 2))
    oracle.emcee(dens, x0[:n1], 1, 0, 1, 2.0, seed=1, store=False, nthreads=1, native=True)   # library load
    t0 = time.perf_counter()
    oracle.emcee(dens, x0[:n1], 1, 0, 1, 2.0, seed=1, store=False, nthreads=1, native=True)
    per_ws1 = max((time.perf_counter() - t0) / n1, 1e-9)
    # 2) all threads on a sub-ensemble sized for ~0.5 s if the threads scaled perfectly (best of 2)
    ncal = int(min(nw, max(n1, 0.5 * nthreads / (2 * per_ws1))))
    ncal -= ncal % 2
    dt = float("inf")
    for _ in range(2):
        t0 = time.perf_counter()
        oracle.emcee(dens, x0[:ncal], 2, 1, 1, 2.0, seed=1, store=False, nthreads=nthreads, native=True)
        dt = min(dt, time.perf_counter() - t0)
    per_ws = max(dt / (2 * ncal), 1e-9)
    nw_s = nw
    if 2 * nw * per_ws > 1.5 * seconds:
        nw_s = int(max(ncal, min(nw, seconds / (2 * per_ws))))
        nw_s -= nw_s % 2
    iters = int(max(2, min(wl["niter_walker"], seconds / (per_ws * nw_s))))
    return dens, x0[:nw_s], nw_s, iters


def _cpu_run(wl, dens, x0, iters, seconds, nthreads, seed):
    """One timed CPU sample; if the calibration was pessimistic (a noisy host makes small OpenMP regions look slow)
    and the run ended in under a third of the budget, lengthen it and time again (at most twice)."""
    from oracle import oracle
    for _ in range(3):
        t0 = time.perf_counter()
        oracle.emcee(dens, x0, iters, iters // 2, max(1, iters // 5), 2.0, seed=seed, store=True, nthreads=nthreads,
                     native=True)
        dt = time.perf_counter() - t0
        if dt >= seconds / 3 or iters >= wl["niter_walker"]:
            break
        iters = int(min(wl["niter_walker"], max(iters + 1, iters * 0.8 * seconds / max(dt, 1e-6))))
    return iters, dt


def cpu_baseline(wl, seconds=15.0):
    nthreads = os.cpu_count() or 1
    dens, x0, nw_s, iters = _cpu_sample(wl, seconds, nthreads)
    iters, dt = _cpu_run(wl, dens, x0, iters, seconds, nthreads, 2)
    return {"value": nw_s * iters / dt, "unit": UNIT, "cores": nthreads, "kind": "port",
            "sample": f"{wl['plugin']} d={wl['d']}, {nw_s} walkers (of {wl['nw']}) x {iters} iterations "
                      f"(of {wl['niter_walker']}), {dt:.1f} s, C restatement of the reference loop with OpenMP"}


def roofline_of(wl, workload, tensor, launch_mode, k_ms, traffic):
    """The roofline object of the dominant kernel of one step of `workload` (SURVEY.md section 8d)."""
    d, nw, nitw, nthin = wl["d"], wl["nw"], wl["niter_walker"], wl["nthin"]
    ns = (nitw - nitw // 2) // nthin
    walker_steps = nw * nitw
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    peaks = json.loads(peaks_path.read_text()) if peaks_path.exists() else {}
    if wl["plugin"] == "logistic":      # tensor-bound nominally: 2*d*N flops per walker-step
        tpeak = peaks.get("bf16_tflops_sustained", 1400.0)
        flops = 2.0 * d * wl["ndata"] * walker_steps
        tflops = flops / (k_ms * 1e-3) / 1e12
        return {"bound": "tensor", "achieved": tflops, "peak": tpeak, "unit": "TFLOP/s", "frac": tflops / tpeak,
                "traffic": traffic, "kernel": "tc::logistic_tc_kernel" if tensor else "logistic_logp_kernel",
                "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback",
                "algorithmic_flops_per_step": flops, "kernel_ms_per_step": k_ms,
                "note": "algorithmic flops 2*d*N per walker-step; the tcgen05 kernel issues 3x that (theta split into 3 "
                        "bf16 pieces) and is bounded by its softplus epilogue"}
    peak = peaks.get("hbm_gbs", 6650.0)
    alg = b_step(d) * walker_steps + (8 * d + 8) * nw * ns
    achieved = alg / (k_ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "kernel": dominant_kernel(wl, tensor, launch_mode),
            "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback (B200_PROFILING.md)",
            "algorithmic_bytes_per_launch": alg, "kernel_ms_per_launch": k_ms,
            "note": "algorithmic bytes = (24d+24) per walker-step + (8d+8) per stored sample; a state that fits L2 / "
                    "shared memory makes frac against the HBM copy peak able to exceed 1"}


def measure_traffic(workload, kernel_regex, timeout=240):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE bench-size launch of the dominant kernel, measured now:
    ncu around a child process that runs one step of the same workload with the same library build.  Returns
    (bytes | None, how)."""
    import hashlib
    import shutil
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not Path(ncu).exists():
        return None, "ncu not found"
    import kissmcmc_b200 as km
    sha = hashlib.sha256(Path(km.LIB_PATH).read_bytes()).hexdigest()[:16]
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "-k",
           f"regex:{kernel_regex}", "-c", "1", "--csv", sys.executable, str(ROOT / "bench.py"), "--traffic-child",
           "--workload", workload]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout)
    except Exception as e:      # noqa: BLE001
        return None, f"ncu failed: {e!r}"
    tot, seen = 0.0, 0
    import csv
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    for row in csv.reader(r.stdout.splitlines()):
        if len(row) > 3 and row[-3] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            try:
                tot += float(row[-1].replace(",", "")) * scale.get(row[-2], 1.0)
                seen += 1
            except ValueError:
                pass
    if seen != 2:
        return None, "ncu gave no dram counters (rc %d): %s" % (r.returncode, (r.stdout + r.stderr)[-200:].replace("\n", " "))
    return tot, f"ncu dram__bytes_read.sum+dram__bytes_write.sum of one {kernel_regex} launch, library sha256 {sha}"


def traffic_child(wl_name):
    """One step of the workload (run under ncu by measure_traffic)."""
    import kissmcmc_b200 as km
    wl = WORKLOADS[wl_name]
    params, x0 = make_inputs(wl, 1000)
    ld = km.LogDensity(wl["plugin"], wl["d"], params, data=wl.get("_data"))
    if wl["plugin"] == "logistic" or (wl["plugin"] == "gaussian" and wl["d"] > 16):
        ld.set_option("tensor_cores", 1)
    s = km.Sampler(ld, x0, wl["niter_walker"], wl["niter_walker"] // 2, wl["nthin"], 2.0, seed=1)
    s.run(-1)
    s.close()
    return 0


class Env:
    """Process-wide plumbing of one bench process (one rank)."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.stream = torch.cuda.Stream()
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier(self):
        # synchronize FIRST: a dist.barrier() issued while this rank's kernels are still queued puts NCCL's kernel between
        # them -- it holds an SM while it waits for the peer, and the next cooperative launch (every SM, all shared memory)
        # cannot start: measured +12 ms per step on one (random) rank of a 2- or 8-GPU run (profiles/r2_call34.log)
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def gather(self, vals):
        """vals of every rank, [world][len(vals)]."""
        if self.world == 1:
            return [list(vals)]
        t = self.torch.tensor(vals, dtype=self.torch.float64, device="cuda")
        out = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [o.tolist() for o in out]

    def max_sum(self, vals):
        t = self.torch.tensor(vals, dtype=self.torch.float64, device="cuda")
        if self.world == 1:
            return vals, vals
        mx, sm = t.clone(), t.clone()
        self.dist.all_reduce(mx, op=self.dist.ReduceOp.MAX)
        self.dist.all_reduce(sm, op=self.dist.ReduceOp.SUM)
        return mx.tolist(), sm.tolist()


def dump_outputs(out_dir, chain, logp, ratio, budget=48_000_000):
    """Writes what one emcee job returns to its caller -- the stored chain [nw, ns, d], its log-densities [nw, ns] and
    the accept ratio of every walker -- as float64 .npy files under out_dir, with walker_index.npy naming the walkers
    written.  When all walkers would exceed `budget` bytes, a fixed seeded sample of walkers (sorted; the same rows in
    every file) is written, so that two builds run with the same arguments can be compared file for file."""
    nw = len(ratio)
    per_walker = 8 * (chain[0].size + logp[0].size + 2)
    keep = np.arange(nw)
    if nw * per_walker > budget:
        keep = np.sort(np.random.default_rng(0).choice(nw, budget // per_walker, replace=False))
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    arrays = {"chain": chain[keep], "log_density": logp[keep], "accept_ratio": ratio[keep], "walker_index": keep}
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a.astype(np.float64))


def run_workload(env, km, workload, steps, warmup, launch_mode=0, tensor_cores=None, e2e_steps=3, keep_outputs=False):
    """Times `steps` steps (complete emcee jobs) of one workload on every rank (independent ensembles).
    Returns the pieces of a bench line: value / ms_per_step / roofline / e2e / clocks / launches, and with
    keep_outputs the (chain, log-densities, accept ratios) of the last timed step."""
    torch = env.torch
    wl = WORKLOADS[workload]
    rank, world, local = env.rank, env.world, env.local
    d, nw, nitw, nthin = wl["d"], wl["nw"], wl["niter_walker"], wl["nthin"]
    nbw = nitw // 2
    ns = (nitw - nbw) // nthin
    params, x0 = make_inputs(wl, 1000 + rank)
    ld = km.LogDensity(wl["plugin"], d, params, data=wl.get("_data"), device=local)
    if tensor_cores is not None:
        ld.set_option("tensor_cores", tensor_cores)
    elif wl["plugin"] == "logistic" or (wl["plugin"] == "gaussian" and d > 16):
        ld.set_option("tensor_cores", 1)          # bench default for configs[2], configs[3]: the tcgen05 kernels (opt-in)
    tensor = ld.info("tensor_cores") == 1.0
    stream, flush = env.stream, env.flush

    def new_sampler(step):
        # independent ensembles: rank-distinct Philox key and walker-id range
        s = km.Sampler(ld, x0, nitw, nbw, nthin, 2.0, seed=(step << 8) | rank, walker_id_base=rank * nw,
                       launch_mode=launch_mode)
        s.set_stream(stream.cuda_stream)
        return s

    walker_steps_per_step = nw * nitw

    # ---- value: device-timed, inputs resident in HBM -------------------------------------
    total = warmup + steps
    samplers = [new_sampler(i) for i in range(total)]
    with torch.cuda.stream(stream):
        for i in range(warmup):
            flush.fill_(i & 0xFF)
            samplers[i].run(-1, sync=False)
    env.barrier()
    clocks = ClockSampler(local)
    clocks.start()
    clocks.wait_ready()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env.barrier()
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for i in range(warmup, total):
            flush.fill_(i & 0xFF)                     # L2 flush between steps (inside the timed region)
            samplers[i].run(-1, sync=False)
        ev1.record(stream)
    env.barrier()
    clk = clocks.stop()
    dev_ms = ev0.elapsed_time(ev1)
    kern_ms, launches = [], 0
    for i in range(warmup, total):
        ms, n = samplers[i].last_run_ms()
        kern_ms.append(ms)
        launches += n
    outputs = samplers[-1].results() if keep_outputs else None
    for s in samplers:
        s.close()

    # ---- e2e: public API, host buffers, H2D + D2H inside the timed region ------------------
    x0_pinned = torch.from_numpy(x0).pin_memory()
    out_th = torch.empty((nw, ns, d), dtype=torch.float64).pin_memory()
    out_lp = torch.empty((nw, ns), dtype=torch.float64).pin_memory()
    out_ar = torch.empty((nw,), dtype=torch.float64).pin_memory()

    def e2e_step(step):
        ta = time.perf_counter()
        s = km.Sampler(ld, x0_pinned.numpy(), nitw, nbw, nthin, 2.0, seed=(step << 8) | rank,
                       walker_id_base=rank * nw, launch_mode=launch_mode)
        tb = time.perf_counter()
        s.run(-1)
        tc = time.perf_counter()
        s.results(out_th.numpy(), out_lp.numpy(), out_ar.numpy())
        td = time.perf_counter()
        s.close()
        if os.environ.get("KMC_BENCH_VERBOSE"):
            print(f"e2e step {step}: create {1e3 * (tb - ta):.1f} run {1e3 * (tc - tb):.1f} results "
                  f"{1e3 * (td - tc):.1f} close {1e3 * (time.perf_counter() - td):.1f} ms", file=sys.stderr)

    e2e_steps = max(1, min(steps, e2e_steps))
    e2e_step(0)
    env.barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(100 + i)
    env.barrier()
    e2e_s = time.perf_counter() - t0
    del x0_pinned, out_th, out_lp, out_ar
    km.lib.kmc_trim()                             # give the cached device blocks back before the next workload

    per_rank = env.gather([statistics.mean(kern_ms), dev_ms / steps, float(clk["sm_mhz"] or 0.0)])
    (dev_ms, e2e_ms, _, _), (_, _, _, launches) = env.max_sum([dev_ms, e2e_s * 1e3, max(kern_ms), float(launches)])
    k_ms = statistics.mean(kern_ms)
    return {
        "wl": wl, "tensor": tensor, "k_ms": k_ms, "outputs": outputs,
        "per_rank": {"kernel_ms": [round(v[0], 3) for v in per_rank], "ms_per_step": [round(v[1], 3) for v in per_rank],
                     "sm_mhz": [v[2] for v in per_rank]},
        "value": world * walker_steps_per_step * steps / (dev_ms * 1e-3),
        "ms_per_step": dev_ms / steps,
        "dtype": "bf16x3 split operands, f32 accumulate (tcgen05); f64 state" if tensor else "f64",
        "e2e": {"value": world * walker_steps_per_step * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": int(x0.nbytes), "d2h_bytes_per_step": int(nw * ns * d * 8 + nw * ns * 8 + nw * 4),
                "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps},
        "gpu_launches": int(launches), "clocks": clk,
        "config": {
            "workload": workload, "tensor_cores": tensor, "description": wl["desc"], "plugin": wl["plugin"], "d": d,
            "nwalkers_per_gpu": nw, "niter_walker": nitw, "nburnin_walker": nbw, "nthin": nthin,
            "samples_per_walker": ns, "a_scale": 2.0, "rng": "philox4x32-10",
            "parallelism": "1 ensemble" if world == 1 else f"{world} independent ensembles (no collective)",
            "launch_mode": "persistent kernel, grid barrier per half-step" if launch_mode == 0
            else "one launch per half-step",
            "l2": "ensemble state is L2-resident by construction across the dependent half-steps of one step; "
                  "L2 flushed (256 MiB fill) between steps, inside the timed region",
        },
    }


def sharded_section(env, km, lg_nw=24, iters=20, warm=4):
    """BASELINE.json configs[4]: ONE 2^24-walker 10-D Gaussian ensemble sharded by walker index over all ranks.
    Rank 0 first times the unsharded ensemble on its GPU (the in-run 1-GPU anchor); then all ranks time the push
    exchange (csrc/kmc_push.cuh: owner-computes packed row pushes over NVLink, no collective) and the NCCL
    all-gather exchange north_star names.  Device time = max over ranks of each rank's CUDA-event time of its own
    kernels (all-gather: events around kernels + collectives on the one stream they share).  Strong scaling: the
    ensemble is fixed; `weak` repeats it with 2^21 walkers per GPU."""
    torch, dist = env.torch, env.dist
    rank, world, local = env.rank, env.world, env.local
    from kissmcmc_b200 import distributed as kd

    def one(nw, with_allgather):
        wl = dict(WORKLOADS["gaussian10d"], nw=nw)
        params, x0 = make_inputs(wl, 1)              # the same ensemble on every rank
        d, nhalf = wl["d"], nw // 2
        ld = km.LogDensity("gaussian", d, params, device=local)
        out = {"nwalkers": nw, "d": d, "iters": iters}
        ms1 = 0.0
        if rank == 0:                                 # 1-GPU anchor: the unsharded ensemble on this rank's GPU
            s = km.Sampler(ld, x0, iters + warm, 0, 10**6, 2.0, 7, device=local)
            s.run(warm)
            s.run(iters)
            ms1, _ = s.last_run_ms()
            s.close()
            km.lib.kmc_trim()
        env.barrier()
        (ms1,), _ = env.max_sum([ms1])
        out["value_1gpu"] = nw * iters / (ms1 * 1e-3)
        out["ms_per_halfstep_1gpu"] = ms1 / (2 * iters)
        if world == 1:
            return out
        begin, count = kd.shard_range(nw, rank, world)
        # ---- push exchange: one persistent kernel per rank
        s = km.Sampler(ld, x0, iters + warm, 0, 10**6, 2.0, 7, device=local, shard=(begin, count),
                       exchange=km.EXCHANGE_PUSH)
        allh = [None] * world
        dist.all_gather_object(allh, s.window_export())
        s.window_attach(allh, rank)
        env.barrier()
        s.run(warm, sync=True)
        env.barrier()
        s.run(iters, sync=True)
        ms, _ = s.last_run_ms()
        env.barrier()
        s.close()
        (msp,), _ = env.max_sum([ms])
        out["value_push"] = nw * iters / (msp * 1e-3)
        out["ms_per_halfstep_push"] = msp / (2 * iters)
        out["efficiency_push"] = out["value_push"] / (world * out["value_1gpu"])
        out["bytes_nvlink_per_halfstep"] = count * 8 * d * (world - 1) // world       # per GPU, each direction
        out["nvlink_gbs_per_gpu"] = out["bytes_nvlink_per_halfstep"] / (msp / (2 * iters) * 1e-3) / 1e9
        if not with_allgather:
            return out
        # ---- NCCL all-gather of the updated half after every half-step (every rank holds the full ensemble)
        km.lib.kmc_trim()
        s = km.Sampler(ld, x0, iters + warm, 0, 10**6, 2.0, 7, device=local, launch_mode=1, shard=(begin, count))
        st = torch.cuda.Stream()
        s.set_stream(st.cuda_stream)
        xt = kd.x_tensor(s)

        def halfsteps(n, h0):
            for h in range(h0, h0 + n):
                s.run_half(1)
                half = xt[(h & 1) * nhalf:((h & 1) + 1) * nhalf]
                dist.all_gather_into_tensor(half.view(-1), half[begin:begin + count].reshape(-1))
        with torch.cuda.stream(st):
            halfsteps(2 * warm, 0)
            env.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            halfsteps(2 * iters, 2 * warm)
            e1.record(st)
            env.barrier()
        (msa,), _ = env.max_sum([e0.elapsed_time(e1)])
        s.close()
        km.lib.kmc_trim()
        out["value_allgather"] = nw * iters / (msa * 1e-3)
        out["ms_per_halfstep_allgather"] = msa / (2 * iters)
        out["allgather_bytes_per_rank_per_halfstep"] = nhalf * d * 8
        return out

    res = one(1 << lg_nw, True)
    res["workload"] = f"gaussian10d, ONE ensemble of 2^{lg_nw} walkers sharded by walker index (strong scaling)"
    if world > 1:
        res["value_peer"] = res["value_push"]         # the fused peer-memory path is the push exchange
        res["efficiency_peer"] = res["efficiency_push"]
        weak = one((1 << 21) * world, False)
        anchor = one(1 << 21, False) if world > 1 else weak
        res["weak"] = {"nwalkers_per_gpu": 1 << 21, "value_1gpu_one_shard": anchor["value_1gpu"],
                       "value_push": weak.get("value_push"),
                       "efficiency": weak["value_push"] / (world * anchor["value_1gpu"]),
                       "ms_per_halfstep_push": weak.get("ms_per_halfstep_push"),
                       "ms_per_halfstep_1gpu_one_shard": anchor["ms_per_halfstep_1gpu"]}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="rosenbrock2d", choices=sorted(WORKLOADS))
    ap.add_argument("--launch-mode", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip the short lines of the other four configs (N=1)")
    ap.add_argument("--no-sharded", action="store_true", help="skip the sharded-ensemble section")
    ap.add_argument("--no-traffic", action="store_true", help="skip the ncu DRAM-traffic measurement (N=1)")
    ap.add_argument("--traffic-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--tensor-cores", type=int, default=None, choices=[0, 1],
                    help="force the tcgen05 (1) or FP64 (0) log-density kernel of the dense plugins")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (chain, log-densities, accept ratios; "
                         "rank 0) to DIR/*.npy as float64, a fixed seeded sample of walkers if all would exceed 48 MB")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, wl)
    if args.traffic_child:
        return traffic_child(args.workload)

    import kissmcmc_b200 as km
    env = Env()
    rank, world = env.rank, env.world

    r = run_workload(env, km, args.workload, args.steps, args.warmup, args.launch_mode, args.tensor_cores,
                     keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *r["outputs"])
    r["outputs"] = None
    default_run = args.workload == "rosenbrock2d" and args.launch_mode == 0 and args.tensor_cores is None

    others = []
    if world == 1 and default_run and not args.no_others:      # the other four configs, short, on the same box
        for name in ("exponential1d", "gaussian100d", "logistic32d", "gaussian10d"):
            o = run_workload(env, km, name, 3, 3, 0, None, e2e_steps=2)
            others.append({"workload": name, "value": o["value"], "unit": UNIT, "steps": 3, "warmup": 3,
                           "ms_per_step": o["ms_per_step"], "dtype": o["dtype"],
                           "roofline": roofline_of(o["wl"], name, o["tensor"], 0, o["k_ms"], None),
                           "e2e": o["e2e"], "clocks": o["clocks"], "gpu_launches": o["gpu_launches"],
                           "description": o["wl"]["desc"]})

    sharded = None
    if default_run and not args.no_sharded:
        sharded = sharded_section(env, km)

    traffic, traffic_how = None, "not measured"
    if rank == 0 and world == 1 and not args.no_traffic:
        env.torch.cuda.synchronize()
        kern = dominant_kernel(r["wl"], r["tensor"], args.launch_mode).split("::")[-1].split(" ")[0]
        traffic, traffic_how = measure_traffic(args.workload, kern)

    if rank == 0:
        roof = roofline_of(r["wl"], args.workload, r["tensor"], args.launch_mode, r["k_ms"], traffic)
        roof["traffic_source"] = traffic_how
        line = {
            "metric": METRIC, "value": r["value"], "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": r["dtype"],
            "data": "synthetic", "config": r["config"], "roofline": roof, "e2e": r["e2e"],
            "gpu_launches": r["gpu_launches"], "clocks": r["clocks"],
        }
        if world > 1:
            line["per_rank"] = r["per_rank"]      # the step time is the slowest rank's: which one, and at what clock
        if others:
            line["others"] = others
        if sharded:
            line["sharded"] = sharded
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(wl)
        print(json.dumps(line))
    if world > 1:
        env.dist.barrier()
        env.dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
