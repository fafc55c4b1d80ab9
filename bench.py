#!/usr/bin/env python
"""Benchmark of the kernel-recombination hot path (BASELINE.json metric: candidate points
recombined per second, N -> n at d = 10).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scaling weak|strong]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one full pass of the hot path over one batch of synthetic candidates: Nystrom basis of
the landmark Gram matrix + the Tchernychova-Lyons / Caratheodory loop (refined passes, DESIGN.md 2)
down to <= n weighted points.
Workload (config.workload): BASELINE config 3 - 10-D Gaussian-mixture setting, batch n = 1000,
M = 1e4 landmarks, RBF kernel, VBQ posterior-covariance kernel object with n_obs = 1002 at the
reference's default likelihood noise (BASQ/_parameters.py:30).  Default scaling is weak (N_rec = 1e7
candidates PER GPU); at N > 1 the line also carries `strong` - the configuration as BASELINE.json
words it, 1e7 candidates in total sharded over the ranks - and `--scaling strong` makes that the
headline instead.
`value` times the device-resident path; `e2e` times the host-buffer C-ABI call including the
host<->device copies; `iteration` times one BASQ iteration with the candidates drawn on the device;
`extra` (N = 1 only) times the other BASELINE configurations and the config-5 acquisition pass.
`--impl reference` times the CPU oracle port of the reference's algorithm on a bounded sample (the
reference is pure Python over gpytorch and does not ship to the GPU box).
`--dump-outputs DIR` writes the quadrature rule the last timed `value` step returned (global candidate
indices and weights) as DIR/indices.npy and DIR/weights.npy, both float64; the inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "candidate points recombined/sec (N->n, d=10)"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    p.add_argument("--N", type=int, default=10_000_000, help="candidates per GPU (weak) / in total (strong)")
    p.add_argument("--M", type=int, default=10_000, help="Nystrom landmarks")
    p.add_argument("--n", type=int, default=1000, help="batch size (points returned)")
    p.add_argument("--d", type=int, default=10)
    p.add_argument("--n-obs", type=int, default=1002)
    p.add_argument("--lengthscale", type=float, default=2.5)
    p.add_argument("--noise", type=float, default=1e-10, help="likelihood noise (reference default 1e-10)")
    p.add_argument("--cpu-sample", type=int, default=100_000, help="candidates in the CPU-baseline sample")
    p.add_argument("--cpu-budget", type=float, default=200.0, help="seconds of timed CPU work in --impl reference")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-extra", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the last timed step's rule as DIR/indices.npy and DIR/weights.npy (float64)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    return a


def dump_outputs(out_dir, idx, w):
    """The rule a caller of the timed path receives: candidate indices (exact in float64) and weights."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "indices.npy"), idx.cpu().to(torch.float64).numpy())
    np.save(os.path.join(out_dir, "weights.npy"), w.cpu().to(torch.float64).numpy())


# ------------------------------------------------------------------------------------------ workload
def make_observations(d, n_obs, seed=11, log=False, sqrt=False):
    """Synthetic GP observations: prior N(0, 2 I_d) inputs, 3-component Gaussian-mixture likelihood
    (the shape of BASQ/experiment/gmm.py), fixed hyper-parameters (SURVEY 8d)."""
    g = torch.Generator().manual_seed(seed)
    X = math.sqrt(2.0) * torch.randn(n_obs, d, generator=g, dtype=torch.float64)
    centres = 1.5 * torch.randn(3, d, generator=g, dtype=torch.float64)
    y = sum(torch.exp(-0.25 * ((X - c) ** 2).sum(-1)) for c in centres) / 3.0
    if log:
        y = torch.log(y + 1e-12)
        y = y - y.max()
    if sqrt:
        y = torch.sqrt(2.0 * y)
    return X, y


def workload_name(a):
    return (f"BASELINE config 3: N_rec={a.N:g}{'/GPU' if a.scaling == 'weak' else ' total'} d={a.d} n={a.n} "
            f"M={a.M} RBF l={a.lengthscale:g} noise={a.noise:g} VBQ predictive-covariance kernel n_obs={a.n_obs}")


def config_of(a, world):
    n_total = a.N * world if a.scaling == "weak" else a.N
    return {"workload": workload_name(a), "N_total": n_total, "parallelism": f"dp{world}",
            "l2_policy": "inputs (640 MB of candidate records per 1e7 candidates) exceed the 126 MB L2"}


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, every 100 ms from a background thread.
    In-process NVML (nvidia_ml_py) when available: forking `nvidia-smi` five times a second from every rank
    perturbs the host-side loop of an 8-rank run (the Nystrom phase measured 36 instead of 21 ms);
    `nvidia-smi` is the fallback.  Only rank 0 samples (it prints the line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, enabled=True):
        self.index, self.rows, self.stop, self.enabled = index, [], threading.Event(), enabled
        self.t = threading.Thread(target=self._run, daemon=True)
        self.nvml = None
        if enabled:
            try:
                import pynvml
                pynvml.nvmlInit()
                # CUDA_VISIBLE_DEVICES may renumber the devices: resolve through the PCI address of the torch device
                try:
                    self.handle = self._by_bus(pynvml, index)
                except Exception:
                    self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
                self.nvml = pynvml
            except Exception:
                self.nvml = None

    @staticmethod
    def _by_bus(pynvml, index):
        p = torch.cuda.get_device_properties(index)
        want = (int(p.pci_domain_id), int(p.pci_bus_id), int(p.pci_device_id))
        for i in range(pynvml.nvmlDeviceGetCount()):
            h = pynvml.nvmlDeviceGetHandleByIndex(i)
            info = pynvml.nvmlDeviceGetPciInfo(h)
            if (int(info.domain), int(info.bus), int(info.device)) == want:
                return h
        return pynvml.nvmlDeviceGetHandleByIndex(index)

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        pw = n.nvmlDeviceGetPowerUsage(h) / 1e3
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        r = int(get(h))
        bit = lambda name, alt: int(getattr(n, name, getattr(n, alt, 0)))
        flags = [("hw_slowdown", bit("nvmlClocksEventReasonHwSlowdown", "nvmlClocksThrottleReasonHwSlowdown")),
                 ("hw_thermal_slowdown", bit("nvmlClocksEventReasonHwThermalSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown")),
                 ("sw_thermal_slowdown", bit("nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwThermalSlowdown")),
                 ("sw_power_cap", bit("nvmlClocksEventReasonSwPowerCap", "nvmlClocksThrottleReasonSwPowerCap"))]
        return [str(sm), str(mx), f"{pw:.1f}"] + ["Active" if (m and (r & m)) else "Not Active" for _, m in flags]

    def _run(self):
        while not self.stop.is_set():
            try:
                if self.nvml is not None:
                    self.rows.append(self._sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                    self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self.stop.wait(0.1 if self.nvml is not None else 0.2)

    def __enter__(self):
        if self.enabled:
            self.t.start()
        return self

    def __exit__(self, *exc):
        self.stop.set()
        if self.enabled:
            self.t.join(timeout=6)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------ reference arm
def host_threads():
    """All host cores: torch.distributed.run exports OMP_NUM_THREADS=1, which would leave the CPU arm
    on one thread."""
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    torch.set_num_threads(max(1, cores))
    return torch.get_num_threads()


def oracle_step(a, n_sample, seed=0, device="cpu"):
    """One pass of the reference's algorithm (oracle port of BASQ/_rchq.py, plain torch ops) over a
    bounded sample of the workload: same d, M, n, kernel object; N reduced to n_sample.  device="cuda"
    runs the same torch-op sequence on the GPU - the reference's own GPU story (`tensor.to(device)`)."""
    from oracle import gp_kernels as ogp
    from oracle import rchq as orchq

    Xo, yo = make_observations(a.d, a.n_obs)
    # matmul_dist: gpytorch's own distance formula (one GEMM per Gram block) - what the reference executes
    model = ogp.ExactGP(Xo, yo, ogp.ScaleKernel(ogp.RBFKernel(a.lengthscale), 1.0, matmul_dist=True),
                        noise=a.noise).to(device)
    kern = ogp.VanillaGP(model).predictive_kernel
    g = torch.Generator().manual_seed(seed)
    X = (math.sqrt(2.0) * torch.randn(n_sample, a.d, generator=g)).double().to(device)
    Z = X[: a.M].clone()
    if device != "cpu":
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    torch.manual_seed(seed)
    idx, w = orchq.recombination(X, Z, a.n, kern, chunk=max(1, (200_000 if device == "cpu" else 50_000) // (2 * a.n)))
    if device != "cpu":
        torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    assert len(idx) <= a.n and bool((w > 0).all())
    return dt


def sample_text(a, n_sample, what):
    return (f"N={n_sample} candidates of the same workload (d={a.d}, M={a.M}, n={a.n}, n_obs={a.n_obs}), {what}")


def run_reference(a, rank, world):
    """The reference arm: the CPU oracle port on all host cores, on a FIXED bounded sample of the
    workload (N = --cpu-sample, never shrunk), as many of the K requested steps as fit --cpu-budget
    seconds (at least one).  A second, smaller sample gives the per-point marginal cost, so that the
    full-size (N = 1e7) time is stated as an explicit extrapolation instead of being implied."""
    if rank != 0:
        return
    cores = host_threads()
    n_sample = max(a.cpu_sample, 4 * a.n, a.M)
    n_small = max(n_sample // 4, 4 * a.n, a.M)
    t_small = oracle_step(a, n_small, seed=100)          # also the warm-up (thread pools, allocator)
    times, t_begin = [], time.perf_counter()
    for s in range(max(1, a.steps)):
        times.append(oracle_step(a, n_sample, seed=s))
        if time.perf_counter() - t_begin + times[-1] > a.cpu_budget:
            break
    t = sum(times) / len(times)
    v = n_sample / t
    marginal = max(t - t_small, 0.0) / max(n_sample - n_small, 1)   # seconds per additional candidate
    fixed = t - marginal * n_sample
    n_full = a.N
    t_full = fixed + marginal * n_full
    sample = sample_text(a, n_sample, "oracle port of BASQ/_rchq.py, fp64 torch CPU")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "points/s", "n_gpus": a.gpus,
        "steps": len(times), "warmup": 1, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": a.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(a, world),
        "cpu_baseline": {"value": v, "unit": "points/s", "cores": cores, "kind": "port", "sample": sample,
                         "seconds": t, "steps_requested": a.steps, "steps_timed": len(times)},
        "extrapolation": {"what": "fixed + marginal cost fitted on two sample sizes; the CPU path's points/s grows "
                                  "with N because the Nystrom basis and the Caratheodory rounds are fixed costs",
                          "n_small": n_small, "seconds_small": t_small, "n_large": n_sample, "seconds_large": t,
                          "fixed_seconds": fixed, "seconds_per_point": marginal,
                          "N_full": n_full, "seconds_full": t_full, "points_per_s_full": n_full / t_full},
        "e2e": {"value": v, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ our arm
def extra_configs(dev, a):
    """The other BASELINE configurations at full size (Nystrom basis + recombination, device-resident)
    and the config-5 acquisition pass; one timed repetition each after one warm-up."""
    from basq_b200 import _lib, gp as bgp, ops, sampler as bsampler
    from basq_b200.kernels import KernelSpec, spec_from_model

    out = {}
    try:
        peak_bf16 = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"]
    except Exception:
        peak_bf16 = 1400.0     # fallback of B200_PROFILING.md (sustained)
    ctx = _lib.context_for(dev)

    def run(name, kern, d, N, M, n, reps=2):
        X = bsampler.sample_mvn(torch.zeros(d), 2.0 * torch.eye(d), N, seed=7, device=dev)
        Z = X[:M].clone()
        Om = torch.randn(M, n - 1, dtype=torch.float64, device=dev, generator=torch.Generator(device=dev).manual_seed(3))

        def step():
            _, U = ops.nystrom_basis(kern, Z, n - 1, omega=Om, want_S=False)
            return ops.recombine(kern, X, Z, U)
        step()
        torch.cuda.synchronize(dev)
        ctx.profile(True)
        ctx.profile_read(reset=True)
        pe0 = ctx.pair_evals
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            idx, w = step()
        e1.record()
        torch.cuda.synchronize(dev)
        prof = ctx.profile_read(reset=True)
        ctx.profile(False)
        ms = e0.elapsed_time(e1) / reps
        assert 1 <= len(idx) <= n and abs(float(w.sum()) - 1.0) < 1e-9
        out[name] = {"ms": round(ms, 3), "points_per_s": N / ms * 1e3, "N": N, "M": M, "n": n, "d": d,
                     "phases_ms": {k: round(v[0] / reps, 2) for k, v in prof.items() if v[0] > 0}}
        if kern.mode in (_lib.WSABI_M, _lib.MMLT_G):
            # the pairwise correction Az k(Xobs, x): 2 n_obs flop per (landmark, candidate) pair on tcgen05
            pairs = (ctx.pair_evals - pe0) / reps
            ss = prof["set_sum"][0] / reps * 1e-3
            n_obs_k = int(kern.Xobs.shape[0])
            ach = 2.0 * n_obs_k * pairs / ss / 1e12
            out[name]["roofline"] = {"bound": "tensor", "kernel": "nlsum_kernel (tcgen05 kind::f16, fp16 hi / lo split: 3 products)",
                                     "unit": "TFLOP/s", "achieved": ach, "peak": peak_bf16, "frac": ach / peak_bf16,
                                     "issued_frac": 3.0 * ach / peak_bf16, "pairs": pairs, "set_sum_s": ss,
                                     "what": "algorithmic 2 n_obs flop per pair over the set-sum phase (kxgen + nlsum "
                                             "launches); peak = MEASURED_PEAKS.json bf16_tflops_sustained"}
        del X, Z, Om

    def model(d, n_obs, seed, ls, noise=None, **kw):
        Xo, yo = make_observations(d, n_obs, seed=seed, **kw)
        return bgp.FixedGP(Xo.to(dev, torch.float32), yo.to(dev), bgp.ScaleKernel(bgp.RBFKernel(ls), 1.0),
                           noise=a.noise if noise is None else noise)

    m1 = model(10, 102, 2, 2.5)
    run("config1_batch_N2e4_M200_n100_vbq", spec_from_model(m1, _lib.PRED_COV), 10, 20_000, 200, 100, reps=5)
    run("config1_quadrature_N1e5_M200_n100_vbq", spec_from_model(m1, _lib.PRED_COV), 10, 100_000, 200, 100, reps=5)
    m2 = model(2, 102, 3, 1.0, noise=max(a.noise, 1e-4))   # 102 observations in 2-D: K_XX + 1e-10 I is not positive definite
    run("config2_d2_N1e6_M1e4_n100_vbq", spec_from_model(m2, _lib.PRED_COV), 2, 1_000_000, 10_000, 100)
    run("config4_d20_matern52_N4e6_M5e3_n500", KernelSpec(_lib.MATERN25, _lib.PLAIN, torch.tensor([4.0]), 1.0),
        20, 4_000_000, 5_000, 500)
    m5 = model(10, 1002, 5, 2.5, sqrt=True)
    run("config5_wsabil_N1e7_M1e4_n1000", spec_from_model(m5, _lib.WSABI_L), 10, 10_000_000, 10_000, 1000)
    run("config5_wsabim_N1e7_M1e4_n1000", spec_from_model(m5, _lib.WSABI_M), 10, 10_000_000, 10_000, 1000, reps=1)
    m5l = model(10, 1002, 6, 2.5, log=True)
    run("config5_mmlt_N1e7_M1e4_n1000", spec_from_model(m5l, _lib.MMLT_G), 10, 10_000_000, 10_000, 1000, reps=1)
    # fp64 inputs (SOBER's global dtype, SOBER/_settings.py:4-11): the all-fp64 CUDA-core path
    # (setsum_kernel<double>: direct differences, fp64 exp; bound by the fp64 pipe - DESIGN.md 4)
    def run64(name, kern, d, N, M, n):
        X = bsampler.sample_mvn(torch.zeros(d), 2.0 * torch.eye(d), N, seed=7, device=dev, dtype=torch.float64)
        Om = torch.randn(M, n - 1, dtype=torch.float64, device=dev, generator=torch.Generator(device=dev).manual_seed(3))

        def step64():
            _, U = ops.nystrom_basis(kern, X[:M], n - 1, omega=Om, want_S=False)
            return ops.recombine(kern, X, X[:M], U)
        step64()
        torch.cuda.synchronize(dev)
        ctx.profile(True)
        ctx.profile_read(reset=True)
        pe0 = ctx.pair_evals
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        idx, w = step64()
        e1.record()
        torch.cuda.synchronize(dev)
        prof = ctx.profile_read(reset=True)
        ctx.profile(False)
        assert 1 <= len(idx) <= n and abs(float(w.sum()) - 1.0) < 1e-9
        ss = prof["set_sum"][0]
        out[name] = {"ms": round(e0.elapsed_time(e1), 3), "phases_ms": {k: round(v[0], 2) for k, v in prof.items() if v[0] > 0},
                     "set_sum_pairs_per_s": (ctx.pair_evals - pe0) / (ss * 1e-3) if ss > 0 else None}
        del X, Om

    run64("config2_fp64_inputs_d2_N1e6_M1e4_n100_vbq", spec_from_model(m2, _lib.PRED_COV), 2, 1_000_000, 10_000, 100)
    run64("config4_fp64_inputs_d20_matern52_N4e6_M5e3_n500", KernelSpec(_lib.MATERN25, _lib.PLAIN, torch.tensor([4.0]), 1.0),
          20, 4_000_000, 5_000, 500)
    # acquisition pass of config 5: GP posterior mean + variance over 1e7 candidates, then calc_weights
    kern = spec_from_model(model(10, 1002, 5, 2.5), _lib.PRED_COV)
    X = bsampler.sample_mvn(torch.zeros(10), 2.0 * torch.eye(10), 10_000_000, seed=9, device=dev)
    ops.gp_predict(kern, X, space=0, want_var=True)     # warm-up at full size (the pool grows once)
    bsampler.calc_weights(kern, X, ratio=0.5)
    torch.cuda.synchronize(dev)
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    mean, var = ops.gp_predict(kern, X, space=0, want_var=True)
    e1.record()
    w = bsampler.calc_weights(kern, X, ratio=0.5)
    e2.record()
    torch.cuda.synchronize(dev)
    assert bool(torch.isfinite(mean).all()) and bool((var > 0).all()) and abs(float(w.sum()) - 1.0) < 1e-9
    ms_var = e0.elapsed_time(e1)
    n_obs = 1002
    out["config5_gp_mean_variance_1e7_candidates"] = {
        "ms": round(ms_var, 3), "candidates_per_s": 1e7 / ms_var * 1e3,
        "calc_weights_ms": round(e1.elapsed_time(e2), 3),
        "what": "posterior mean + exact variance (fused tcgen05 kernel gpvar_fused_kernel), then calc_weights = the "
                "same moments again + one elementwise pass",
        "roofline": {"bound": "tensor", "unit": "TFLOP/s", "peak": peak_bf16,
                     "what": "algorithmic n_obs^2 flop per candidate (triangular solve v = L^-1 k, |v|^2) over the "
                             "call time; the kernel issues 3x that (fp16 hi / lo split products for fp32 accuracy)",
                     "achieved": 1e7 * n_obs * n_obs / (ms_var * 1e-3) / 1e12,
                     "frac": 1e7 * n_obs * n_obs / (ms_var * 1e-3) / 1e12 / peak_bf16,
                     "issued_frac": 3e7 * n_obs * n_obs / (ms_var * 1e-3) / 1e12 / peak_bf16,
                     "traffic": "algorithmic: candidates in (40 B each) + moments out (16 B each); ncu r02: 92 MB per 2e6 candidates"}}
    return out


def run_ours(a, rank, world, local_rank):
    import torch.distributed as dist

    import basq_b200  # noqa: F401
    from basq_b200 import _lib, gp as bgp, ops, sharded

    assert torch.cuda.is_available(), "bench.py --impl ours needs a CUDA device (no CPU fallback)"
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    ctx = _lib.context_for(dev)
    q = a.n - 1

    # GP model (replicated): fixed hyper-parameters, caches built once outside the timed region
    Xo, yo = make_observations(a.d, a.n_obs)
    model = bgp.FixedGP(Xo.to(dev, torch.float32), yo.to(dev), bgp.ScaleKernel(bgp.RBFKernel(a.lengthscale), 1.0),
                        noise=a.noise)
    from basq_b200.kernels import spec_from_model
    kern = spec_from_model(model, _lib.PRED_COV)

    # synthetic candidates: rank-local shard, pinned host copy for the end-to-end leg
    if a.scaling == "weak":
        N_loc, N_glob, base = a.N, a.N * world, rank * a.N
    else:
        lo, hi = sharded.shard_bounds(a.N, world, rank)
        N_loc, N_glob, base = hi - lo, a.N, lo
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    X = math.sqrt(2.0) * torch.randn(N_loc, a.d, generator=g, device=dev, dtype=torch.float32)
    Z = X[: a.M].clone()
    if world > 1:
        dist.broadcast(Z, 0)
    gO = torch.Generator(device=dev).manual_seed(7)
    Omega = torch.randn(a.M, q, generator=gO, device=dev, dtype=torch.float64)

    shard_basis = world > 1 and os.environ.get("BASQ_BENCH_SHARD_NYSTROM", "1") != "0"

    def basis(k, Zb, omega=None, seed=None):
        """Nystrom basis: at N > 1 the rows of K(Z, Z) are sharded over the ranks (basq_nystrom_basis_sharded)."""
        if shard_basis:
            return sharded.nystrom_basis_sharded(k, Zb, q, omega=omega, seed=seed)
        if world > 1 and omega is None and seed is None:
            seed = sharded._shared_seed(None, True, dev)      # every rank must draw the same test matrix
        return ops.nystrom_basis(k, Zb, q, omega=omega, want_S=False, seed=seed)[1]

    def step_device():
        U = basis(kern, Z, omega=Omega)
        if world == 1:
            return ops.recombine(kern, X, Z, U)
        return sharded.recombination_sharded(X, Z, a.n, kern, N_glob, base, U)

    X_host = Z_host = None
    side_stream = torch.cuda.Stream(dev)
    if not a.no_e2e:
        X_host = torch.empty(N_loc, a.d, dtype=torch.float32).pin_memory()
        X_host.copy_(X)
        Z_host = Z.cpu().pin_memory()
        # no test matrix travels: like torch.svd_lowrank inside the reference, the library draws it on the device

    def step_e2e():
        if world == 1:
            return ops.recombine_host(kern, X_host, Z_host, q, device=dev, seed=7)
        # candidates through the C ABI's host entry of the sharded path, underneath
        # the Nystrom phase - what basq_recombine_host does inside the C call at N = 1
        Zd = Z_host.to(dev, non_blocking=True)                # 0.4 MB of landmarks first: the copy engine is FIFO
        staged = ops.stage_candidates(X_host, device=dev)     # basq_ctx_stage_candidates: the shard travels on a side stream
        U = basis(kern, Zd, seed=7)                            # every rank draws the same matrix
        idx, w = sharded.recombination_sharded(None, Zd, a.n, kern, N_glob, base, U, staged=staged)
        return idx.cpu(), w.cpu()

    # BASELINE metric (2), "BASQ iteration time": candidates drawn on the device from the prior (every
    # rank its slice of one Philox stream), landmarks = leading rows, Nystrom basis, recombination
    # (GP hyper-parameter refit excluded, as in the reference's tutorial timing - SURVEY 8d)
    from basq_b200 import sampler as bsampler
    prior_mean = torch.zeros(a.d, dtype=torch.float64)
    prior_tril = math.sqrt(2.0) * torch.eye(a.d, dtype=torch.float64)
    it_count = [0]

    def step_iteration():
        it_count[0] += 1
        seed = 4242 + it_count[0]
        Xs = bsampler.sample_mvn(prior_mean, None, N_loc, seed=seed, offset=base, device=dev, scale_tril=prior_tril)
        Zs = Xs[: a.M] if world == 1 else bsampler.sample_mvn(prior_mean, None, a.M, seed=seed, offset=0, device=dev,
                                                              scale_tril=prior_tril)
        U = basis(kern, Zs)      # the library draws the test matrix (rank 0's torch generator seeds every rank)
        if world == 1:
            return ops.recombine(kern, Xs, Zs, U)
        return sharded.recombination_sharded(Xs, Zs, a.n, kern, N_glob, base, U)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    debug = os.environ.get("BASQ_BENCH_DEBUG") == "1"

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)] if debug else None
        e0.record()
        out = None
        for i in range(steps):
            if debug:
                marks[i].record()
            out = fn()
        if debug:
            marks[steps].record()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if debug:   # per-step device times from events recorded without synchronising (diagnostic runs)
            per = [marks[i].elapsed_time(marks[i + 1]) for i in range(steps)]
            print(f"[bench debug] rank {rank} {fn.__name__}: " + " ".join(f"{t:.1f}" for t in per), file=sys.stderr, flush=True)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms / steps, out

    for _ in range(max(a.warmup, 3)):
        out = step_device()
    # phase spans are recorded as CUDA-event pairs on the library's stream (= torch's current stream)
    # without synchronising, so they are taken live inside the timed region and read afterwards
    ctx.profile(True)
    ctx.profile_read(reset=True)
    launches0, pe0 = ctx.launches, ctx.pair_evals
    with ClockSampler(local_rank, enabled=(rank == 0)) as clk:
        ms_step, out = timed(step_device, a.steps)
    launches = ctx.launches - launches0
    pairs_step = (ctx.pair_evals - pe0) / a.steps
    prof = ctx.profile_read(reset=True)
    ctx.profile(False)
    idx, w = out
    assert 1 <= len(idx) <= a.n and bool((w > 0).all()), "invalid quadrature rule"
    assert abs(float(w.sum()) - 1.0) < 1e-9, float(w.sum())
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, idx, w)
    value = N_glob / (ms_step * 1e-3)

    e2e = None
    if not a.no_e2e:
        step_e2e()
        ms_e2e, out2 = timed(step_e2e, a.steps)
        h2d = X_host.numel() * 4 + Z_host.numel() * 4
        d2h = len(out2[0]) * 16
        # what this box's PCIe link gives the candidate copy on its own (outside the timed region): explains
        # the gap between `e2e` and `value` when the copy is longer than the Nystrom phase it hides under
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        Xtmp = torch.empty(X_host.shape, dtype=X_host.dtype, device=dev)   # allocate first: only the copy is timed
        torch.cuda.synchronize(dev)
        e0.record()
        Xtmp.copy_(X_host, non_blocking=True)
        e1.record()
        torch.cuda.synchronize(dev)
        h2d_ms = e0.elapsed_time(e1)
        del Xtmp
        e2e = {"value": N_glob / (ms_e2e * 1e-3), "unit": "points/s", "ms_per_step": ms_e2e,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "candidate_copy_alone_ms": round(h2d_ms, 2),
               "pcie_h2d_GBps": round(X_host.numel() * 4 / (h2d_ms * 1e-3) / 1e9, 1)}

    step_iteration()
    ms_iter, out3 = timed(step_iteration, a.steps)
    assert 1 <= len(out3[0]) <= a.n and abs(float(out3[1].sum()) - 1.0) < 1e-9

    # the configuration as BASELINE.json words it: a.N candidates IN TOTAL sharded over the ranks
    strong = None
    if world > 1 and a.scaling == "weak":
        lo, hi = sharded.shard_bounds(a.N, world, rank)
        Xs_ = X[: hi - lo]

        def step_strong():
            U = basis(kern, Z, omega=Omega)
            return sharded.recombination_sharded(Xs_, Z, a.n, kern, a.N, lo, U)
        step_strong()
        ctx.profile(True)
        ctx.profile_read(reset=True)
        ms_strong, out4 = timed(step_strong, a.steps)
        prof_s = ctx.profile_read(reset=True)
        ctx.profile(False)
        assert 1 <= len(out4[0]) <= a.n and abs(float(out4[1].sum()) - 1.0) < 1e-9
        strong = {"scaling": "strong", "N_total": a.N, "ms_per_step": ms_strong, "value": a.N / (ms_strong * 1e-3),
                  "unit": "points/s", "phases_ms": {k: round(v[0] / a.steps, 3) for k, v in prof_s.items()},
                  "what": "BASELINE config 3 as worded: 1e7 candidates in total sharded over the ranks; the Nystrom "
                          "basis and the Caratheodory levels are replicated work (Amdahl)"}

    # BASELINE config 5 as worded (Tutorial 03 models on 8 x B200): 1e7 candidates in total sharded over the ranks,
    # WSABI-M and MMLT kernels (the pairwise tensor-core set sums shard with the candidates)
    extra_multi = None
    if world > 1 and not a.no_extra:
        extra_multi = {}
        lo, hi = sharded.shard_bounds(a.N, world, rank)
        Xs5 = X[: hi - lo]
        for tag, mode, kw in (("wsabim", _lib.WSABI_M, {"sqrt": True}), ("mmlt", _lib.MMLT_G, {"log": True})):
            Xo5, yo5 = make_observations(a.d, a.n_obs, seed=5 if tag == "wsabim" else 6, **kw)
            m5 = bgp.FixedGP(Xo5.to(dev, torch.float32), yo5.to(dev), bgp.ScaleKernel(bgp.RBFKernel(a.lengthscale), 1.0),
                             noise=a.noise)
            k5 = spec_from_model(m5, mode)

            def step5():
                U = basis(k5, Z, omega=Omega)
                return sharded.recombination_sharded(Xs5, Z, a.n, k5, a.N, lo, U)
            step5()
            ms5, out5 = timed(step5, 2)
            assert 1 <= len(out5[0]) <= a.n and abs(float(out5[1].sum()) - 1.0) < 1e-9
            extra_multi[f"config5_{tag}_N1e7_total_sharded"] = {"ms": round(ms5, 3), "points_per_s": a.N / (ms5 * 1e-3)}

    line = None
    if rank == 0:
        ss_ms_tot, ss_calls = prof["set_sum"]
        ss_ms = ss_ms_tot / a.steps                    # set-sum kernel time per step (one launch per pass)
        n_rounds = ss_calls // a.steps
        ss_launch_ms = ss_ms_tot / max(ss_calls, 1)    # average launch duration
        pairs_launch = pairs_step / max(n_rounds, 1)   # kernel evaluations k(z, x) per launch (average)
        clocks = clk.summary()
        sm_mhz = clocks.get("sm_mhz") or 1965.0
        mufu_peak = 148 * 16 * sm_mhz * 1e6            # ex2.approx lanes/s: 16 per clock per SM
        pair_rate = pairs_launch / (ss_launch_ms * 1e-3) if ss_ms > 0 else None
        traffic = None
        try:   # per-launch DRAM bytes of this kernel from the committed ncu --set full capture
            traffic = json.load(open(os.path.join(ROOT, "profiles", "setsum_traffic.json")))["dram_bytes_per_launch_avg"]
        except Exception:
            pass
        flop_per_pair = 2 * a.d + 4
        line = {
            "metric": METRIC, "value": value, "unit": "points/s",
            "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
            "dtype": "f32 kernel evaluation (fp16 hi/lo split distance contraction, 3 products), f64 accumulation/projection/Caratheodory",
            "data": "synthetic", "config": config_of(a, world),
            "clocks": clocks, "gpu_launches": int(launches), "e2e": e2e,
            "iteration": {"ms": ms_iter, "unit": "ms per BASQ iteration",
                          "what": "device prior sampling (Philox MVN) + Nystrom basis + recombination to n points; "
                                  "GP refit excluded (BASELINE metric part 2)"},
            "phases_ms": {k: round(v[0] / a.steps, 3) for k, v in prof.items()}, "rounds": n_rounds,
            "roofline": {
                "bound": "mufu",
                "kernel": "setsum_mma_kernel<RBF, 10> (tcgen05 kind::f16 distance contraction on fp16 hi/lo split operands, ex2 + fp64 set-sum epilogue)",
                "achieved": pair_rate / 1e9 if pair_rate else None, "peak": mufu_peak / 1e9,
                "unit": "G kernel evaluations/s", "frac": (pair_rate / mufu_peak) if pair_rate else None,
                "traffic": traffic,
                "peak_source": "148 SMs x 16 ex2.approx lanes/clk x SM clock measured during the timed region "
                               "(scripts/mufu_probe.cu measured 15.7/clk/SM); neither HBM nor the tensor pipe binds this "
                               "kernel: one transcendental per (landmark, candidate) pair does",
                "pairs_per_launch_avg": pairs_launch, "launch_ms_avg": ss_launch_ms,
                "pairs_per_step": pairs_step, "set_sum_ms_per_step": ss_ms, "set_sum_launches_per_step": n_rounds,
                "tensor_pipe": {"algorithmic_flop_per_pair": flop_per_pair,
                                "achieved_tflops": (pair_rate * flop_per_pair / 1e12) if pair_rate else None,
                                "note": "the distance contraction issues 96 fp16 MMA flop per pair (K = 48: lo hi, hi lo, hi hi "
                                        "of the split operands); far from the tensor peak by design"},
                "hbm": {"algorithmic_bytes_per_step": None if not pairs_step else int(2 * 64 * N_loc * 1.04),
                        "note": "records are re-read per 256-landmark group from L2 (DESIGN.md 4)"},
            },
        }
        if strong is not None:
            line["strong"] = strong
        if extra_multi:
            line["extra"] = extra_multi
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cores = host_threads()
        n_sample = max(a.cpu_sample, 4 * a.n, a.M)
        t = oracle_step(a, n_sample)
        line["cpu_baseline"] = {"value": n_sample / t, "unit": "points/s", "cores": cores, "kind": "port", "seconds": t,
                                "sample": sample_text(a, n_sample, "oracle port of BASQ/_rchq.py, fp64 torch CPU")}
        # the reference's own GPU story: the same torch-op sequence with the tensors on the B200
        try:
            oracle_step(a, max(4 * a.n, a.M), device=str(dev))
            n_gpu = max(4 * n_sample, 4 * a.n, a.M)
            tg = oracle_step(a, n_gpu, device=str(dev))
            line["gpu_baseline"] = {"value": n_gpu / tg, "unit": "points/s", "kind": "port", "seconds": tg,
                                    "sample": sample_text(a, n_gpu, "oracle port of BASQ/_rchq.py, fp64 torch ops on "
                                                                    "the same B200 (the reference's device=cuda path)")}
        except Exception as exc:   # reported, never fatal for the bench line
            line["gpu_baseline"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    if rank == 0 and world == 1 and not a.no_extra:
        try:
            del X
            torch.cuda.empty_cache()
            line["extra"] = extra_configs(dev, a)
        except Exception as exc:
            line["extra"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    if rank == 0:
        try:    # scratch memory the library holds at the end of the run (block cache + host-call buffer)
            cached, live, n_alloc = ctx.memory()
            line["scratch_memory"] = {"cached_GB": round(cached / 1e9, 2), "live_GB": round(live / 1e9, 2),
                                      "driver_allocations": n_alloc}
        except Exception:
            pass
        print(json.dumps(line), flush=True)


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank, max(world, a.gpus))
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    try:
        run_ours(a, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
