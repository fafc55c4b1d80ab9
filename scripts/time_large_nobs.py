"""Time the fp32 posterior variance and its L^-1 preparation on GPs of 1002 .. 16002 observations, and one
config-5 MMLT recombination on a GP of 8002 observations, on one GPU.

    python scripts/time_large_nobs.py [--out FILE] [--n-obs 1002,4002,8002,16002]

A BASQ run appends every batch to the GP, so at batch 1000 the k-th iteration sees 2 + 1000 k observations.
The GPs are built as bench.py builds its config-5 GP: d = 10, RBF lengthscale 2.5, outputscale 1, noise 1e-10,
observations from N(0, 2 I), Gaussian-mixture targets; basq_b200.gp.FixedGP on the device.  Where the Cholesky
of K + 1e-10 I fails, the smallest jitter of 1e-8, 1e-6, 1e-4 that passes is added and recorded.

Per GP size, one JSON entry with
  - prep_ms: the L^-1 preparation on the device, from the first kernel of a gp_predict call to the start of the
    variance kernel (torch.profiler trace of its own call);
  - var_kernel_ms: the variance kernel (gpvar_fused_kernel) in that trace, over 1e7 fp32 candidates, and
    var_kernel_tflops = 1e7 n_obs^2 / var_kernel_ms (algorithmic flop; the kernel issues three products each);
  - predict_ms: gp_predict mean + variance over the same 1e7 candidates, CUDA events, profiler off;
  - max_var_err / max_mean_rel_err: against fp64 torch on 1e5 candidates (the GP's own W and mean cache);
  - mmlt: kappa of an MMLT session (N = 2e5, M = 2000, n = 200) on the log-target GP of the same size and
    whether the conditioning guard promoted it to fp64 (basq_ctx_conditioning).
Prints one JSON object (also written to FILE) that starts with the GPU's name and power limit."""
import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import basq_b200  # noqa: E402
from basq_b200 import _lib, gp as bgp, ops, sampler as bsampler  # noqa: E402
from basq_b200.kernels import spec_from_model  # noqa: E402
from oracle import gp_kernels as ogp  # noqa: E402

DEV = torch.device("cuda:0")
D, LS, NOISE = 10, 2.5, 1e-10


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def observations(n_obs, seed, log=False):
    """bench.py make_observations: N(0, 2 I) inputs, 3-component Gaussian-mixture targets."""
    g = torch.Generator().manual_seed(seed)
    X = math.sqrt(2.0) * torch.randn(n_obs, D, generator=g, dtype=torch.float64)
    centres = 1.5 * torch.randn(3, D, generator=g, dtype=torch.float64)
    y = sum(torch.exp(-0.25 * ((X - c) ** 2).sum(-1)) for c in centres) / 3.0
    if log:
        y = torch.log(y + 1e-12)
        y = y - y.max()
    return X, y


def model(n_obs, seed, log=False):
    Xo, yo = observations(n_obs, seed, log)
    for jitter in (0.0, 1e-8, 1e-6, 1e-4):
        try:
            m = bgp.FixedGP(Xo.to(DEV, torch.float32), yo.to(DEV), bgp.ScaleKernel(bgp.RBFKernel(LS), 1.0),
                            noise=NOISE, jitter=jitter)
            return m, jitter
        except torch.linalg.LinAlgError:
            continue
    raise RuntimeError(f"no jitter up to 1e-4 makes K + noise I positive definite at n_obs = {n_obs}")


def reference(m, X):
    """fp64 posterior mean / variance with the oracle's kernel function on the GP's own W and mean cache."""
    twin = ogp.ScaleKernel(ogp.RBFKernel(LS), 1.0, matmul_dist=True)
    Xobs = m.train_inputs[0].double()
    S = m.prediction_strategy.covar_cache
    W = S @ S.T
    alpha = m.prediction_strategy.mean_cache
    means, vars_ = [], []
    for c in torch.split(X.double(), 5000):
        K = twin.forward(c, Xobs)
        means.append(float(m.mean_module.constant) + K @ alpha)
        vars_.append(1.0 + NOISE - ((K @ W) * K).sum(-1))
    return torch.cat(means), torch.cat(vars_)


def trace_predict(spec, X):
    """(prep_ms, var_kernel_ms) of one gp_predict call from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ops.gp_predict(spec, X, space=0, want_var=True)
        torch.cuda.synchronize(DEV)
    kern = sorted(((e.time_range.start, e.time_range.end, e.name) for e in prof.events()
                   if e.device_type == torch.autograd.DeviceType.CUDA), key=lambda t: t[0])
    var = [k for k in kern if "gpvar_fused_kernel" in k[2]]
    assert kern and len(var) == 1, [k[2] for k in kern]
    return (var[0][0] - kern[0][0]) / 1e3, (var[0][1] - var[0][0]) / 1e3


def timed(fn, reps=3):
    fn()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize(DEV)
        ms.append(e0.elapsed_time(e1))
    return sorted(ms)[len(ms) // 2]


def mmlt_session(n_obs):
    """kappa and promotion of one MMLT recombination session (N = 2e5, M = 2000, n = 200)."""
    ctx = _lib.context_for(DEV)
    ml, jitter = model(n_obs, 6, log=True)
    spec = spec_from_model(ml, _lib.MMLT_G)
    X = bsampler.sample_mvn(torch.zeros(D), 2.0 * torch.eye(D), 200_000, seed=7, device=DEV)
    Z = X[:2000].clone()
    _, prom0 = ctx.conditioning()
    _, U = ops.nystrom_basis(spec, Z, 199, want_S=False)
    idx, w = ops.recombine(spec, X, Z, U)
    kappa, prom1 = ctx.conditioning()
    return {"kappa": kappa, "promoted": prom1 > prom0, "jitter": jitter, "rule_points": len(idx),
            "weight_sum": float(w.double().sum())}


def config5_mmlt(n_obs):
    ctx = _lib.context_for(DEV)
    ml, jitter = model(n_obs, 6, log=True)
    spec = spec_from_model(ml, _lib.MMLT_G)
    N, M, n = 10_000_000, 10_000, 1000
    X = bsampler.sample_mvn(torch.zeros(D), 2.0 * torch.eye(D), N, seed=7, device=DEV)
    Z = X[:M].clone()
    Om = torch.randn(M, n - 1, dtype=torch.float64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))

    def step():
        _, U = ops.nystrom_basis(spec, Z, n - 1, omega=Om, want_S=False)
        return ops.recombine(spec, X, Z, U)
    step()
    torch.cuda.synchronize(DEV)
    _, prom0 = ctx.conditioning()
    ctx.profile(True)
    ctx.profile_read(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    idx, w = step()
    e1.record()
    torch.cuda.synchronize(DEV)
    prof = ctx.profile_read(reset=True)
    ctx.profile(False)
    kappa, prom1 = ctx.conditioning()
    return {"n_obs": n_obs, "N": N, "M": M, "n": n, "jitter": jitter, "ms": round(e0.elapsed_time(e1), 3),
            "phases_ms": {k: round(v[0], 2) for k, v in prof.items() if v[0] > 0},
            "kappa": kappa, "promoted": prom1 > prom0, "rule_points": len(idx), "weight_sum": float(w.double().sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--n-obs", default="1002,4002,8002,16002")
    ap.add_argument("--config5-n-obs", type=int, default=8002)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_large_nobs.py needs a CUDA device"
    res = {"gpu": gpu_info(), "candidates": 10_000_000, "sizes": {}}
    X = bsampler.sample_mvn(torch.zeros(D), 2.0 * torch.eye(D), 10_000_000, seed=9, device=DEV)
    Xe = X[:100_000]
    for n_obs in (int(s) for s in args.n_obs.split(",")):
        m, jitter = model(n_obs, 5)
        spec = spec_from_model(m, _lib.PRED_COV)
        ops.gp_predict(spec, X, space=0, want_var=True)        # warm-up at full size (the pool grows once)
        prep_ms, var_ms = trace_predict(spec, X)
        predict_ms = timed(lambda: ops.gp_predict(spec, X, space=0, want_var=True))
        mean, var = ops.gp_predict(spec, Xe, space=0, want_var=True)
        m_ref, v_ref = reference(m, Xe)
        flop = 1e7 * n_obs * n_obs
        res["sizes"][str(n_obs)] = {
            "jitter": jitter, "prep_ms": round(prep_ms, 3), "var_kernel_ms": round(var_ms, 3),
            "var_kernel_tflops": flop / (var_ms * 1e-3) / 1e12, "predict_ms": round(predict_ms, 3),
            "predict_tflops": flop / (predict_ms * 1e-3) / 1e12,
            "max_var_err": float((var - v_ref).abs().max()), "var_ref_min": float(v_ref.min()),
            "max_mean_rel_err": float((mean - m_ref).abs().max() / m_ref.abs().max()),
            "mmlt": mmlt_session(n_obs)}
        print(json.dumps({n_obs: res["sizes"][str(n_obs)]}), flush=True)
        del m, spec, mean, var, m_ref, v_ref
        torch.cuda.empty_cache()
    s = res["sizes"]
    if "1002" in s and "8002" in s:
        res["tflops_ratio_8002_over_1002"] = s["8002"]["var_kernel_tflops"] / s["1002"]["var_kernel_tflops"]
    del X, Xe
    torch.cuda.empty_cache()
    if args.config5_n_obs > 0:
        res["config5_mmlt_recombination"] = config5_mmlt(args.config5_n_obs)
    out = json.dumps(res, indent=1)
    print(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
