"""Time the weighted kernel double sums (ops.kernel_quadform / gp.worst_case_error) on one GPU, next to the set-sum
pair rate of one config-3 recombination (N = 1e7, d = 10, M = 11 002, q = 999) measured in the same run.

    python scripts/time_quadform.py [--out FILE]

Prints one JSON object (also written to FILE): the GPU's name and power limit, then per case the milliseconds
of one call (CUDA events after a warm-up call, median of the repeats), the kernel evaluations of the set-sum
kernels (ctx.pair_evals) and their rate, and the kernel launches per call."""
import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import basq_b200  # noqa: E402
from basq_b200 import _lib, gp, ops  # noqa: E402
from basq_b200.kernels import KernelSpec  # noqa: E402
from oracle import gp_kernels as ogp  # noqa: E402

DEV = torch.device("cuda:0")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn, reps):
    ctx = _lib.context_for(DEV)
    fn()                                              # warm-up: module loads, block cache
    ms, pairs, launches = [], 0, 0
    for _ in range(reps):
        p0, l0 = ctx.pair_evals, ctx.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
        pairs, launches = ctx.pair_evals - p0, ctx.launches - l0
    ms.sort()
    med = ms[len(ms) // 2]
    return {"ms": med, "ms_min": ms[0], "ms_max": ms[-1], "reps": reps, "pair_evals": pairs,
            "pairs_per_s": pairs / (med * 1e-3), "launches": launches}


def gp_model(d, n_obs, noise):
    return ogp.make_gp(d, n_obs, lengthscale=1.5 * math.sqrt(d / 2.0), outputscale=1.0, noise=noise, mean_const=0.1,
                       seed=3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    d = 10
    res = {"gpu": gpu_info(), "cases": {}}
    g = torch.Generator(device=DEV).manual_seed(0)
    ctx = _lib.context_for(DEV)

    # yardstick: the set-sum phase of one config-3 recombination
    N3, M3, q3 = 10_000_000, 11_002, 999
    X3 = math.sqrt(2.0) * torch.randn(N3, d, generator=g, device=DEV)
    U3 = torch.linalg.qr(torch.randn(M3, q3, generator=g, device=DEV, dtype=torch.float64)).Q.T.contiguous()
    plain = KernelSpec(_lib.RBF, _lib.PLAIN, torch.tensor([2.5]), 1.0)
    ops.recombine(plain, X3, X3[:M3].clone(), U3)
    torch.cuda.synchronize()
    ctx.profile(True)
    ctx.profile_read(True)
    p0 = ctx.pair_evals
    ops.recombine(plain, X3, X3[:M3].clone(), U3)
    prof = ctx.profile_read(True)
    ctx.profile(False)
    ss_ms = prof["set_sum"][0]
    res["yardstick_config3_recombine"] = {"set_sum_ms": ss_ms, "pair_evals": ctx.pair_evals - p0,
                                          "pairs_per_s": (ctx.pair_evals - p0) / (ss_ms * 1e-3)}
    del X3, U3
    torch.cuda.empty_cache()

    model = gp_model(d, 100, 1e-2)
    vbq = ogp.VanillaGP(model).predictive_kernel
    for N in (100_000, 1_000_000):
        X = math.sqrt(2.0) * torch.randn(N, d, generator=g, device=DEV)
        a = torch.randn(N, generator=g, device=DEV, dtype=torch.float64)
        res["cases"][f"pred_cov_f32_N{N:.0e}"] = timed(lambda: ops.kernel_quadform(vbq, X, a), 5 if N > 100_000 else 20)
        if N == 1_000_000:
            # the set-sum phase alone, for the comparison with the yardstick's rate
            ctx.profile(True)
            ctx.profile_read(True)
            p0 = ctx.pair_evals
            ops.kernel_quadform(vbq, X, a)
            prof = ctx.profile_read(True)
            ctx.profile(False)
            ms = prof["set_sum"][0]
            res["cases"][f"pred_cov_f32_N{N:.0e}"]["set_sum_phase"] = {
                "ms": ms, "pair_evals": ctx.pair_evals - p0, "pairs_per_s": (ctx.pair_evals - p0) / (ms * 1e-3)}
        if N == 100_000:
            X64 = X.double()
            res["cases"][f"pred_cov_f64_N{N:.0e}"] = timed(lambda: ops.kernel_quadform(vbq, X64, a), 5)
        del X, a
    y = res["yardstick_config3_recombine"]["pairs_per_s"]
    r = res["cases"]["pred_cov_f32_N1e+06"]
    r["set_sum_rate_over_yardstick"] = r["set_sum_phase"]["pairs_per_s"] / y
    r["call_rate_over_yardstick"] = r["pairs_per_s"] / y
    wsabim = ogp.WsabiGP(model, alpha=0.05).wsabim_kernel
    X = math.sqrt(2.0) * torch.randn(100_000, d, generator=g, device=DEV)
    a = torch.randn(100_000, generator=g, device=DEV, dtype=torch.float64)
    res["cases"]["wsabi_m_f32_N1e+05"] = timed(lambda: ops.kernel_quadform(wsabim, X, a), 5)
    res["cases"]["wsabi_m_f32_N1e+05"]["kappa"] = ctx.conditioning()[0]
    del X, a

    # worst-case error of a config-1 rule (N = 2e4, M = 200, n = 100, VBQ)
    gc = torch.Generator().manual_seed(0)
    N1, M1, n1 = 20_000, 200, 100
    X1 = (math.sqrt(2.0) * torch.randn(N1, d, generator=gc)).to(DEV)
    m1 = ogp.make_gp(d, 102, lengthscale=2.5, outputscale=1.0, noise=1e-4, seed=1)
    k1 = ogp.VanillaGP(m1).predictive_kernel
    torch.manual_seed(0)
    idx, w = basq_b200.recombination(X1, X1[:M1].clone(), n1, k1, DEV)
    case = timed(lambda: gp.worst_case_error(k1, X1, idx, w), 20)
    case["value"] = gp.worst_case_error(k1, X1, idx, w)
    res["cases"]["worst_case_error_config1"] = case

    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
